// gae_kernel.cu -- GAE advantages + returns over a time-major [T][N] rollout, one thread per environment.
//
// Restates PPO.compute_gae (reference src/ppo.py:107-120) and the identical loop inlined in
// FOMAML.compute_loss (src/fomaml.py:116-123) / src/utils/utils_rl.py:11-30:
//     mask  = 1 - done[t]
//     delta = rew[t] + gamma * next_val * mask - val[t]          next_val = last_value at t = T-1
//     gae   = delta + gamma * lam * mask * gae
//     adv[t] = gae ;  ret[t] = val[t] + adv[t]
// The reference evaluates this in fp32 with python-float (double) hyper-parameters, so `gamma * lam` and
// `gamma * last_value` are formed in double and rounded once; every other product/sum is a separately
// rounded fp32 operation.  The kernel keeps that operation order and forbids FMA contraction
// (__fmul_rn/__fadd_rn/__fsub_rn), which makes it bit-identical to the reference loops on the fixtures.
//
// HBM-streaming: 20 B per (t, env) (3 reads + 2 writes of f32), reads coalesced across envs; the reverse
// scan is sequential in t by nature, parallel over envs.
#include <cuda_runtime.h>
#include <stdint.h>

#include "env_kernels.cuh"

namespace merlin {

template <int kChunk>
__global__ void __launch_bounds__(128) gae_kernel(const float* __restrict__ rew, const float* __restrict__ val,
                                                  const float* __restrict__ done, const float* __restrict__ last_val,
                                                  float* __restrict__ adv, float* __restrict__ ret, const int T,
                                                  const int N, const double gamma, const float g32, const float gl32) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float gae = 0.f;
  // gamma * next_val for t = T-1: python double product, rounded to f32 when it meets the f32 mask
  float gnext = (float)(gamma * (double)last_val[n]);
  // The recurrence is serial in t but its loads are not: fetch kChunk time steps (3 x kChunk independent, coalesced
  // loads in flight per thread) before running the kChunk dependent updates, so a short rollout (a few thousand envs,
  // one warp per SM) is bound by the arithmetic chain rather than by kChunk-times-fewer memory round trips.
  // Measured on B200 (profiles/r01_gae_chunk_variants.txt): kChunk = 32 for small rollouts (kGaeChunkSmall; T=128 x
  // N=4096: 14.3 us vs 20.5 with 8 -- 4 memory round trips per thread instead of 16; 149 registers do not matter at one
  // warp per SM), 16 for rollouts that fill the machine (kGaeChunkLarge; T=64 x N=1M: 0.90 of the HBM copy peak vs 0.885
  // with 8 and 0.87 with 4).
  int t = T - 1;
  for (; t >= kChunk - 1; t -= kChunk) {
    float r[kChunk], v[kChunk], d[kChunk];
#pragma unroll
    for (int j = 0; j < kChunk; ++j) {
      const size_t k = (size_t)(t - j) * N + n;
      r[j] = __ldcs(rew + k); v[j] = __ldcs(val + k); d[j] = __ldcs(done + k);
    }
#pragma unroll
    for (int j = 0; j < kChunk; ++j) {
      const size_t k = (size_t)(t - j) * N + n;
      const float mask = __fsub_rn(1.0f, d[j]);
      const float delta = __fsub_rn(__fadd_rn(r[j], __fmul_rn(gnext, mask)), v[j]);
      gae = __fadd_rn(delta, __fmul_rn(__fmul_rn(gl32, mask), gae));
      __stcs(adv + k, gae);
      __stcs(ret + k, __fadd_rn(v[j], gae));
      gnext = __fmul_rn(g32, v[j]);  // gamma * values[t] is the next_val term of step t-1
    }
  }
  for (; t >= 0; --t) {
    const size_t k = (size_t)t * N + n;
    const float r = rew[k], v = val[k], d = done[k];
    const float mask = __fsub_rn(1.0f, d);
    const float delta = __fsub_rn(__fadd_rn(r, __fmul_rn(gnext, mask)), v);
    gae = __fadd_rn(delta, __fmul_rn(__fmul_rn(gl32, mask), gae));
    adv[k] = gae;
    ret[k] = __fadd_rn(v, gae);
    gnext = __fmul_rn(g32, v);
  }
}

// Small rollouts (a few thousand envs: one warp or less per SM in the kernel above, whose run time is then T / kChunk
// dependent memory round trips plus the chain): a CTA of 8 warps owns 32 envs and a window of 128 time steps at once.
//   phase 1  ALL warps load the window's rew / val / done rows -- 16 rows per warp, every load of the window in flight
//            together -- and compute what does not depend on the scan, delta[t] and c[t] = (gamma * lam) * mask[t],
//            into shared memory;
//   phase 2  ONE warp (lane = env) runs the recurrence gae = delta[t] + c[t] * gae from shared memory, 16 steps per
//            batch of shared-memory reads: two dependent fp32 operations per step; adv[t] and ret[t] = val[t] + adv[t]
//            leave from there as coalesced 128-byte stores.
// Same operations in the same order as gae_kernel (and the reference loop): bit-identical results.
constexpr int kGaeRows = 16;                 // rows per warp per window (phase 1), steps per batch (phase 2)
constexpr int kGaeWindow = 8 * kGaeRows;     // 128 time steps x 32 envs x 3 arrays x 4 B = 48 KB of shared memory
__global__ void __launch_bounds__(256) gae_tile_kernel(const float* __restrict__ rew, const float* __restrict__ val,
                                                       const float* __restrict__ done, const float* __restrict__ last_val,
                                                       float* __restrict__ adv, float* __restrict__ ret, const int T,
                                                       const int N, const double gamma, const float g32, const float gl32) {
  __shared__ float s_delta[kGaeWindow * 32], s_c[kGaeWindow * 32], s_v[kGaeWindow * 32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int n = blockIdx.x * 32 + lane;
  const bool ok = n < N;
  float gae = 0.f;
  for (int t_hi = T - 1; t_hi >= 0; t_hi -= kGaeWindow) {
    const int len = min(kGaeWindow, t_hi + 1), t_lo = t_hi - len + 1;
    if (ok) {
      float r[kGaeRows], v[kGaeRows], d[kGaeRows], vn[kGaeRows];
#pragma unroll
      for (int i = 0; i < kGaeRows; ++i) {       // rows j = w + 8 i of the window
        const int j = w + 8 * i, t = t_lo + j;
        if (j < len) {
          const size_t k = (size_t)t * N + n;
          r[i] = rew[k]; v[i] = val[k]; d[i] = done[k];
          vn[i] = t == T - 1 ? 0.f : val[k + N];
        }
      }
#pragma unroll
      for (int i = 0; i < kGaeRows; ++i) {
        const int j = w + 8 * i, t = t_lo + j;
        if (j < len) {
          // gamma * next_val: python double product rounded to f32 at t = T-1, else gamma(f32) * values[t+1]
          const float gnext = t == T - 1 ? (float)(gamma * (double)last_val[n]) : __fmul_rn(g32, vn[i]);
          const float mask = __fsub_rn(1.0f, d[i]);
          s_delta[j * 32 + lane] = __fsub_rn(__fadd_rn(r[i], __fmul_rn(gnext, mask)), v[i]);
          s_c[j * 32 + lane] = __fmul_rn(gl32, mask);
          s_v[j * 32 + lane] = v[i];
        }
      }
    }
    __syncthreads();
    if (w == 0 && ok) {
      int j = len - 1;
      for (; j >= kGaeRows - 1; j -= kGaeRows) {
        float dl[kGaeRows], c[kGaeRows], v[kGaeRows];
#pragma unroll
        for (int i = 0; i < kGaeRows; ++i) {
          dl[i] = s_delta[(j - i) * 32 + lane]; c[i] = s_c[(j - i) * 32 + lane]; v[i] = s_v[(j - i) * 32 + lane];
        }
#pragma unroll
        for (int i = 0; i < kGaeRows; ++i) {
          const size_t k = (size_t)(t_lo + j - i) * N + n;
          gae = __fadd_rn(dl[i], __fmul_rn(c[i], gae));
          adv[k] = gae;
          ret[k] = __fadd_rn(v[i], gae);
        }
      }
      for (; j >= 0; --j) {
        const size_t k = (size_t)(t_lo + j) * N + n;
        gae = __fadd_rn(s_delta[j * 32 + lane], __fmul_rn(s_c[j * 32 + lane], gae));
        adv[k] = gae;
        ret[k] = __fadd_rn(s_v[j * 32 + lane], gae);
      }
    }
    __syncthreads();   // the next window overwrites the shared arrays
  }
}

// Where the tile kernel runs.  32 calls replayed from a CUDA graph, L2-warm (tools/bench_gae.py, T = 128), tile kernel vs
// one thread per env: 6.06 vs 5.61 us at 32 envs (one CTA: nothing to spread), 6.06 vs 7.57 at 1024, 6.14 vs 7.61 at 4096,
// 12.2 vs 11.8 at 16 384 (512 CTAs of 48 KB: four rounds per SM).
constexpr int kGaeTileMinEnvs = 128, kGaeTileMaxEnvs = 8192;
constexpr int kGaeChunkSmall = 32, kGaeChunkLarge = 16;   // see gae_kernel

cudaError_t launch_gae(const float* rew, const float* val, const float* done, const float* last_val, float* adv,
                       float* ret, int T, int N, double gamma, double lam, cudaStream_t stream) {
  // small rollouts: 32-thread blocks spread the envs over more SMs (4096 envs -> 128 blocks instead of 32)
  if (N >= kGaeTileMinEnvs && N <= kGaeTileMaxEnvs) {
    gae_tile_kernel<<<(N + 31) / 32, 256, 0, stream>>>(rew, val, done, last_val, adv, ret, T, N, gamma, (float)gamma,
                                                       (float)(gamma * lam));
    return cudaGetLastError();
  }
  const bool large = N >= 32768;
  const int threads = N >= 128 * 148 * 4 ? 128 : 32;
  const int blocks = (N + threads - 1) / threads;
  if (large)
    gae_kernel<kGaeChunkLarge><<<blocks, threads, 0, stream>>>(rew, val, done, last_val, adv, ret, T, N, gamma,
                                                               (float)gamma, (float)(gamma * lam));
  else
    gae_kernel<kGaeChunkSmall><<<blocks, threads, 0, stream>>>(rew, val, done, last_val, adv, ret, T, N, gamma,
                                                               (float)gamma, (float)(gamma * lam));
  return cudaGetLastError();
}

}  // namespace merlin
