// env_kernels_tile.cu -- the CTA-tile step kernels for sm_100a: env_kernel_tile (the headline mapping: RGB observations
// from ~25 000 envs up) and env_kernel_tile_tma (its frame phase through the TMA unit; measured, not adopted).
// Same per-env work as every step kernel (see env_kernels.cu); the state phase is env_state_phase.cuh.
#include <cuda_runtime.h>
#include <stdint.h>

#include "env_kernels.cuh"
#include "env_kernels_common.cuh"
#include "env_state_phase.cuh"

namespace merlin {

// ---------------------------------------------------------------------------------------------------
// env_kernel_tile<T, STEP>: a CTA owns a tile of T <= 32 consecutive envs; warp 0 runs the state phase, every
// warp of the CTA takes frames of the tile; co-resident CTAs overlap one tile's state phase with others' frames.
// Shape (B200, 1M envs, RGB), all with tiles handed out in order (see the ticket scheduler below):
//   T=16, 128 threads x 4 CTAs/SM   1.08 of the measured HBM copy peak (7.3e8 env-steps/s)   <- used
//   T=32, 128 x 3: 1.08    T=32, 256 x 2: 1.06    T=32, 128 x 4: 1.06    T=16, 64 x 6: 1.07    T=8, 64 x 8: 1.04
//   T=16, 128 x 5 (96 registers): 1.03    T=16, 128 x 6 (80 registers): 0.95    T=16, 256 x 2: 0.87
// With the static `tile += gridDim.x` assignment the best shape (T=32, 256 x 2) reached 0.99 and every other one
// 0.69-0.96.  Also slower: the blit map in shared memory (-7 %), overlapping the next tile's state phase inside the
// CTA, all warps writing ONE frame at a time, plain / .cg / 256-bit stores instead of st.global.cs.v4, and a separate
// state kernel + high-occupancy frame kernel with static assignment.  Padding the shared-memory atlas slots to remove
// the 17 % bank conflicts changes nothing (the store stream, not the LSU, is the limit).  A plain vectorised fill reaches 7.4-7.6 TB/s on
// this part and frames streamed in order without any env logic 7.4 TB/s (tools/cuda/write_pattern_bench.cu): the fused
// kernel's 7.1 TB/s is 95 % of that.
__host__ __device__ constexpr int tile_smem_bytes(int T) {
  return kAtlasBytes + ((T * kKindStride + T * kSymBytes + 15) & ~15) + 16;
}

template <int T, int STEP, bool SWAR = false>
__global__ void __launch_bounds__(kTileThreads, kTileCtasPerSm) env_kernel_tile(const EnvParams p, const int n_tiles) {
  extern __shared__ __align__(16) uint8_t smem[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int warps_per_cta = blockDim.x >> 5;
  Flags f(p);
  if (SWAR) f.doors = pool_has_doors(p.tile_present);
  uint8_t* atlas_s = smem;
  uint8_t* kinds_s = smem + kAtlasBytes;   // [T][kKindStride]
  uint8_t* sym_s = kinds_s + T * kKindStride;              // [T][147]
  unsigned* mask_s = reinterpret_cast<unsigned*>(smem + tile_smem_bytes(T) - 16);

  uint32_t lut[kChunksPerLane];
  if (f.want_rgb) {
    stage_atlas(p, atlas_s);
    load_lut(p, lane, lut);
  }

  // Tiles are handed out IN ORDER from a ticket counter rather than round-robin by CTA index: the CTAs' write fronts
  // then stay inside one narrow, advancing window of the observation buffer, which is what keeps HBM writes near the
  // plain-fill rate (measured with tools/cuda/write_pattern_bench.cu: 7.4 TB/s in order vs 6.4 TB/s with the static
  // `tile += gridDim.x` assignment, whose CTAs drift apart).  Thread 32 draws the next ticket while warp 0 runs the
  // state phase; the last CTA to finish rearms the counters for the next launch (also under CUDA-graph replay).
  __shared__ int s_next;
  if (threadIdx.x == 0) s_next = (int)atomicAdd(&p.sched[0], 1u);
  __syncthreads();
  int tile = s_next;
  while (tile < n_tiles) {
    const int e0 = tile * T;
    if (warp == 0) {
      const unsigned m = state_phase<T, STEP, SWAR>(p, f, e0, lane, kinds_s, sym_s);
      if (lane == 0) *mask_s = m;
    } else if (threadIdx.x == 32) {
      s_next = (int)atomicAdd(&p.sched[0], 1u);
    }
    __syncthreads();  // kinds / sym / mask of this tile, the next ticket (and, first time round, the atlas) are in smem
    const unsigned render_mask = *mask_s;
    const int next = s_next;
    if (f.want_sym && render_mask)
      emit_sym_rows(p.obs_sym + (size_t)e0 * kSymBytes, sym_s, min(T, p.N - e0), render_mask, threadIdx.x, blockDim.x);
    if (f.want_rgb) {
      for (int i = warp; i < T; i += warps_per_cta)
        if ((render_mask >> i) & 1)
          blit_frame(atlas_s, kinds_s + i * kKindStride, lut, p.obs_rgb + (size_t)(e0 + i) * kImgBytes, lane);
    }
    __syncthreads();  // the tile buffers and the ticket slot are rewritten in the next round
    tile = next;
  }
  if (threadIdx.x == 0 && atomicAdd(&p.sched[1], 1u) == gridDim.x - 1) {
    p.sched[0] = 0;  // every CTA has drawn its last ticket: safe to rearm
    p.sched[1] = 0;
  }
}

// ---------------------------------------------------------------------------------------------------
// env_kernel_tile_tma<STEP>: env_kernel_tile with the frame phase routed through the TMA unit.
// A warp assembles a frame in one of its kTmaNbuf shared-memory staging buffers (the same atlas reads, 16-byte shared
// stores instead of global ones), makes it visible to the async proxy and ONE lane issues a single 9408-byte
// cp.async.bulk.global.shared::cta for it; the buffer is reused once its bulk group has been read.  The copy engine
// streams whole frames to HBM while warp 0 is already in the next tile's state phase, and the LSU no longer carries
// the 10 GB/launch store stream (ncu on env_kernel_tile: L1/TEX 78 % busy next to 85 % DRAM).
// MEASURED AND NOT ADOPTED (B200, 1M envs, RGB, fraction of the HBM copy peak; env_kernel_tile<16>: 1.08):
//   T=32, 128 thr x 3 CTAs, 1 buffer/warp  0.96      T=32, 128 x 2, 2 buffers  0.87      T=16, 128 x 3, 1 buffer  0.82
//   T=32, 256 x 2, 1 buffer  0.82    T=16, 64 x 3, 2 buffers  0.78    T=16, 128 x 2, 2 buffers  0.70    T=16, 256 x 1, 2 buffers  0.48
// The copy engine itself is not the problem -- tools/cuda/tma_store_bench.cu streams staged frames at 7.56-7.60 TB/s
// with as little as ONE 64-thread CTA per SM (per-lane st.global.cs.v4: 7.49) -- but every frame byte now crosses
// shared memory three times (atlas read, staging write, engine read) instead of once, and the staging buffers
// (9.4 KB per frame in flight) cost a resident CTA per SM (profiles/r01_tile_tma_variants.txt).  Kept selectable (kernel
// choice 4) with its parity tests, in the best shape of the table.
constexpr int kTmaT = 32, kTmaThreads = 128, kTmaCtas = 3, kTmaNbuf = 1;

__device__ __forceinline__ void bulk_store_frame(uint8_t* gdst, const uint8_t* ssrc) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst),
               "r"((uint32_t)__cvta_generic_to_shared(ssrc)), "n"(kImgBytes)
               : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
template <int PENDING>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(PENDING) : "memory");
}

// Frame phase into shared memory: `stage` receives the frame exactly as blit_frame would write it to global memory.
__device__ __forceinline__ void blit_frame_smem(const uint8_t* atlas_s, const uint8_t* kp, const uint32_t (&lut)[kChunksPerLane],
                                                uint8_t* stage, int lane) {
  const uint2* atlas64 = reinterpret_cast<const uint2*>(atlas_s);
#pragma unroll
  for (int k = 0; k < kChunksPerLane; ++k) {
    const int c = lane + 32 * k;
    if (c < kChunks) {
      const uint32_t q = lut[k];
      const uint32_t k0 = kp[q & 0xff], k1 = kp[(q >> 16) & 0xff];
      const uint2 a = atlas64[k0 * (kTileBytes / 8) + ((q >> 8) & 0xff)];
      const uint2 b = atlas64[k1 * (kTileBytes / 8) + (q >> 24)];
      *reinterpret_cast<uint4*>(stage + c * 16) = make_uint4(a.x, a.y, b.x, b.y);
    }
  }
}

constexpr int kTmaSmemBytes = tile_smem_bytes(kTmaT) + (kTmaThreads / 32) * kTmaNbuf * kImgBytes;

template <int STEP>
__global__ void __launch_bounds__(kTmaThreads, kTmaCtas) env_kernel_tile_tma(const EnvParams p, const int n_tiles) {
  extern __shared__ __align__(16) uint8_t smem[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  constexpr int warps_per_cta = kTmaThreads / 32;
  const Flags f(p);
  uint8_t* atlas_s = smem;
  uint8_t* kinds_s = smem + kAtlasBytes;
  uint8_t* sym_s = kinds_s + kTmaT * kKindStride;
  unsigned* mask_s = reinterpret_cast<unsigned*>(smem + tile_smem_bytes(kTmaT) - 16);
  uint8_t* stage_s = smem + tile_smem_bytes(kTmaT) + warp * kTmaNbuf * kImgBytes;   // this warp's kTmaNbuf frame buffers

  uint32_t lut[kChunksPerLane];
  if (f.want_rgb) {
    stage_atlas(p, atlas_s);
    load_lut(p, lane, lut);
  }
  int buf = 0;
  __shared__ int s_next;
  if (threadIdx.x == 0) s_next = (int)atomicAdd(&p.sched[0], 1u);
  __syncthreads();
  int tile = s_next;
  while (tile < n_tiles) {
    const int e0 = tile * kTmaT;
    if (warp == 0) {
      const unsigned m = state_phase<kTmaT, STEP>(p, f, e0, lane, kinds_s, sym_s);
      if (lane == 0) *mask_s = m;
    } else if (threadIdx.x == 32) {
      s_next = (int)atomicAdd(&p.sched[0], 1u);
    }
    __syncthreads();
    const unsigned render_mask = *mask_s;
    const int next = s_next;
    if (f.want_sym && render_mask)
      emit_sym_rows(p.obs_sym + (size_t)e0 * kSymBytes, sym_s, min(kTmaT, p.N - e0), render_mask, threadIdx.x, blockDim.x);
    if (f.want_rgb) {
      for (int i = warp; i < kTmaT; i += warps_per_cta) {
        if (!((render_mask >> i) & 1)) continue;
        uint8_t* stage = stage_s + buf * kImgBytes;
        if (lane == 0) bulk_wait_read<kTmaNbuf - 1>();   // the bulk group that last read this buffer is done with it
        __syncwarp();
        blit_frame_smem(atlas_s, kinds_s + i * kKindStride, lut, stage, lane);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> visible to the copy engine
        __syncwarp();
        if (lane == 0) bulk_store_frame(p.obs_rgb + (size_t)(e0 + i) * kImgBytes, stage);
        buf = (buf + 1 == kTmaNbuf) ? 0 : buf + 1;
      }
    }
    __syncthreads();
    tile = next;
  }
  if (lane == 0) bulk_wait_read<0>();   // shared memory must outlive the engine's reads
  if (threadIdx.x == 0 && atomicAdd(&p.sched[1], 1u) == gridDim.x - 1) {
    p.sched[0] = 0;
    p.sched[1] = 0;
  }
}

template <int T, int STEP, bool SWAR>
static cudaError_t launch_tile_kernel_impl(const EnvParams& p, const LaunchCtx& ctx, cudaStream_t stream) {
  const int n_tiles = (p.N + T - 1) / T;
  const size_t smem = tile_smem_bytes(T);
  int ctas;
  if (cudaError_t err = resident_ctas(ctx, env_kernel_tile<T, STEP, SWAR>, kTileThreads, smem, ctas, kTileCtasPerSm))
    return err;
  const int grid = min(ctx.sm_count * ctas, n_tiles);
  env_kernel_tile<T, STEP, SWAR><<<grid, kTileThreads, smem, stream>>>(p, n_tiles);
  return cudaGetLastError();
}
template <int T, int STEP>
static cudaError_t launch_tile_kernel_step(const EnvParams& p, const LaunchCtx& ctx, cudaStream_t stream) {
  return use_swar(p, ctx, true) ? launch_tile_kernel_impl<T, STEP, true>(p, ctx, stream)
                                : launch_tile_kernel_impl<T, STEP, false>(p, ctx, stream);
}

template <int STEP>
static cudaError_t launch_tile_tma_kernel_step(const EnvParams& p, const LaunchCtx& ctx, cudaStream_t stream) {
  const int n_tiles = (p.N + kTmaT - 1) / kTmaT;
  int ctas;
  if (cudaError_t err = resident_ctas(ctx, env_kernel_tile_tma<STEP>, kTmaThreads, kTmaSmemBytes, ctas, kTmaCtas))
    return err;
  const int grid = min(ctx.sm_count * ctas, n_tiles);
  env_kernel_tile_tma<STEP><<<grid, kTmaThreads, kTmaSmemBytes, stream>>>(p, n_tiles);
  return cudaGetLastError();
}

cudaError_t launch_tile_kernel(int T, int step, const EnvParams& p, const LaunchCtx& ctx, cudaStream_t stream) {
  if (T == 16) {
    if (step == 0) return launch_tile_kernel_step<16, 0>(p, ctx, stream);
    if (step == 1) return launch_tile_kernel_step<16, 1>(p, ctx, stream);
    return launch_tile_kernel_step<16, 2>(p, ctx, stream);
  }
  if (step == 0) return launch_tile_kernel_step<8, 0>(p, ctx, stream);
  if (step == 1) return launch_tile_kernel_step<8, 1>(p, ctx, stream);
  return launch_tile_kernel_step<8, 2>(p, ctx, stream);
}
cudaError_t launch_tile_tma_kernel(int step, const EnvParams& p, const LaunchCtx& ctx, cudaStream_t stream) {
  if (step == 0) return launch_tile_tma_kernel_step<0>(p, ctx, stream);
  if (step == 1) return launch_tile_tma_kernel_step<1>(p, ctx, stream);
  return launch_tile_tma_kernel_step<2>(p, ctx, stream);
}

}  // namespace merlin
