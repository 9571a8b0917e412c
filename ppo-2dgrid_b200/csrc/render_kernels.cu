// render_kernels.cu -- frames from stored symbolic observations (render_kernel: u8, both layouts; render_f32_kernel: the
// first layer's float32 input) and the fully observable symbolic observation, for sm_100a.
#include <cuda_runtime.h>
#include <stdint.h>

#include "env_kernels.cuh"
#include "env_kernels_common.cuh"
#include "env_logic.cuh"

namespace merlin {

// ---------------------------------------------------------------------------------------------------
// render_kernel<BLOCKED>: frames from stored symbolic observations, one warp per frame, optional row gather.
// Rollouts can then keep 147 B per step instead of 9408 B and expand minibatches on read.
//
// One frame from `atlas` (the CTA's staged copy in shared memory, or the u8 atlas in global memory) and its 49 kinds.
template <bool BLOCKED>
__device__ __forceinline__ void render_frame(const uint8_t* atlas, const uint8_t* kp, const uint32_t (&lut)[kChunksPerLane],
                                             uint8_t* frame, int lane) {
  if (BLOCKED) {
    const uint4* atlas128 = reinterpret_cast<const uint4*>(atlas);
#pragma unroll
    for (int k = 0; k < kChunksPerLane; ++k) {
      const int c = lane + 32 * k;
      if (c < kChunks) {
        const uint32_t q = lut[k];
        const uint4 v = atlas128[kp[q & 0xff] * (kTileBytes / 16) + (q >> 8)];
        st_stream_v4(frame + c * 16, v.x, v.y, v.z, v.w);
      }
    }
  } else {
    blit_frame(atlas, kp, lut, frame, lane);
  }
}

template <bool BLOCKED>
__global__ void __launch_bounds__(256, 2) render_kernel(const RenderParams p) {
  extern __shared__ __align__(16) uint8_t smem[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int warps_per_cta = blockDim.x >> 5;
  uint8_t* atlas_s = smem;
  uint8_t* kp = smem + kAtlasBytes + warp * kWarpKindStride;
  {
    const int4* src = reinterpret_cast<const int4*>(p.atlas);
    int4* dst = reinterpret_cast<int4*>(atlas_s);
    for (int i = threadIdx.x; i < kAtlasBytes / 16; i += blockDim.x) {
      const int tile = i / (kTileBytes / 16);
      if (tile_bit(p.tile_present, tile)) dst[i] = __ldg(src + i);
    }
  }
  uint32_t lut[kChunksPerLane];
#pragma unroll
  for (int k = 0; k < kChunksPerLane; ++k) lut[k] = __ldg(p.lut + k * 32 + lane);
  __syncthreads();

  // groups of consecutive frames are drawn in order from a ticket counter (see env_kernel_tile): 32 frames per ticket
  // for large batches (the write fronts of all CTAs stay in one narrow window), 8 -- one per warp -- for minibatch-sized
  // ones (16 384 frames are 512 groups of 32 on 296 CTAs: two rounds, the second 73 % full; 2048 groups of 8 are 6.9)
  const int kRenderGroup = p.group_frames;
  __shared__ int s_next;
  const int n_groups = (p.M + kRenderGroup - 1) / kRenderGroup;
  if (threadIdx.x == 0) s_next = (int)atomicAdd(&p.sched[0], 1u);
  __syncthreads();
  int group = s_next;
  while (group < n_groups) {
    __syncthreads();  // everyone has read the ticket
    if (threadIdx.x == 0) s_next = (int)atomicAdd(&p.sched[0], 1u);
    for (int m = group * kRenderGroup + warp; m < min(p.M, (group + 1) * kRenderGroup); m += warps_per_cta) {
      long long row = p.index ? p.index[m] : m;
      if (p.n_rows && (row < 0 || row >= p.n_rows)) row = 0;  // never read outside the buffer; callers validate indices
      const uint8_t* sym = p.sym + (size_t)row * kSymBytes;
      bool staged = true;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int k = lane + 32 * h;  // cell index vi*7 + vj, the order Grid.encode stores them
        if (k < kCells) {
          const uint32_t t = sym[3 * k], c = sym[3 * k + 1], st = sym[3 * k + 2];
          const uint32_t kind = kind_of_sym(t, c, st, k == (kView / 2) * kView + (kView - 1));
          kp[k] = (uint8_t)kind;
          staged = staged && tile_bit(p.tile_present, kind);
        }
      }
      // Only the tiles the current pool can show were staged.  A stored image may show others (it was stepped under an
      // earlier pool, or never came from this handle at all): such a frame is read from the atlas in global memory.
      const bool all_staged = __all_sync(0xffffffffu, staged);
      __syncwarp();
      uint8_t* frame = p.out + (size_t)m * kImgBytes;
      if (all_staged) render_frame<BLOCKED>(atlas_s, kp, lut, frame, lane);
      else render_frame<BLOCKED>(p.atlas, kp, lut, frame, lane);
      __syncwarp();  // kp is reused by this warp's next frame
    }
    __syncthreads();  // the next ticket is in shared memory
    group = s_next;
  }
  if (threadIdx.x == 0 && atomicAdd(&p.sched[1], 1u) == gridDim.x - 1) {
    p.sched[0] = 0;
    p.sched[1] = 0;
  }
}

constexpr int kRenderGroup32MinFrames = 65536;
cudaError_t launch_render(const RenderParams& p, bool blocked, int sm_count, cudaStream_t stream) {
  if (p.M <= 0) return cudaSuccess;
  constexpr int threads = 256, warps = threads / 32;
  const size_t smem = kAtlasBytes + warps * kWarpKindStride;
  RenderParams q = p;
  q.group_frames = p.M >= kRenderGroup32MinFrames ? 32 : warps;
  const int grid = min(sm_count * 2, (p.M + q.group_frames - 1) / q.group_frames);
  if (blocked) render_kernel<true><<<grid, threads, smem, stream>>>(q);
  else render_kernel<false><<<grid, threads, smem, stream>>>(q);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------
// render_f32_kernel: the blocked frame as float32 -- f32[M][14][14][48], optionally pixel / 255.0f -- i.e. the very
// tensor the actor-critic's first layer reads (reference src/actor_critic.py:21 forms `x / 255.0` from a float32 copy
// of the frame on every evaluation).  Writing it here replaces three passes of the learner's minibatch path (u8 frame
// write, u8 read + f32 write of the cast, and the layout copy) by one 37 632-byte streaming write per frame.
//
// One warp per frame.  The atlas slots the layout pool can show are converted ONCE per CTA into a float atlas in
// shared memory (compacted: slot_of_kind[128]; 768 B per staged tile, `cap_tiles` of them), so a 16-byte output chunk
// is one u16 map read (shared by 4 lanes), one slot read and one 16-byte shared-memory read.  A kind that is not
// staged (a CUDA graph replayed after a re-upload brought new tile kinds) is converted on the fly from the u8 atlas.
// HBM-bound: 147 (+8) B read, 37 632 B written per frame.
constexpr int kF32Chunks = kImgBytes / 4;                  // 2352 float4 chunks per frame
constexpr int kF32Iters = (kF32Chunks + 31) / 32;          // 74
constexpr int kRenderF32Group = 8;                          // frames per ticket: 301 KB, like the u8 kernels' groups
constexpr int kRenderF32Threads = 256;
constexpr int kRenderF32CtaFramesMax = 8192;

__host__ __device__ constexpr size_t render_f32_smem(int cap_tiles) {
  return (size_t)cap_tiles * kTileBytes * 4 + 128 + 592 * 2 + (kRenderF32Threads / 32) * 128;
}

// normalise: 0 = the pixel value, 1 = pixel / 255.0f (IEEE division: what torch's CPU kernels compute for `x / 255.0`),
// 2 = pixel * (1.0f / 255.0f) (what torch's CUDA kernel computes for a tensor divided by a Python scalar)
__device__ __forceinline__ float pixel_f32(uint32_t b, int normalise) {
  const float v = (float)b;
  if (normalise == 1) return __fdiv_rn(v, 255.0f);
  if (normalise == 2) return __fmul_rn(v, __fdiv_rn(1.0f, 255.0f));
  return v;
}

__global__ void __launch_bounds__(kRenderF32Threads, 3) render_f32_kernel(const RenderParams p) {
  extern __shared__ __align__(16) uint8_t smem[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  constexpr int warps_per_cta = kRenderF32Threads / 32;
  float* atlas_f = reinterpret_cast<float*>(smem);
  uint8_t* slot_s = smem + (size_t)p.cap_tiles * kTileBytes * 4;
  uint16_t* map_s = reinterpret_cast<uint16_t*>(slot_s + 128);
  uint8_t* kp = reinterpret_cast<uint8_t*>(map_s + 592) + warp * 128;   // [0..48] slots, [64..112] kinds
  const int normalise = p.normalise;

  if (threadIdx.x < kAtlasTiles) {  // compact the present tiles: slot = number of present tiles below this one
    const int t = threadIdx.x;
    int below = 0;
    for (int w = 0; w < (t >> 5); ++w) below += __popc(__ldg(p.tile_present + w));
    below += __popc(__ldg(p.tile_present + (t >> 5)) & ((1u << (t & 31)) - 1u));
    slot_s[t] = (tile_bit(p.tile_present, t) && below < p.cap_tiles) ? (uint8_t)below : (uint8_t)255;
  }
  for (int c = threadIdx.x; c < kChunks; c += blockDim.x) map_s[c] = (uint16_t)chunk_lut_blocked(c);
  __syncthreads();
  for (int t = warp; t < kAtlasTiles; t += warps_per_cta) {
    const uint32_t slot = slot_s[t];
    if (slot == 255) continue;
    for (int i = lane; i < kTileBytes; i += 32)
      atlas_f[slot * kTileBytes + i] = pixel_f32(__ldg(p.atlas + t * kTileBytes + i), normalise);
  }
  __syncthreads();

  // one frame's float4 chunk f: one u16 map read (shared by 4 lanes), one slot read, one 16-byte atlas read, one store
  auto emit_chunk = [&](const uint8_t* kpw, float* frame, int f) {
    const uint32_t q = map_s[f >> 2];
    const uint32_t cell = q & 0xff, off = (q >> 8) * 16 + (f & 3) * 4;   // element offset inside the tile
    const uint32_t slot = kpw[cell];
    float4 v;
    if (slot != 255) {
      v = *reinterpret_cast<const float4*>(atlas_f + slot * kTileBytes + off);
    } else {
      const uint32_t w = __ldg(reinterpret_cast<const uint32_t*>(p.atlas + (uint32_t)kpw[64 + cell] * kTileBytes + off));
      v = make_float4(pixel_f32(w & 0xff, normalise), pixel_f32((w >> 8) & 0xff, normalise),
                      pixel_f32((w >> 16) & 0xff, normalise), pixel_f32(w >> 24, normalise));
    }
    st_stream_v4(frame + f * 4, __float_as_uint(v.x), __float_as_uint(v.y), __float_as_uint(v.z), __float_as_uint(v.w));
  };
  auto load_kinds = [&](uint8_t* kpw, int m, int t) {   // thread t < 64 of the caller's group handles cells t (and < 49)
    long long row = p.index ? p.index[m] : m;
    if (p.n_rows && (row < 0 || row >= p.n_rows)) row = 0;
    const uint8_t* sym = p.sym + (size_t)row * kSymBytes;
    if (t < kCells) {
      const uint32_t kind = kind_of_sym(sym[3 * t], sym[3 * t + 1], sym[3 * t + 2], t == (kView / 2) * kView + (kView - 1));
      kpw[t] = slot_s[kind];
      kpw[64 + t] = (uint8_t)kind;
    }
  };

  if (p.frame_per_cta) {
    // few frames (a policy-input render for a small batch: launch latency is what counts): one CTA per frame, all
    // eight warps share its 2352 chunks -- 10 chunk rounds per thread instead of 74 per lane
    for (int m = blockIdx.x; m < p.M; m += gridDim.x) {
      __syncthreads();  // kp of the previous frame has been consumed
      load_kinds(kp - warp * 128, m, threadIdx.x);
      __syncthreads();
      float* frame = p.out_f32 + (size_t)m * kImgBytes;
      for (int f = threadIdx.x; f < kF32Chunks; f += kRenderF32Threads) emit_chunk(kp - warp * 128, frame, f);
    }
    return;
  }

  __shared__ int s_next;
  const int n_groups = (p.M + kRenderF32Group - 1) / kRenderF32Group;
  if (threadIdx.x == 0) s_next = (int)atomicAdd(&p.sched[0], 1u);
  __syncthreads();
  int group = s_next;
  while (group < n_groups) {
    __syncthreads();  // everyone has read the ticket
    if (threadIdx.x == 0) s_next = (int)atomicAdd(&p.sched[0], 1u);
    for (int m = group * kRenderF32Group + warp; m < min(p.M, (group + 1) * kRenderF32Group); m += warps_per_cta) {
      load_kinds(kp, m, lane);
      load_kinds(kp, m, lane + 32);
      __syncwarp();
      float* frame = p.out_f32 + (size_t)m * kImgBytes;
#pragma unroll 4
      for (int k = 0; k < kF32Iters; ++k) {
        const int f = lane + 32 * k;
        if (f < kF32Chunks) emit_chunk(kp, frame, f);
      }
      __syncwarp();  // kp is reused by this warp's next frame
    }
    __syncthreads();  // the next ticket is in shared memory
    group = s_next;
  }
  if (threadIdx.x == 0 && atomicAdd(&p.sched[1], 1u) == gridDim.x - 1) {
    p.sched[0] = 0;
    p.sched[1] = 0;
  }
}

cudaError_t launch_render_f32(const RenderParams& p, int sm_count, cudaStream_t stream) {
  if (p.M <= 0) return cudaSuccess;
  const size_t smem = render_f32_smem(p.cap_tiles);
  if (smem > 48 * 1024) {  // every atlas slot staged (7-action handles): opt in, per device (the call is cheap)
    cudaError_t err = cudaFuncSetAttribute(render_f32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)render_f32_smem(kAtlasTiles));
    if (err != cudaSuccess) return err;
  }
  const int per_sm = smem > 72 * 1024 ? 2 : 3;
  RenderParams q = p;
  // Few frames -- up to a few rounds of (resident CTAs x 8 warps): a CTA renders a frame with all its warps and strides
  // over the frames (no ticket counter involved).  With a warp per frame, 4096 frames are 1.15 rounds of the 3552 resident
  // warps, i.e. two rounds of which the second is 15 % full; with a CTA per frame they are 9.2 rounds of 444 CTAs, i.e. ten.
  // Above: groups of 8 frames per ticket, one warp per frame.
  q.frame_per_cta = p.M <= kRenderF32CtaFramesMax ? 1 : 0;
  const int grid = q.frame_per_cta ? min(p.M, sm_count * per_sm)
                                   : min(sm_count * per_sm, (p.M + kRenderF32Group - 1) / kRenderF32Group);
  render_f32_kernel<<<grid, kRenderF32Threads, smem, stream>>>(q);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------
// full_obs_kernel: the fully observable symbolic observation (minigrid FullyObsWrapper; selected by
// `observation.fully_observable: true` in the reference's scenario.yaml, src/scenario_creator/scenario_creator.py:45-46).
// One thread per output cell, output-order indexing (coalesced 3-byte cells; the 256-byte grids are read through L1).
__global__ void __launch_bounds__(256) full_obs_kernel(const EnvParams p, uint8_t* __restrict__ out) {
  const long long cells_per_env = (long long)p.W * p.H;
  const long long total = cells_per_env * p.N;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int e = (int)(i / cells_per_env);
    const int c = (int)(i - (long long)e * cells_per_env);
    const int x = c / p.H, y = c - x * p.H;  // output index [x][y]
    const int4 st = p.state[e];
    EnvState s{};
    unpack_state(st.x, st.y, st.z, st.w, s);
    const uint8_t* grid = p.cells ? p.cells + (size_t)e * p.cell_stride
                                  : p.pool_cells + (size_t)(s.layout < 0 ? ~s.layout : s.layout) * p.cell_stride;
    uint8_t t, col, stt;
    if (x == s.x && y == s.y) { t = (uint8_t)T_AGENT; col = 0; stt = (uint8_t)s.dir; }
    else sym_of_code(grid[y * p.W + x], t, col, stt);
    out[i * 3 + 0] = t; out[i * 3 + 1] = col; out[i * 3 + 2] = stt;
  }
}

cudaError_t launch_full_obs(const EnvParams& p, uint8_t* out, int sm_count, cudaStream_t stream) {
  const long long total = (long long)p.W * p.H * p.N;
  const int grid = (int)min((long long)sm_count * 8, (total + 255) / 256);
  full_obs_kernel<<<grid, 256, 0, stream>>>(p, out);
  return cudaGetLastError();
}

}  // namespace merlin
