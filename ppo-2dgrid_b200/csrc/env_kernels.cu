// env_kernels.cu -- fused MERLIN env kernels for sm_100a: the launch policy (which mapping serves which batch) and the
// group / ordered-group / symbolic-only step kernels.  The other mappings live in their own translation units so that
// the library builds side by side: env_kernels_tile.cu (CTA tiles -- the headline mapping), env_kernels_small.cu (one
// warp per env, four envs per warp), render_kernels.cu (frames from stored symbolic observations); shared device
// helpers in env_kernels_common.cuh, the lane-per-env state phase in env_state_phase.cuh.
//
// Every step kernel does the same work per environment -- step + wrappers + auto-reset (STEP = 1: actions given;
// STEP = 2: actions drawn in the kernel from the policy's logits, merlin_env_policy_step; STEP = 3 / 4: the same two,
// also writing the symbolic image of every terminal state before its restart) or a masked reset (STEP = 0), then
// gen_obs (+process_vis), the symbolic encode and the RGB frame -- and differs only in how environments are mapped onto
// the machine.  Two phases:
//
//   state phase   step logic, reward shaping, restart, 49-cell window gather, bitmask visibility -> the 49 tile
//                 kinds (and 147 symbolic bytes) of the env, in shared memory.  ~20 warp-instructions per env when
//                 run one env per LANE (state_phase<G>), ~600 when one WARP serves one env cooperatively.
//   frame phase   the 9408-byte frame as 588 coalesced 16-byte streaming stores per env, each assembled from two
//                 8-byte reads of the tile atlas in shared memory (blit_frame); always one warp per env.
//
//   env_kernel<G>        a warp owns G consecutive envs for both phases (G = 32 at scale).  Cheapest in instructions;
//                        the unit of work is G frames (300 KB at G = 32), so it wants many groups per warp.
//   env_kernel_tile<T>   a CTA owns a tile of T envs: warp 0 runs the state phase one env per lane, then ALL warps
//                        of the CTA share the T frames.  Same cheap state phase, 8x finer frame-phase granularity:
//                        fills the SMs from a few thousand envs up and has no tail at a few tiles per CTA.
//   env_kernel_warp      one warp per env, cooperative state phase (two window cells per lane, warp ballots for the
//                        transparency mask).  Lowest latency for batches too small to give each SM a tile.
//   env_kernel_sym       state phase only (symbolic observations), one warp per 32 envs.
//
// HBM-bound streaming writers; tensor cores are not involved (there is no contraction on this path).
// Algorithmic HBM bytes per env-step (16x16, RGB): 9408 obs + 256 grid + 32 state + 8 action + 6 = 9710.
#include <cuda_runtime.h>
#include <stdint.h>

#include "env_kernels.cuh"
#include "env_kernels_common.cuh"
#include "env_state_phase.cuh"

namespace merlin {

// ---------------------------------------------------------------------------------------------------
// env_kernel<G, STEP>: a warp owns G consecutive envs.
template <int G, int STEP>
__global__ void __launch_bounds__(kThreads, 1) env_kernel(const EnvParams p, const int n_groups) {
  extern __shared__ __align__(16) uint8_t smem[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const Flags f(p);
  uint8_t* atlas_s = smem;
  uint8_t* warp_s = smem + kAtlasBytes + warp * warp_smem_bytes(G);
  uint8_t* kinds_s = warp_s;                       // [G][kKindStride]
  uint8_t* sym_s = warp_s + G * kKindStride;       // [G][147] contiguous, same layout as the output rows

  uint32_t lut[kChunksPerLane];
  if (f.want_rgb) {
    stage_atlas(p, atlas_s);
    load_lut(p, lane, lut);
  }
  __syncthreads();

  const int warps_per_cta = blockDim.x >> 5;
  for (int g = blockIdx.x * warps_per_cta + warp; g < n_groups; g += gridDim.x * warps_per_cta) {
    const int e0 = g * G;
    const unsigned render_mask = state_phase<G, STEP>(p, f, e0, lane, kinds_s, sym_s);
    if (f.want_sym && render_mask)
      emit_sym_rows(p.obs_sym + (size_t)e0 * kSymBytes, sym_s, min(G, p.N - e0), render_mask, lane, 32);
    if (f.want_rgb) {
      unsigned m = render_mask;
      while (m) {
        const int i = __ffs(m) - 1;
        m &= m - 1;
        blit_frame(atlas_s, kinds_s + i * kKindStride, lut, p.obs_rgb + (size_t)(e0 + i) * kImgBytes, lane);
      }
    }
    __syncwarp();  // smem rows are reused by the next group
  }
}

// ---------------------------------------------------------------------------------------------------
// env_kernel_ordered<STEP>: env_kernel's mapping (a warp owns kOrdG consecutive envs for both phases)
// with the groups handed out IN ORDER, one ticket per warp, from the same self-resetting counter the tile kernel
// uses.  Every warp of the SM runs its own state phase (no warp-0 bottleneck, no CTA barrier in the loop): the
// dependent-load chain of a state phase (~10 us) is hidden by all resident warps instead of one per CTA, while the
// write fronts still advance together.  The next ticket is drawn before the work so its latency is off the path.
// MEASURED AND NOT ADOPTED (B200, 1M envs, RGB, fraction of the HBM copy peak; env_kernel_tile<16>: 1.08):
//   G=8, 128 thr x 3 CTAs  1.046    G=16, 128 x 3  1.045    G=32, 128 x 3  1.041    G=8, 128 x 4 (spills)  1.033
//   G=8, 256 x 2  1.034    G=16, 256 x 2  1.024    G=16, 128 x 4  1.021    G=4, 128 x 4  0.920
// i.e. in-order hand-out lifts the group mapping from 0.92 (static assignment) to 1.05, but more concurrent state phases
// buy nothing over the tile kernel: its limit is the store stream, not the state-phase chain
// (profiles/r01_ordered_group_variants.txt).  Kept selectable (choice 6) in the first shape of the table.
constexpr int kOrdG = 8, kOrdThreads = 128, kOrdCtas = 3;
template <int STEP, bool SWAR = false>
__global__ void __launch_bounds__(kOrdThreads, kOrdCtas) env_kernel_ordered(const EnvParams p, const int n_groups) {
  extern __shared__ __align__(16) uint8_t smem[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  Flags f(p);
  if (SWAR) f.doors = pool_has_doors(p.tile_present);
  uint8_t* atlas_s = smem;
  uint8_t* warp_s = smem + kAtlasBytes + warp * warp_smem_bytes(kOrdG);
  uint8_t* kinds_s = warp_s;
  uint8_t* sym_s = warp_s + kOrdG * kKindStride;

  uint32_t lut[kChunksPerLane];
  if (f.want_rgb) {
    stage_atlas(p, atlas_s);
    load_lut(p, lane, lut);
  }
  __syncthreads();

  int g = 0;
  if (lane == 0) g = draw_ticket(p.sched);
  g = __shfl_sync(0xffffffffu, g, 0);
  while (g < n_groups) {
    int next = 0;
    if (lane == 0) next = draw_ticket(p.sched);
    const int e0 = g * kOrdG;
    const unsigned render_mask = state_phase<kOrdG, STEP, SWAR>(p, f, e0, lane, kinds_s, sym_s);
    if (f.want_sym && render_mask)
      emit_sym_rows(p.obs_sym + (size_t)e0 * kSymBytes, sym_s, min(kOrdG, p.N - e0), render_mask, lane, 32);
    if (f.want_rgb) {
      unsigned m = render_mask;
      while (m) {
        const int i = __ffs(m) - 1;
        m &= m - 1;
        blit_frame(atlas_s, kinds_s + i * kKindStride, lut, p.obs_rgb + (size_t)(e0 + i) * kImgBytes, lane);
      }
    }
    __syncwarp();  // smem rows are reused by the next group
    g = __shfl_sync(0xffffffffu, next, 0);
  }
  // every warp of the grid has drawn its last ticket once all of them have passed here: the last one rearms
  if (lane == 0) rearm_tickets(p.sched, gridDim.x * (kOrdThreads / 32));
}

// ---------------------------------------------------------------------------------------------------
// env_kernel_sym<STEP>: symbolic observations only (no frame phase): one warp per 32 envs, plain grid.  Without the
// blit map and the frame loop the state phase fits in ~72 registers, so six to seven 128-thread CTAs are resident per
// SM instead of one 256-thread CTA of env_kernel<32>: this mode is instruction/latency-bound (449 B per env-step), and
// occupancy is what it needs.
__host__ __device__ constexpr int sym_kernel_warp_smem(bool swar) {
  return swar ? 32 * kSymBytes : warp_smem_bytes(32);
}

// Resident CTAs the row-parallel form is compiled for: 48 registers, 40 warps/SM, 1.16e10 env-steps/s at 1M envs
// (unconstrained, 56 registers: 1.11e10; 12 CTAs, 40 registers + spills: 1.04e10;
// profiles/r01_symbolic_kernel_occupancy_variants.txt).
constexpr int kSymSwarCtas = 10;
template <int STEP, bool SWAR = false>
__global__ void __launch_bounds__(128, SWAR ? kSymSwarCtas : 1) env_kernel_sym(const EnvParams p, const int n_groups) {
  extern __shared__ __align__(16) uint8_t smem[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  Flags f(p);
  f.want_rgb = false;  // no frame phase here: tile kinds are not produced either
  if (SWAR) f.doors = pool_has_doors(p.tile_present);
  // the row-parallel form keeps the window in registers; only the per-cell form stages the 49 codes per env
  uint8_t* warp_s = smem + warp * sym_kernel_warp_smem(SWAR);
  uint8_t* kinds_s = SWAR ? nullptr : warp_s;
  uint8_t* sym_s = SWAR ? warp_s : warp_s + 32 * kKindStride;
  const int g = blockIdx.x * (blockDim.x >> 5) + warp;
  if (g >= n_groups) return;
  const int e0 = g * 32;
  const unsigned render_mask = state_phase<32, STEP, SWAR>(p, f, e0, lane, kinds_s, sym_s);
  if (f.want_sym && render_mask)
    emit_sym_rows(p.obs_sym + (size_t)e0 * kSymBytes, sym_s, min(32, p.N - e0), render_mask, lane, 32);
}

template <int STEP>
static cudaError_t launch_sym_kernel(const EnvParams& p, const LaunchCtx& ctx, cudaStream_t stream) {
  constexpr int threads = 128, warps = threads / 32;
  const int n_groups = (p.N + 31) / 32;
  const int grid = (n_groups + warps - 1) / warps;
  if (use_swar(p, ctx, false))
    env_kernel_sym<STEP, true><<<grid, threads, warps * sym_kernel_warp_smem(true), stream>>>(p, n_groups);
  else
    env_kernel_sym<STEP, false><<<grid, threads, warps * sym_kernel_warp_smem(false), stream>>>(p, n_groups);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------
// launch helpers: persistent grids of (SMs x resident CTAs), capped by the work available (resident_ctas:
// env_kernels_common.cuh).
template <int G, int STEP>
static cudaError_t launch_group_kernel(const EnvParams& p, const LaunchCtx& ctx, cudaStream_t stream) {
  const int n_groups = (p.N + G - 1) / G;
  const size_t smem = cta_smem_bytes(G);
  int ctas;
  if (cudaError_t err = resident_ctas(ctx, env_kernel<G, STEP>, kThreads, smem, ctas)) return err;
  const int grid = min(ctx.sm_count * ctas, (n_groups + kWarps - 1) / kWarps);
  env_kernel<G, STEP><<<grid, kThreads, smem, stream>>>(p, n_groups);
  return cudaGetLastError();
}

template <int STEP, bool SWAR>
static cudaError_t launch_ordered_kernel_impl(const EnvParams& p, const LaunchCtx& ctx, cudaStream_t stream) {
  constexpr int warps = kOrdThreads / 32;
  const int n_groups = (p.N + kOrdG - 1) / kOrdG;
  const size_t smem = kAtlasBytes + warps * warp_smem_bytes(kOrdG);
  int ctas;
  if (cudaError_t err = resident_ctas(ctx, env_kernel_ordered<STEP, SWAR>, kOrdThreads, smem, ctas, kOrdCtas))
    return err;
  const int grid = min(ctx.sm_count * ctas, (n_groups + warps - 1) / warps);
  env_kernel_ordered<STEP, SWAR><<<grid, kOrdThreads, smem, stream>>>(p, n_groups);
  return cudaGetLastError();
}
template <int STEP>
static cudaError_t launch_ordered_kernel(const EnvParams& p, const LaunchCtx& ctx, cudaStream_t stream) {
  return use_swar(p, ctx, true) ? launch_ordered_kernel_impl<STEP, true>(p, ctx, stream)
                                : launch_ordered_kernel_impl<STEP, false>(p, ctx, stream);
}

// Automatic choice, from the B200 sweeps in profiles/.  RGB observations: the warp kernel while every env of the batch
// is resident at once or nearly so, the tile kernel above.  The quad kernel (choice 7) is not picked: under CUDA-graph
// replay it is 7 % faster at 8192 envs (14.6 vs 15.7 us), equal at 5120-6144, slower below (8.8 vs 8.3 us at 4096) and
// above (22.4 vs 20.6 us at 12 288), and slower everywhere when launched eagerly (profiles/r02_quad_vs_warp.txt).
// Symbolic-only observations are instruction-bound: the state phase alone, at high occupancy -- except for batches so
// small that one env's chain of ~1800 dependent instructions IS the run time: there a warp per env (the same chain
// spread over 32 lanes) is 1.3 us faster (2.9 vs 4.2 us at 32 envs, 3.4 vs 4.7 us at 1024; equal at ~3000).
constexpr int kRgbWarpMaxEnvs = 24576;
constexpr int kSymWarpMaxEnvs = 2048;

StepKernel select_step_kernel(int n_envs, bool rgb, bool lean, bool final, const LaunchCtx& ctx) {
  int choice = ctx.kernel_choice;
  if (choice == kChoiceAuto) {
    if (rgb) choice = n_envs <= kRgbWarpMaxEnvs ? kChoiceWarp : kChoiceTile;
    else choice = n_envs <= kSymWarpMaxEnvs ? kChoiceWarp : kChoiceSym;
  }
  switch (choice) {
    case kChoiceGroup: {
      // the largest group size that still yields >= ~8 warps per SM; tiny batches use smaller groups
      const long long want_warps = (long long)ctx.sm_count * 8;
      for (int G = 32; G > 4; G /= 2)
        if (n_envs / G >= want_warps) return {kChoiceGroup, G};
      return {kChoiceGroup, 4};
    }
    case kChoiceTile:
      // tiles of 16 envs once every resident CTA gets one; smaller tiles spread a small batch over more CTAs
      return {kChoiceTile, n_envs >= ctx.sm_count * kTileCtasPerSm * 16 ? 16 : 8};
    case kChoiceQuad:
      return {lean && rgb && !final ? kChoiceQuad : kChoiceWarp, 0};
    default:
      return {choice, 0};
  }
}

const char* step_kernel_name(StepKernel k) {
  switch (k.choice) {
    case kChoiceGroup:
      return k.size == 32 ? "merlin::env_kernel<32,true>" : k.size == 16 ? "merlin::env_kernel<16,true>"
           : k.size == 8  ? "merlin::env_kernel<8,true>"  : "merlin::env_kernel<4,true>";
    case kChoiceTile: return k.size == 16 ? "merlin::env_kernel_tile<16,true>" : "merlin::env_kernel_tile<8,true>";
    case kChoiceTileTma: return "merlin::env_kernel_tile_tma<true>";
    case kChoiceSym: return "merlin::env_kernel_sym<true>";
    case kChoiceOrdered: return "merlin::env_kernel_ordered<true>";
    case kChoiceQuad: return "merlin::env_kernel_quad<true>";
    default: return "merlin::env_kernel_warp<true>";
  }
}

template <int STEP>
static cudaError_t launch_sized(const EnvParams& p, const LaunchCtx& ctx, cudaStream_t stream) {
  const StepKernel k = select_step_kernel(p.N, p.obs_rgb != nullptr, lean_config(p.flags), step_final(STEP), ctx);
  switch (k.choice) {
    case kChoiceGroup:
      if (k.size == 32) return launch_group_kernel<32, STEP>(p, ctx, stream);
      if (k.size == 16) return launch_group_kernel<16, STEP>(p, ctx, stream);
      if (k.size == 8) return launch_group_kernel<8, STEP>(p, ctx, stream);
      return launch_group_kernel<4, STEP>(p, ctx, stream);
    case kChoiceTile:
      return k.size == 16 ? launch_tile_kernel<16, STEP>(p, ctx, stream) : launch_tile_kernel<8, STEP>(p, ctx, stream);
    case kChoiceTileTma: return launch_tile_tma_kernel<STEP>(p, ctx, stream);
    case kChoiceSym: return launch_sym_kernel<STEP>(p, ctx, stream);
    case kChoiceOrdered: return launch_ordered_kernel<STEP>(p, ctx, stream);
    case kChoiceQuad:
      if constexpr (STEP == 1 || STEP == 2) return launch_quad_kernel<STEP>(p, ctx, stream);
      return launch_warp_kernel<STEP>(p, ctx, stream);   // the quad kernel only steps, without final observations
    default: return launch_warp_kernel<STEP>(p, ctx, stream);
  }
}

cudaError_t launch_env_step(const EnvParams& p, const LaunchCtx& ctx, cudaStream_t stream) {
  if (p.final_sym != nullptr) return p.logits != nullptr ? launch_sized<4>(p, ctx, stream) : launch_sized<3>(p, ctx, stream);
  return p.logits != nullptr ? launch_sized<2>(p, ctx, stream) : launch_sized<1>(p, ctx, stream);
}
cudaError_t launch_env_reset(const EnvParams& p, const LaunchCtx& ctx, cudaStream_t stream) {
  return launch_sized<0>(p, ctx, stream);
}

}  // namespace merlin


