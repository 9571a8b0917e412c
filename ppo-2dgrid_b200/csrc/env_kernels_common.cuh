// env_kernels_common.cuh -- device helpers and launch helpers shared by the kernel translation units
// (env_kernels.cu: the group / ordered / symbolic-only step kernels and the launch policy; env_kernels_tile.cu: the
// CTA-tile step kernels; env_kernels_small.cu: the small-batch step kernels; render_kernels.cu: frames from stored
// symbolic observations).  Every per-env building block the six step-kernel mappings share -- the step outputs, the
// restart, a window cell, the tile kind an observed cell shows, the work tickets -- is defined here once, and so are
// the declarations of the launchers env_kernels.cu calls in the other translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "env_kernels.cuh"
#include "env_logic.cuh"

namespace merlin {

// Streaming (evict-first) 16-byte store.  Measured on B200 at 1M envs: .cs 0.99 of the HBM copy peak, plain / .cg
// stores 0.93, 256-bit st.global.v8.b32 (with or without L2::evict_first) 0.92-0.94.
__device__ __forceinline__ void st_stream_v4(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// Grid loads carry an L2 cache policy: evict-LAST when the grid is an entry of the shared layout pool.  The pool
// (16 MB at the benchmark's 65 536 layouts) is re-read by every step while 10 GB of frames stream through the same L2
// between two uses of a line; tagged evict-last it stays resident.  Measured on B200, 1M envs, RGB, 65 536 layouts:
// 1.484 -> 1.418 ms per step (7.07e8 -> 7.39e8 env-steps/s, +4.6 %); with the 8192-layout pool of round 1 +0.9 %
// (profiles/r02_pool_evict_last_ab.txt).  Private (mutable) grids -- 256 B per env, no reuse across envs -- keep the
// normal policy.
__device__ __forceinline__ uint64_t grid_policy(bool shared_pool) {
  uint64_t last, normal;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(last));
  asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(normal));
  return shared_pool ? last : normal;
}
__device__ __forceinline__ uint32_t ld_cell(const uint8_t* p, uint64_t pol) {
  uint32_t v;
  asm volatile("ld.global.L2::cache_hint.u8 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
  return v;
}

constexpr int kWarpKindStride = 64;   // per-warp slot for the 49 tile kinds of one env

// bit `tile` of the 128-bit "present" mask (four device words, read through the read-only path; they live in device
// memory rather than in the kernel parameters so that a captured CUDA graph sees a re-uploaded layout pool's mask)
__device__ __forceinline__ bool tile_bit(const uint32_t* m, int tile) {
  return (__ldg(m + (tile >> 5)) >> (tile & 31)) & 1u;
}

// Can a closed / locked door occur in a grid of this handle?  Read from the device-resident "present" mask (codes
// type | colour << 4 with type 11 / 12; mutable grids set every bit), so a CUDA graph captured before a re-upload
// still sees the current pool.  Without doors, walls are the only opaque cells and Grid.encode needs no state byte:
// the row-parallel observation takes its short path (warp-uniform branch).
__device__ __forceinline__ bool pool_has_doors(const uint32_t* present) {
  constexpr uint32_t kDoorBits = (1u << T_DOOR_CLOSED) | (1u << T_DOOR_LOCKED);
  constexpr uint32_t kMask = kDoorBits | (kDoorBits << 16);   // colours 2w and 2w + 1 share word w
  return ((__ldg(present) | __ldg(present + 1) | __ldg(present + 2) | __ldg(present + 3)) & kMask) != 0;
}

struct Flags {
  int n_actions;
  bool mutable_grid, stuck_on, explore_on, auto_reset, advance, want_rgb, want_sym;
  bool doors = true;   // set by the kernels that run the row-parallel observation
  uint64_t pol;        // L2 cache policy of the grid loads (grid_policy)
  __device__ __forceinline__ explicit Flags(const EnvParams& p)
      : n_actions((p.flags & MERLIN_F_SEVEN_ACTIONS) ? 7 : 3), mutable_grid(p.cells != nullptr),
        stuck_on(p.flags & MERLIN_F_STUCK_PENALTY), explore_on(p.flags & MERLIN_F_EXPLORE_BONUS),
        auto_reset(p.flags & MERLIN_F_AUTO_RESET), advance(!(p.flags & MERLIN_F_RESET_SAME)),
        want_rgb(p.obs_rgb != nullptr), want_sym(p.obs_sym != nullptr), pol(grid_policy(p.cells == nullptr)) {}
};

// The action env e takes this step: read from `actions`, or -- policy I/O -- drawn here from the policy's logits
// (sample_policy, env_logic.cuh).  `commit`: this thread stores the action / log-probability / value rows and advances
// the env's draw counter (one lane per env in the lane-per-env kernels, lane 0 in the warp-per-env kernel, where every
// lane computes the same sample from the same warp-uniform loads).
struct ActionDraw {
  long long action;
  float logp;
  uint32_t draw;
};
// The step kernels are instantiated five times: STEP = 0 (masked reset), 1 (step, actions given), 2 (step, actions
// drawn here from the policy's logits), 3 and 4 (1 and 2 that also write the final observation of every episode that
// ends, EnvParams::final_sym).  The policy code exists only in the instances that draw, the final-observation code only
// in STEP 3 / 4: compiled into the others -- even behind a uniform branch, even out of line -- it degrades the register
// allocation of the frame kernels' state phase, which runs under a 128-register cap (B200, 1M envs: 1461 us per step vs
// 1434 us without the policy code; profiles/r02_tile_kernel_ab.txt).
__host__ __device__ constexpr bool step_given(int STEP) { return STEP == 1 || STEP == 3; }   // actions from `actions`
__host__ __device__ constexpr bool step_draws(int STEP) { return STEP == 2 || STEP == 4; }   // drawn from `logits`
__host__ __device__ constexpr bool step_final(int STEP) { return STEP >= 3; }                // writes `final_sym`
template <bool POLICY>
__device__ __forceinline__ ActionDraw draw_action(const EnvParams& p, int n_actions, int e) {
  ActionDraw d;
  d.logp = 0.f;
  d.draw = 0;
  if (!POLICY) {
    d.action = p.actions[e];
    return d;
  }
  float lg[kMaxActions];
  const float* row = p.logits + (size_t)e * p.logits_stride;
#pragma unroll
  for (int a = 0; a < kMaxActions; ++a) lg[a] = a < n_actions ? row[a] : 0.f;
  float u = 0.f;
  if (!p.greedy) {
    d.draw = p.draws[e];
    u = sampler_uniform(p.seed_lo, p.seed_hi, (uint32_t)e, d.draw);
  }
  const PolicySample smp = sample_policy(lg, n_actions, u, p.greedy != 0);
  d.action = smp.action;
  d.logp = smp.logp;
  return d;
}
template <bool POLICY>
__device__ __forceinline__ void commit_action(const EnvParams& p, int e, const ActionDraw& d) {
  if (!POLICY) return;
  if (!p.greedy) p.draws[e] = d.draw + 1u;
  p.out_action[e] = d.action;
  p.out_logp[e] = d.logp;
  if (p.out_value) p.out_value[e] = p.value_in[(size_t)e * p.value_stride];
}
// First-episode record of deterministic evaluation (see EnvParams::rec_finished).
template <bool POLICY>
__device__ __forceinline__ void record_first_episode(const EnvParams& p, int e, bool done, bool goal, float ep_ret, int len) {
  if (!POLICY || p.rec_finished == nullptr || !done || p.rec_finished[e]) return;
  p.rec_finished[e] = 1;
  p.rec_return[e] = ep_ret;
  p.rec_length[e] = len;
  p.rec_goal[e] = goal ? 1 : 0;
}

// Per-env outputs of a step: reward, the termination flags, and the optional episode-end / stuck / done rows.
__device__ __forceinline__ void store_step_outputs(const EnvParams& p, int e, float rew, bool terminated, bool truncated,
                                                   float ep_ret, int len, bool stuck) {
  const bool done = terminated || truncated;
  p.reward[e] = rew;
  p.terminated[e] = terminated ? 1 : 0;
  p.truncated[e] = truncated ? 1 : 0;
  if (p.out_ep_return) p.out_ep_return[e] = done ? ep_ret : 0.f;
  if (p.out_ep_length) p.out_ep_length[e] = done ? len : 0;
  if (p.out_stuck) p.out_stuck[e] = stuck ? 1 : 0;
  if (p.out_done) p.out_done[e] = done ? 1.f : 0.f;
}

// Restart: the pool slot an env loads -- its pending first layout, else the next (PPO) or the same (FOMAML) one.
__device__ __forceinline__ int restart_layout(const EnvParams& p, bool advance, int layout) {
  return layout < 0 ? ~layout
                    : (advance ? (int)(((unsigned)layout + (unsigned)p.cursor_stride) % (unsigned)p.n_layouts) : layout);
}
// Restart pose from the pool's agent table, counters cleared.
__device__ __forceinline__ void restart_state(const EnvParams& p, int layout, EnvState& s) {
  const uint32_t a = p.pool_agent[layout];
  s.x = a & 0xff; s.y = (a >> 8) & 0xff; s.dir = (a >> 16) & 3; s.carry = 0;
  s.step_count = 0; s.stay = 0; s.last_x = s.x; s.last_y = s.y;
}
// Restart of a mutable grid: env e's private grid <- pool slot `layout`, by the 32 lanes of a warp.
__device__ __forceinline__ void copy_pool_grid(const EnvParams& p, size_t e, int layout, int lane) {
  const int4* from = reinterpret_cast<const int4*>(p.pool_cells + (size_t)layout * p.cell_stride);
  int4* to = reinterpret_cast<int4*>(p.cells + e * p.cell_stride);
  for (int i = lane; i < p.cell_stride / 16; i += 32) to[i] = from[i];
}
// Restart of the exploration bonus: env e's visited map <- only the cell (x, y), by the 32 lanes of a warp.
__device__ __forceinline__ void reset_visited(const EnvParams& p, size_t e, int x, int y, int lane) {
  const int cell = y * p.W + x;
  for (int i = lane; i < p.vis_words; i += 32)
    p.visited[e * p.vis_words + i] = (i == (cell >> 5)) ? (1u << (cell & 31)) : 0u;
}

// Code of grid cell (wx, wy); outside the grid it is a wall (Grid.slice).
__device__ __forceinline__ uint32_t grid_cell(const uint8_t* grid, int W, int H, uint64_t pol, int wx, int wy) {
  return ((unsigned)wx < (unsigned)W && (unsigned)wy < (unsigned)H) ? ld_cell(grid + wy * W + wx, pol) : CODE_WALL;
}
// Code of the cell `a` ahead of and `b` right of (x, y) for heading (fx, fy): window cell (vi, vj) is
// a = 6 - vj, b = vi - 3.
__device__ __forceinline__ uint32_t window_cell(const uint8_t* grid, int W, int H, uint64_t pol, int x, int y, int fx,
                                                int fy, int a, int b) {
  return grid_cell(grid, W, H, pol, x + a * fx - b * fy, y + a * fy + b * fx);
}

// One observed cell, `code` being what Grid.encode shows there -- at the agent cell what the agent carries
// (carried_code).  shown_kind: the atlas slot of its tile -- the agent with its load at the agent cell, the unseen tile
// where the cell is not visible, else the code.
__device__ __forceinline__ uint32_t carried_code(uint32_t carry) { return carry ? carry : CODE_EMPTY; }
__device__ __forceinline__ uint32_t shown_kind(uint32_t code, bool seen, bool agent_cell, uint32_t carry) {
  return agent_cell ? agent_kind(carry) : (seen ? code : KIND_UNSEEN);
}

// In-order work tickets (tile, tile-TMA and ordered kernels): draw the next one; the last of `participants` to be done
// drawing rearms the counters for the next launch (also under CUDA-graph replay).
__device__ __forceinline__ int draw_ticket(unsigned* sched) { return (int)atomicAdd(&sched[0], 1u); }
__device__ __forceinline__ void rearm_tickets(unsigned* sched, unsigned participants) {
  if (atomicAdd(&sched[1], 1u) == participants - 1) {
    sched[0] = 0;
    sched[1] = 0;
  }
}

// Stage the tile atlas: only the slots a frame of this handle's layout pool can show (5 of 128 for the MERLIN
// scenarios: 960 B instead of 24 KB), at their usual offsets.  All threads of the CTA take part.
__device__ __forceinline__ void stage_atlas(const EnvParams& p, uint8_t* atlas_s) {
  const int4* src = reinterpret_cast<const int4*>(p.atlas);
  int4* dst = reinterpret_cast<int4*>(atlas_s);
  for (int i = threadIdx.x; i < kAtlasBytes / 16; i += blockDim.x) {
    const int tile = i / (kTileBytes / 16);
    if (tile_bit(p.tile_present, tile)) dst[i] = __ldg(src + i);
  }
}

// Per-lane blit map: chunk c = lane + 32*k -> (cell0, off0, cell1, off1), from the table built at handle creation.
__device__ __forceinline__ void load_lut(const EnvParams& p, int lane, uint32_t (&lut)[kChunksPerLane]) {
#pragma unroll
  for (int k = 0; k < kChunksPerLane; ++k) lut[k] = __ldg(p.blit_lut + k * 32 + lane);
}

// Frame phase for one env: `kp` = its 49 tile kinds in shared memory.
__device__ __forceinline__ void blit_frame(const uint8_t* atlas_s, const uint8_t* kp, const uint32_t (&lut)[kChunksPerLane],
                                           uint8_t* frame, int lane) {
  const uint2* atlas64 = reinterpret_cast<const uint2*>(atlas_s);
#pragma unroll
  for (int k = 0; k < kChunksPerLane; ++k) {
    const int c = lane + 32 * k;
    if (c < kChunks) {
      const uint32_t q = lut[k];
      const uint32_t k0 = kp[q & 0xff], k1 = kp[(q >> 16) & 0xff];
      const uint2 a = atlas64[k0 * (kTileBytes / 8) + ((q >> 8) & 0xff)];
      const uint2 b = atlas64[k1 * (kTileBytes / 8) + (q >> 24)];
      st_stream_v4(frame + c * 16, a.x, a.y, b.x, b.y);
    }
  }
}

// Symbolic rows of `n_here` consecutive envs from shared memory (same layout as the output), by `nthreads` threads.
__device__ __forceinline__ void emit_sym_rows(uint8_t* out, const uint8_t* sym_s, int n_here, unsigned render_mask,
                                              int tid, int nthreads) {
  const unsigned full = n_here >= 32 ? 0xffffffffu : ((1u << n_here) - 1u);
  if (render_mask == full && ((reinterpret_cast<uintptr_t>(out) & 15) == 0) && (n_here * kSymBytes) % 16 == 0) {
    const int4* src = reinterpret_cast<const int4*>(sym_s);
    int4* dst = reinterpret_cast<int4*>(out);
    for (int i = tid; i < n_here * kSymBytes / 16; i += nthreads) dst[i] = src[i];
  } else {
    for (int b = tid; b < n_here * kSymBytes; b += nthreads) {
      const int i = b / kSymBytes;
      if ((render_mask >> i) & 1) out[b] = sym_s[b];
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// launch helper: resident CTAs per SM of `kernel` launched with `threads` threads and `smem` bytes of dynamic shared
// memory, at most `max_ctas` -- the persistent kernels launch SMs x that many CTAs, capped by the work available.  The
// first launch of an instance through a handle sets its shared-memory attribute and queries the occupancy; the count is
// kept in the HANDLE's cache (LaunchCtx::occ): a process may drive several handles on several devices from several
// threads, so nothing here is process-wide.
template <typename Kernel>
static cudaError_t resident_ctas(const LaunchCtx& ctx, Kernel kernel, int threads, size_t smem, int& ctas,
                                 int max_ctas = 1 << 30) {
  OccupancyCache& c = *ctx.occ;
  const void* key = reinterpret_cast<const void*>(kernel);
  for (int i = 0; i < c.n; ++i) {
    if (c.kernel[i] == key) {
      ctas = c.ctas[i];
      return cudaSuccess;
    }
  }
  cudaError_t err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (err != cudaSuccess) return err;
  err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas, kernel, threads, smem);
  if (err != cudaSuccess) return err;
  ctas = max(1, min(ctas, max_ctas));
  if (c.n < OccupancyCache::kEntries) {
    c.kernel[c.n] = key;
    c.ctas[c.n] = ctas;
    c.n += 1;
  }
  return cudaSuccess;
}

// Launchers of the step kernels outside env_kernels.cu, instantiated in their own translation units for STEP = 0 masked
// reset, 1 step with given actions, 2 policy step, 3 / 4 the same two recording final observations (the quad kernel:
// 1 and 2 only).  CTA tiles (env_kernels_tile.cu): T = 16 or 8 envs per tile.
constexpr int kTileThreads = 128;
constexpr int kTileCtasPerSm = 4;
template <int T, int STEP>
cudaError_t launch_tile_kernel(const EnvParams& p, const LaunchCtx& ctx, cudaStream_t stream);
template <int STEP>
cudaError_t launch_tile_tma_kernel(const EnvParams& p, const LaunchCtx& ctx, cudaStream_t stream);
// small-batch kernels (env_kernels_small.cu)
template <int STEP>
cudaError_t launch_warp_kernel(const EnvParams& p, const LaunchCtx& ctx, cudaStream_t stream);
template <int STEP>
cudaError_t launch_quad_kernel(const EnvParams& p, const LaunchCtx& ctx, cudaStream_t stream);

}  // namespace merlin
