// env_kernels_small.cu -- the small-batch step kernels for sm_100a: env_kernel_warp (one warp per env) and
// env_kernel_quad (four envs per warp), with their launch shapes.  Same per-env work as the kernels of env_kernels.cu
// (see the header there); these mappings serve batches whose envs are all resident at once, where the run time is launch
// latency + one env's dependent chain + its stores.
#include <cuda_runtime.h>
#include <stdint.h>

#include "env_kernels.cuh"
#include "env_kernels_common.cuh"
#include "env_logic.cuh"

namespace merlin {

// ---------------------------------------------------------------------------------------------------
// env_kernel_warp<STEP, PDL, LEAN>: one WARP per environment -- the small-batch mapping (N <= 24 576: every env of the
// batch is resident at once or nearly so, and the run time is launch latency + one env's dependent chain + its stores).
//   * state / action / forward cell are loaded at warp-uniform addresses (one broadcast transaction each) and the
//     step logic runs redundantly on all lanes; lane 0 alone writes the per-env outputs and the new state.  The first
//     env's state and action are requested BEFORE the atlas is staged, so both round trips overlap.
//   * LEAN (three actions, no shaping wrapper => immutable grids; launch_warp_kernel): the step needs TWO dependent
//     round trips instead of three -- see the block at `if (LEAN)`.
//   * the 49-cell window is gathered two cells per lane; transparency goes through two warp ballots into the same
//     49-bit mask the visibility routine consumes; every lane then knows the visibility of its own cells.
//   * frame phase without a blit map: the frame is 28 pairs of pixel rows; a pair is 336 bytes = 21 16-byte chunks, and
//     chunk l of EVERY pair covers the same (cell column, tile part) twice over -- so lane l < 21 owns chunk l of all 28
//     pairs, its two (vi, part) are loop constants, the tile row (vj, py) is the loop counter, and after unrolling
//     every shared-memory and global address is `lane register + immediate`: 3 instructions per chunk (two 8-byte
//     atlas reads, one 16-byte store) plus 4 per tile row for the two kinds, ~115 per frame instead of ~480 with the
//     588-entry chunk map (ncu at 4096 envs, profiles/r02_warp_n4096_v2_ncu_details.csv: 1387 -> 791 warp instructions per env).
//     The kinds are kept premultiplied (kind * 192, the tile's byte offset in the atlas) as 16-bit words.
//   * atlas staging touches only the slots the pool can show: thread t tests tile t / 2 and copies half of it.
constexpr int kWarpKernelThreads = 256, kWarpCtas = 4;
// RGB batches of at least this many envs launch the warp kernel with programmatic dependent launch (see the kernel)
constexpr int kWarpPdlMinEnvs = 4096;
constexpr int kWarpKindBytes = 128;          // 49 premultiplied kinds (u16) per warp, padded
constexpr int kPairChunks = 2 * kUnitsPerRow / 2;   // 21 16-byte chunks per pair of pixel rows

// Final observation of one env, one warp per env (STEP = 3 / 4): the 49 window codes of its terminal state, code0 in
// mask order c = lane and code1 at c = lane + 32, encoded into the global row `out` -- the same ballots, visibility and
// bytes as the observation part of env_kernel_warp.
__device__ __forceinline__ void warp_store_final(uint32_t code0, uint32_t code1, int lane, uint32_t carry, uint8_t* out) {
  const int c1 = lane + 32;
  const unsigned t0 = __ballot_sync(0xffffffffu, !((M_OPAQUE >> (code0 & 0xf)) & 1u));
  const unsigned t1 = __ballot_sync(0xffffffffu, c1 < kCells && !((M_OPAQUE >> (code1 & 0xf)) & 1u));
  const uint64_t vis = visibility((uint64_t)t0 | ((uint64_t)t1 << 32));
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int c = h ? c1 : lane;
    if (c >= kCells) break;
    const int vj = (c * 37) >> 8, vi = c - vj * kView;   // c / 7 for c < 64
    const bool agent_cell = (vi == kView / 2 && vj == kView - 1);
    const uint32_t code = agent_cell ? (carry ? carry : CODE_EMPTY) : (h ? code1 : code0);
    uint8_t t = 0, col = 0, stt = 0;
    if ((vis >> c) & 1) sym_of_code(code, t, col, stt);
    uint8_t* o = out + (vi * kView + vj) * 3;
    o[0] = t; o[1] = col; o[2] = stt;
  }
}

template <int STEP, bool PDL, bool LEAN = false>
__global__ void __launch_bounds__(kWarpKernelThreads, kWarpCtas) env_kernel_warp(const EnvParams p) {
  extern __shared__ __align__(16) uint8_t smem[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int warps_per_cta = blockDim.x >> 5;
  const Flags f(p);
  uint8_t* atlas_s = smem;
  uint16_t* kq = reinterpret_cast<uint16_t*>(smem + kAtlasBytes + warp * kWarpKindBytes);   // this warp's 49 kinds * 192

  int e = blockIdx.x * warps_per_cta + warp;
  int4 st_next = make_int4(0, 0, 0, 0);
  long long act_next = 0;
  if (PDL) {
    // Programmatic dependent launch (RGB batches of >= 4096 envs): the kernel is launched with
    // cudaLaunchAttributeProgrammaticStreamSerialization, so its CTAs may be scheduled while the PREVIOUS kernel of the
    // stream is still draining its stores.  Everything up to griddepcontrol.wait touches only data no kernel writes (the
    // atlas and the tile mask are written by synchronous uploads): launch latency and the two-round-trip atlas staging
    // overlap the predecessor's tail.  After the wait the predecessor has completed and its writes (state, the policy's
    // logits, ...) are visible.  launch_dependents at once: a following env step may start its own prologue under THIS
    // kernel's store phase (all CTAs of a <= 24 576-env batch are resident together: early arrivals cannot starve it).
    // Measured (B200, CUDA-graph replay / eager back to back, us per step): 4096 envs 10.4 -> 9.7 / 12.3 -> 10.0,
    // 16 384 envs 28.1 -> 27.2 / 29.9 -> 27.5, 24 576 envs 40.9 -> 40.0; at 1024 envs graph replay gets SLOWER (4.9 ->
    // 8.0: the programmatic edge costs more than it hides), hence the size threshold.
    asm volatile("griddepcontrol.launch_dependents;");
  } else if (e < p.N) {
    // first env's state / action: in flight while the atlas is staged
    st_next = p.state[e];
    if (step_given(STEP)) act_next = p.actions[e];
  }
  if (f.want_rgb) {
    // thread t tests tile t / 2 and copies half of it (6 int4); a 128-thread CTA takes two rounds
    for (int t = threadIdx.x; t < 2 * kAtlasTiles; t += blockDim.x) {
      const int tile = t >> 1, half = t & 1;
      if (tile_bit(p.tile_present, tile)) {
        const int4* src = reinterpret_cast<const int4*>(p.atlas) + tile * (kTileBytes / 16) + half * 6;
        int4* dst = reinterpret_cast<int4*>(atlas_s) + tile * (kTileBytes / 16) + half * 6;
#pragma unroll
        for (int i = 0; i < 6; ++i) dst[i] = __ldg(src + i);
      }
    }
  }
  if (PDL) {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (e < p.N) {
      st_next = p.state[e];
      if (step_given(STEP)) act_next = p.actions[e];
    }
  }
  __syncthreads();

  // this lane's two window cells, in mask order c = vj*7 + vi
  const int c0 = lane, c1 = lane + 32;
  const int vj0 = (c0 * 37) >> 8, vi0 = c0 - vj0 * kView;                       // c / 7 for c < 64
  const int vj1 = c1 < kCells ? (c1 * 37) >> 8 : 0, vi1 = c1 < kCells ? c1 - vj1 * kView : 0;
  const int a0 = (kView - 1) - vj0, b0 = vi0 - kView / 2, a1 = (kView - 1) - vj1, b1 = vi1 - kView / 2;
  // lean step: second cell of the 8-row window, ext index lane + 32 < 56 (row j = x / 7 counted from the far end)
  const int vj1x = (c1 * 37) >> 8, a1x = (kView - 1) - vj1x, b1x = c1 - vj1x * kView - kView / 2;
  // frame phase constants of this lane: chunk `lane` of every row pair = units 2*lane and 2*lane + 1 of 42
  const int u0 = 2 * lane, u1 = 2 * lane + 1;
  const int r0 = u0 >= kUnitsPerRow, r1 = u1 >= kUnitsPerRow;          // second row of the pair?
  const int w0 = u0 - r0 * kUnitsPerRow, w1 = u1 - r1 * kUnitsPerRow;
  const int cv0 = (w0 * 11) >> 5, cv1 = (w1 * 11) >> 5;                 // w / 3 for w < 21: the cell column vi
  const uint16_t* kq0 = kq + cv0 * kView;                               // + vj
  const uint16_t* kq1 = kq + cv1 * kView;
  const uint8_t* at0 = atlas_s + (w0 - 3 * cv0) * 8 + r0 * 24;          // + kind * 192 + (py & ~1) * 24
  const uint8_t* at1 = atlas_s + (w1 - 3 * cv1) * 8 + r1 * 24;

  for (; e < p.N; e += gridDim.x * warps_per_cta) {
    EnvState s{};
    const int4 st = st_next;
    const long long act_in = act_next;
    {
      const int en = e + gridDim.x * warps_per_cta;   // prefetch the next env of this warp
      if (en < p.N) {
        st_next = p.state[en];
        if (step_given(STEP)) act_next = p.actions[en];
      }
    }
    unpack_state(st.x, st.y, st.z, st.w, s);
    float ep_ret = p.ep_return[e];
    bool restart = false, render = true;
    uint32_t code0, code1 = CODE_WALL;   // this lane's two window cells (mask order c0 = lane, c1 = lane + 32)

    if (LEAN) {
      // Lean step (the reference's own configuration: ThreeActionWrapper, no reward-shaping wrapper => immutable grids):
      // TWO dependent round trips instead of three.  The action is known together with the state, hence the new
      // heading; the agent then stands on its old cell or one cell ahead of it.  Both windows lie inside 8 rows x 7
      // columns in front of the OLD cell (rows a = 7..0 ahead, ext index x = (7 - a) * 7 + vi): loaded at once, two
      // cells per lane (56 <= 64), BEFORE the forward cell has been looked at -- it is ext cell 45 itself.  The window
      // of an agent that moved is ext rows 0..6 (cell c = x: the lane's own loads); of one that did not, rows 1..7
      // (c = x - 7: one lane rotation by 7).
      ActionDraw act;
      if (step_draws(STEP)) act = draw_action<true>(p, 3, e);
      else { act.action = act_in; act.logp = 0.f; act.draw = 0; }
      const bool bad = act.action < 0 || act.action >= 3;
      const int a = bad ? A_DONE : (int)act.action;
      s.dir = a == A_LEFT ? (s.dir + 3) & 3 : (a == A_RIGHT ? (s.dir + 1) & 3 : s.dir);
      const uint8_t* grid = p.pool_cells + (size_t)s.layout * p.cell_stride;
      const int fx = dir_dx(s.dir), fy = dir_dy(s.dir);
      const uint32_t e0 = window_cell(grid, p.W, p.H, f.pol, s.x, s.y, fx, fy, a0 + 1, b0);
      uint32_t e1 = CODE_WALL;
      if (lane + 32 < kCells + kView) e1 = window_cell(grid, p.W, p.H, f.pol, s.x, s.y, fx, fy, a1x + 1, b1x);
      const uint32_t ft = __shfl_sync(0xffffffffu, e1, 45 - 32) & 0xf;   // the cell ahead: ext row 6, column 3
      s.step_count += 1;
      const bool fwd_act = a == A_FORWARD;
      const bool moved = fwd_act && ((M_OVERLAP >> ft) & 1u);
      const bool goal = fwd_act && ft == T_GOAL;
      const bool terminated = goal || (fwd_act && ft == T_LAVA);
      const bool truncated = s.step_count >= p.max_steps;
      float rew = 0.f;
      if (goal) rew = (float)(1 - 0.9 * ((double)s.step_count / (double)p.max_steps));   // MiniGridEnv._reward in float64
      if (moved) { s.x += fx; s.y += fy; }
      ep_ret += rew;
      const bool done = terminated || truncated;
      if (lane == 0) {
        commit_action<step_draws(STEP)>(p, e, act);
        record_first_episode<step_draws(STEP)>(p, e, done, goal && rew > 0.f, ep_ret, s.step_count);
        if (bad) atomicAdd(p.bad_actions, 1ull);
        store_step_outputs(p, e, rew, terminated, truncated, ep_ret, s.step_count, false);
      }
      restart = done && f.auto_reset;
      const int rot = (lane + kView) & 31;
      const uint32_t r0 = __shfl_sync(0xffffffffu, e0, rot), r1 = __shfl_sync(0xffffffffu, e1, rot);
      code0 = moved ? e0 : (lane + kView < 32 ? r0 : r1);
      code1 = moved ? e1 : r1;
      // the window just assembled is the terminal state's: its final image, before the restart below (warp-uniform)
      if constexpr (step_final(STEP)) {
        if (done) warp_store_final(code0, code1, lane, s.carry, p.final_sym + (size_t)e * kSymBytes);
      }
    } else if (STEP) {
      const uint8_t* grid = f.mutable_grid ? p.cells + (size_t)e * p.cell_stride
                                           : p.pool_cells + (size_t)s.layout * p.cell_stride;
      const int fx = s.x + dir_dx(s.dir), fy = s.y + dir_dy(s.dir);
      const bool inb = (unsigned)fx < (unsigned)p.W && (unsigned)fy < (unsigned)p.H;
      const int fidx = fy * p.W + fx;
      const uint32_t fwd = inb ? ld_cell(grid + fidx, f.pol) : CODE_WALL;
      ActionDraw act;
      if (step_draws(STEP)) act = draw_action<true>(p, f.n_actions, e);
      else { act.action = act_in; act.logp = 0.f; act.draw = 0; }
      StepResult r = step_logic(s, act.action, f.n_actions, fwd, inb, fidx, p.max_steps);
      uint32_t vword = 0;
      const int cell = s.y * p.W + s.x;
      uint32_t* vptr = nullptr;
      if (f.explore_on) { vptr = p.visited + (size_t)e * p.vis_words + (cell >> 5); vword = *vptr; }
      bool stuck = false;
      const uint32_t vword_in = vword;
      const double rew_d = shape_reward(s, r.reward, f.stuck_on, p.stuck_max_stay, p.stuck_penalty, f.explore_on,
                                        p.explore_bonus, vword, cell & 31, stuck);
      const float rew = (float)rew_d;
      ep_ret += rew;
      const bool done = r.terminated || r.truncated;
      __syncwarp();  // every lane has read the old grid cell / visited word / draw counter before lane 0 overwrites them
      if (lane == 0) {
        commit_action<step_draws(STEP)>(p, e, act);
        record_first_episode<step_draws(STEP)>(p, e, done, r.terminated && r.reward > 0.0, ep_ret, s.step_count);
        if (r.bad_action) atomicAdd(p.bad_actions, 1ull);
        if (r.write_idx >= 0 && f.mutable_grid) p.cells[(size_t)e * p.cell_stride + r.write_idx] = (uint8_t)r.write_code;
        if (f.explore_on && vword != vword_in) *vptr = vword;
        store_step_outputs(p, e, rew, r.terminated, r.truncated, ep_ret, s.step_count, stuck);
      }
      // final image (warp-uniform): the window after lane 0's grid write above, before the restart copy below
      if constexpr (step_final(STEP)) {
        if (done) {
          __syncwarp();
          const int fx = dir_dx(s.dir), fy = dir_dy(s.dir);
          const uint32_t w0 = window_cell(grid, p.W, p.H, f.pol, s.x, s.y, fx, fy, a0, b0);
          uint32_t w1 = CODE_WALL;
          if (c1 < kCells) w1 = window_cell(grid, p.W, p.H, f.pol, s.x, s.y, fx, fy, a1, b1);
          warp_store_final(w0, w1, lane, s.carry, p.final_sym + (size_t)e * kSymBytes);
        }
      }
      restart = done && f.auto_reset;
    } else {
      restart = p.reset_mask == nullptr || p.reset_mask[e] != 0;
      render = restart;
    }

    if (restart) {  // warp-uniform
      const int load_cur = restart_layout(p, f.advance, s.layout);
      restart_state(p, load_cur, s);
      ep_ret = 0.f;
      s.layout = load_cur;
      if (!LEAN && f.mutable_grid) {
        __syncwarp();
        copy_pool_grid(p, (size_t)e, load_cur, lane);
      }
      if (!LEAN && f.explore_on) {
        __syncwarp();
        reset_visited(p, (size_t)e, s.x, s.y, lane);
      }
    }
    if (lane == 0 && (STEP || restart)) {
      int4 o;
      pack_state(s, o.x, o.y, o.z, o.w);
      p.state[e] = o;
      p.ep_return[e] = ep_ret;
    }
    if (!render || !(f.want_rgb || f.want_sym)) continue;
    __syncwarp();  // grid writes of this step (pickup/drop/toggle, restart copy) are visible to the gather below

    // observation, part 1: two window cells per lane -> ballot -> visibility -> tile kinds (+ symbolic bytes)
    if (!LEAN || restart) {   // the lean step holds the window already unless the env restarted (warp-uniform)
      const uint8_t* grid = (!LEAN && f.mutable_grid) ? p.cells + (size_t)e * p.cell_stride
                                           : p.pool_cells + (size_t)s.layout * p.cell_stride;
      const int fx = dir_dx(s.dir), fy = dir_dy(s.dir);
      const int rx = -fy, ry = fx;
      // window_cell's arithmetic spelled with the right vector (rx, ry): this form keeps the lean STEP = 4 instances at
      // their instruction count (through window_cell they take 8 more)
      code1 = CODE_WALL;
      code0 = grid_cell(grid, p.W, p.H, f.pol, s.x + a0 * fx + b0 * rx, s.y + a0 * fy + b0 * ry);
      if (c1 < kCells) code1 = grid_cell(grid, p.W, p.H, f.pol, s.x + a1 * fx + b1 * rx, s.y + a1 * fy + b1 * ry);
    }
    const unsigned t0 = __ballot_sync(0xffffffffu, !((M_OPAQUE >> (code0 & 0xf)) & 1u));
    const unsigned t1 = __ballot_sync(0xffffffffu, c1 < kCells && !((M_OPAQUE >> (code1 & 0xf)) & 1u));
    const uint64_t vis = visibility((uint64_t)t0 | ((uint64_t)t1 << 32));
    uint8_t* sym_out = f.want_sym ? p.obs_sym + (size_t)e * kSymBytes : nullptr;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int c = h ? c1 : c0;
      if (c >= kCells) break;
      const int vi = h ? vi1 : vi0, vj = h ? vj1 : vj0;
      uint32_t code = h ? code1 : code0;
      const bool seen = (vis >> c) & 1;
      const bool agent_cell = (vi == kView / 2 && vj == kView - 1);
      if (agent_cell) code = carried_code(s.carry);
      const int k = vi * kView + vj;
      kq[k] = (uint16_t)((agent_cell ? agent_kind(s.carry) : (seen ? code : KIND_UNSEEN)) * kTileBytes);
      if (f.want_sym) {
        uint8_t t = 0, col = 0, stt = 0;
        if (seen) sym_of_code(code, t, col, stt);
        sym_out[k * 3 + 0] = t; sym_out[k * 3 + 1] = col; sym_out[k * 3 + 2] = stt;
      }
    }
    __syncwarp();
    if (f.want_rgb && lane < kPairChunks) {
      uint8_t* out = p.obs_rgb + (size_t)e * kImgBytes + lane * 16;
#pragma unroll
      for (int vj = 0; vj < kView; ++vj) {
        const uint8_t* t0p = at0 + kq0[vj];
        const uint8_t* t1p = at1 + kq1[vj];
#pragma unroll
        for (int q = 0; q < kTile / 2; ++q) {   // row pair vj*4 + q: pixel rows py = 2q, 2q + 1 of tile row vj
          const uint2 a = *reinterpret_cast<const uint2*>(t0p + q * 48);
          const uint2 b = *reinterpret_cast<const uint2*>(t1p + q * 48);
          st_stream_v4(out + (vj * (kTile / 2) + q) * (2 * kRowBytes), a.x, a.y, b.x, b.y);
        }
      }
    }
    __syncwarp();  // kq is reused by this warp's next env
  }
}

// ---------------------------------------------------------------------------------------------------
// env_kernel_quad<STEP> (kernel choice 7): one warp per FOUR environments, eight lanes per env -- a small-batch mapping
// for the reference's own configuration (ThreeActionWrapper => immutable grids, no reward-shaping wrapper; RGB frames).
// MEASURED AND NOT ADOPTED as a default (profiles/r02_quad_vs_warp.txt): it executes 328 instead of 773 instructions per
// env, but the small-batch step is bound by the latency of one env's dependent chain, not by issue slots (ncu at 4096
// envs: env_kernel_warp 33 % of the issue slots busy, 15.8 cycles per issued instruction per warp) -- fewer, longer-
// running warps hide less of it: 8.8 vs 8.3 us per step at 4096 envs, 22.4 vs 20.6 at 12 288, faster only around 8192
// (14.6 vs 15.7).  Kept selectable and held to the parity bar (tests/test_gpu_variants.py).
// In env_kernel_warp one instruction stream serves one env and every lane repeats the warp-uniform step logic.  Here one
// stream serves four envs -- everything below is uniform within a group of eight lanes and differs between the groups:
//   * lane r of a group loads ROW r of the 8-row x 7-column region in front of the agent's old cell (seven byte loads,
//     all in flight together with the other rows'): both candidate windows -- the agent stays, or moves one cell ahead --
//     lie inside it, so the step needs two dependent round trips (state + action, then cells), and the cell ahead is
//     byte 3 of row 6 (one shuffle);
//   * the lane's row arrives as 7 codes in a 64-bit register with its 7-bit transparency mask computed in place (no
//     ballots); the window row vj is ext row vj (agent moved) or vj + 1 (not moved): one lane-shifted shuffle;
//   * the seven row masks meet in shared memory (one byte each, one 8-byte read per lane); every lane runs
//     `visibility_rows` on them, takes its own row of the result and writes its seven tile kinds;
//   * frame phase as in env_kernel_warp (map-free row pairs), one env after the other.
// Quads are dealt to warps CTA-minor (quad q -> warp q / gridDim of CTA q % gridDim), so a batch that needs 1.3 rounds
// leaves every SM with the same share of second-round quads.
constexpr int kQuadCtas = 4;
constexpr int kQuadKindBytes = 4 * 128 + 32;   // per warp: 4 envs x 49 premultiplied kinds (u16, padded to 64) + 4 x 8 row masks

// Row `r` (0 = farthest, 7 = the agent's own row) of the 8 x 7 region in front of pose (x, y, heading f): codes of its
// seven cells, byte vi, and the transparency mask, bit vi.  Outside the grid = wall (Grid.slice).
__device__ __forceinline__ void load_ext_row(const EnvParams& p, const uint8_t* grid, uint64_t pol, int x, int y, int fx,
                                             int fy, int r, uint64_t& codes, uint32_t& transp) {
  const int ae = kView - r;
  int wx = x + ae * fx + (kView / 2) * fy, wy = y + ae * fy - (kView / 2) * fx;
  uint32_t c[kView];
#pragma unroll
  for (int vi = 0; vi < kView; ++vi) {
    c[vi] = grid_cell(grid, p.W, p.H, pol, wx, wy);
    wx -= fy; wy += fx;
  }
  codes = 0; transp = 0;
#pragma unroll
  for (int vi = 0; vi < kView; ++vi) {
    codes |= (uint64_t)c[vi] << (8 * vi);
    transp |= (((M_OPAQUE >> (c[vi] & 0xf)) & 1u) ^ 1u) << vi;
  }
}

template <int STEP, bool PDL>
__global__ void __launch_bounds__(kWarpKernelThreads, kQuadCtas) env_kernel_quad(const EnvParams p) {
  static_assert(STEP == 1 || STEP == 2, "the quad kernel steps; resets and final-observation steps run the warp kernel");
  extern __shared__ __align__(16) uint8_t smem[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int warps_per_cta = blockDim.x >> 5;
  const int g = lane >> 3, r = lane & 7;
  uint8_t* atlas_s = smem;
  uint16_t* kq = reinterpret_cast<uint16_t*>(smem + kAtlasBytes + warp * kQuadKindBytes);   // [4][64]
  uint8_t* tmask = smem + kAtlasBytes + warp * kQuadKindBytes + 4 * 128;                    // [4][8] row masks
  const uint64_t pol = grid_policy(true);
  const bool auto_reset = p.flags & MERLIN_F_AUTO_RESET, advance = !(p.flags & MERLIN_F_RESET_SAME);
  const int n_quads = (p.N + 3) >> 2;
  const int stride = gridDim.x * warps_per_cta;

  int q = warp * gridDim.x + blockIdx.x;
  int4 st_next = make_int4(0, 0, 0, 0);
  long long act_next = 0;
  if (PDL) {
    asm volatile("griddepcontrol.launch_dependents;");   // see env_kernel_warp
  } else if (q < n_quads) {
    const int e = min(4 * q + g, p.N - 1);
    st_next = p.state[e];
    if (step_given(STEP)) act_next = p.actions[e];
  }
  for (int t = threadIdx.x; t < 2 * kAtlasTiles; t += blockDim.x) {
    const int tile = t >> 1, half = t & 1;
    if (tile_bit(p.tile_present, tile)) {
      const int4* src = reinterpret_cast<const int4*>(p.atlas) + tile * (kTileBytes / 16) + half * 6;
      int4* dst = reinterpret_cast<int4*>(atlas_s) + tile * (kTileBytes / 16) + half * 6;
#pragma unroll
      for (int i = 0; i < 6; ++i) dst[i] = __ldg(src + i);
    }
  }
  if (PDL) {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (q < n_quads) {
      const int e = min(4 * q + g, p.N - 1);
      st_next = p.state[e];
      if (step_given(STEP)) act_next = p.actions[e];
    }
  }
  __syncthreads();

  // frame phase constants of this lane (see env_kernel_warp): chunk `lane` of every row pair
  const int u0 = 2 * lane, u1 = 2 * lane + 1;
  const int r0 = u0 >= kUnitsPerRow, r1 = u1 >= kUnitsPerRow;
  const int w0 = u0 - r0 * kUnitsPerRow, w1 = u1 - r1 * kUnitsPerRow;
  const int cv0 = (w0 * 11) >> 5, cv1 = (w1 * 11) >> 5;
  const int ko0 = cv0 * kView, ko1 = cv1 * kView;
  const uint8_t* at0 = atlas_s + (w0 - 3 * cv0) * 8 + r0 * 24;
  const uint8_t* at1 = atlas_s + (w1 - 3 * cv1) * 8 + r1 * 24;

  for (; q < n_quads; q += stride) {
    const bool valid = 4 * q + g < p.N;           // a ragged last quad: its surplus groups shadow env N - 1, store nothing
    const int e = valid ? 4 * q + g : p.N - 1;
    const int4 st = st_next;
    const long long act_in = act_next;
    if (q + stride < n_quads) {
      const int en = min(4 * (q + stride) + g, p.N - 1);
      st_next = p.state[en];
      if (step_given(STEP)) act_next = p.actions[en];
    }
    int x = st.x & 0xff, y = (st.x >> 8) & 0xff, dir = (st.x >> 16) & 3;
    uint32_t carry = ((uint32_t)st.x >> 24) & 0x7f;
    int step_count = st.y, layout = st.z, sw = st.w;
    float ep_ret = p.ep_return[e];

    ActionDraw act;
    if (step_draws(STEP)) act = draw_action<true>(p, 3, e);
    else { act.action = act_in; act.logp = 0.f; act.draw = 0; }
    const bool bad = act.action < 0 || act.action >= 3;
    const int a = bad ? A_DONE : (int)act.action;
    dir = a == A_LEFT ? (dir + 3) & 3 : (a == A_RIGHT ? (dir + 1) & 3 : dir);
    int fx = dir_dx(dir), fy = dir_dy(dir);
    uint64_t codes;
    uint32_t transp_row;
    load_ext_row(p, p.pool_cells + (size_t)layout * p.cell_stride, pol, x, y, fx, fy, r, codes, transp_row);
    const uint32_t ft = __shfl_sync(0xffffffffu, (uint32_t)(codes >> 24), (lane & 24) | (kView - 1)) & 0xf;  // row 6, column 3

    step_count += 1;
    const bool fwd_act = a == A_FORWARD;
    bool moved = fwd_act && ((M_OVERLAP >> ft) & 1u);
    const bool goal = fwd_act && ft == T_GOAL;
    const bool terminated = goal || (fwd_act && ft == T_LAVA);
    const bool truncated = step_count >= p.max_steps;
    float rew = 0.f;
    if (goal) rew = (float)(1 - 0.9 * ((double)step_count / (double)p.max_steps));   // MiniGridEnv._reward, float64
    if (moved) { x += fx; y += fy; }
    ep_ret += rew;
    const bool done = terminated || truncated;
    if (r == 0 && valid) {
      commit_action<step_draws(STEP)>(p, e, act);
      record_first_episode<step_draws(STEP)>(p, e, done, goal && rew > 0.f, ep_ret, step_count);
      if (bad) atomicAdd(p.bad_actions, 1ull);
      store_step_outputs(p, e, rew, terminated, truncated, ep_ret, step_count, false);
    }
    if (done && auto_reset) {   // uniform within the group
      const int load_cur = restart_layout(p, advance, layout);
      const uint32_t pa = p.pool_agent[load_cur];
      x = pa & 0xff; y = (pa >> 8) & 0xff; dir = (pa >> 16) & 3; carry = 0;
      step_count = 0; sw = (x << 16) | (int)((uint32_t)y << 24);
      ep_ret = 0.f;
      layout = load_cur;
      fx = dir_dx(dir); fy = dir_dy(dir);
      load_ext_row(p, p.pool_cells + (size_t)layout * p.cell_stride, pol, x, y, fx, fy, r, codes, transp_row);
      moved = false;
    }
    if (r == 0 && valid) {
      p.state[e] = make_int4(x | (y << 8) | (dir << 16) | (int)(carry << 24), step_count, layout, sw);
      p.ep_return[e] = ep_ret;
    }

    // window row vj = r (r < 7): ext row r when the agent moved, r + 1 when it did not
    const int src = (lane + (moved ? 0 : 1)) & 31;
    const uint32_t wlo = __shfl_sync(0xffffffffu, (uint32_t)codes, src);
    const uint32_t whi = __shfl_sync(0xffffffffu, (uint32_t)(codes >> 32), src);
    const uint32_t wt = __shfl_sync(0xffffffffu, transp_row, src);
    // the group's seven row masks, one byte each, through shared memory (a redux.sync on an 8-lane member mask is not
    // one instruction: REDUX reduces the whole warp, sub-warp masks take a loop)
    tmask[lane] = (uint8_t)wt;
    __syncwarp();
    const uint64_t vis = visibility_rows(*reinterpret_cast<const uint64_t*>(tmask + (lane & 24)));
    if (r < kView) {
      const uint32_t visrow = (uint32_t)(vis >> (8 * r)) & 0x7f;
      const uint64_t w = (uint64_t)wlo | ((uint64_t)whi << 32);
      uint16_t* kd = kq + g * 64 + r;
      uint8_t* so = (p.obs_sym != nullptr && valid) ? p.obs_sym + (size_t)e * kSymBytes + r * 3 : nullptr;
#pragma unroll
      for (int vi = 0; vi < kView; ++vi) {
        const bool seen = (visrow >> vi) & 1u;
        const bool agent_cell = vi == kView / 2 && r == kView - 1;
        uint32_t code = (uint32_t)(w >> (8 * vi)) & 0xff;
        if (agent_cell) code = carried_code(carry);
        kd[vi * kView] = (uint16_t)(shown_kind(code, seen, agent_cell, carry) * kTileBytes);
        if (so) {   // Grid.encode of the cell, (0, 0, 0) when not visible: bytes (vi * 7 + vj) * 3 ..
          uint8_t t = 0, col = 0, stt = 0;
          if (seen) sym_of_code(code, t, col, stt);
          so[vi * kView * 3 + 0] = t; so[vi * kView * 3 + 1] = col; so[vi * kView * 3 + 2] = stt;
        }
      }
    }
    __syncwarp();
    if (lane < kPairChunks) {
      const int n_here = min(4, p.N - 4 * q);
      uint8_t* out = p.obs_rgb + (size_t)(4 * q) * kImgBytes + lane * 16;
      const uint16_t* kf = kq;
#pragma unroll 1
      for (int fr = 0; fr < n_here; ++fr, out += kImgBytes, kf += 64) {
#pragma unroll
        for (int vj = 0; vj < kView; ++vj) {
          const uint8_t* t0p = at0 + kf[ko0 + vj];
          const uint8_t* t1p = at1 + kf[ko1 + vj];
#pragma unroll
          for (int h = 0; h < kTile / 2; ++h) {
            const uint2 a2 = *reinterpret_cast<const uint2*>(t0p + h * 48);
            const uint2 b2 = *reinterpret_cast<const uint2*>(t1p + h * 48);
            st_stream_v4(out + (vj * (kTile / 2) + h) * (2 * kRowBytes), a2.x, a2.y, b2.x, b2.y);
          }
        }
      }
    }
    __syncwarp();  // kq is reused by this warp's next quad
  }
}

// Shape of a warp-kernel launch.  Batches that fit the machine in one round (N <= SMs x resident CTAs x 8 warps) are
// BALANCED: with 8-warp CTAs, 4096 envs are 512 CTAs on 148 SMs -- 68 SMs get four CTAs (32 envs), 80 get three (24),
// and the launch lasts as long as the SMs with 32.  Instead the CTA shape follows the batch: the fewest envs per SM
// that cover it, ceil(N / SMs), split into c <= resident CTAs of w <= 8 warps (4096 envs: 4 x 7 warps, 28 envs on
// (almost) every SM).  Larger batches loop over rounds of full CTAs, where the imbalance is a few percent at most.
static void warp_kernel_shape(int N, int sm_count, int blocks_per_sm, int& grid, int& threads, bool few_ctas = false) {
  constexpr int max_warps = kWarpKernelThreads / 32;
  threads = kWarpKernelThreads;
  grid = min(sm_count * blocks_per_sm, (N + max_warps - 1) / max_warps);
  if (N > sm_count * blocks_per_sm * max_warps) return;
  const int per_sm = (N + sm_count - 1) / sm_count;
  int best_w = max_warps, best_cost = 1 << 30;
  for (int c = blocks_per_sm; c >= 1; --c) {   // ties: more, smaller CTAs (each clears its staging barrier sooner)
    const int w = (per_sm + c - 1) / c;
    if (w > max_warps) continue;
    if (c * w < best_cost || (few_ctas && c * w == best_cost)) { best_cost = c * w; best_w = w; }
  }
  threads = best_w * 32;
  grid = (N + best_w - 1) / best_w;
}

template <typename Kernel>
static cudaError_t launch_maybe_pdl(Kernel kernel, bool pdl, int grid, int threads, size_t smem, cudaStream_t stream,
                                    const EnvParams& p) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(threads); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, p);
}

template <int STEP, bool LEAN>
static cudaError_t launch_warp_kernel_impl(const EnvParams& p, const LaunchCtx& ctx, cudaStream_t stream) {
  const size_t smem = kAtlasBytes + (kWarpKernelThreads / 32) * kWarpKindBytes;
  const bool pdl = p.obs_rgb != nullptr && p.N >= kWarpPdlMinEnvs;
  const auto kernel = pdl ? env_kernel_warp<STEP, true, LEAN> : env_kernel_warp<STEP, false, LEAN>;
  int ctas;
  if (cudaError_t err = resident_ctas(ctx, kernel, kWarpKernelThreads, smem, ctas)) return err;
  int grid, threads;
  warp_kernel_shape(p.N, ctx.sm_count, ctas, grid, threads);
  return launch_maybe_pdl(kernel, pdl, grid, threads, smem, stream, p);
}
// The lean step (two dependent round trips, see the kernel) serves the lean configuration (lean_config) while every env
// of the batch is resident at once or nearly so: from 16 384 envs up (3.5 rounds of resident warps, chains hidden behind
// other warps' stores) the lean form's 56-cell region and shuffles cost 1.5 % (27.5 vs 27.0 us).
constexpr int kWarpLeanMaxEnvs = 12288;
template <int STEP>
cudaError_t launch_warp_kernel(const EnvParams& p, const LaunchCtx& ctx, cudaStream_t stream) {
  if constexpr (STEP != 0) {
    if (p.N <= kWarpLeanMaxEnvs && lean_config(p.flags)) return launch_warp_kernel_impl<STEP, true>(p, ctx, stream);
  }
  return launch_warp_kernel_impl<STEP, false>(p, ctx, stream);
}

// The quad kernel is launched with programmatic dependent launch only when its CTAs fill every resident slot of the
// machine: a grid that leaves room lets its successors (which signal launch_dependents on entry themselves) pile up
// resident behind it, and a step then takes twice as long (4096 envs = 147 CTAs: 16 us instead of 9).
constexpr int kQuadPdlMinEnvs = 16384;
template <int STEP>
cudaError_t launch_quad_kernel(const EnvParams& p, const LaunchCtx& ctx, cudaStream_t stream) {
  const size_t smem = kAtlasBytes + (kWarpKernelThreads / 32) * kQuadKindBytes;
  const bool pdl = p.N >= kQuadPdlMinEnvs;
  const auto kernel = pdl ? env_kernel_quad<STEP, true> : env_kernel_quad<STEP, false>;
  int ctas;
  if (cudaError_t err = resident_ctas(ctx, kernel, kWarpKernelThreads, smem, ctas, kQuadCtas)) return err;
  int grid, threads;
  warp_kernel_shape((p.N + 3) >> 2, ctx.sm_count, ctas, grid, threads, /*few_ctas=*/true);   // one warp per quad
  return launch_maybe_pdl(kernel, pdl, grid, threads, smem, stream, p);
}

template cudaError_t launch_warp_kernel<0>(const EnvParams&, const LaunchCtx&, cudaStream_t);
template cudaError_t launch_warp_kernel<1>(const EnvParams&, const LaunchCtx&, cudaStream_t);
template cudaError_t launch_warp_kernel<2>(const EnvParams&, const LaunchCtx&, cudaStream_t);
template cudaError_t launch_warp_kernel<3>(const EnvParams&, const LaunchCtx&, cudaStream_t);
template cudaError_t launch_warp_kernel<4>(const EnvParams&, const LaunchCtx&, cudaStream_t);
template cudaError_t launch_quad_kernel<1>(const EnvParams&, const LaunchCtx&, cudaStream_t);
template cudaError_t launch_quad_kernel<2>(const EnvParams&, const LaunchCtx&, cudaStream_t);

}  // namespace merlin
