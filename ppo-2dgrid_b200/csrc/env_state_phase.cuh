// env_state_phase.cuh -- the lane-per-env state phase shared by the large-batch step kernels (env_kernels.cu: group,
// ordered and symbolic-only kernels; env_kernels_tile.cu: CTA-tile kernels), and the observation-path switch.
#pragma once
#include "env_kernels_common.cuh"
#include "obs_swar.cuh"

namespace merlin {

// One env's 147-byte symbolic image from its seven visible-code groups (obs_swar.cuh) into shared memory at `row`
// (any alignment: rows of consecutive lanes are 147 bytes apart).  The image is assembled as 37 little-endian words in
// registers, funnel-shifted by this lane's misalignment and stored as 35 aligned words; the words that straddle the
// row's two ends are shared with the neighbouring lanes' rows and go out as single bytes.
__device__ __forceinline__ void store_sym_row(uint8_t* row, const uint64_t (&g)[kView], bool doors) {
  uint32_t r[38];
  {
    uint64_t acc = 0;
    int have = 0, n = 0;  // compile-time after unrolling: every shift below is an immediate
#pragma unroll
    for (int vi = 0; vi < kView; ++vi) {
      uint32_t w[6];
      encode_group(g[vi], w, doors);
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        acc |= (uint64_t)w[i] << (8 * have);
        have += i < 5 ? 4 : 1;
        if (have >= 4) { r[n++] = (uint32_t)acc; acc >>= 32; have -= 4; }
      }
    }
    r[n++] = (uint32_t)acc;  // bytes 144..146 (+ one zero)
    r[n] = 0;                // n == 37
  }
  const uint32_t addr = (uint32_t)__cvta_generic_to_shared(row);
  const uint32_t s = addr & 3u, sh = 8u * s;
  uint8_t* base = row - s;  // word-aligned
  uint32_t prev = 0;
#pragma unroll
  for (int k = 0; k < 38; ++k) {
    const uint32_t word = __funnelshift_l(prev, r[k], sh);  // bytes 4k - s .. 4k - s + 3 of the image
    prev = r[k];
    if (k >= 1 && k <= 35) {
      *reinterpret_cast<uint32_t*>(base + 4 * k) = word;
    } else {
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int i = 4 * k + b - (int)s;  // image byte held by byte b of this word
        if (i >= 0 && i < kSymBytes) base[4 * k + b] = (uint8_t)(word >> (8 * b));
      }
    }
  }
}

// Grid.encode image of one env's view, cell by cell, straight into a global row: the final observation of an episode
// that ends (STEP = 3 / 4).  Two passes over the window -- the transparency mask by view rows, then the encode by view
// columns -- with the seven loads of a row or column in flight together: 14 round trips, and few enough registers that
// the caller's allocation does not grow (every cell at once costs the register-capped tile and symbolic kernels
// hundreds of bytes of spills).  Same bytes as the observation part of state_phase (either form).  About
// N / max_steps lanes of a step take this path.
static __device__ __noinline__ void store_final_row(const EnvState& s, const uint8_t* grid, int W, int H, uint64_t pol,
                                                    uint8_t* out) {
  const int fx = dir_dx(s.dir), fy = dir_dy(s.dir);
  const auto cell = [&](int vi, int vj) -> uint32_t {
    return window_cell(grid, W, H, pol, s.x, s.y, fx, fy, (kView - 1) - vj, vi - kView / 2);
  };
  uint64_t transp = 0;
#pragma unroll 1
  for (int vj = 0; vj < kView; ++vj) {
#pragma unroll
    for (int vi = 0; vi < kView; ++vi)
      if (!((M_OPAQUE >> (cell(vi, vj) & 0xf)) & 1u)) transp |= (uint64_t)1 << (vj * kView + vi);
  }
  const uint64_t vis = visibility(transp);
#pragma unroll 1
  for (int vi = 0; vi < kView; ++vi) {
#pragma unroll
    for (int vj = 0; vj < kView; ++vj) {
      const bool agent_cell = (vi == kView / 2 && vj == kView - 1);
      const uint32_t code = agent_cell ? carried_code(s.carry) : cell(vi, vj);
      uint8_t t = 0, col = 0, stt = 0;
      if ((vis >> (vj * kView + vi)) & 1) sym_of_code(code, t, col, stt);
      uint8_t* o = out + (vi * kView + vj) * 3;
      o[0] = t; o[1] = col; o[2] = stt;
    }
  }
}

// State phase, one env per lane, for the G envs e0 .. e0+G-1 (lanes >= G idle).  Must be called by a full warp.
// Leaves kinds_s[lane][kKindStride] / sym_s[lane][147] filled for the envs whose bit is set in the returned mask.
// SWAR = true: the observation is computed on window rows (obs_swar.cuh; needs W >= 7), else cell by cell.
template <int G, int STEP, bool SWAR = false>
__device__ __forceinline__ unsigned state_phase(const EnvParams& p, const Flags& f, int e0, int lane, uint8_t* kinds_s,
                                                uint8_t* sym_s) {
  const int e = e0 + lane;
  const bool active = lane < G && e < p.N;
  EnvState s{};
  bool restart = false;   // this lane's env (re)loads a layout now
  bool render = active;   // this lane's env gets its observation written
  if (active) {
    const int4 st = p.state[e];
    unpack_state(st.x, st.y, st.z, st.w, s);
  }
  float ep_ret = active ? p.ep_return[e] : 0.f;

  if (STEP) {
    if (active) {
      const uint8_t* grid = f.mutable_grid ? p.cells + (size_t)e * p.cell_stride
                                           : p.pool_cells + (size_t)s.layout * p.cell_stride;
      const int fx = s.x + dir_dx(s.dir), fy = s.y + dir_dy(s.dir);
      const bool inb = (unsigned)fx < (unsigned)p.W && (unsigned)fy < (unsigned)p.H;
      const int fidx = fy * p.W + fx;
      const uint32_t fwd = inb ? ld_cell(grid + fidx, f.pol) : CODE_WALL;
      const ActionDraw act = draw_action<step_draws(STEP)>(p, f.n_actions, e);
      commit_action<step_draws(STEP)>(p, e, act);
      StepResult r = step_logic(s, act.action, f.n_actions, fwd, inb, fidx, p.max_steps);
      if (r.bad_action) atomicAdd(p.bad_actions, 1ull);
      if (r.write_idx >= 0 && f.mutable_grid) p.cells[(size_t)e * p.cell_stride + r.write_idx] = (uint8_t)r.write_code;

      uint32_t vword = 0;
      const int cell = s.y * p.W + s.x;
      uint32_t* vptr = nullptr;
      if (f.explore_on) { vptr = p.visited + (size_t)e * p.vis_words + (cell >> 5); vword = *vptr; }
      bool stuck = false;
      const uint32_t vword_in = vword;
      const double rew_d = shape_reward(s, r.reward, f.stuck_on, p.stuck_max_stay, p.stuck_penalty, f.explore_on,
                                        p.explore_bonus, vword, cell & 31, stuck);
      if (f.explore_on && vword != vword_in) *vptr = vword;
      const float rew = (float)rew_d;
      ep_ret += rew;
      const bool done = r.terminated || r.truncated;
      store_step_outputs(p, e, rew, r.terminated, r.truncated, ep_ret, s.step_count, stuck);
      record_first_episode<step_draws(STEP)>(p, e, done, r.terminated && r.reward > 0.0, ep_ret, s.step_count);
      // the final image: after this lane's own grid write above, before the restart below replaces pose and grid
      if constexpr (step_final(STEP)) {
        if (done) store_final_row(s, grid, p.W, p.H, f.pol, p.final_sym + (size_t)e * kSymBytes);
      }
      restart = done && f.auto_reset;
    }
  } else {
    restart = active && (p.reset_mask == nullptr || p.reset_mask[e] != 0);
    render = restart;
  }

  // (re)start: pose from the pool, counters cleared, cursor advanced; mutable grids / visited maps are
  // re-initialised by the whole warp with coalesced copies
  const unsigned restart_mask = __ballot_sync(0xffffffffu, restart);
  if (restart_mask) {
    const int load_cur = restart_layout(p, f.advance, s.layout);
    if (restart) {
      restart_state(p, load_cur, s);
      ep_ret = 0.f;
    }
    if (f.mutable_grid || f.explore_on) {
      unsigned m = restart_mask;
      while (m) {
        const int src = __ffs(m) - 1;
        m &= m - 1;
        const int cur = __shfl_sync(0xffffffffu, load_cur, src);
        const int sx = __shfl_sync(0xffffffffu, s.x, src), sy = __shfl_sync(0xffffffffu, s.y, src);
        const size_t ee = (size_t)(e0 + src);
        if (f.mutable_grid) copy_pool_grid(p, ee, cur, lane);
        if (f.explore_on) reset_visited(p, ee, sx, sy, lane);
      }
      __syncwarp();
    }
    if (restart) s.layout = load_cur;
  }

  if (active && (STEP || restart)) {
    int4 st;
    pack_state(s, st.x, st.y, st.z, st.w);
    p.state[e] = st;
    p.ep_return[e] = ep_ret;
  }

  // observation, part 1 (per lane): window gather -> visibility -> tile kinds (+ symbolic bytes) in smem
  if ((f.want_rgb || f.want_sym) && render) {
    const uint8_t* grid = f.mutable_grid ? p.cells + (size_t)e * p.cell_stride
                                         : p.pool_cells + (size_t)s.layout * p.cell_stride;
    uint8_t* kind = kinds_s + lane * kKindStride;
    if (SWAR) {
      uint64_t g[kView], seen[kView];
      observe_swar(s, grid, p.W, p.H, g, seen, f.doors, f.pol);
      if (f.want_rgb) {
        uint32_t kw[13];
        kind_words(g, s.carry, kw);
        uint32_t* kdst = reinterpret_cast<uint32_t*>(kind);  // kKindStride = 52: word-aligned rows
#pragma unroll
        for (int i = 0; i < 13; ++i) kdst[i] = kw[i];
      }
      if (f.want_sym) store_sym_row(sym_s + lane * kSymBytes, g, f.doors);
    } else {
      const uint64_t pol = f.pol;
      const uint64_t transp = gather_view(s, p.W, p.H, [&](int idx) -> uint32_t { return ld_cell(grid + idx, pol); }, kind);
      const uint64_t vis = visibility(transp);
      uint8_t* sym = sym_s + lane * kSymBytes;
#pragma unroll
      for (int vi = 0; vi < kView; ++vi) {
#pragma unroll
        for (int vj = 0; vj < kView; ++vj) {
          const int c = vi * kView + vj;
          const bool seen = (vis >> (vj * kView + vi)) & 1;
          uint32_t code = kind[c];
          const bool agent_cell = (vi == kView / 2 && vj == kView - 1);
          if (agent_cell) code = carried_code(s.carry);
          kind[c] = (uint8_t)shown_kind(code, seen, agent_cell, s.carry);
          if (f.want_sym) {
            uint8_t t = 0, col = 0, stt = 0;
            if (seen) sym_of_code(code, t, col, stt);
            sym[c * 3 + 0] = t; sym[c * 3 + 1] = col; sym[c * 3 + 2] = stt;
          }
        }
      }
    }
  }
  __syncwarp();
  return __ballot_sync(0xffffffffu, render);
}

// Observation path.  Measured on B200 at 1M envs: the row-parallel form (obs_swar.cuh, 30 % fewer instructions, 48
// instead of 72 registers) lifts the symbolic-only kernel from 7.6e9 to 1.19e10 env-steps/s (0.52 -> 0.82 of the HBM
// roofline of its 449 B/step): that kernel is ALU-bound and runs 40 warps per SM.  The frame kernels are indifferent
// (tile kernel 1.083 per-cell vs 1.076 row form, ordered-group kernel 1.05 either way): their limit is the store
// stream.  (With the window loads behind per-row branches the tile kernel dropped to 1.01 -- its single state-phase
// warp paid one L2 round trip per row; window_rows() is straight-line for that reason.)  Hence: 0 = automatic =
// row-parallel in the symbolic-only kernel only, 1 = per-cell everywhere, 2 = row-parallel in every kernel that has it
// (symbolic-only, tile, ordered; tests, A/B).
static bool use_swar(const EnvParams& p, const LaunchCtx& ctx, bool frame_kernel) {
  if (p.W < kView || ctx.observation_path == 1) return false;
  return ctx.observation_path == 2 || !frame_kernel;
}

}  // namespace merlin
