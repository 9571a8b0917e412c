// layout_kernels.cu -- on-device generation of MERLIN layouts (the `_gen_grid` routines of the five difficulties),
// one warp per layout, straight into the handle's layout pool.
//
// What it restates (reference file:line; upstream place_obj / place_agent / wall_rect semantics as in SURVEY 8c.2):
//   easy        src/custom_envs/easy_env.py:19-39         medium      src/custom_envs/medium_env.py:19-33
//   mediumhard  src/custom_envs/medium_hard_env.py:12-74   hard        src/custom_envs/hard_env.py:11-97
//   hardest     src/custom_envs/hardest_env.py:20-96
// Same algorithms and the same draw ORDER as the host generators (merlin_b200/layouts.py), fed by one of two streams:
//   SplitMixRng  (merlin_env_generate_layouts) a counter-based generator, SplitMix64 keyed by seed and layout number: the
//                same distributions, but NOT the layout `env.reset(seed=s)` builds in the reference.  Fresh layouts for
//                training.  Validated by structural invariants, by statistics against the host generator and by driving
//                the oracle with the generated pool (tests/test_gpu_layoutgen.py).
//   NumpyRng     (merlin_env_generate_seeded_layouts) numpy's default_rng(seed) stream (np_random.cuh), one fresh
//                generator per layout: exactly the layout `env.reset(seed=s)` builds, byte for byte
//                (tests/test_gpu_seeded_layouts.py).  Where the host generator raises or never returns, the layout is
//                flagged instead of built (NumpyRng::failed).
// The routines are templates on the stream; the two streams differ only in `integers`, in the k distinct rows of hard's
// `choice(replace=False)` and in what a failed placement means.
//
// Mapping: every lane of the warp executes the identical draw sequence (uniform control flow, same-value stores), so
// rejection sampling needs no communication; only the two data-parallel parts are split over lanes: building the
// bordered room and the reachability flood fill (iterative relaxation over the cells, reached = bit 7 of the cell byte,
// warp vote for convergence), which replaces the reference's BFS queue.
#include <cuda_runtime.h>
#include <stdint.h>

#include "env_kernels.cuh"
#include "env_logic.cuh"
#include "np_random.cuh"

namespace merlin {

namespace {

constexpr uint32_t CODE_GOAL = T_GOAL | (1u << 4);
constexpr uint8_t kReached = 0x80;
constexpr int kAgentTries = 1 << 20;  // the cap on place_obj(max_tries=inf)
// CTAs of 4 warps that must fit on one SM: caps both kernels at 48 registers, where ptxas keeps every value in a
// register (left to its own heuristic it spills a few at 40 registers)
constexpr int kMinCtas = 10;

struct SplitMixRng {
  uint64_t s;
  __device__ __forceinline__ uint64_t next() {  // SplitMix64
    uint64_t z = (s += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
  }
  // uniform integer in [lo, hi) (np_random.integers); a degenerate range yields lo
  __device__ __forceinline__ int integers(int lo, int hi) {
    if (hi <= lo + 1) { next(); return lo; }
    return lo + (int)(((next() >> 32) * (uint64_t)(uint32_t)(hi - lo)) >> 32);
  }
  // np_random.choice(range(lo, hi), size=k, replace=False): distinct values, uniformly, by rejection
  __device__ __forceinline__ void distinct(int lo, int hi, int k, int* out) {
    for (int i = 0; i < k; ++i) {
      for (;;) {
        const int r = integers(lo, hi);
        bool dup = false;
        for (int j = 0; j < i; ++j) dup |= out[j] == r;
        if (!dup || hi - lo <= i) { out[i] = r; break; }
      }
    }
  }
  // a placement that ran out of tries is a failed attempt of the routine; the layout is always built
  __device__ __forceinline__ void fail() {}
  __device__ __forceinline__ bool failed() const { return false; }
};

struct NumpyRng {
  NpRandom g;
  bool bad;  // the host generator raises (or never returns) on this seed
  __device__ __forceinline__ int integers(int lo, int hi) {
    if (hi <= lo) { bad = true; return lo; }  // numpy: ValueError (high <= low)
    return (int)g.integers(lo, hi);
  }
  __device__ __forceinline__ void distinct(int lo, int hi, int k, int* out) {
    if (k > hi - lo) { bad = true; return; }  // numpy: ValueError (a larger sample than the population)
    g.choice(hi - lo, k, out);
    for (int i = 0; i < k; ++i) out[i] += lo;
  }
  __device__ __forceinline__ void fail() { bad = true; }  // place_obj raises RecursionError / loops forever
  __device__ __forceinline__ bool failed() const { return bad; }
};

template <class Rng>
struct Builder {
  uint8_t* g;      // this layout's cells, row-major [y*W + x]
  int W, H, lane;
  int ax, ay, adir;  // agent pose; (-1,-1) until placed -- survives retries, like self.agent_pos in the reference
  Rng rng;

  __device__ __forceinline__ void room() {  // Grid(W,H) + wall_rect(0,0,W,H)
    __syncwarp();
    for (int c = lane; c < W * H; c += 32) {
      const int x = c % W, y = c / W;
      g[c] = (x == 0 || y == 0 || x == W - 1 || y == H - 1) ? (uint8_t)CODE_WALL : (uint8_t)CODE_EMPTY;
    }
    __syncwarp();
  }
  __device__ __forceinline__ uint32_t at(int x, int y) const { return g[y * W + x] & 0x7f; }
  __device__ __forceinline__ void set(int x, int y, uint32_t code) { g[y * W + x] = (uint8_t)code; }

  // minigrid place_obj: rejection-sample an empty cell that is not the agent's; x drawn before y.  `code` 0 = only pick.
  __device__ __forceinline__ bool place(uint32_t code, int tx, int ty, int sx, int sy, int max_tries, int& px, int& py) {
    if (rng.failed()) return false;
    tx = max(tx, 0); ty = max(ty, 0);
    for (int tries = 0; tries <= max_tries; ++tries) {
      const int x = rng.integers(tx, min(tx + sx, W));
      const int y = rng.integers(ty, min(ty + sy, H));
      if (at(x, y) != CODE_EMPTY) continue;
      if (x == ax && y == ay) continue;
      if (code) set(x, y, code);
      px = x; py = y;
      return true;
    }
    rng.fail();
    return false;  // upstream raises RecursionError here
  }
  __device__ __forceinline__ bool place_agent(int tx, int ty, int sx, int sy) {
    ax = ay = -1;
    int x, y;
    if (!place(0, tx, ty, sx, sy, kAgentTries, x, y)) return false;
    ax = x; ay = y;
    adir = rng.integers(0, 4);
    return true;
  }

  // _is_reachable: 4-neighbour connectivity over empty / goal cells, as a warp-wide relaxation
  __device__ bool reachable(int gx, int gy) {
    __syncwarp();
    if (ax < 0 || ay < 0) return false;   // no agent was placed (warp-uniform: every lane runs the same draws)
    if (lane == 0) g[ay * W + ax] |= kReached;
    __syncwarp();
    for (;;) {
      bool changed = false;
      for (int c = lane; c < W * H; c += 32) {
        const uint32_t v = g[c];
        if (v & kReached) continue;
        const uint32_t t = v & 0xf;
        const int x = c % W, y = c / W;
        if (!(t == T_EMPTY || t == T_GOAL || (x == gx && y == gy))) continue;
        const bool near = (x > 0 && (g[c - 1] & kReached)) || (x < W - 1 && (g[c + 1] & kReached)) ||
                          (y > 0 && (g[c - W] & kReached)) || (y < H - 1 && (g[c + W] & kReached));
        if (near) { g[c] = (uint8_t)(v | kReached); changed = true; }
      }
      __syncwarp();
      if (!__any_sync(0xffffffffu, changed)) break;
    }
    const bool ok = g[gy * W + gx] & kReached;
    __syncwarp();
    for (int c = lane; c < W * H; c += 32) g[c] &= 0x7f;
    __syncwarp();
    return ok;
  }

  __device__ void fallback() {  // the empty-room fallback of every generator
    if (rng.failed()) return;
    int x, y;
    room();
    // an empty room always has free interior cells; should 2^20 draws still miss them all, the pose is pinned to the
    // first interior cell rather than left at (-1, -1) (the pool must never hold a pose outside the grid)
    if (!place_agent(0, 0, W, H)) { ax = 1; ay = 1; adir = 0; }
    place(CODE_GOAL, 0, 0, W, H, kAgentTries, x, y);
  }
};

// Every attempt loop stops at the first failure of the seeded stream (for SplitMixRng `failed()` is constant false).

template <class Rng>
__device__ void gen_easy(Builder<Rng>& b) {
  b.room();
  if (!b.place_agent(0, 0, b.W, b.H)) { b.ax = 1; b.ay = 1; b.adir = 0; }   // an empty room: cannot fail in practice
  b.set(b.W - 5, b.H - 5, CODE_GOAL);
}

template <class Rng>
__device__ void gen_medium(Builder<Rng>& b) {
  int x, y;
  b.room();
  if (!b.place_agent(0, 0, b.W, b.H)) { b.ax = 1; b.ay = 1; b.adir = 0; }
  b.place(CODE_GOAL, 0, 0, b.W, b.H, kAgentTries, x, y);
}

template <class Rng>
__device__ void gen_mediumhard(Builder<Rng>& b) {
  const int interior = (b.W - 2) * (b.H - 2);
  const int lo = max(1, (int)(interior * 0.10)), hi = max(1, (int)(interior * 0.20)) + 1;
  for (int attempt = 0; attempt < 100 && !b.rng.failed(); ++attempt) {
    b.room();
    const int n = b.rng.integers(lo, hi);
    int x, y;
    bool ok = true;
    for (int i = 0; i < n && ok; ++i) ok = b.place(CODE_WALL, 0, 0, b.W, b.H, 100, x, y);  // rejects the previous attempt's agent cell
    if (!ok) continue;
    if (!b.place_agent(0, 0, b.W, b.H)) continue;   // no free cell found: a failed attempt, as in gen_hard
    int gx, gy;
    if (!b.place(CODE_GOAL, 0, 0, b.W, b.H, kAgentTries, gx, gy)) continue;
    if (b.reachable(gx, gy)) return;
  }
  b.fallback();
}

template <class Rng>
__device__ void gen_hard(Builder<Rng>& b) {
  const int W = b.W, H = b.H, mid = W / 2;
  const bool big = W > 10;
  for (int attempt = 0; attempt < 100 && !b.rng.failed(); ++attempt) {
    b.room();
    const int n_gaps = big ? b.rng.integers(2, 6) : 1;
    int gaps[5];
    b.rng.distinct(1, H - 1, n_gaps, gaps);  // np_random.choice(range(1, H-1), size=n_gaps, replace=False)
    if (b.rng.failed()) return;
    for (int j = 1; j < H - 1; ++j) {
      bool gap = false;
      for (int k = 0; k < n_gaps; ++k) gap |= gaps[k] == j;
      if (!gap) b.set(mid, j, CODE_WALL);
    }
    if (big) {
      const int extra = b.rng.integers(6, 13);
      for (int i = 0; i < extra; ++i)
        for (int t = 0; t < 10; ++t) {
          const int x = b.rng.integers(1, W - 1), y = b.rng.integers(1, H - 1);
          if (x != mid && b.at(x, y) == CODE_EMPTY) { b.set(x, y, CODE_WALL); break; }
        }
    }
    int gx, gy;
    if (!b.place(CODE_GOAL, mid + 1, 0, W - mid - 1, H, kAgentTries, gx, gy)) continue;
    if (!b.place_agent(1, 1, mid - 1, H - 2)) continue;
    if (b.reachable(gx, gy)) return;
  }
  b.fallback();
}

template <class Rng>
__device__ void gen_hardest(Builder<Rng>& b) {
  const int W = b.W, H = b.H, mx = W / 2, my = H / 2;
  for (int attempt = 0; attempt < 100 && !b.rng.failed(); ++attempt) {
    b.room();
    for (int y = 1; y < H - 1; ++y) b.set(mx, y, CODE_WALL);
    for (int x = 1; x < W - 1; ++x) b.set(x, my, CODE_WALL);
    b.set(mx, b.rng.integers(2, my - 1), CODE_EMPTY);
    b.set(mx, b.rng.integers(my + 1, H - 2), CODE_EMPTY);
    b.set(b.rng.integers(2, mx - 1), my, CODE_EMPTY);
    b.set(b.rng.integers(mx + 1, W - 2), my, CODE_EMPTY);
    const int n = b.rng.integers(6, 13);
    for (int i = 0; i < n; ++i) {
      const int x = b.rng.integers(1, W - 1), y = b.rng.integers(1, H - 1);
      if (b.at(x, y) == CODE_EMPTY && x != mx && y != my) b.set(x, y, CODE_WALL);
    }
    if (!b.place_agent(0, 0, W, H)) continue;
    int gx, gy;
    if (!b.place(CODE_GOAL, 0, 0, W, H, kAgentTries, gx, gy)) continue;
    if (b.reachable(gx, gy)) return;
  }
  b.fallback();
}

// one `_gen_grid` call into pool slot `slot`, then the row padding and the packed agent pose
template <class Rng>
__device__ void build_layout(Builder<Rng>& b, int difficulty, int cell_stride, uint32_t* pool_agent, int slot) {
  b.ax = b.ay = -1; b.adir = 0;
  switch (difficulty) {
    case 0: gen_easy(b); break;
    case 1: gen_medium(b); break;
    case 2: gen_mediumhard(b); break;
    case 3: gen_hard(b); break;
    default: gen_hardest(b); break;
  }
  __syncwarp();
  for (int c = b.W * b.H + b.lane; c < cell_stride; c += 32) b.g[c] = (uint8_t)CODE_EMPTY;  // row padding
  if (b.lane == 0) pool_agent[slot] = (uint32_t)b.ax | ((uint32_t)b.ay << 8) | ((uint32_t)b.adir << 16);
}

__global__ void __launch_bounds__(128, kMinCtas)
layout_kernel(uint8_t* pool_cells, uint32_t* pool_agent, int cell_stride, int W, int H, int difficulty, uint64_t seed,
              long long first_number, int first_slot, int count) {
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  for (int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < count; i += warps) {
    Builder<SplitMixRng> b;
    b.g = pool_cells + (size_t)(first_slot + i) * cell_stride;
    b.W = W; b.H = H; b.lane = lane;
    // one independent stream per (seed, layout number): the number, not the pool slot, keys the stream, so a pool can
    // be refilled with the NEXT layouts of the same run
    b.rng.s = seed * 0xD1342543DE82EF95ull + (uint64_t)(first_number + i) * 0x2545F4914F6CDD1Dull + 0x632BE59BD9B4E019ull;
    b.rng.next();
    build_layout(b, difficulty, cell_stride, pool_agent, first_slot + i);
  }
}

// slot i <- the layout of reset(seed=seeds[i]); *first_failed <- the smallest slot the host generator could not build
__global__ void __launch_bounds__(128, kMinCtas)
seeded_layout_kernel(uint8_t* pool_cells, uint32_t* pool_agent, int cell_stride, int W, int H, int difficulty,
                     const uint64_t* seeds, int count, int* first_failed) {
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  for (int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < count; i += warps) {
    Builder<NumpyRng> b;
    b.g = pool_cells + (size_t)i * cell_stride;
    b.W = W; b.H = H; b.lane = lane;
    b.rng.g.seed(seeds[i]);
    b.rng.bad = false;
    build_layout(b, difficulty, cell_stride, pool_agent, i);
    if (lane == 0 && b.rng.failed()) atomicMin(first_failed, i);
  }
}

int layout_grid(int count, int sm_count) {
  const int warps_per_cta = 128 / 32;
  const int grid = (count + warps_per_cta - 1) / warps_per_cta;
  return grid > sm_count * 16 ? sm_count * 16 : grid;
}

}  // namespace

cudaError_t launch_layouts(uint8_t* pool_cells, uint32_t* pool_agent, int cell_stride, int W, int H, int difficulty,
                           uint64_t seed, long long first_number, int first_slot, int count, int sm_count,
                           cudaStream_t stream) {
  if (count <= 0) return cudaSuccess;
  layout_kernel<<<layout_grid(count, sm_count), 128, 0, stream>>>(pool_cells, pool_agent, cell_stride, W, H, difficulty,
                                                                  seed, first_number, first_slot, count);
  return cudaGetLastError();
}

cudaError_t launch_seeded_layouts(uint8_t* pool_cells, uint32_t* pool_agent, int cell_stride, int W, int H,
                                  int difficulty, const uint64_t* seeds, int count, int* first_failed, int sm_count,
                                  cudaStream_t stream) {
  if (count <= 0) return cudaSuccess;
  seeded_layout_kernel<<<layout_grid(count, sm_count), 128, 0, stream>>>(pool_cells, pool_agent, cell_stride, W, H,
                                                                         difficulty, seeds, count, first_failed);
  return cudaGetLastError();
}

}  // namespace merlin
