// capi.cu -- the C ABI declared in include/merlin_b200.h: handle lifetime, host->device uploads,
// argument validation and kernel launches.  No compute happens on the host; without a CUDA device
// every entry point fails (there is no CPU fallback by design).
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "env_kernels.cuh"

using namespace merlin;

namespace {

thread_local std::string g_last_error;

int fail(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}
int cuda_fail(cudaError_t err, const char* what) {
  return fail(MERLIN_ECUDA, std::string(what) + ": " + cudaGetErrorString(err));
}

struct DeviceGuard {  // the caller (e.g. torch) owns the current-device setting; restore it on exit
  int prev = -1;
  bool ok = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) return;
    ok = (prev == dev) || (cudaSetDevice(dev) == cudaSuccess);
  }
  ~DeviceGuard() {
    int cur = -1;
    if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
  }
};

// process-wide DEFAULTS of the two tuning knobs (merlin_set_kernel_choice / merlin_set_observation_path): what a handle
// uses until merlin_env_set_kernel_choice / merlin_env_set_observation_path give it a setting of its own
std::atomic<int> g_default_kernel_choice{0};
std::atomic<int> g_default_observation_path{0};

constexpr int kRenderRing = 16;                    // ticket-counter pairs the render launches rotate through
constexpr int kSchedWords = 2 * (1 + kRenderRing); // pair 0: step / reset; pairs 1..16: render

}  // namespace

struct merlin_env {
  merlin_env_config_t cfg{};
  int sm_count = 0;
  int cell_stride = 0;
  int vis_words = 0;
  int n_layouts = 0;
  bool mutable_grid = false;
  bool has_atlas = false;
  int n_present = kAtlasTiles;           // atlas slots the current layout pool can show (host copy of the popcount)
  bool was_reset = false;
  bool pool_failed = false;              // the last seeded generation hit a seed it could not build: no reset until a new pool
  int64_t launches = 0;
  // per-handle tuning knobs (-1 = follow the process-wide default) and occupancy cache
  int kernel_choice = -1;
  int observation_path = -1;
  OccupancyCache occ;
  // action sampler (merlin_env_policy_step)
  uint64_t sampler_seed = 0x9E3779B97F4A7C15ull;
  uint32_t* draws = nullptr;             // [N] draws made so far per env
  // stream ordering of the launches that share a ticket counter: class 0 = reset / step, class 1 = render
  cudaStream_t last_stream[2] = {nullptr, nullptr};
  bool last_stream_valid[2] = {false, false};
  cudaEvent_t order_event = nullptr;
  unsigned render_seq = 0;
  // device memory
  int4* state = nullptr;
  float* ep_return = nullptr;
  uint8_t* cells = nullptr;
  uint32_t* visited = nullptr;
  uint8_t* pool_cells = nullptr;
  uint32_t* pool_agent = nullptr;
  uint8_t* atlas = nullptr;
  unsigned* sched = nullptr;             // [2] in-order tile scheduler of env_kernel_tile
  uint32_t* blit_lut = nullptr;
  uint8_t* atlas_blocked = nullptr;      // the atlas with every tile re-laid as four 4x4-pixel, channel-major blocks
  uint32_t* blit_lut_blocked = nullptr;
  uint32_t* tile_present = nullptr;      // [4] device words, rewritten by upload_layouts
  unsigned long long* bad_actions = nullptr;
};

static int count_present(const uint32_t (&present)[4]) {
  int n = 0;
  for (uint32_t w : present) n += __builtin_popcount(w);
  return n;
}

static EnvParams base_params(const merlin_env* h) {
  EnvParams p{};
  p.N = h->cfg.n_envs; p.W = h->cfg.width; p.H = h->cfg.height; p.max_steps = h->cfg.max_steps;
  p.cell_stride = h->cell_stride; p.n_layouts = h->n_layouts; p.vis_words = h->vis_words;
  p.stuck_max_stay = h->cfg.stuck_max_stay; p.flags = h->cfg.flags;
  // every restart must bring a different layout when the pool has more than one: N mod L, or 1 when L divides N
  p.cursor_stride = h->n_layouts > 0 ? p.N % h->n_layouts : 0;
  if (p.cursor_stride == 0 && h->n_layouts > 1) p.cursor_stride = 1;
  p.stuck_penalty = h->cfg.stuck_penalty; p.explore_bonus = h->cfg.explore_bonus;
  p.state = h->state; p.ep_return = h->ep_return; p.cells = h->cells; p.visited = h->visited;
  p.pool_cells = h->pool_cells; p.pool_agent = h->pool_agent; p.atlas = h->atlas; p.bad_actions = h->bad_actions;
  p.blit_lut = h->blit_lut;
  p.tile_present = h->tile_present;
  p.sched = h->sched;
  p.draws = h->draws;
  return p;
}

static LaunchCtx launch_ctx(merlin_env* h) {
  LaunchCtx c;
  c.sm_count = h->sm_count;
  c.kernel_choice = h->kernel_choice >= 0 ? h->kernel_choice : g_default_kernel_choice.load();
  c.observation_path = h->observation_path >= 0 ? h->observation_path : g_default_observation_path.load();
  c.occ = &h->occ;
  return c;
}

// Launches of one class (0 = reset / step, 1 = render) draw tickets from handle-owned counters, so they must not
// overlap.  On one stream they cannot; when the caller moves to another stream, that stream is made to wait for
// everything submitted to the previous one (an event recorded at its tail).  Streams under capture are left alone: the
// captured graph's own dependencies order its launches, and replays are the caller's to order (header, "Conventions").
static void order_streams(merlin_env* h, int cls, cudaStream_t s) {
  if (h->last_stream_valid[cls] && h->last_stream[cls] != s && h->order_event) {
    cudaStreamCaptureStatus a = cudaStreamCaptureStatusNone, b = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(s, &a) == cudaSuccess && a == cudaStreamCaptureStatusNone &&
        cudaStreamIsCapturing(h->last_stream[cls], &b) == cudaSuccess && b == cudaStreamCaptureStatusNone) {
      if (cudaEventRecord(h->order_event, h->last_stream[cls]) == cudaSuccess) cudaStreamWaitEvent(s, h->order_event, 0);
    }
    cudaGetLastError();  // a stale stream handle is the caller's business; never leave an error behind
  }
  h->last_stream[cls] = s;
  h->last_stream_valid[cls] = true;
}

static unsigned* render_sched(merlin_env* h) {
  // consecutive render launches use different counter pairs: two renders that overlap on two streams (a policy-input
  // render beside a minibatch render) would otherwise share one ticket counter
  unsigned* s = h->sched + 2 * (1 + (h->render_seq % kRenderRing));
  h->render_seq += 1;
  return s;
}

// A launch that failed leaves the self-rearming ticket counters in an unknown state if an earlier kernel of this handle
// died mid-flight: clear them (best effort, on the same stream) so the next launch does not silently skip tiles.
static int launch_failed(merlin_env* h, cudaError_t err, const char* what, void* stream) {
  cudaGetLastError();
  cudaMemsetAsync(h->sched, 0, kSchedWords * sizeof(unsigned), static_cast<cudaStream_t>(stream));
  cudaGetLastError();
  return cuda_fail(err, what);
}

// Storage for a pool of n_layouts.  A pool of another size gets new storage; an equal-sized pool is overwritten in
// place, so device pointers (and CUDA graphs captured over them) stay valid across uploads and generations.
static int pool_storage(merlin_env* h, int n_layouts) {
  if (n_layouts == h->n_layouts) return MERLIN_OK;
  uint8_t* d_cells = nullptr;
  uint32_t* d_agent = nullptr;
  if (cudaMalloc(&d_cells, (size_t)n_layouts * h->cell_stride) != cudaSuccess ||
      cudaMalloc(&d_agent, (size_t)n_layouts * sizeof(uint32_t)) != cudaSuccess) {
    cudaFree(d_cells);
    return cuda_fail(cudaGetLastError(), "layout pool allocation");
  }
  cudaFree(h->pool_cells); cudaFree(h->pool_agent);
  h->pool_cells = d_cells; h->pool_agent = d_agent; h->n_layouts = n_layouts;
  return MERLIN_OK;
}

// Arguments of the two device generators.  The seeded one also rejects hard below 5 (its routine raises or never
// returns there for some seeds; the other generator treats such draws as failed attempts).
static int check_generation(merlin_env* h, int difficulty, int n_layouts, bool seeded) {
  if (!h) return fail(MERLIN_EINVAL, "null handle");
  if (difficulty < MERLIN_D_EASY || difficulty > MERLIN_D_HARDEST) return fail(MERLIN_EINVAL, "unknown difficulty id");
  if (n_layouts < 1)
    return fail(MERLIN_EINVAL, seeded ? "merlin_env_generate_seeded_layouts: no seeds"
                                      : "merlin_env_generate_layouts: bad count / first_number");
  const int W = h->cfg.width, H = h->cfg.height;
  int min_side = difficulty == MERLIN_D_HARDEST ? 8 : (difficulty == MERLIN_D_EASY ? 6 : 4);
  if (seeded && difficulty == MERLIN_D_HARD) min_side = 5;
  if (W < min_side || H < min_side) return fail(MERLIN_EINVAL, "grid too small for this difficulty's layout routine");
  return MERLIN_OK;
}

// The shared tail of a device generation that built every slot: the atlas slots a generated pool can show (the
// invisible tile, highlighted empty, the agent, wall and goal), the cursors reset; reset() must follow.
static int generated_pool_ready(merlin_env* h) {
  uint32_t present[4] = {(1u << KIND_UNSEEN) | (1u << CODE_EMPTY) | (1u << KIND_AGENT), 0, 0, 0};
  const uint32_t goal = T_GOAL | (1u << 4);
  present[CODE_WALL >> 5] |= 1u << (CODE_WALL & 31);
  present[goal >> 5] |= 1u << (goal & 31);
  if (h->mutable_grid) present[0] = present[1] = present[2] = present[3] = 0xffffffffu;
  const cudaError_t err = cudaMemcpy(h->tile_present, present, sizeof present, cudaMemcpyHostToDevice);
  if (err != cudaSuccess) return cuda_fail(err, "layout generation (mask)");
  h->n_present = count_present(present);
  h->launches += 1;
  h->was_reset = false;
  h->pool_failed = false;
  return merlin_env_set_cursors(h, nullptr);
}

extern "C" {

void merlin_env_default_config(merlin_env_config_t* cfg) {
  if (!cfg) return;
  std::memset(cfg, 0, sizeof(*cfg));
  cfg->device = 0; cfg->n_envs = 1; cfg->width = 16; cfg->height = 16; cfg->max_steps = 0;
  cfg->view = kView; cfg->tile = kTile; cfg->flags = MERLIN_F_AUTO_RESET;
  cfg->stuck_max_stay = 3; cfg->stuck_penalty = -0.1; cfg->explore_bonus = 0.0;
}

int merlin_env_create(const merlin_env_config_t* cfg, merlin_env_t** out) {
  if (!cfg || !out) return fail(MERLIN_EINVAL, "merlin_env_create: null argument");
  *out = nullptr;
  if (cfg->n_envs < 1) return fail(MERLIN_EINVAL, "n_envs must be >= 1");
  if (cfg->width < 3 || cfg->width > 255 || cfg->height < 3 || cfg->height > 255)
    return fail(MERLIN_EINVAL, "width/height must be in [3,255]");
  if (cfg->view != kView) return fail(MERLIN_EINVAL, "only agent_view_size 7 is built");
  if (cfg->tile != kTile) return fail(MERLIN_EINVAL, "only tile size 8 is built");
  if (cfg->max_steps < 0) return fail(MERLIN_EINVAL, "max_steps must be >= 0");
  if (cfg->stuck_max_stay < 0 || cfg->stuck_max_stay > 0xffff) return fail(MERLIN_EINVAL, "stuck_max_stay out of range");
  int n_dev = 0;
  cudaError_t err = cudaGetDeviceCount(&n_dev);
  if (err != cudaSuccess || n_dev == 0)
    return fail(MERLIN_ECUDA, "no CUDA device: libmerlin_b200 has no CPU fallback");
  if (cfg->device < 0 || cfg->device >= n_dev) return fail(MERLIN_EINVAL, "bad device ordinal");
  DeviceGuard guard(cfg->device);
  if (!guard.ok) return fail(MERLIN_ECUDA, "cudaSetDevice failed");

  merlin_env* h = new (std::nothrow) merlin_env();
  if (!h) return fail(MERLIN_ENOMEM, "host allocation failed");
  h->cfg = *cfg;
  if (h->cfg.max_steps == 0) h->cfg.max_steps = 4 * cfg->width * cfg->height;  // base_env.py:32-33
  h->cell_stride = (cfg->width * cfg->height + 15) & ~15;
  h->mutable_grid = (cfg->flags & MERLIN_F_SEVEN_ACTIONS) != 0;  // only pickup/drop/toggle write the grid
  h->vis_words = (cfg->width * cfg->height + 31) / 32;
  cudaDeviceProp prop{};
  if ((err = cudaGetDeviceProperties(&prop, cfg->device)) != cudaSuccess) { delete h; return cuda_fail(err, "cudaGetDeviceProperties"); }
  h->sm_count = prop.multiProcessorCount;

  const size_t N = (size_t)cfg->n_envs;
  // every CUDA call of the set-up is checked; the first failure wins and the remaining steps are skipped
  const char* what = "device allocation";
  bool alloc_failed = false;
  err = cudaSuccess;
#define MERLIN_TRY(call, w)                                  \
  do {                                                       \
    if (err == cudaSuccess) {                                \
      const cudaError_t e_ = (call);                         \
      if (e_ != cudaSuccess) { err = e_; what = (w); }       \
    }                                                        \
  } while (0)
#define MERLIN_ALLOC(ptr, bytes)                                              \
  do {                                                                        \
    if (err == cudaSuccess) {                                                 \
      const cudaError_t e_ = cudaMalloc((void**)&(ptr), (bytes));             \
      if (e_ != cudaSuccess) { err = e_; what = "device allocation"; alloc_failed = true; } \
    }                                                                         \
  } while (0)
  MERLIN_ALLOC(h->state, N * sizeof(int4));
  MERLIN_ALLOC(h->ep_return, N * sizeof(float));
  MERLIN_ALLOC(h->draws, N * sizeof(uint32_t));
  MERLIN_ALLOC(h->bad_actions, sizeof(unsigned long long));
  MERLIN_ALLOC(h->atlas, kAtlasBytes);
  MERLIN_ALLOC(h->sched, kSchedWords * sizeof(unsigned));
  MERLIN_ALLOC(h->blit_lut, kChunksPerLane * 32 * sizeof(uint32_t));
  MERLIN_ALLOC(h->blit_lut_blocked, kChunksPerLane * 32 * sizeof(uint32_t));
  MERLIN_ALLOC(h->atlas_blocked, kAtlasBytes);
  MERLIN_ALLOC(h->tile_present, 4 * sizeof(uint32_t));
  if (h->mutable_grid) MERLIN_ALLOC(h->cells, N * h->cell_stride);
  if (cfg->flags & MERLIN_F_EXPLORE_BONUS) MERLIN_ALLOC(h->visited, N * h->vis_words * sizeof(uint32_t));
  MERLIN_TRY(cudaEventCreateWithFlags(&h->order_event, cudaEventDisableTiming), "event creation");
  MERLIN_TRY(cudaMemset(h->state, 0, N * sizeof(int4)), "state init");
  MERLIN_TRY(cudaMemset(h->ep_return, 0, N * sizeof(float)), "episode-return init");
  MERLIN_TRY(cudaMemset(h->draws, 0, N * sizeof(uint32_t)), "sampler init");
  MERLIN_TRY(cudaMemset(h->bad_actions, 0, sizeof(unsigned long long)), "counter init");
  MERLIN_TRY(cudaMemset(h->atlas, 0, kAtlasBytes), "atlas init");
  MERLIN_TRY(cudaMemset(h->sched, 0, kSchedWords * sizeof(unsigned)), "scheduler init");
  {
    uint32_t lut[kChunksPerLane * 32];
    for (int c = 0; c < kChunksPerLane * 32; ++c) lut[c] = c < kChunks ? chunk_lut(c) : 0u;
    MERLIN_TRY(cudaMemcpy(h->blit_lut, lut, sizeof lut, cudaMemcpyHostToDevice), "blit map upload");
    for (int c = 0; c < kChunksPerLane * 32; ++c) lut[c] = c < kChunks ? chunk_lut_blocked(c) : 0u;
    MERLIN_TRY(cudaMemcpy(h->blit_lut_blocked, lut, sizeof lut, cudaMemcpyHostToDevice), "blocked blit map upload");
    MERLIN_TRY(cudaMemset(h->atlas_blocked, 0, kAtlasBytes), "blocked atlas init");
    MERLIN_TRY(cudaMemset(h->tile_present, 0xff, 4 * sizeof(uint32_t)), "tile mask init");
  }
  if (h->cells) MERLIN_TRY(cudaMemset(h->cells, CODE_EMPTY, N * h->cell_stride), "grid init");
  if (h->visited) MERLIN_TRY(cudaMemset(h->visited, 0, N * h->vis_words * sizeof(uint32_t)), "visited-map init");
  MERLIN_TRY(cudaDeviceSynchronize(), "init");
#undef MERLIN_TRY
#undef MERLIN_ALLOC
  if (err != cudaSuccess) {
    cudaGetLastError();
    merlin_env_destroy(h);
    if (alloc_failed) return fail(MERLIN_ENOMEM, std::string("device allocation failed: ") + cudaGetErrorString(err));
    return cuda_fail(err, what);
  }
  *out = h;
  return MERLIN_OK;
}

int merlin_env_destroy(merlin_env_t* h) {
  if (!h) return MERLIN_OK;
  DeviceGuard guard(h->cfg.device);
  cudaFree(h->state); cudaFree(h->ep_return); cudaFree(h->cells); cudaFree(h->visited);
  cudaFree(h->pool_cells); cudaFree(h->pool_agent); cudaFree(h->atlas); cudaFree(h->bad_actions);
  cudaFree(h->blit_lut); cudaFree(h->blit_lut_blocked); cudaFree(h->atlas_blocked); cudaFree(h->tile_present); cudaFree(h->sched);
  cudaFree(h->draws);
  if (h->order_event) cudaEventDestroy(h->order_event);
  delete h;
  return MERLIN_OK;
}

int merlin_env_upload_layouts(merlin_env_t* h, const uint8_t* cells, const int32_t* agent_xyd, int32_t n_layouts) {
  if (!h || !cells || !agent_xyd || n_layouts < 1) return fail(MERLIN_EINVAL, "merlin_env_upload_layouts: bad argument");
  const int W = h->cfg.width, H = h->cfg.height, HW = W * H;
  std::vector<uint8_t> packed((size_t)n_layouts * h->cell_stride, (uint8_t)CODE_EMPTY);
  std::vector<uint32_t> agent((size_t)n_layouts);
  // atlas slots a frame of this pool can show: the invisible tile, highlighted empty, the agent, every code present
  uint32_t present[4] = {(1u << KIND_UNSEEN) | (1u << CODE_EMPTY) | (1u << KIND_AGENT), 0, 0, 0};
  for (int l = 0; l < n_layouts; ++l) {
    for (int k = 0; k < HW; ++k) {
      const uint8_t c = cells[(size_t)l * HW + k];
      const uint32_t t = c & 0xf, col = (c >> 4) & 7;
      const bool type_ok = (t >= T_EMPTY && t <= T_LAVA) || t == T_DOOR_CLOSED || t == T_DOOR_LOCKED;
      if (!type_ok || col > 5 || (c & 0x80)) {
        char msg[128];
        std::snprintf(msg, sizeof msg, "layout %d cell %d: invalid packed code 0x%02x", l, k, c);
        return fail(MERLIN_EINVAL, msg);
      }
      packed[(size_t)l * h->cell_stride + k] = c;
      present[c >> 5] |= 1u << (c & 31);
    }
    const int x = agent_xyd[3 * l], y = agent_xyd[3 * l + 1], d = agent_xyd[3 * l + 2];
    if (x < 0 || x >= W || y < 0 || y >= H || d < 0 || d > 3) return fail(MERLIN_EINVAL, "agent pose outside the grid");
    const uint32_t under = packed[(size_t)l * h->cell_stride + y * W + x] & 0xf;
    if (!((M_OVERLAP >> under) & 1u)) return fail(MERLIN_EINVAL, "agent placed on a non-overlappable cell");
    agent[l] = (uint32_t)x | ((uint32_t)y << 8) | ((uint32_t)d << 16);
  }
  DeviceGuard guard(h->cfg.device);
  // pickup/drop/toggle create codes the pool does not hold (door states, carried objects): stage the whole atlas then
  if (h->mutable_grid) present[0] = present[1] = present[2] = present[3] = 0xffffffffu;
  cudaError_t err = cudaDeviceSynchronize();  // nothing may still be reading the old pool
  if (err != cudaSuccess) return cuda_fail(err, "layout upload (sync)");
  if (const int rc = pool_storage(h, n_layouts)) return rc;
  err = cudaMemcpy(h->pool_cells, packed.data(), packed.size(), cudaMemcpyHostToDevice);
  if (err == cudaSuccess) err = cudaMemcpy(h->pool_agent, agent.data(), agent.size() * sizeof(uint32_t), cudaMemcpyHostToDevice);
  if (err == cudaSuccess) err = cudaMemcpy(h->tile_present, present, sizeof present, cudaMemcpyHostToDevice);
  if (err != cudaSuccess) return cuda_fail(err, "layout upload");
  h->n_present = count_present(present);
  h->was_reset = false;
  h->pool_failed = false;
  cudaMemset(h->sched, 0, kSchedWords * sizeof(unsigned));  // the device is idle here: a cheap place to rearm the tickets
  return merlin_env_set_cursors(h, nullptr);
}

int merlin_env_generate_layouts(merlin_env_t* h, int32_t difficulty, uint64_t seed, int64_t first_number,
                                int32_t n_layouts, void* stream) {
  if (const int rc = check_generation(h, difficulty, n_layouts, false)) return rc;
  if (first_number < 0) return fail(MERLIN_EINVAL, "merlin_env_generate_layouts: bad count / first_number");
  DeviceGuard guard(h->cfg.device);
  cudaError_t err = cudaDeviceSynchronize();  // nothing may still be reading the old pool
  if (err != cudaSuccess) return cuda_fail(err, "layout generation (sync)");
  if (const int rc = pool_storage(h, n_layouts)) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  err = launch_layouts(h->pool_cells, h->pool_agent, h->cell_stride, h->cfg.width, h->cfg.height, difficulty, seed,
                       first_number, 0, n_layouts, h->sm_count, s);
  if (err == cudaSuccess) err = cudaStreamSynchronize(s);
  if (err != cudaSuccess) return cuda_fail(err, "layout generation");
  return generated_pool_ready(h);
}

int merlin_env_generate_seeded_layouts(merlin_env_t* h, int32_t difficulty, const uint64_t* seeds, int32_t n_layouts,
                                       void* stream) {
  if (h && !seeds) return fail(MERLIN_EINVAL, "merlin_env_generate_seeded_layouts: null seeds");
  if (const int rc = check_generation(h, difficulty, n_layouts, true)) return rc;
  DeviceGuard guard(h->cfg.device);
  cudaError_t err = cudaDeviceSynchronize();  // nothing may still be reading the old pool
  if (err != cudaSuccess) return cuda_fail(err, "seeded layout generation (sync)");
  if (const int rc = pool_storage(h, n_layouts)) return rc;
  // from here on the pool is being rewritten: it counts as failed until the kernel has built every slot
  h->pool_failed = true;
  h->was_reset = false;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  uint64_t* d_seeds = nullptr;
  int* d_first_failed = nullptr;
  int first_failed = n_layouts;
  if (cudaMalloc(&d_seeds, (size_t)n_layouts * sizeof(uint64_t)) != cudaSuccess ||
      cudaMalloc(&d_first_failed, sizeof(int)) != cudaSuccess) {
    cudaFree(d_seeds);
    return cuda_fail(cudaGetLastError(), "seeded layout generation (allocation)");
  }
  err = cudaMemcpyAsync(d_seeds, seeds, (size_t)n_layouts * sizeof(uint64_t), cudaMemcpyHostToDevice, s);
  if (err == cudaSuccess) err = cudaMemcpyAsync(d_first_failed, &first_failed, sizeof(int), cudaMemcpyHostToDevice, s);
  if (err == cudaSuccess)
    err = launch_seeded_layouts(h->pool_cells, h->pool_agent, h->cell_stride, h->cfg.width, h->cfg.height, difficulty,
                                d_seeds, n_layouts, d_first_failed, h->sm_count, s);
  if (err == cudaSuccess) err = cudaMemcpyAsync(&first_failed, d_first_failed, sizeof(int), cudaMemcpyDeviceToHost, s);
  if (err == cudaSuccess) err = cudaStreamSynchronize(s);
  cudaFree(d_seeds); cudaFree(d_first_failed);
  if (err != cudaSuccess) return cuda_fail(err, "seeded layout generation");
  if (first_failed < n_layouts) {
    static const char* const kNames[] = {"easy", "medium", "mediumhard", "hard", "hardest"};
    char msg[224];
    std::snprintf(msg, sizeof msg, "seed %llu (slot %d): the %s %dx%d layout routine raises or never returns for it; "
                  "the pool is incomplete until the next upload or generation",
                  (unsigned long long)seeds[first_failed], first_failed, kNames[difficulty], h->cfg.width, h->cfg.height);
    return fail(MERLIN_EINVAL, msg);
  }
  return generated_pool_ready(h);
}

int merlin_env_read_layouts(merlin_env_t* h, uint8_t* cells, int32_t* agent_xyd) {
  if (!h) return fail(MERLIN_EINVAL, "null handle");
  if (h->n_layouts < 1) return fail(MERLIN_ESTATE, "no layout pool");
  DeviceGuard guard(h->cfg.device);
  cudaError_t err = cudaDeviceSynchronize();
  const size_t HW = (size_t)h->cfg.width * h->cfg.height, L = (size_t)h->n_layouts;
  if (err == cudaSuccess && cells) err = cudaMemcpy2D(cells, HW, h->pool_cells, h->cell_stride, HW, L, cudaMemcpyDeviceToHost);
  if (err == cudaSuccess && agent_xyd) {
    std::vector<uint32_t> a(L);
    err = cudaMemcpy(a.data(), h->pool_agent, L * sizeof(uint32_t), cudaMemcpyDeviceToHost);
    for (size_t l = 0; l < L && err == cudaSuccess; ++l) {
      agent_xyd[3 * l] = a[l] & 0xff; agent_xyd[3 * l + 1] = (a[l] >> 8) & 0xff; agent_xyd[3 * l + 2] = (a[l] >> 16) & 3;
    }
  }
  if (err != cudaSuccess) return cuda_fail(err, "layout read-back");
  return MERLIN_OK;
}

int merlin_env_layout_count(merlin_env_t* h) { return h ? h->n_layouts : 0; }

int merlin_env_set_tile_atlas(merlin_env_t* h, const uint8_t* tiles, int32_t n_tiles) {
  if (!h || !tiles || n_tiles != kAtlasTiles) return fail(MERLIN_EINVAL, "atlas must hold exactly 128 tiles of 8x8x3");
  DeviceGuard guard(h->cfg.device);
  cudaError_t err = cudaMemcpy(h->atlas, tiles, kAtlasBytes, cudaMemcpyHostToDevice);
  if (err != cudaSuccess) return cuda_fail(err, "atlas upload");
  // blocked copy: tile[py][px][c] -> [sub = (py/4)*2 + px/4][c*16 + (py%4)*4 + px%4]
  std::vector<uint8_t> blocked(kAtlasBytes);
  for (int t = 0; t < kAtlasTiles; ++t)
    for (int py = 0; py < kTile; ++py)
      for (int px = 0; px < kTile; ++px)
        for (int c = 0; c < 3; ++c)
          blocked[(size_t)t * kTileBytes + ((py >> 2) * 2 + (px >> 2)) * 48 + c * 16 + (py & 3) * 4 + (px & 3)] =
              tiles[(size_t)t * kTileBytes + (py * kTile + px) * 3 + c];
  err = cudaMemcpy(h->atlas_blocked, blocked.data(), kAtlasBytes, cudaMemcpyHostToDevice);
  if (err != cudaSuccess) return cuda_fail(err, "blocked atlas upload");
  h->has_atlas = true;
  return MERLIN_OK;
}

int merlin_env_set_cursors(merlin_env_t* h, const int32_t* cursor) {
  if (!h) return fail(MERLIN_EINVAL, "null handle");
  if (h->n_layouts < 1) return fail(MERLIN_ESTATE, "upload layouts first");
  if (h->pool_failed) return fail(MERLIN_ESTATE, "the layout pool is incomplete: the last seeded generation failed");
  const int N = h->cfg.n_envs;
  std::vector<int4> st((size_t)N);
  for (int e = 0; e < N; ++e) {
    const int c = cursor ? cursor[e] : e % h->n_layouts;
    if (c < 0 || c >= h->n_layouts) return fail(MERLIN_EINVAL, "cursor outside the layout pool");
    st[e] = make_int4(0, 0, ~c, 0);  // negative layout = pending first load
  }
  DeviceGuard guard(h->cfg.device);
  cudaError_t err = cudaMemcpy(h->state, st.data(), st.size() * sizeof(int4), cudaMemcpyHostToDevice);
  if (err != cudaSuccess) return cuda_fail(err, "cursor upload");
  h->was_reset = false;
  return MERLIN_OK;
}

int merlin_env_reset(merlin_env_t* h, const uint8_t* mask, uint8_t* obs_rgb, uint8_t* obs_sym, void* stream) {
  if (!h) return fail(MERLIN_EINVAL, "null handle");
  if (h->n_layouts < 1) return fail(MERLIN_ESTATE, "reset before layouts were uploaded");
  if (h->pool_failed) return fail(MERLIN_ESTATE, "the layout pool is incomplete: the last seeded generation failed");
  if (obs_rgb && !h->has_atlas) return fail(MERLIN_ESTATE, "RGB observation requested before the tile atlas was set");
  if (mask && !h->was_reset) return fail(MERLIN_ESTATE, "the first reset must cover every env (mask = NULL)");
  if (obs_rgb && (reinterpret_cast<uintptr_t>(obs_rgb) & 15)) return fail(MERLIN_EINVAL, "obs_rgb must be 16-byte aligned");
  DeviceGuard guard(h->cfg.device);
  EnvParams p = base_params(h);
  p.reset_mask = mask; p.obs_rgb = obs_rgb; p.obs_sym = obs_sym;
  order_streams(h, 0, static_cast<cudaStream_t>(stream));
  cudaError_t err = launch_env_reset(p, launch_ctx(h), static_cast<cudaStream_t>(stream));
  if (err != cudaSuccess) return launch_failed(h, err, "env reset launch", stream);
  h->launches += 1;
  h->was_reset = true;
  return MERLIN_OK;
}

static int step_common(merlin_env_t* h, const int64_t* actions, const merlin_policy_io_t* pol, uint8_t* obs_rgb,
                       uint8_t* obs_sym, float* reward, uint8_t* terminated, uint8_t* truncated,
                       const merlin_step_extras_t* extras, uint8_t* final_sym, void* stream) {
  if (!reward || !terminated || !truncated) return fail(MERLIN_EINVAL, "reward/terminated/truncated are required");
  if (!h->was_reset) return fail(MERLIN_ESTATE, "step before reset");
  if (obs_rgb && !h->has_atlas) return fail(MERLIN_ESTATE, "RGB observation requested before the tile atlas was set");
  if (obs_rgb && (reinterpret_cast<uintptr_t>(obs_rgb) & 15)) return fail(MERLIN_EINVAL, "obs_rgb must be 16-byte aligned");
  DeviceGuard guard(h->cfg.device);
  EnvParams p = base_params(h);
  p.actions = actions; p.obs_rgb = obs_rgb; p.obs_sym = obs_sym;
  p.reward = reward; p.terminated = terminated; p.truncated = truncated;
  p.final_sym = final_sym;
  if (extras) { p.out_ep_return = extras->episode_return; p.out_ep_length = extras->episode_length; p.out_stuck = extras->stuck; p.out_done = extras->done; }
  if (pol) {
    p.logits = pol->logits; p.value_in = pol->value; p.out_action = pol->action; p.out_logp = pol->logprob;
    p.out_value = pol->value_out; p.greedy = pol->greedy ? 1 : 0;
    p.logits_stride = pol->logits_stride > 0 ? pol->logits_stride : ((h->cfg.flags & MERLIN_F_SEVEN_ACTIONS) ? 7 : 3);
    p.value_stride = pol->value_stride > 0 ? pol->value_stride : 1;
    p.seed_lo = (uint32_t)h->sampler_seed; p.seed_hi = (uint32_t)(h->sampler_seed >> 32);
    p.rec_finished = pol->finished; p.rec_return = pol->first_return; p.rec_length = pol->first_length;
    p.rec_goal = pol->first_goal;
  }
  order_streams(h, 0, static_cast<cudaStream_t>(stream));
  cudaError_t err = launch_env_step(p, launch_ctx(h), static_cast<cudaStream_t>(stream));
  if (err != cudaSuccess) return launch_failed(h, err, "env step launch", stream);
  h->launches += 1;
  return MERLIN_OK;
}

int merlin_env_step(merlin_env_t* h, const int64_t* actions, uint8_t* obs_rgb, uint8_t* obs_sym, float* reward,
                    uint8_t* terminated, uint8_t* truncated, const merlin_step_extras_t* extras, void* stream) {
  if (!h) return fail(MERLIN_EINVAL, "null handle");
  if (!actions) return fail(MERLIN_EINVAL, "actions/reward/terminated/truncated are required");
  return step_common(h, actions, nullptr, obs_rgb, obs_sym, reward, terminated, truncated, extras, nullptr, stream);
}

int merlin_env_step_final(merlin_env_t* h, const int64_t* actions, uint8_t* obs_rgb, uint8_t* obs_sym, float* reward,
                          uint8_t* terminated, uint8_t* truncated, const merlin_step_extras_t* extras,
                          uint8_t* final_sym, void* stream) {
  if (!h) return fail(MERLIN_EINVAL, "null handle");
  if (!actions) return fail(MERLIN_EINVAL, "actions/reward/terminated/truncated are required");
  return step_common(h, actions, nullptr, obs_rgb, obs_sym, reward, terminated, truncated, extras, final_sym, stream);
}

static int check_policy_io(merlin_env_t* h, const merlin_policy_io_t* pol) {
  if (!pol || !pol->logits || !pol->action || !pol->logprob)
    return fail(MERLIN_EINVAL, "merlin_env_policy_step: logits, action and logprob are required");
  if (pol->value_out && !pol->value) return fail(MERLIN_EINVAL, "merlin_env_policy_step: value_out needs value");
  if (pol->logits_stride < 0 || pol->value_stride < 0) return fail(MERLIN_EINVAL, "merlin_env_policy_step: negative stride");
  if (pol->logits_stride > 0 && pol->logits_stride < ((h->cfg.flags & MERLIN_F_SEVEN_ACTIONS) ? 7 : 3))
    return fail(MERLIN_EINVAL, "merlin_env_policy_step: logits_stride smaller than the action count");
  if (pol->finished && (!pol->first_return || !pol->first_length || !pol->first_goal))
    return fail(MERLIN_EINVAL, "merlin_env_policy_step: the first-episode record needs all four arrays");
  return MERLIN_OK;
}

int merlin_env_policy_step(merlin_env_t* h, const merlin_policy_io_t* pol, uint8_t* obs_rgb, uint8_t* obs_sym,
                           float* reward, uint8_t* terminated, uint8_t* truncated, const merlin_step_extras_t* extras,
                           void* stream) {
  if (!h) return fail(MERLIN_EINVAL, "null handle");
  if (const int rc = check_policy_io(h, pol)) return rc;
  return step_common(h, nullptr, pol, obs_rgb, obs_sym, reward, terminated, truncated, extras, nullptr, stream);
}

int merlin_env_policy_step_final(merlin_env_t* h, const merlin_policy_io_t* pol, uint8_t* obs_rgb, uint8_t* obs_sym,
                                 float* reward, uint8_t* terminated, uint8_t* truncated,
                                 const merlin_step_extras_t* extras, uint8_t* final_sym, void* stream) {
  if (!h) return fail(MERLIN_EINVAL, "null handle");
  if (const int rc = check_policy_io(h, pol)) return rc;
  return step_common(h, nullptr, pol, obs_rgb, obs_sym, reward, terminated, truncated, extras, final_sym, stream);
}

int merlin_env_seed_sampler(merlin_env_t* h, uint64_t seed) {
  if (!h) return fail(MERLIN_EINVAL, "null handle");
  DeviceGuard guard(h->cfg.device);
  cudaError_t err = cudaDeviceSynchronize();  // no step may still be drawing
  if (err == cudaSuccess) err = cudaMemset(h->draws, 0, (size_t)h->cfg.n_envs * sizeof(uint32_t));
  if (err != cudaSuccess) return cuda_fail(err, "sampler reseed");
  h->sampler_seed = seed;
  return MERLIN_OK;
}

int merlin_env_rearm(merlin_env_t* h, void* stream) {
  if (!h) return fail(MERLIN_EINVAL, "null handle");
  DeviceGuard guard(h->cfg.device);
  cudaError_t err = cudaMemsetAsync(h->sched, 0, kSchedWords * sizeof(unsigned), static_cast<cudaStream_t>(stream));
  if (err != cudaSuccess) return cuda_fail(err, "scheduler rearm");
  return MERLIN_OK;
}

int merlin_env_render(merlin_env_t* h, const uint8_t* obs_sym, int64_t n_rows, const int64_t* index, int32_t m,
                      uint8_t* out, int32_t blocked, void* stream) {
  if (!h || !obs_sym || !out) return fail(MERLIN_EINVAL, "merlin_env_render: null argument");
  if (m < 0 || n_rows < 0) return fail(MERLIN_EINVAL, "merlin_env_render: negative size");
  if (!h->has_atlas) return fail(MERLIN_ESTATE, "frames requested before the tile atlas was set");
  if (reinterpret_cast<uintptr_t>(out) & 15) return fail(MERLIN_EINVAL, "out must be 16-byte aligned");
  if (!index && n_rows && m > n_rows) return fail(MERLIN_EINVAL, "merlin_env_render: more frames than observation rows");
  DeviceGuard guard(h->cfg.device);
  RenderParams p{};
  p.sym = obs_sym; p.index = index; p.out = out; p.M = m; p.n_rows = n_rows;
  p.atlas = blocked ? h->atlas_blocked : h->atlas;
  p.lut = blocked ? h->blit_lut_blocked : h->blit_lut;
  p.tile_present = h->tile_present;
  p.sched = render_sched(h);
  order_streams(h, 1, static_cast<cudaStream_t>(stream));
  cudaError_t err = launch_render(p, blocked != 0, h->sm_count, static_cast<cudaStream_t>(stream));
  if (err != cudaSuccess) return launch_failed(h, err, "render launch", stream);
  h->launches += 1;
  return MERLIN_OK;
}

int merlin_env_render_f32(merlin_env_t* h, const uint8_t* obs_sym, int64_t n_rows, const int64_t* index, int32_t m,
                          float* out, int32_t normalise, void* stream) {
  if (!h || !obs_sym || !out) return fail(MERLIN_EINVAL, "merlin_env_render_f32: null argument");
  if (m < 0 || n_rows < 0) return fail(MERLIN_EINVAL, "merlin_env_render_f32: negative size");
  if (!h->has_atlas) return fail(MERLIN_ESTATE, "frames requested before the tile atlas was set");
  if (reinterpret_cast<uintptr_t>(out) & 15) return fail(MERLIN_EINVAL, "out must be 16-byte aligned");
  if (normalise < 0 || normalise > 2) return fail(MERLIN_EINVAL, "merlin_env_render_f32: normalise must be 0, 1 or 2");
  if (!index && n_rows && m > n_rows) return fail(MERLIN_EINVAL, "merlin_env_render_f32: more frames than observation rows");
  DeviceGuard guard(h->cfg.device);
  RenderParams p{};
  p.sym = obs_sym; p.index = index; p.out_f32 = out; p.M = m; p.n_rows = n_rows;
  p.atlas = h->atlas_blocked;
  p.tile_present = h->tile_present;
  p.sched = render_sched(h);
  p.normalise = normalise;
  p.cap_tiles = h->n_present < 8 ? 8 : (h->n_present > kAtlasTiles ? kAtlasTiles : h->n_present);
  order_streams(h, 1, static_cast<cudaStream_t>(stream));
  cudaError_t err = launch_render_f32(p, h->sm_count, static_cast<cudaStream_t>(stream));
  if (err != cudaSuccess) return launch_failed(h, err, "render_f32 launch", stream);
  h->launches += 1;
  return MERLIN_OK;
}

int merlin_env_full_obs(merlin_env_t* h, uint8_t* out, void* stream) {
  if (!h || !out) return fail(MERLIN_EINVAL, "merlin_env_full_obs: null argument");
  if (!h->was_reset) return fail(MERLIN_ESTATE, "full observation requested before reset");
  DeviceGuard guard(h->cfg.device);
  EnvParams p = base_params(h);
  cudaError_t err = launch_full_obs(p, out, h->sm_count, static_cast<cudaStream_t>(stream));
  if (err != cudaSuccess) return cuda_fail(err, "full observation launch");
  h->launches += 1;
  return MERLIN_OK;
}

int merlin_env_state_ptrs(merlin_env_t* h, int32_t** state, uint8_t** cells, int32_t* cell_stride, float** episode_return) {
  if (!h) return fail(MERLIN_EINVAL, "null handle");
  if (state) *state = reinterpret_cast<int32_t*>(h->state);
  if (cells) *cells = h->cells;
  if (cell_stride) *cell_stride = h->cell_stride;
  if (episode_return) *episode_return = h->ep_return;
  return MERLIN_OK;
}

int merlin_env_read_state(merlin_env_t* h, int32_t* state, uint8_t* cells, float* episode_return) {
  if (!h) return fail(MERLIN_EINVAL, "null handle");
  if (cells && !h->cells) return fail(MERLIN_ESTATE, "grids are immutable: index the layout pool by state[e][2]");
  DeviceGuard guard(h->cfg.device);
  const size_t N = (size_t)h->cfg.n_envs;
  cudaError_t err = cudaDeviceSynchronize();
  if (err == cudaSuccess && state) err = cudaMemcpy(state, h->state, N * sizeof(int4), cudaMemcpyDeviceToHost);
  if (err == cudaSuccess && episode_return) err = cudaMemcpy(episode_return, h->ep_return, N * sizeof(float), cudaMemcpyDeviceToHost);
  if (err == cudaSuccess && cells) {
    const size_t HW = (size_t)h->cfg.width * h->cfg.height;
    err = cudaMemcpy2D(cells, HW, h->cells, h->cell_stride, HW, N, cudaMemcpyDeviceToHost);
  }
  if (err != cudaSuccess) return cuda_fail(err, "state read-back");
  return MERLIN_OK;
}

int merlin_env_write_state(merlin_env_t* h, const int32_t* state, const uint8_t* cells, const float* episode_return) {
  if (!h) return fail(MERLIN_EINVAL, "null handle");
  if (!h->was_reset) return fail(MERLIN_ESTATE, "write_state before the first reset");
  if (cells && !h->cells) return fail(MERLIN_ESTATE, "grids are immutable: an env's grid is the pool entry state[e][2] names");
  const size_t N = (size_t)h->cfg.n_envs;
  const int W = h->cfg.width, H = h->cfg.height;
  if (state) {
    for (size_t e = 0; e < N; ++e) {
      EnvState s{};
      unpack_state(state[4 * e], state[4 * e + 1], state[4 * e + 2], state[4 * e + 3], s);
      const int layout = s.layout < 0 ? ~s.layout : s.layout;
      if (s.x >= W || s.y >= H || layout >= h->n_layouts || s.step_count < 0 || s.step_count >= h->cfg.max_steps) {
        char msg[160];
        std::snprintf(msg, sizeof msg, "env %zu: state outside the grid / pool / episode (x %d y %d layout %d step_count %d)",
                      e, s.x, s.y, layout, s.step_count);
        return fail(MERLIN_EINVAL, msg);
      }
    }
  }
  DeviceGuard guard(h->cfg.device);
  cudaError_t err = cudaDeviceSynchronize();
  if (err == cudaSuccess && state) err = cudaMemcpy(h->state, state, N * sizeof(int4), cudaMemcpyHostToDevice);
  if (err == cudaSuccess && episode_return) err = cudaMemcpy(h->ep_return, episode_return, N * sizeof(float), cudaMemcpyHostToDevice);
  if (err == cudaSuccess && cells) {
    const size_t HW = (size_t)W * H;
    err = cudaMemcpy2D(h->cells, h->cell_stride, cells, HW, HW, N, cudaMemcpyHostToDevice);
  }
  if (err != cudaSuccess) return cuda_fail(err, "state write");
  return MERLIN_OK;
}

int merlin_env_bad_actions(merlin_env_t* h, uint64_t* count) {
  if (!h || !count) return fail(MERLIN_EINVAL, "null argument");
  DeviceGuard guard(h->cfg.device);
  unsigned long long v = 0;
  cudaError_t err = cudaMemcpy(&v, h->bad_actions, sizeof v, cudaMemcpyDeviceToHost);
  if (err != cudaSuccess) return cuda_fail(err, "bad-action counter read");
  *count = v;
  return MERLIN_OK;
}

int64_t merlin_env_launch_count(merlin_env_t* h) { return h ? h->launches : 0; }

const char* merlin_env_step_kernel(merlin_env_t* h, int rgb) {
  if (!h) return "";
  return step_kernel_name(
      select_step_kernel(h->cfg.n_envs, (rgb & 1) != 0, lean_config(h->cfg.flags), false, launch_ctx(h)));
}

const char* merlin_env_final_step_kernel(merlin_env_t* h, int rgb) {
  if (!h) return "";
  return step_kernel_name(
      select_step_kernel(h->cfg.n_envs, (rgb & 1) != 0, lean_config(h->cfg.flags), true, launch_ctx(h)));
}

static int check_kernel_choice(int choice, int lowest) {
  if (choice < lowest || choice > 7)
    return fail(MERLIN_EINVAL, "kernel choice must be 0 (auto), 1 (group), 2 (warp), 3 (tile), 4 (tile, TMA frame stores), 5 (symbolic-only), 6 (ordered groups) or 7 (four envs per warp)");
  return MERLIN_OK;
}
static int check_observation_path(int path, int lowest) {
  if (path < lowest || path > 2)
    return fail(MERLIN_EINVAL, "observation path must be 0 (automatic), 1 (per-cell form) or 2 (row-parallel form wherever built)");
  return MERLIN_OK;
}

int merlin_set_kernel_choice(int choice) {
  if (int rc = check_kernel_choice(choice, 0)) return rc;
  g_default_kernel_choice.store(choice);
  return MERLIN_OK;
}

int merlin_set_observation_path(int path) {
  if (int rc = check_observation_path(path, 0)) return rc;
  g_default_observation_path.store(path);
  return MERLIN_OK;
}

int merlin_env_set_kernel_choice(merlin_env_t* h, int choice) {
  if (!h) return fail(MERLIN_EINVAL, "null handle");
  if (int rc = check_kernel_choice(choice, -1)) return rc;
  h->kernel_choice = choice;
  return MERLIN_OK;
}

int merlin_env_set_observation_path(merlin_env_t* h, int path) {
  if (!h) return fail(MERLIN_EINVAL, "null handle");
  if (int rc = check_observation_path(path, -1)) return rc;
  h->observation_path = path;
  return MERLIN_OK;
}

int merlin_gae(const float* rew, const float* val, const float* done, const float* last_val, float* adv, float* ret,
               int32_t T, int32_t N, double gamma, double lam, void* stream) {
  if (!rew || !val || !done || !last_val || !adv || !ret) return fail(MERLIN_EINVAL, "merlin_gae: null pointer");
  if (T < 0 || N < 0) return fail(MERLIN_EINVAL, "merlin_gae: negative size");
  if (T == 0 || N == 0) return MERLIN_OK;
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0)
    return fail(MERLIN_ECUDA, "no CUDA device: libmerlin_b200 has no CPU fallback");
  cudaError_t err = launch_gae(rew, val, done, last_val, adv, ret, T, N, gamma, lam, static_cast<cudaStream_t>(stream));
  if (err != cudaSuccess) return cuda_fail(err, "gae launch");
  return MERLIN_OK;
}

uint8_t merlin_pack_cell(int type, int color, int state) {
  uint32_t t = (uint32_t)type & 0xf;
  if (t == 0) t = T_EMPTY;
  if (t == 4) t = state == 1 ? T_DOOR_CLOSED : (state == 2 ? T_DOOR_LOCKED : T_DOOR_OPEN);
  uint32_t c = (uint32_t)color & 7;
  if (t == T_GOAL) c = 1;                   // upstream Goal() is always green, Lava() red, None has no colour
  if (t == T_LAVA || t == T_EMPTY) c = 0;
  return (uint8_t)(t | (c << 4));
}

const char* merlin_last_error(void) { return g_last_error.c_str(); }
const char* merlin_version(void) { return "merlin_b200 0.1 (sm_100a)"; }

}  // extern "C"
