// env_kernels.cuh -- launch interface between the C ABI (capi.cu) and the kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/merlin_b200.h"
#include "env_logic.cuh"

namespace merlin {

constexpr int kThreads = 256;                 // 8 warps per CTA
constexpr int kWarps = kThreads / 32;
constexpr int kAtlasBytes = kAtlasTiles * kTileBytes;   // 24576
constexpr int kKindStride = 52;               // 49 tile kinds per env, padded: odd word stride -> conflict-free lanes
constexpr int kChunksPerLane = (kChunks + 31) / 32;     // 19

__host__ __device__ constexpr int warp_smem_bytes(int G) {
  return (G * kKindStride + G * kSymBytes + 15) & ~15;
}
__host__ __device__ constexpr int cta_smem_bytes(int G) { return kAtlasBytes + kWarps * warp_smem_bytes(G); }

struct EnvParams {
  // geometry / behaviour
  int N, W, H, max_steps, cell_stride, n_layouts, vis_words, stuck_max_stay;
  int cursor_stride;           // a restarting env moves on by this many pool slots: N mod L, or 1 when L divides N
  uint32_t flags;
  double stuck_penalty, explore_bonus;
  // handle-owned device state
  int4* state;                 // [N] pose | step_count | layout | stuck
  float* ep_return;            // [N] running episode return
  uint8_t* cells;              // [N][cell_stride] private grids, or nullptr when grids are immutable
  uint32_t* visited;           // [N][vis_words] per-episode visited bitmap, or nullptr
  const uint8_t* pool_cells;   // [L][cell_stride]
  const uint32_t* pool_agent;  // [L] x | y<<8 | dir<<16
  unsigned* sched;             // [2] tile ticket counter + finished-CTA counter of the tile kernel (self-resetting)
  const uint8_t* atlas;        // [128][192]
  const uint32_t* blit_lut;    // [kChunksPerLane][32] chunk -> (cell0, off0, cell1, off1), see chunk_lut()
  const uint32_t* tile_present;  // [4] device words; bit t set: atlas slot t can appear in a frame of this handle's pool
  unsigned long long* bad_actions;
  // caller-owned I/O
  const int64_t* actions;
  const uint8_t* reset_mask;
  uint8_t* obs_rgb;
  uint8_t* obs_sym;
  float* reward;
  uint8_t* terminated;
  uint8_t* truncated;
  float* out_ep_return;
  int32_t* out_ep_length;
  uint8_t* out_stuck;
  float* out_done;
  // policy I/O (merlin_env_policy_step): `logits` != nullptr replaces `actions` -- the action of env e is sampled in the
  // kernel from logits[e][0..n_actions) (or is their argmax when `greedy`) and stored with its log-probability
  const float* logits;         // [N][n_actions]
  const float* value_in;       // [N] or nullptr
  int64_t* out_action;         // [N]
  float* out_logp;             // [N]
  float* out_value;            // [N] or nullptr: copy of value_in (row t of a rollout's value tensor)
  uint32_t* draws;             // [N] handle-owned: how many actions env e has drawn (the Philox counter)
  uint32_t seed_lo, seed_hi;   // sampler key
  int greedy;
  int logits_stride, value_stride;   // in floats; rows of `logits` / elements of `value_in`
  // first-episode record (deterministic evaluation, "freeze after done"): when env e finishes an episode and
  // rec_finished[e] == 0, its return / length / terminated flag are stored and rec_finished[e] becomes 1
  uint8_t* rec_finished;       // [N] in/out, or nullptr
  float* rec_return;           // [N]
  int32_t* rec_length;         // [N]
  uint8_t* rec_goal;           // [N] 1 = the episode ended by termination with a positive reward (goal reached)
};

// Resident CTAs per SM of every kernel instance a handle has launched eagerly, keyed by the kernel's address (graph
// replays run no host code).  Filled on first use by resident_ctas (env_kernels_common.cuh); the step kernels have
// fewer than 50 instances.
struct OccupancyCache {
  static constexpr int kEntries = 64;
  const void* kernel[kEntries] = {};
  int ctas[kEntries] = {};
  int n = 0;
};

// Per-handle launch context: kernel choice, observation path and the occupancy cache live in the handle (a process may
// hold several handles on several devices, driven from different threads).
struct LaunchCtx {
  int sm_count;
  int kernel_choice;      // 0 = automatic, 1..7 as merlin_set_kernel_choice
  int observation_path;   // 0 = automatic, 1 = per-cell, 2 = row-parallel wherever built
  OccupancyCache* occ;
};

// kernel choice (merlin_set_kernel_choice)
enum KernelChoice : int {
  kChoiceAuto = 0,
  kChoiceGroup = 1,     // env_kernel<G>: a warp owns a group of G envs
  kChoiceWarp = 2,      // env_kernel_warp: a warp per env
  kChoiceTile = 3,      // env_kernel_tile<T>: a CTA owns a tile of T envs
  kChoiceTileTma = 4,   // env_kernel_tile_tma: the tile kernel with its frames stored through cp.async.bulk
  kChoiceSym = 5,       // env_kernel_sym: state phase only -- any RGB output pointer is ignored
  kChoiceOrdered = 6,   // env_kernel_ordered: the group kernel with groups handed out in order
  kChoiceQuad = 7,      // env_kernel_quad: four envs per warp; steps of the lean configuration with RGB frames --
                        // anything else asked of it runs kChoiceWarp
};
// observation path: 0 = automatic (row-parallel obs_swar.cuh in the symbolic-only kernel when W >= 7), 1 = per-cell
// everywhere, 2 = row-parallel in every kernel that has it (symbolic-only, tile, ordered)

// The lean configuration (the reference's own): three actions (=> immutable grids), no stuck penalty, no exploration
// bonus.  The quad kernel and the lean form of the warp kernel serve only this configuration.
inline bool lean_config(uint32_t flags) {
  return (flags & (MERLIN_F_SEVEN_ACTIONS | MERLIN_F_STUCK_PENALTY | MERLIN_F_EXPLORE_BONUS)) == 0;
}

// The step kernel a step of n_envs envs runs: `choice` is never kChoiceAuto, `size` is G (kChoiceGroup) or T
// (kChoiceTile) and 0 otherwise.  A reset sent to kChoiceQuad runs kChoiceWarp.
struct StepKernel {
  int choice;
  int size;
};
StepKernel select_step_kernel(int n_envs, bool rgb, bool lean, const LaunchCtx& ctx);
const char* step_kernel_name(StepKernel k);
cudaError_t launch_env_step(const EnvParams& p, const LaunchCtx& ctx, cudaStream_t stream);
cudaError_t launch_env_reset(const EnvParams& p, const LaunchCtx& ctx, cudaStream_t stream);
// Frames from stored symbolic observations (RGBImgPartialObsWrapper.observation as a batch op, with an optional
// row gather): out[m] = frame(sym[index ? index[m] : m]).  blocked = false: u8[M][56][56][3] as the env kernel writes
// them; blocked = true: u8[M][14][14][48], every 4x4 pixel block contiguous with channel index c*16 + dy*4 + dx (the
// layout the actor-critic's first layer consumes).  `atlas` / `lut` must be the pair matching `blocked`.
struct RenderParams {
  const uint8_t* sym;        // [*][147]
  const int64_t* index;      // [M] or nullptr
  uint8_t* out;              // [M][9408]
  const uint8_t* atlas;      // [128][192]
  const uint32_t* lut;       // [kChunksPerLane][32]
  const uint32_t* tile_present;  // [4] device words
  unsigned* sched;           // [2] in-order ticket counter + finished-CTA counter (self-resetting)
  int M;
  long long n_rows;          // rows of `sym` (index bound), 0 = unchecked
  // float32 variant only (launch_render_f32): blocked layout, `atlas` = the blocked u8 atlas
  float* out_f32;            // [M][14][14][48]
  int normalise;             // 0: the pixel value; 1: pixel / 255.0f (IEEE division); 2: pixel * (1.0f / 255.0f)
  int cap_tiles;             // atlas slots the float atlas in shared memory can hold (8..128)
  int frame_per_cta;         // set by launch_render_f32: 1 = few frames, one CTA renders one frame with all its warps
  int group_frames;          // set by launch_render: frames per work ticket of the u8 kernels
};
cudaError_t launch_render(const RenderParams& p, bool blocked, int sm_count, cudaStream_t stream);
cudaError_t launch_render_f32(const RenderParams& p, int sm_count, cudaStream_t stream);
// On-device layout generation (layout_kernels.cu): fills pool slots first_slot .. first_slot+count-1 with layouts number
// first_number .. of the stream `seed`; difficulty 0 easy, 1 medium, 2 mediumhard, 3 hard, 4 hardest.
cudaError_t launch_layouts(uint8_t* pool_cells, uint32_t* pool_agent, int cell_stride, int W, int H, int difficulty,
                           uint64_t seed, long long first_number, int first_slot, int count, int sm_count,
                           cudaStream_t stream);
// FullyObsWrapper.observation for every env: Grid.encode() of the current grid, u8[N][W][H][3] indexed [x][y][c],
// with the agent's cell replaced by (OBJECT_TO_IDX["agent"] = 10, COLOR_TO_IDX["red"] = 0, agent_dir).
cudaError_t launch_full_obs(const EnvParams& p, uint8_t* out, int sm_count, cudaStream_t stream);
cudaError_t launch_gae(const float* rew, const float* val, const float* done, const float* last_val, float* adv,
                       float* ret, int T, int N, double gamma, double lam, cudaStream_t stream);

}  // namespace merlin
