/* merlin_b200.h -- C ABI of the B200-native MERLIN rollout hot path (libmerlin_b200.so).
 *
 * The reference (borangundogan/PPO-2DGrid) has no FFI layer: its boundary for this path is the
 * Python API of gymnasium/minigrid environments.  Each entry point below states which reference
 * call it replaces (file:line are relative to the reference checkout):
 *
 *   merlin_env_create / destroy   gym.make(env_id, size=...) + wrapper stack
 *                                 src/scenario_creator/scenario_creator.py:35-57 ; constants from
 *                                 src/custom_envs/base_env.py:32-41 (max_steps = 4*size^2, view 7)
 *   merlin_env_upload_layouts     the result of MiniGridEnv.reset() -> _gen_grid()
 *                                 src/custom_envs/medium_hard_env.py:12-45 (and the four siblings)
 *   merlin_env_generate_layouts   the same `_gen_grid` routines run on the device (fresh layouts without a host pool)
 *   merlin_env_generate_seeded_layouts   env.reset(seed=s) -> _gen_grid() for a list of seeds, on the device: the
 *                                 `_gen_grid` routines fed by numpy's default_rng(s) stream, restated
 *   merlin_env_set_tile_atlas     Grid.render_tile cache used by RGBImgPartialObsWrapper
 *                                 (src/scenario_creator/scenario_creator.py:48, tile_size 8)
 *   merlin_env_reset              env.reset()   src/ppo.py:35,65,96 ; src/fomaml.py:63,92,184
 *   merlin_env_step               env.step(a)   src/ppo.py:76 ; src/fomaml.py:71 -- through
 *                                 ThreeActionWrapper (src/wrappers/three_action_wrapper.py:10-17),
 *                                 optionally StuckPenaltyWrapper (src/wrappers/stuck_penalty_wrapper.py:29-58)
 *   merlin_env_step_final / merlin_env_policy_step_final   the same two, also returning the observation of every
 *                                 terminal state before its auto-reset (src/ppo.py:76,93-96: env.step(a), then env.reset())
 *   merlin_env_policy_step        the whole rollout transition "act -> sample -> step -> store": Categorical(logits).sample(),
 *                                 .log_prob(a) (src/actor_critic.py:80-99 act()), env.step(a) and RolloutBuffer.add /
 *                                 the trajectory lists (src/ppo.py:70-86 ; src/fomaml.py:65-84) in ONE launch; with
 *                                 `greedy` + the first-episode record it is one step of the deterministic evaluation
 *                                 loops (ppo/ppo_train.py:43-69 ; src/sweep_checkpoints.py:58-78)
 *   merlin_env_render             RGBImgPartialObsWrapper.observation on stored symbolic observations (batched,
 *                                 gathered) -- the read side of a compact RolloutBuffer (src/rollout_buffer.py:3-32)
 *   merlin_env_render_f32         the same, written as the float32 `x / 255.0` tensor CNNFeatureExtractor.forward
 *                                 consumes (src/actor_critic.py:21), in the blocked layout of its first layer
 *   merlin_gae                    PPO.compute_gae src/ppo.py:107-120 ; FOMAML src/fomaml.py:116-123
 *
 * Conventions
 *   - Every function returns 0 on success and a negative MERLIN_E* code on failure;
 *     merlin_last_error() returns a thread-local message for the last failure.
 *   - All data pointers passed to reset/step/gae are CALLER-OWNED DEVICE pointers on the handle's
 *     device; the library neither frees nor retains them.  Upload functions take HOST pointers
 *     and copy.  Env state lives in device memory owned by the handle.
 *   - reset/step/gae are asynchronous on `stream` (a cudaStream_t passed as void*; NULL = the
 *     legacy default stream), allocate nothing, never synchronise, and may be captured in a CUDA graph.
 *   - A handle is not thread-safe: one caller thread per handle at a time.  Any number of handles may live in one
 *     process, on the same or on different devices, each driven by its own thread; nothing in the library is shared
 *     between handles except the two process-wide DEFAULTS of the tuning knobs below.
 *   - Launches of one handle are stream-ordered: reset/step (which own the env state) and the render calls draw work
 *     tickets from handle-owned counters.  On one stream nothing needs doing.  When a call arrives on a different
 *     stream than the previous call of its kind, the library orders the new stream after the old one with an event
 *     (eager launches only).  CUDA-graph replays are invisible to it: order a replay against eager calls on other
 *     streams yourself.  Consecutive render launches use different counters, so a render may overlap a step.
 *   - If a launch ever fails, the ticket counters are cleared on the failing call's stream; merlin_env_rearm() does the
 *     same on demand (e.g. after a device-side fault was cleared by the application).
 *   - There is no CPU fallback: without a CUDA device every entry point fails with MERLIN_ECUDA.
 *
 * Packed cell code (1 byte per grid cell, row-major [y*W + x]):
 *   bits 3..0  type: minigrid OBJECT_TO_IDX (1 empty, 2 wall, 3 floor, 4 door OPEN, 5 key, 6 ball,
 *                    7 box, 8 goal, 9 lava) plus 11 = door CLOSED, 12 = door LOCKED
 *   bits 6..4  colour: minigrid COLOR_TO_IDX (0 red 1 green 2 blue 3 purple 4 yellow 5 grey)
 *   merlin_pack_cell(type, color, state) converts one minigrid (type, color, state) triple.
 */
#ifndef MERLIN_B200_H
#define MERLIN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MERLIN_OK 0
#define MERLIN_EINVAL (-1)   /* bad argument */
#define MERLIN_ECUDA (-2)    /* CUDA runtime / launch failure, or no device */
#define MERLIN_ESTATE (-3)   /* call out of order (e.g. step before layouts were uploaded) */
#define MERLIN_ENOMEM (-4)

/* flags for merlin_env_create */
#define MERLIN_F_AUTO_RESET 0x1u      /* finished envs restart inside step(); obs is the new episode's */
#define MERLIN_F_RESET_SAME 0x2u      /* restart on the SAME layout (FOMAML, src/fomaml.py:92); default: move on by n_envs pool
                                         slots modulo the pool size -- by ONE slot when the pool size divides n_envs, so that a
                                         restart always brings a different layout */
#define MERLIN_F_SEVEN_ACTIONS 0x4u   /* full MiniGrid action set 0..6; default: ThreeActionWrapper {left,right,forward} */
#define MERLIN_F_STUCK_PENALTY 0x8u   /* StuckPenaltyWrapper semantics (off in the reference's training path) */
#define MERLIN_F_EXPLORE_BONUS 0x10u  /* first-visit-per-episode bonus (not in the reference; builder-specified) */

typedef struct merlin_env merlin_env_t;

typedef struct merlin_env_config {
  int32_t device;          /* CUDA device ordinal */
  int32_t n_envs;          /* N >= 1 */
  int32_t width, height;   /* grid W,H in [3,255] */
  int32_t max_steps;       /* episode cap; 0 => 4*W*H (src/custom_envs/base_env.py:32-33) */
  int32_t view;            /* agent_view_size; only 7 is built */
  int32_t tile;            /* RGB tile size in pixels; only 8 is built */
  uint32_t flags;          /* MERLIN_F_* */
  int32_t stuck_max_stay;  /* default 3  (stuck_penalty_wrapper.py:12) */
  double stuck_penalty;    /* default -0.1 */
  double explore_bonus;    /* used when MERLIN_F_EXPLORE_BONUS */
} merlin_env_config_t;

/* Optional outputs of step(); any pointer may be NULL. */
typedef struct merlin_step_extras {
  float* episode_return;   /* [N] sum of rewards of the episode that ended this step, else 0.  Accumulated on the device in
                              float32, one rounding per step; the reference sums Python floats, i.e. float64
                              (src/ppo.py:88, src/fomaml.py:76).  A logging quantity only -- rewards themselves are formed in
                              float64 and rounded once, bit-identical to the reference's float32 buffer entries -- and the
                              two sums agree to ~1e-7 relative per step (tests/helpers.py compares them at 1e-5) */
  int32_t* episode_length; /* [N] its length, else 0 */
  uint8_t* stuck;          /* [N] info["stuck"] of StuckPenaltyWrapper */
  float* done;             /* [N] 1.0f where terminated or truncated, else 0.0f: the `done` the reference's learners store
                              (src/ppo.py:77,85; src/fomaml.py:72,81), written straight into a rollout row */
} merlin_step_extras_t;

void merlin_env_default_config(merlin_env_config_t* cfg);
int merlin_env_create(const merlin_env_config_t* cfg, merlin_env_t** out);
int merlin_env_destroy(merlin_env_t* h);

/* HOST inputs. cells: [n_layouts][H*W] packed codes; agent_xyd: [n_layouts][3] = x, y, dir. Replaces the pool and
 * resets the cursors (reset() must follow).  A pool of the SAME size is overwritten in place: device addresses, and
 * CUDA graphs captured over reset/step, stay valid; a different size reallocates and invalidates such graphs. */
int merlin_env_upload_layouts(merlin_env_t* h, const uint8_t* cells, const int32_t* agent_xyd, int32_t n_layouts);
/* Generate the pool ON THE DEVICE: n_layouts layouts of `difficulty` (the reference's `_gen_grid` routines,
 * src/custom_envs/{easy,medium,medium_hard,hard,hardest}_env.py, same algorithm and distributions) from a counter-based
 * generator keyed by (seed, first_number + slot).  NOT the layouts numpy's PCG64 stream would give for a reference seed:
 * use merlin_env_generate_seeded_layouts (or merlin_env_upload_layouts with host-generated layouts) to reproduce
 * `env.reset(seed=s)`.  Replaces the pool (in place when n_layouts is unchanged), resets the cursors.  Synchronous.
 * Sides below 6 (easy), 8 (hardest) or 4 (the others) are rejected. */
#define MERLIN_D_EASY 0
#define MERLIN_D_MEDIUM 1
#define MERLIN_D_MEDIUMHARD 2
#define MERLIN_D_HARD 3
#define MERLIN_D_HARDEST 4
int merlin_env_generate_layouts(merlin_env_t* h, int32_t difficulty, uint64_t seed, int64_t first_number,
                                int32_t n_layouts, void* stream);
/* Generate the pool ON THE DEVICE from reference seeds: slot i gets the layout of `env.reset(seed=seeds[i])` -> `_gen_grid`
 * (src/custom_envs/{easy,medium,medium_hard,hard,hardest}_env.py), byte for byte the layout the reference and
 * merlin_b200.layouts.generate build.  The routines are those of merlin_env_generate_layouts, fed by a restatement of
 * numpy's `default_rng(seed)`: SeedSequence -> PCG64 (XSL-RR), `Generator.integers` (Lemire's bounded method on the
 * buffered next_uint32) and `Generator.choice(replace=False)` (Floyd's algorithm + shuffle), pinned to numpy 2.3.5.
 * seeds: HOST u64[n_layouts].  Same pool semantics as merlin_env_generate_layouts: replaced in place when n_layouts is
 * unchanged (CUDA graphs captured over reset/step stay valid), cursors reset, the same atlas mask.  Synchronous.
 * Rejects what merlin_env_generate_layouts rejects, and hard below 5.
 * Where the reference's routine raises or never returns for a seed (a `place_obj` that exhausts max_tries=100, or 2^20
 * tries for max_tries=inf; `integers` or `choice` on an empty range), returns MERLIN_EINVAL and merlin_last_error()
 * names the first such seed.  The pool then holds the layouts of the other seeds and garbage in the failed slots:
 * reset() and set_cursors() fail with MERLIN_ESTATE (so does step(), which needs a reset) until the next successful
 * upload or generation; read_layouts() still works.  Graphs captured earlier are not stopped: do not replay them. */
int merlin_env_generate_seeded_layouts(merlin_env_t* h, int32_t difficulty, const uint64_t* seeds, int32_t n_layouts,
                                       void* stream);
/* Synchronous copy of the current pool to HOST buffers (either may be NULL): cells u8[n_layouts][H*W], agent_xyd
 * i32[n_layouts][3]; merlin_env_layout_count gives n_layouts. */
int merlin_env_read_layouts(merlin_env_t* h, uint8_t* cells, int32_t* agent_xyd);
int merlin_env_layout_count(merlin_env_t* h);
/* HOST input. tiles: [128][tile*tile*3] u8, indexed by packed code (0 = unseen cell, 10 = agent on empty,
 * 13/14/15 | colour<<4 = agent carrying key/ball/box). Required before an RGB observation is requested. */
int merlin_env_set_tile_atlas(merlin_env_t* h, const uint8_t* tiles, int32_t n_tiles);
/* HOST input or NULL. cursor[e] = pool index env e loads at its next reset. Default e % n_layouts. */
int merlin_env_set_cursors(merlin_env_t* h, const int32_t* cursor);

/* (Re)start envs. mask: DEVICE u8[N] or NULL (= all). obs_rgb: DEVICE u8[N][56][56][3] or NULL;
 * obs_sym: DEVICE u8[N][7][7][3] or NULL. Only restarted envs have their observation rows written. */
int merlin_env_reset(merlin_env_t* h, const uint8_t* mask, uint8_t* obs_rgb, uint8_t* obs_sym, void* stream);

/* One step of every env. actions: DEVICE i64[N]. reward f32[N], terminated/truncated u8[N] required.
 * Out-of-range actions are executed as `done` (no-op) and counted (merlin_env_bad_actions). */
int merlin_env_step(merlin_env_t* h, const int64_t* actions, uint8_t* obs_rgb, uint8_t* obs_sym, float* reward,
                    uint8_t* terminated, uint8_t* truncated, const merlin_step_extras_t* extras, void* stream);

/* Policy outputs in, sampled actions out: one rollout transition in one launch.  All pointers DEVICE.
 *   logits      f32[N][A]  the actor head's output (A = 3, or 7 with MERLIN_F_SEVEN_ACTIONS); row e starts at
 *                          logits + e * logits_stride floats (logits_stride = 0 means A: dense rows)
 *   value       f32[N]     the critic's output, or NULL; element e at value + e * value_stride (0 means 1: dense) -- the
 *                          strides let both heads be slices of ONE fused output matrix
 *   action      i64[N]     OUT the action taken (row t of the rollout's action tensor)
 *   logprob     f32[N]     OUT log_softmax(logits)[action] in float32: (l_a - max) - log(sum exp(l - max))
 *   value_out   f32[N]     OUT copy of `value` (row t of the rollout's value tensor), or NULL
 *   greedy      0: sample from Categorical(logits); 1: argmax (first maximum), the deterministic evaluation policy
 *   finished / first_return / first_length / first_goal   u8 / f32 / i32 / u8 [N], all or none: the first-episode record
 *               of an evaluation sweep ("freeze after done"): when env e ends an episode and finished[e] == 0, its return,
 *               length and goal flag are stored and finished[e] becomes 1; later episodes of that env change nothing.
 * Sampling is specified, not borrowed (torch's generator stream cannot be reproduced): u = Philox4x32-10(key = sampler
 * seed, counter = (env, number of draws env has made, 0, 0)) word 0, top 24 bits; the action is the first a with
 * cumsum(exp(l - max))[a] > u * sum, in float32, left to right.  Draw numbers advance by one per sampled step and are
 * reset by merlin_env_seed_sampler (synchronous).  The result does not depend on the kernel mapping. */
typedef struct merlin_policy_io {
  const float* logits;
  const float* value;
  int64_t* action;
  float* logprob;
  float* value_out;
  int32_t greedy;
  int32_t logits_stride;
  int32_t value_stride;
  uint8_t* finished;
  float* first_return;
  int32_t* first_length;
  uint8_t* first_goal;
} merlin_policy_io_t;
int merlin_env_policy_step(merlin_env_t* h, const merlin_policy_io_t* policy, uint8_t* obs_rgb, uint8_t* obs_sym,
                           float* reward, uint8_t* terminated, uint8_t* truncated, const merlin_step_extras_t* extras,
                           void* stream);
int merlin_env_seed_sampler(merlin_env_t* h, uint64_t seed);

/* Final observations of auto-reset episodes (gymnasium's info["final_obs"]; what the reference's env.step(a) returns
 * before its caller runs env.reset(), src/ppo.py:76,93-96).  merlin_env_step / merlin_env_policy_step plus
 *   final_sym   DEVICE u8[N][7][7][3]: when env e's episode ends in this step (terminated or truncated), row e receives
 *               the Grid.encode image of env e's state after the action and before the auto-reset -- byte for byte the
 *               obs_sym row the same step writes with MERLIN_F_AUTO_RESET off.  Rows of the other envs are not written.
 * Every other output, the env state and the draw counters are exactly those of the call without final_sym;
 * final_sym == NULL is that call.  Asynchronous, allocates nothing, capturable.  No RGB frame is written for the
 * terminal state: merlin_env_render(final_sym, index = the done rows) gives exactly the frame such a step would write.
 * Time-limit bootstrapping (reward += gamma * V(final observation) on truncated steps) needs this image. */
int merlin_env_step_final(merlin_env_t* h, const int64_t* actions, uint8_t* obs_rgb, uint8_t* obs_sym, float* reward,
                          uint8_t* terminated, uint8_t* truncated, const merlin_step_extras_t* extras,
                          uint8_t* final_sym, void* stream);
int merlin_env_policy_step_final(merlin_env_t* h, const merlin_policy_io_t* policy, uint8_t* obs_rgb,
                                 uint8_t* obs_sym, float* reward, uint8_t* terminated, uint8_t* truncated,
                                 const merlin_step_extras_t* extras, uint8_t* final_sym, void* stream);
/* Clear the in-kernel work-ticket counters of this handle on `stream` (see Conventions). */
int merlin_env_rearm(merlin_env_t* h, void* stream);

/* Frames from STORED symbolic observations -- RGBImgPartialObsWrapper.observation (get_frame(tile_size=8,
 * agent_pov=True), src/scenario_creator/scenario_creator.py:48) as a batch op with an optional row gather, so a
 * rollout can keep the 147-byte symbolic image per step and expand minibatches on read (the reference's RolloutBuffer
 * keeps 37 632 B of float32 per step, src/rollout_buffer.py:5).  obs_sym: DEVICE u8[n_rows][7][7][3] as step()/reset()
 * write them -- any image Grid.encode can produce renders correctly, also one stepped under an earlier layout pool or
 * showing objects the current pool does not hold; index: DEVICE i64[m] row numbers or NULL (= rows 0..m-1), a row
 * outside [0, n_rows) renders row 0; out: DEVICE u8[m][9408].
 * blocked = 0: u8[m][56][56][3], identical to the obs_rgb of step();  blocked = 1: u8[m][14][14][48], every 4x4 pixel
 * block contiguous with channel index c*16 + dy*4 + dx (space-to-depth; what the actor-critic's first layer reads). */
int merlin_env_render(merlin_env_t* h, const uint8_t* obs_sym, int64_t n_rows, const int64_t* index, int32_t m,
                      uint8_t* out, int32_t blocked, void* stream);

/* The same frames as the float32 tensor the policy's first layer reads: out: DEVICE f32[m][14][14][48] in the blocked
 * layout of merlin_env_render(blocked = 1).  normalise = 0: the pixel value 0..255 as float32;  1: pixel / 255.0f (IEEE
 * float32 division) and 2: pixel * (1.0f / 255.0f) -- the two things `x / 255.0` in CNNFeatureExtractor.forward
 * (src/actor_critic.py:21) evaluates to, in torch's CPU and CUDA kernels respectively (frames reach it as float32 through
 * PPO._obs_to_tensor, src/ppo.py:58-62, and RolloutBuffer.states, src/rollout_buffer.py:5).  One 37 632-byte streaming
 * write per frame instead of a u8 frame plus a cast pass plus a layout copy on the learner's minibatch path. */
int merlin_env_render_f32(merlin_env_t* h, const uint8_t* obs_sym, int64_t n_rows, const int64_t* index, int32_t m,
                          float* out, int32_t normalise, void* stream);

/* The fully observable symbolic observation of every env's CURRENT state -- minigrid FullyObsWrapper.observation,
 * which the reference selects with `observation.fully_observable: true` (src/scenario_creator/scenario_creator.py:45-46):
 * out: DEVICE u8[N][W][H][3], Grid.encode() indexed [x][y][type, colour, state], the agent's cell = (10, 0, agent_dir). */
int merlin_env_full_obs(merlin_env_t* h, uint8_t* out, void* stream);

/* State views: DEVICE pointers owned by the handle (valid until destroy). */
int merlin_env_state_ptrs(merlin_env_t* h, int32_t** state_xyds /* int4[N]: pose,step_count,cursor,stuck */,
                          uint8_t** cells /* [N][cell_stride] or NULL when grids are immutable */,
                          int32_t* cell_stride, float** episode_return);
/* Synchronous copy of the env state to HOST buffers (any may be NULL): state i32[N][4], cells u8[N][H*W]
 * (fails with MERLIN_ESTATE when grids are immutable -- index the pool by state[e][2] instead), episode_return f32[N]. */
int merlin_env_read_state(merlin_env_t* h, int32_t* state, uint8_t* cells, float* episode_return);
/* The inverse: overwrite the env state from HOST buffers laid out as merlin_env_read_state returns them (any may be NULL)
 * -- resume a saved rollout state, or start a benchmark from staggered episode clocks.  Synchronous; validated (poses
 * inside the grid, layout indices inside the pool, 0 <= step_count < max_steps).  The next step()'s observation is
 * computed from the new state; the observation buffers themselves are not touched. */
int merlin_env_write_state(merlin_env_t* h, const int32_t* state, const uint8_t* cells, const float* episode_return);
int merlin_env_bad_actions(merlin_env_t* h, uint64_t* count); /* synchronises the device */
int64_t merlin_env_launch_count(merlin_env_t* h);             /* kernels launched so far by this handle */
/* Per-handle tuning knobs: same values as the two process-wide knobs below, or -1 = follow the process-wide default
 * (the initial state of every handle). */
int merlin_env_set_kernel_choice(merlin_env_t* h, int choice);
int merlin_env_set_observation_path(merlin_env_t* h, int path);
/* Tuning/testing knob, process-wide DEFAULT for handles without their own setting: 0 = automatic (default), 1 = warp-owns-a-group kernel, 2 = warp-per-env kernel,
 * 3 = CTA-tile kernel, 4 = CTA-tile kernel with the frames stored by the TMA unit (cp.async.bulk), 5 = symbolic-only
 * kernel (writes no RGB frames; what "automatic" picks when obs_rgb is NULL), 6 = group kernel with in-order hand-out,
 * 7 = four envs per warp (steps of the three-action / no-shaping-wrapper configuration with RGB frames; anything else
 * asked of it runs kernel 2).
 * All kernels produce identical results for the outputs they write; "automatic" never picks 4, 6 or 7 (measured slower). */
int merlin_set_kernel_choice(int choice);
/* Tuning/testing knob, process-wide DEFAULT for handles without their own setting: how gen_obs is computed.  0 = automatic (default): the symbolic-only kernel works
 * on seven window cells per 64-bit register (csrc/obs_swar.cuh; grids at least 7 wide), the frame kernels cell by cell
 * (csrc/env_logic.cuh) -- the faster choice for each, measured;  1 = cell by cell everywhere;  2 = the row-parallel form
 * in every kernel that has it (symbolic-only, tile, ordered).  Identical results. */
int merlin_set_observation_path(int path);
/* Name of the kernel merlin_env_step launches for this handle (rgb != 0: with an RGB observation). */
const char* merlin_env_step_kernel(merlin_env_t* h, int rgb);
/* The same for merlin_env_step_final / merlin_env_policy_step_final with a final_sym buffer (kernel choice 7 runs the
 * warp-per-env kernel there). */
const char* merlin_env_final_step_kernel(merlin_env_t* h, int rgb);

/* GAE + returns over a time-major [T][N] rollout (all DEVICE f32). done = terminated|truncated as 0/1.
 * adv[t] = delta_t + gamma*lam*(1-done_t)*adv[t+1]; ret = val + adv.  fp32, unfused, reference op order.
 * The outputs must not alias the inputs (rows are re-read after later rows have been written). */
int merlin_gae(const float* rew, const float* val, const float* done, const float* last_val, float* adv, float* ret,
               int32_t T, int32_t N, double gamma, double lam, void* stream);

uint8_t merlin_pack_cell(int type, int color, int state);
const char* merlin_last_error(void);
const char* merlin_version(void);

#ifdef __cplusplus
}
#endif
#endif /* MERLIN_B200_H */
