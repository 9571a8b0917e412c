"""BatchedMerlinEnv -- N MiniGrid/MERLIN environments stepped by one fused CUDA kernel per call.

Host-side mirror of the reference env interface for the batched case: `reset()` / `step(actions)` with the
gymnasium 5-tuple, observations as the policy consumes them (`u8[N, 56, 56, 3]`, the
RGBImgPartialObsWrapper + ImgObsWrapper output of src/scenario_creator/scenario_creator.py:45-50), the
ThreeActionWrapper action set (src/wrappers/three_action_wrapper.py) and optional StuckPenaltyWrapper
semantics (src/wrappers/stuck_penalty_wrapper.py).  Everything stays on the device; this class only owns
tensors and forwards pointers through the C ABI (include/merlin_b200.h).
"""
from __future__ import annotations

import ctypes as C
import operator

import numpy as np
import torch

from . import _lib, codes, tiles

VIEW, TILE = 7, 8
OBS_SHAPE = (VIEW * TILE, VIEW * TILE, 3)
SYM_SHAPE = (VIEW, VIEW, 3)


class StepBuffers:
    """Caller-owned per-step outputs of `BatchedMerlinEnv.step` (all `[N]`, on the env's device).  Any of them may be
    a row of a rollout tensor (`StepBuffers(N, dev, reward=rewards[t], done=dones[t], ...)`): the step kernel then
    writes the rollout directly and no copy kernels are needed."""

    def __init__(self, num_envs, device, reward=None, terminated=None, truncated=None, episode_return=None,
                 episode_length=None, stuck=None, done=None):
        N, dev = num_envs, device

        def own(t, dtype):
            if t is None:
                return torch.empty(N, dtype=dtype, device=dev)
            if t.shape != (N,) or t.dtype != dtype or not t.is_contiguous() or t.device != torch.device(dev):
                raise ValueError(f"step output must be a contiguous {dtype} tensor of shape ({N},) on {dev}")
            return t

        self.reward = own(reward, torch.float32)
        self.terminated = own(terminated, torch.bool)
        self.truncated = own(truncated, torch.bool)
        self.episode_return = own(episode_return, torch.float32)
        self.episode_length = own(episode_length, torch.int32)
        self.stuck = own(stuck, torch.bool)
        self.done = own(done, torch.float32)
        self._extras = _lib.StepExtras(self.episode_return.data_ptr(), self.episode_length.data_ptr(),
                                       self.stuck.data_ptr(), self.done.data_ptr())


class _PolicyIO:
    """Tensors + the C struct of one fused policy transition (BatchedMerlinEnv.make_policy_io)."""
    __slots__ = ("logits", "value", "action", "logprob", "value_out", "record", "_c")


class BatchedMerlinEnv:
    def __init__(self, num_envs, cells=None, agent=None, *, enc=None, width=None, height=None, max_steps=None,
                 device="cuda", n_actions=3, auto_reset=True, reset_mode="next", stuck_penalty=False,
                 stuck_max_stay=3, stuck_penalty_value=-0.1, exploration_bonus=0.0, want_symbolic=True,
                 want_rgb=True, generate=None, generate_seeded=None, episode_stats=True):
        """cells: packed u8[L, H*W] (merlin_b200.codes) or `enc`: Grid.encode() arrays u8[L, W, H, 3];
        agent: i32[L, 3] = (x, y, dir).  Instead of a pool: `generate=(difficulty, seed, n_layouts)` generates one on
        the device (`generate_layouts`), `generate_seeded=(difficulty, seeds)` the reference's layouts of `seeds` on the
        device (`generate_seeded_layouts`); both need width/height.
        `reset_mode`: "next" advances each env's pool cursor by num_envs at
        every restart, modulo the pool size (by one slot when the pool size divides num_envs) (PPO: a fresh layout per episode), "same" replays the same layout (FOMAML task)."""
        self.device = torch.device(device)
        if self.device.type != "cuda" or not torch.cuda.is_available():
            raise RuntimeError("BatchedMerlinEnv needs a CUDA device (no CPU fallback)")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        if reset_mode not in ("next", "same"):
            raise ValueError("reset_mode must be 'next' or 'same'")
        if n_actions not in (3, 7):
            raise ValueError("n_actions must be 3 (ThreeActionWrapper) or 7 (full MiniGrid set)")
        if enc is not None:
            enc = np.asarray(enc)
            width, height = enc.shape[1], enc.shape[2]
            cells = codes.pack_encoding(enc)
        if generate is not None and generate_seeded is not None:
            raise ValueError("generate and generate_seeded are exclusive")
        if generate is not None or generate_seeded is not None:
            if width is None:
                raise ValueError("width/height are required with generate=(difficulty, seed, n_layouts) or "
                                 "generate_seeded=(difficulty, seeds)")
        elif cells is None or agent is None:
            raise ValueError("a layout pool (cells or enc, and agent), generate=(difficulty, seed, n_layouts) or "
                             "generate_seeded=(difficulty, seeds) is required")
        else:
            cells = np.ascontiguousarray(cells, dtype=np.uint8)
            if width is None:
                width = height = int(round(cells.shape[1] ** 0.5))
        self.num_envs, self.width, self.height = int(num_envs), int(width), int(height)
        # what evaluators need to rebuild this env's layouts for other seeds: the layout routine (known when the pool was
        # generated here or the env came from ScenarioCreator.create_batched_env, else None) and the grid size
        self.difficulty = next((g[0] for g in (generate, generate_seeded) if g is not None), None)
        self.size = self.width
        self.n_actions = n_actions
        self.want_symbolic, self.want_rgb = want_symbolic, want_rgb
        # episode_stats=False: step() skips the optional per-env outputs (episode return / length, stuck, done): the
        # gymnasium 5-tuple only, 17 bytes less written per env-step
        self.episode_stats = bool(episode_stats)
        self.auto_reset = auto_reset

        self._lib = _lib.load()
        cfg = _lib.EnvConfig()
        self._lib.merlin_env_default_config(C.byref(cfg))
        cfg.device = self.device.index
        cfg.n_envs, cfg.width, cfg.height = self.num_envs, self.width, self.height
        cfg.max_steps = int(max_steps) if max_steps else 0
        flags = 0
        flags |= _lib.F_AUTO_RESET if auto_reset else 0
        flags |= _lib.F_RESET_SAME if reset_mode == "same" else 0
        flags |= _lib.F_SEVEN_ACTIONS if n_actions == 7 else 0
        flags |= _lib.F_STUCK_PENALTY if stuck_penalty else 0
        flags |= _lib.F_EXPLORE_BONUS if exploration_bonus != 0.0 else 0
        cfg.flags = flags
        cfg.stuck_max_stay, cfg.stuck_penalty = int(stuck_max_stay), float(stuck_penalty_value)
        cfg.explore_bonus = float(exploration_bonus)
        self.max_steps = cfg.max_steps or 4 * self.width * self.height
        self._h = C.c_void_p()
        _lib.check(self._lib.merlin_env_create(C.byref(cfg), C.byref(self._h)))
        # the tile atlas is always installed (24 KB): `render` expands stored symbolic observations to frames even for
        # envs that never write frames themselves (want_rgb=False only skips the [N, 56, 56, 3] observation buffer)
        atlas = np.ascontiguousarray(tiles.build_atlas(TILE))
        _lib.check(self._lib.merlin_env_set_tile_atlas(self._h, atlas.ctypes.data, atlas.shape[0]))
        if generate is not None:
            self.generate_layouts(*generate)
        elif generate_seeded is not None:
            self.generate_seeded_layouts(*generate_seeded)
        else:
            self.upload_layouts(cells, agent)

        N, dev = self.num_envs, self.device
        self.obs = torch.empty((N,) + OBS_SHAPE, dtype=torch.uint8, device=dev) if want_rgb else None
        self.obs_symbolic = torch.empty((N,) + SYM_SHAPE, dtype=torch.uint8, device=dev) if want_symbolic else None
        self.reward = torch.empty(N, dtype=torch.float32, device=dev)
        self.terminated = torch.empty(N, dtype=torch.bool, device=dev)
        self.truncated = torch.empty(N, dtype=torch.bool, device=dev)
        self.episode_return = torch.empty(N, dtype=torch.float32, device=dev)
        self.episode_length = torch.empty(N, dtype=torch.int32, device=dev)
        self.stuck = torch.empty(N, dtype=torch.bool, device=dev)
        self.done = torch.empty(N, dtype=torch.float32, device=dev)
        self._extras = _lib.StepExtras(self.episode_return.data_ptr(), self.episode_length.data_ptr(),
                                       self.stuck.data_ptr(), self.done.data_ptr())
        self.final_obs_symbolic = None   # env-owned final-observation buffer (`step(..., final_obs=True)`)
        self.n_envs = self.num_envs
        # the in-kernel action sampler follows torch's seeding: key = hash(torch.initial_seed()) -- reproducible after
        # torch.manual_seed and different per rank when ranks seed differently; nothing is drawn from torch's generators.
        # Seeded here, never inside a (capturable) step; `seed_sampler` re-keys it.
        z = (int(torch.initial_seed()) + 0x9E3779B97F4A7C15) & (2**64 - 1)
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & (2**64 - 1)
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & (2**64 - 1)
        self.seed_sampler(z ^ (z >> 31))

    def make_step_buffers(self, **tensors):
        """A private set of per-step outputs (reward, flags, done, episode stats) for `step(..., out=...)`: lets a caller
        keep several steps in flight, or -- passing rows of its rollout tensors as keyword arguments -- have the step
        kernel write the rollout directly."""
        return StepBuffers(self.num_envs, self.device, **tensors)

    # ---- pool ------------------------------------------------------------------------------------
    def upload_layouts(self, cells, agent):
        cells = np.ascontiguousarray(cells, dtype=np.uint8)
        agent = np.ascontiguousarray(agent, dtype=np.int32).reshape(-1, 3)
        if cells.ndim != 2 or cells.shape[1] != self.width * self.height or cells.shape[0] != agent.shape[0]:
            raise ValueError(f"layout pool shape {cells.shape} does not match {self.width}x{self.height} / agent {agent.shape}")
        _lib.check(self._lib.merlin_env_upload_layouts(self._h, cells.ctypes.data, agent.ctypes.data, cells.shape[0]))
        self.n_layouts = cells.shape[0]
        self._pool_cells_host = cells

    DIFFICULTY_IDS = {"easy": 0, "medium": 1, "mediumhard": 2, "hard": 3, "hardest": 4}

    def generate_layouts(self, difficulty, seed, n_layouts, first_number=0):
        """Fill the pool on the device with `n_layouts` fresh layouts of `difficulty` (layouts number first_number..
        of the stream `seed`; same generators and distributions as merlin_b200.layouts, different random stream --
        not the reference's `reset(seed=s)` layouts).  Resets the cursors; call `reset()` afterwards."""
        if difficulty not in self.DIFFICULTY_IDS:
            raise ValueError(f"Unknown difficulty: {difficulty}")
        _lib.check(self._lib.merlin_env_generate_layouts(self._h, self.DIFFICULTY_IDS[difficulty], int(seed) & (2**64 - 1),
                                                         int(first_number), int(n_layouts), self._stream()))
        self.n_layouts = int(n_layouts)
        self._pool_cells_host = None

    def generate_seeded_layouts(self, difficulty, seeds):
        """Fill the pool on the device with the layouts of `env.reset(seed=s)` for every s in `seeds` (Python ints in
        [0, 2^64)): byte for byte what `merlin_b200.layouts.generate(difficulty, size, seeds)` builds on the host.
        Resets the cursors; call `reset()` afterwards.  Raises ValueError for a bad seed, an empty list, or a seed whose
        layout routine raises or never returns in the reference (the pool is then unusable until the next upload or
        generation)."""
        if difficulty not in self.DIFFICULTY_IDS:
            raise ValueError(f"Unknown difficulty: {difficulty}")
        if isinstance(seeds, (str, bytes)):
            raise ValueError("seeds must be an iterable of ints")
        try:
            seeds = [operator.index(s) for s in seeds]
        except TypeError as e:
            raise ValueError(f"seeds must be ints in [0, 2^64): {e}") from None
        if not seeds:
            raise ValueError("seeds is empty")
        bad = next((s for s in seeds if not 0 <= s < 2**64), None)
        if bad is not None:
            raise ValueError(f"seed {bad} is outside [0, 2^64)")
        arr = np.array(seeds, dtype=np.uint64)
        try:
            _lib.check(self._lib.merlin_env_generate_seeded_layouts(self._h, self.DIFFICULTY_IDS[difficulty],
                                                                    arr.ctypes.data, len(seeds), self._stream()))
        finally:
            self.n_layouts = int(self._lib.merlin_env_layout_count(self._h))
            self._pool_cells_host = None

    def layouts_numpy(self):
        """Host copy of the current pool: (cells u8[L, H*W], agent i32[L, 3])."""
        L = int(self._lib.merlin_env_layout_count(self._h))
        cells = np.empty((L, self.width * self.height), dtype=np.uint8)
        agent = np.empty((L, 3), dtype=np.int32)
        _lib.check(self._lib.merlin_env_read_layouts(self._h, cells.ctypes.data, agent.ctypes.data))
        return cells, agent

    def set_cursors(self, cursor=None):
        """cursor[e] = pool index env e loads at its next (full) reset; None = e % n_layouts."""
        if cursor is None:
            _lib.check(self._lib.merlin_env_set_cursors(self._h, None))
        else:
            cur = np.ascontiguousarray(cursor, dtype=np.int32)
            if cur.shape != (self.num_envs,):
                raise ValueError("cursor must have one entry per env")
            _lib.check(self._lib.merlin_env_set_cursors(self._h, cur.ctypes.data))

    # ---- stepping --------------------------------------------------------------------------------
    def _stream(self):
        # the raw handle of torch's current stream on this device (the private getter skips building a Stream object:
        # ~2 us per step, which matters for eager loops over small batches)
        raw = getattr(torch._C, "_cuda_getCurrentRawStream", None)
        if raw is not None:
            return raw(self.device.index)
        return torch.cuda.current_stream(self.device).cuda_stream

    def reset(self, mask=None, out_obs=None, out_symbolic=None, frames=True):
        """(Re)start all envs (mask=None) or those with mask[e] != 0.  Returns (obs_rgb, obs_symbolic).
        `frames=False`: no RGB frames for this call (the symbolic-only kernel runs; obs_rgb is None)."""
        obs = (out_obs if out_obs is not None else self.obs) if frames else None
        sym = out_symbolic if out_symbolic is not None else self.obs_symbolic
        mptr = None
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            mptr = mask.data_ptr()
        _lib.check(self._lib.merlin_env_reset(self._h, mptr, obs.data_ptr() if obs is not None else None,
                                              sym.data_ptr() if sym is not None else None, self._stream()))
        return obs, sym

    def _final_buffer(self, final_obs):
        """The u8[N, 7, 7, 3] tensor a step writes final observations into (`final_obs` of step / policy_step)."""
        if final_obs is True:
            if self.final_obs_symbolic is None:
                if torch.cuda.is_current_stream_capturing():
                    raise RuntimeError("final_obs=True allocates its buffer on first use: call it once before capture")
                self.final_obs_symbolic = torch.empty((self.num_envs,) + SYM_SHAPE, dtype=torch.uint8,
                                                      device=self.device)
            return self.final_obs_symbolic
        t = final_obs
        if (not torch.is_tensor(t) or tuple(t.shape) != (self.num_envs,) + SYM_SHAPE or t.dtype != torch.uint8
                or not t.is_contiguous() or t.device != self.device):
            raise ValueError(f"final_obs must be True or a contiguous torch.uint8 tensor of shape "
                             f"{(self.num_envs,) + SYM_SHAPE} on {self.device}")
        return t

    def step(self, actions, out_obs=None, out_symbolic=None, out=None, frames=True, final_obs=None):
        """actions: int64 CUDA tensor [N] (numpy/int lists are copied over).  Returns the gymnasium 5-tuple
        (obs u8[N,56,56,3], reward f32[N], terminated bool[N], truncated bool[N], info) with device tensors that
        are REUSED by the next call unless `out_obs` / `out_symbolic` point into caller storage (e.g. a rollout slot).
        `frames=False`: this call writes no RGB frames (obs is None; the symbolic-only kernel runs) -- for callers that
        expand the symbolic image themselves (`render(..., dtype=torch.float32)` straight into the policy's input).
        `final_obs`: a contiguous u8[N, 7, 7, 3] tensor on the env's device (e.g. a row of a [T, N, 7, 7, 3] rollout
        tensor), or True for an env-owned one.  Row e then receives the symbolic observation of env e's terminal state
        when its episode ends in this step -- before the auto-reset, as gymnasium's info["final_obs"] -- and is not
        written otherwise; `info["final_obs_symbolic"]` is that tensor.  Everything else is exactly what the call
        without it returns.  Frames of the terminal states: `render(info["final_obs_symbolic"], index=done_rows)`."""
        if not torch.is_tensor(actions):
            actions = torch.as_tensor(np.asarray(actions), dtype=torch.int64)
        if actions.device != self.device or actions.dtype != torch.int64 or not actions.is_contiguous():
            actions = actions.to(device=self.device, dtype=torch.int64).contiguous()
        if actions.numel() != self.num_envs:
            raise ValueError(f"expected {self.num_envs} actions, got {actions.numel()}")
        obs = (out_obs if out_obs is not None else self.obs) if frames else None
        sym = out_symbolic if out_symbolic is not None else self.obs_symbolic
        b = out if out is not None else self
        args = (obs.data_ptr() if obs is not None else None, sym.data_ptr() if sym is not None else None,
                b.reward.data_ptr(), b.terminated.data_ptr(), b.truncated.data_ptr(),
                C.byref(b._extras) if self.episode_stats else None)
        fin = None if final_obs is None else self._final_buffer(final_obs)
        if fin is None:
            _lib.check(self._lib.merlin_env_step(self._h, actions.data_ptr(), *args, self._stream()))
        else:
            _lib.check(self._lib.merlin_env_step_final(self._h, actions.data_ptr(), *args, fin.data_ptr(),
                                                       self._stream()))
        info = {"episode_return": b.episode_return, "episode_length": b.episode_length, "stuck": b.stuck,
                "done": b.done, "obs_symbolic": sym}
        if fin is not None:
            info["final_obs_symbolic"] = fin
        return obs, b.reward, b.terminated, b.truncated, info

    # ---- fused policy transition ------------------------------------------------------------------
    def seed_sampler(self, seed):
        """Key of the in-kernel action sampler (Philox4x32-10); resets every env's draw counter.  Synchronous."""
        _lib.check(self._lib.merlin_env_seed_sampler(self._h, int(seed) & (2**64 - 1)))

    def make_policy_io(self, logits, value=None, action=None, logprob=None, value_out=None, greedy=False, record=None):
        """Bind the tensors of one fused transition once (pointers are baked in; reuse the object every step or
        capture it in a CUDA graph).  `logits` f32[N, A], `value` f32[N]; outputs `action` i64[N], `logprob` f32[N],
        `value_out` f32[N] may be rows of rollout tensors (allocated here when None).  `record`: dict with tensors
        finished (bool/u8), first_return (f32), first_length (i32), first_goal (bool/u8), all [N]: first-episode record."""
        N, dev = self.num_envs, self.device

        def need(t, dtype, shape, name):
            if t is None:
                return torch.empty(shape, dtype=dtype, device=dev)
            ok_dtype = t.dtype == dtype or (dtype == torch.uint8 and t.dtype == torch.bool)
            if tuple(t.shape) != tuple(shape) or not ok_dtype or not t.is_contiguous() or t.device != dev:
                raise ValueError(f"{name} must be a contiguous {dtype} tensor of shape {tuple(shape)} on {dev}")
            return t

        def strided(t, cols, name):
            # [N, cols] (or [N]) float32 with unit inner stride and any row stride: a slice of a fused output matrix
            shape = (N, cols) if cols else (N,)
            if (t.dtype != torch.float32 or tuple(t.shape) != shape or t.device != dev
                    or (cols > 1 and t.stride(1) != 1) or (N > 1 and t.stride(0) < max(cols, 1))):
                raise ValueError(f"{name} must be float32 of shape {shape} on {dev} with unit inner stride")
            return t, int(t.stride(0))

        io = _PolicyIO()
        io.logits, ls = strided(logits, self.n_actions, "logits")
        io.value, vs = (None, 0) if value is None else strided(value, 0, "value")
        io.action = need(action, torch.int64, (N,), "action")
        io.logprob = need(logprob, torch.float32, (N,), "logprob")
        io.value_out = None if (value is None) else need(value_out, torch.float32, (N,), "value_out")
        io.record = None
        c = _lib.PolicyIO(io.logits.data_ptr(), io.value.data_ptr() if io.value is not None else None,
                          io.action.data_ptr(), io.logprob.data_ptr(),
                          io.value_out.data_ptr() if io.value_out is not None else None, 1 if greedy else 0, ls, vs,
                          None, None, None, None)
        if record is not None:
            io.record = {"finished": need(record["finished"], torch.uint8, (N,), "finished"),
                         "first_return": need(record["first_return"], torch.float32, (N,), "first_return"),
                         "first_length": need(record["first_length"], torch.int32, (N,), "first_length"),
                         "first_goal": need(record["first_goal"], torch.uint8, (N,), "first_goal")}
            c.finished, c.first_return = io.record["finished"].data_ptr(), io.record["first_return"].data_ptr()
            c.first_length, c.first_goal = io.record["first_length"].data_ptr(), io.record["first_goal"].data_ptr()
        io._c = c
        return io

    def policy_step(self, io, out_obs=None, out_symbolic=None, out=None, frames=True, final_obs=None):
        """One rollout transition in ONE launch: sample an action per env from `io.logits` (or argmax), store action /
        log-probability / value into `io`'s tensors, step every env and write the next observation.  Returns the same
        5-tuple as `step`; the action taken is `io.action`.  Replaces Categorical(logits).sample() + log_prob + env.step +
        the rollout stores of src/ppo.py:70-86 and src/fomaml.py:65-84.  `final_obs` as in `step`."""
        obs = (out_obs if out_obs is not None else self.obs) if frames else None
        sym = out_symbolic if out_symbolic is not None else self.obs_symbolic
        b = out if out is not None else self
        args = (obs.data_ptr() if obs is not None else None, sym.data_ptr() if sym is not None else None,
                b.reward.data_ptr(), b.terminated.data_ptr(), b.truncated.data_ptr(),
                C.byref(b._extras) if self.episode_stats else None)
        fin = None if final_obs is None else self._final_buffer(final_obs)
        if fin is None:
            _lib.check(self._lib.merlin_env_policy_step(self._h, C.byref(io._c), *args, self._stream()))
        else:
            _lib.check(self._lib.merlin_env_policy_step_final(self._h, C.byref(io._c), *args, fin.data_ptr(),
                                                              self._stream()))
        info = {"episode_return": b.episode_return, "episode_length": b.episode_length, "stuck": b.stuck,
                "done": b.done, "obs_symbolic": sym}
        if fin is not None:
            info["final_obs_symbolic"] = fin
        return obs, b.reward, b.terminated, b.truncated, info

    def set_kernel_choice(self, choice):
        """This env's step-kernel mapping (0 automatic .. 6, see merlin_b200.set_kernel_choice); -1 = follow the
        process-wide default again."""
        _lib.check(self._lib.merlin_env_set_kernel_choice(self._h, int(choice)))

    def set_observation_path(self, path):
        _lib.check(self._lib.merlin_env_set_observation_path(self._h, int(path)))

    def rearm(self):
        """Clear the in-kernel work-ticket counters (after an application-level recovery from a device fault)."""
        _lib.check(self._lib.merlin_env_rearm(self._h, self._stream()))

    def full_observation(self, out=None):
        """FullyObsWrapper's observation of every env's current state: u8[N, W, H, 3] (`Grid.encode()` indexed [x][y],
        the agent's cell = (10, 0, agent_dir))."""
        shape = (self.num_envs, self.width, self.height, 3)
        if out is None:
            out = torch.empty(shape, dtype=torch.uint8, device=self.device)
        elif tuple(out.shape) != shape or out.dtype != torch.uint8 or not out.is_contiguous():
            raise ValueError(f"out must be a contiguous uint8 tensor of shape {shape}")
        _lib.check(self._lib.merlin_env_full_obs(self._h, out.data_ptr(), self._stream()))
        return out

    def render(self, obs_symbolic, index=None, out=None, blocked=False, dtype=torch.uint8, normalise=False):
        """Frames from stored symbolic observations: `obs_symbolic` u8[R, 7, 7, 3] (any leading shape, contiguous),
        `index` optional int64[M] rows to render (a minibatch gather fused with the rendering).
        Returns u8[M, 56, 56, 3] (bit-identical to what `step` wrote for those states) or, with `blocked=True`,
        u8[M, 14, 14, 48] (4x4 pixel blocks, channel-major: the actor-critic's space-to-depth input).
        `dtype=torch.float32` (blocked only): f32[M, 14, 14, 48] holding the pixel values 0..255 (what
        CNNActorCritic takes) or the reference's `x / 255.0` (src/actor_critic.py:21): `normalise="divide"` (or True)
        = IEEE division, torch's CPU result; `normalise="reciprocal"` = x * (1/255), torch's CUDA result -- the
        first layer's input tensor written by the kernel itself, no cast or layout pass afterwards."""
        sym = obs_symbolic
        if sym.dtype != torch.uint8 or sym.device != self.device or not sym.is_contiguous():
            raise ValueError("obs_symbolic must be a contiguous uint8 tensor on the env's device")
        if dtype not in (torch.uint8, torch.float32):
            raise ValueError("dtype must be torch.uint8 or torch.float32")
        modes = {False: 0, None: 0, "none": 0, True: 1, "divide": 1, "reciprocal": 2}
        if normalise not in modes:
            raise ValueError("normalise must be False, True / 'divide' or 'reciprocal'")
        as_f32 = dtype == torch.float32
        if as_f32 and not blocked:
            raise ValueError("float32 frames are written in the blocked layout only (blocked=True)")
        rows = sym.numel() // (VIEW * VIEW * 3)
        if index is not None:
            if index.dtype != torch.int64 or index.device != self.device or not index.is_contiguous():
                index = index.to(device=self.device, dtype=torch.int64).contiguous()
            m = index.numel()
        else:
            m = rows
        shape = (m, 2 * VIEW, 2 * VIEW, 48) if blocked else (m,) + OBS_SHAPE
        if out is None:
            out = torch.empty(shape, dtype=dtype, device=self.device)
        elif (out.numel() != m * VIEW * TILE * VIEW * TILE * 3 or out.dtype != dtype or not out.is_contiguous()
              or out.device != self.device):
            raise ValueError(f"out must be a contiguous {dtype} tensor of m * 9408 elements on the env's device")
        if m == 0:
            return out
        idx_ptr = index.data_ptr() if index is not None else None
        if as_f32:
            _lib.check(self._lib.merlin_env_render_f32(self._h, sym.data_ptr(), rows, idx_ptr, m, out.data_ptr(),
                                                       modes[normalise], self._stream()))
        else:
            _lib.check(self._lib.merlin_env_render(self._h, sym.data_ptr(), rows, idx_ptr, m, out.data_ptr(),
                                                   1 if blocked else 0, self._stream()))
        return out

    # ---- state views (synchronous host copies; debugging / tests / gym adapter) ------------------
    def state_numpy(self):
        """Host copy of the packed per-env state: dict of x, y, dir, carry, step_count, layout, stay, episode_return."""
        a = np.empty((self.num_envs, 4), dtype=np.int32)
        epr = np.empty(self.num_envs, dtype=np.float32)
        _lib.check(self._lib.merlin_env_read_state(self._h, a.ctypes.data, None, epr.ctypes.data))
        pose = a[:, 0].astype(np.int64) & 0xFFFFFFFF
        stuck = a[:, 3].astype(np.int64) & 0xFFFFFFFF
        return {"x": (pose & 0xFF).astype(np.int32), "y": ((pose >> 8) & 0xFF).astype(np.int32),
                "dir": ((pose >> 16) & 3).astype(np.int32), "carry": ((pose >> 24) & 0x7F).astype(np.int32),
                "step_count": a[:, 1].copy(), "layout": a[:, 2].copy(), "stay": (stuck & 0xFFFF).astype(np.int32),
                "episode_return": epr}

    def state_raw(self):
        """Host copy of the packed state exactly as the device holds it: (i32[N, 4], episode_return f32[N]) -- what
        `load_state_raw` takes back (save / resume a rollout state)."""
        a = np.empty((self.num_envs, 4), dtype=np.int32)
        epr = np.empty(self.num_envs, dtype=np.float32)
        _lib.check(self._lib.merlin_env_read_state(self._h, a.ctypes.data, None, epr.ctypes.data))
        return a, epr

    def load_state_raw(self, state, episode_return=None, cells=None):
        """Overwrite the env state (synchronous, validated): `state` i32[N, 4] as `state_raw` returns it; column 1 is
        the episode clock `step_count`."""
        st = np.ascontiguousarray(state, dtype=np.int32)
        if st.shape != (self.num_envs, 4):
            raise ValueError("state must be int32[num_envs, 4]")
        epr = None if episode_return is None else np.ascontiguousarray(episode_return, dtype=np.float32)
        cl = None if cells is None else np.ascontiguousarray(cells, dtype=np.uint8)
        _lib.check(self._lib.merlin_env_write_state(self._h, st.ctypes.data, cl.ctypes.data if cl is not None else None,
                                                    epr.ctypes.data if epr is not None else None))

    def stagger_episode_clocks(self, seed=0):
        """Give every env a random episode clock in [0, max_steps): a batch that was reset together then truncates at
        the steady-state rate (N / max_steps envs per step) instead of all at once (benchmarks, SURVEY 8d)."""
        st, epr = self.state_raw()
        st[:, 1] = np.random.default_rng(seed).integers(0, self.max_steps, self.num_envs, dtype=np.int32)
        self.load_state_raw(st, epr)

    def pose_numpy(self):
        s = self.state_numpy()
        return np.stack([s["x"], s["y"], s["dir"], s["step_count"]], axis=1)

    def cells_numpy(self):
        """Host copy of every env's current grid as packed cells [N, H*W]."""
        if self.n_actions == 3:  # immutable grids: envs read the pool in place
            if self._pool_cells_host is None:
                self._pool_cells_host = self.layouts_numpy()[0]
            return self._pool_cells_host[self.state_numpy()["layout"]]
        out = np.empty((self.num_envs, self.width * self.height), dtype=np.uint8)
        _lib.check(self._lib.merlin_env_read_state(self._h, None, out.ctypes.data, None))
        return out

    def bad_actions(self):
        n = C.c_uint64()
        _lib.check(self._lib.merlin_env_bad_actions(self._h, C.byref(n)))
        return n.value

    def step_kernel(self, final=False):
        """Name of the CUDA kernel `step` launches for this batch size / observation mode (`final`: with final_obs)."""
        fn = self._lib.merlin_env_final_step_kernel if final else self._lib.merlin_env_step_kernel
        return fn(self._h, 1 if self.want_rgb else 0).decode()

    def launch_count(self):
        return int(self._lib.merlin_env_launch_count(self._h))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.merlin_env_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
