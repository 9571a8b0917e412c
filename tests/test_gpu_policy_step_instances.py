"""GPU tests of every policy-step kernel instance (run with -m gpu on a B200).

`merlin_env_policy_step` (act -> sample -> step -> store in one launch) runs the STEP = 2 instance of the step-kernel
mapping the handle selects; those instances are separate code from the STEP = 1 ones the parity suites check.  Each of
the 19 is driven here at a batch size that selects it (computed from the device's SM count, as
test_gpu_kernel_selection.py does), under the flags training uses, and proven launched from the profiler with all its
template arguments.  Every step is checked two ways:

  * env half: the oracle replays the kernel's own actions (`io.action`); rewards, flags, episode statistics, symbolic
    observations and frames are bit-exact;
  * sampler half: the uniforms are restated (oracle/sampler.py, draw number = sampled steps since `seed_sampler`); the
    action equals the float32 restatement wherever the draw is more than 1e-5 from a CDF boundary, and for EVERY env is
    one the float64 distribution allows, with its log-probability within float32 rounding of log_softmax in float64.

No assertion is statistical: softmax frequencies have their own tests."""
from __future__ import annotations

import re
from collections import namedtuple

import numpy as np
import pytest
import torch
from torch.autograd import DeviceType
from torch.profiler import ProfilerActivity, profile

import helpers
from oracle import fast, sampler
from test_gpu_parity import _object_layouts

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SEED = 0x9E3779B97F4A7C15            # the high word of the key matters
SEED_HI = SEED ^ (0x5A5A5A5A << 32)  # differs from SEED in the high word only
SENT_ACT, SENT_F = -7, -1234.5       # guard-band sentinels around the bound rollout rows

CONFIGS = {
    "lean": dict(n_actions=3),
    "seven": dict(n_actions=7),
    "stuck": dict(n_actions=3, stuck_penalty=True),
    "explore": dict(n_actions=3, exploration_bonus=0.02),
    "seven_stuck_explore": dict(n_actions=7, stuck_penalty=True, stuck_max_stay=2, stuck_penalty_value=-0.25,
                                exploration_bonus=0.01),
}

# One row per STEP = 2 instance: the launched kernel (base name, template arguments), the kernel choice and observation
# path that select it, RGB frames or symbolic only, the env configuration, the batch size as a function of the SM
# count, and whether the logits are bound as a [N, 8] slice instead of the [2, N, A] head tensor.
#   group G: the largest of 32 / 16 / 8 with N / G >= 8 x SMs, else 4; tile T = 16 from N >= SMs x 4 x 16;
#   SWAR (row-parallel observation): path 2 in the frame kernels, path 0 or 2 in the symbolic-only kernel;
#   warp PDL: RGB and N >= 4096, LEAN: the lean configuration and N <= 12 288; quad PDL: N >= 16 384.
Case = namedtuple("Case", "kernel args choice path rgb cfg n wide")
CASES = [
    Case("env_kernel", ("4", "2"), 1, 0, True, "seven", lambda s: 1000, False),
    Case("env_kernel", ("8", "2"), 1, 0, True, "lean", lambda s: 64 * s + 5, True),
    Case("env_kernel", ("16", "2"), 1, 0, True, "stuck", lambda s: 128 * s + 3, False),
    Case("env_kernel", ("32", "2"), 1, 0, True, "lean", lambda s: 256 * s + 7, False),
    Case("env_kernel_tile", ("8", "2", "false"), 3, 1, True, "explore", lambda s: 2000, False),
    Case("env_kernel_tile", ("8", "2", "true"), 3, 2, True, "seven", lambda s: 1500, True),
    Case("env_kernel_tile", ("16", "2", "false"), 3, 0, True, "lean", lambda s: 64 * s + 1, False),
    Case("env_kernel_tile", ("16", "2", "true"), 3, 2, True, "seven_stuck_explore", lambda s: 64 * s + 100, False),
    Case("env_kernel_tile_tma", ("2",), 4, 0, True, "seven", lambda s: 3000, False),
    Case("env_kernel_ordered", ("2", "false"), 6, 0, True, "lean", lambda s: 2500, False),
    Case("env_kernel_ordered", ("2", "true"), 6, 2, True, "explore", lambda s: 2600, True),
    Case("env_kernel_sym", ("2", "false"), 5, 1, False, "seven", lambda s: 5000, True),
    Case("env_kernel_sym", ("2", "true"), 5, 0, False, "lean", lambda s: 20000, False),
    Case("env_kernel_warp", ("2", "false", "false"), 2, 0, True, "seven", lambda s: 1000, False),
    Case("env_kernel_warp", ("2", "false", "true"), 2, 0, False, "lean", lambda s: 3000, False),
    Case("env_kernel_warp", ("2", "true", "true"), 2, 0, True, "lean", lambda s: 6000, True),
    Case("env_kernel_warp", ("2", "true", "false"), 2, 0, True, "stuck", lambda s: 4500, False),
    Case("env_kernel_quad", ("2", "false"), 7, 0, True, "lean", lambda s: 3001, False),
    Case("env_kernel_quad", ("2", "true"), 7, 0, True, "lean", lambda s: 16385, True),
]


def _case_id(c):
    return f"{c.kernel[len('env_kernel'):].lstrip('_') or 'group'}<{','.join(c.args)}>"


def _np(x):
    return x.detach().cpu().numpy()


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _launched_key(name):
    """(base name, all template arguments) of a launched kernel, from its demangled or its mangled name; booleans read
    "true" / "false" either way."""
    m = re.search(r"merlin::(\w+)<([^>]*)>", name)
    if m:
        return m.group(1), tuple(a.strip() for a in m.group(2).split(","))
    m = re.search(r"_ZN6merlin(\d+)", name)
    rest = name[m.end():]
    ident = rest[:int(m.group(1))]
    args = re.match(r"I((?:L[ib]\d+E)+)E", rest[len(ident):]).group(1)
    return ident, tuple({"b1": "true", "b0": "false"}.get(k + v, v) for k, v in re.findall(r"L([ib])(\d+)E", args))


def _step_arg(key):
    """STEP of a launched instance: 0 masked reset, 1 step, 2 policy step (after G or T in the group and tile kernels)."""
    base, args = key
    return args[1] if base in ("env_kernel", "env_kernel_tile") else args[0]


def _assert_policy_steps_launched(prof, case, n_policy_steps):
    """Every policy step launched exactly the case's instance; the only other step-kernel launches are resets."""
    keys = [_launched_key(e.name) for e in prof.events() if e.device_type == DeviceType.CUDA and "env_kernel" in e.name]
    policy = [k for k in keys if _step_arg(k) == "2"]
    assert all(_step_arg(k) == "0" for k in keys if _step_arg(k) != "2"), keys
    assert len(policy) == n_policy_steps, (len(policy), n_policy_steps)
    assert set(policy) == {(case.kernel, case.args)}, set(policy)


@pytest.fixture(scope="module")
def pools():
    from merlin_b200 import codes, layouts
    cells, agent = layouts.generate("mediumhard", 16, range(4200, 4264))
    merlin = (codes.unpack_to_encoding(cells, 16, 16), agent)
    objects = _object_layouts(np.random.default_rng(3), 96, 11)   # lava, doors, keys, balls, boxes
    return {"merlin": merlin, "objects": objects}


def _logits(rng, N, A):
    """A seeded mix of rows: scales 0.1, 2 and 20, exact ties, a -inf action, a forward / pickup / toggle bias with
    seven actions, and about 1 % non-finite rows (NaN, +inf, all -inf).  Returns (logits f32[N, A], finite-row mask)."""
    l = (rng.standard_normal((N, A)) * rng.choice([0.1, 2.0, 20.0], (N, 1))).astype(np.float32)
    if A == 7:
        l[:, [2, 3, 5]] += 1.5
    tie = rng.random(N) < 0.08
    l[tie, A - 1] = l[tie].max(axis=1)                     # the last action ties the row's maximum
    tie_all = rng.random(N) < 0.04
    l[tie_all] = np.round(l[tie_all, :1])                   # every action equal
    masked = rng.random(N) < 0.1
    l[masked, rng.integers(0, A, int(masked.sum()))] = -np.inf
    bad = rng.random(N) < 0.01
    kind = rng.integers(0, 3, N)
    col = rng.integers(0, A, N)
    for e in np.nonzero(bad)[0]:
        if kind[e] == 2:
            l[e] = -np.inf
        else:
            l[e, col[e]] = np.nan if kind[e] == 0 else np.inf
    finite = ~(np.isnan(l).any(axis=1) | np.isposinf(l).any(axis=1) | np.isneginf(l).all(axis=1))
    return l, finite


def _check_sampler(L, finite, a, lp, seed, draw):
    """Sampler half of one step: actions `a` / log-probabilities `lp` the kernel wrote for logits `L`, draw `draw`."""
    N, A = L.shape
    assert ((a >= 0) & (a < A)).all()
    ract, _, margin = sampler.sample_batch(L, seed, np.full(N, draw))
    safe = finite & (margin > 1e-5)
    assert np.array_equal(a[safe], ract[safe]), np.nonzero(a[safe] != ract[safe])[0][:10]
    u = sampler.uniform_batch(seed, np.arange(N), draw)
    _check_allowed(L[finite], a[finite], lp[finite], u[finite])


def _check_allowed(L, a, lp, u):
    n = np.arange(len(a))
    _, logp64, allowed = sampler.reference_f64(L, u)
    assert allowed[n, a].all(), np.nonzero(~allowed[n, a])[0][:10]
    assert not np.isneginf(L[n, a]).any()
    _check_logp(L, a, lp, logp64)


def _check_logp(L, a, lp, logp64):
    n = np.arange(len(a))
    l64 = L.astype(np.float64)
    mx = l64.max(axis=1)
    lse = np.log(np.exp(l64 - mx[:, None]).sum(axis=1))
    err = np.abs(lp.astype(np.float64) - logp64[n, a])
    assert (err <= 2e-6 + 4 * 2.0 ** -24 * (np.abs(l64[n, a] - mx) + np.abs(lse))).all(), err.max()


class _Run:
    """One handle of a case, its oracle, and the policy-head tensors bound the way training binds them."""

    def __init__(self, case, pool, N, max_steps):
        from merlin_b200 import BatchedMerlinEnv
        enc, agent = pool
        cfg = CONFIGS[case.cfg]
        self.case, self.N, self.A, self.rgb = case, N, cfg["n_actions"], case.rgb
        self.env = BatchedMerlinEnv(N, enc=enc, agent=agent, max_steps=max_steps, device=DEV, want_rgb=case.rgb,
                                    episode_stats=True, **cfg)
        self.env.set_kernel_choice(case.choice)
        self.env.set_observation_path(case.path)
        self.ref = fast.OracleVecEnv(N, enc, agent, max_steps=max_steps, want_rgb=case.rgb, **cfg)
        obs, sym = self.env.reset(frames=case.rgb)
        robs, rsym = self.ref.reset()
        assert np.array_equal(_np(sym), rsym)
        if case.rgb:
            assert np.array_equal(_np(obs), robs)
        # logits and value: strided views of one [2, N, A] head tensor (src/ppo.py), or logits as a [N, 8] slice
        self.heads = torch.zeros((2, N, self.A), device=DEV)
        self.wide = torch.zeros((N, 8), device=DEV)
        self.logits = self.wide[:, :self.A] if case.wide else self.heads[0]
        self.value = self.heads[1, :, 0]
        z = lambda dt: torch.zeros(N, dtype=dt, device=DEV)
        self.rec = {"finished": z(torch.bool), "first_return": z(torch.float32), "first_length": z(torch.int32),
                    "first_goal": z(torch.bool)}
        self.book = {"finished": np.zeros(N, bool), "first_return": np.zeros(N, np.float32),
                     "first_length": np.zeros(N, np.int32), "first_goal": np.zeros(N, bool)}
        self.steps = 0

    def load(self, rng):
        L, finite = _logits(rng, self.N, self.A)
        V = rng.standard_normal(self.N).astype(np.float32)
        self.logits.copy_(torch.from_numpy(L))
        self.value.copy_(torch.from_numpy(V))
        return L, finite, V

    def step(self, io, frames_now):
        """One policy step, its env half checked against the oracle's replay; returns the actions taken."""
        self.env.policy_step(io, frames=self.rgb)
        self.steps += 1
        a = _np(io.action)
        A = self.A
        assert ((a >= 0) & (a < A)).all()
        self.ref.want_rgb = self.rgb and frames_now
        robs, rr, rte, rtr, rinfo = self.ref.step(a)
        env = self.env
        t = self.steps
        assert np.array_equal(_np(env.reward), rr), t
        assert np.array_equal(_np(env.terminated), rte) and np.array_equal(_np(env.truncated), rtr), t
        assert np.array_equal(_np(env.episode_return), rinfo["episode_return"]), t
        assert np.array_equal(_np(env.episode_length), rinfo["episode_length"]), t
        assert np.array_equal(_np(env.stuck), rinfo["stuck"]), t
        assert np.array_equal(_np(env.done), (rte | rtr).astype(np.float32)), t
        assert np.array_equal(_np(env.obs_symbolic), rinfo["obs_symbolic"]), t
        if self.rgb and frames_now:
            assert np.array_equal(_np(env.obs), robs), t
        # the first-episode record, kept in Python (the bookkeeping src/evaluation.py used to do)
        b = self.book
        first = (rinfo["episode_length"] > 0) & ~b["finished"]
        b["first_return"] = np.where(first, rinfo["episode_return"], b["first_return"])
        b["first_length"] = np.where(first, rinfo["episode_length"], b["first_length"])
        b["first_goal"] |= first & rte & (rinfo["reward_env"] > 0)
        b["finished"] |= first
        return a

    def check_record(self):
        for k, v in self.book.items():
            assert np.array_equal(_np(self.rec[k]), v), k

    def check_end(self):
        assert np.array_equal(self.env.pose_numpy(), helpers.get_pose(self.ref))
        if self.A == 7:
            from merlin_b200 import codes
            W = self.ref.W
            got = codes.unpack_to_encoding(self.env.cells_numpy(), W, W)
            want = np.stack([self.ref.gt, self.ref.gc, self.ref.gs], axis=-1).reshape(self.N, W, W, 3).transpose(0, 2, 1, 3)
            assert np.array_equal(got, want)
        assert self.env.bad_actions() == 0


def _rows(T, N, dtype, sentinel):
    """T rollout rows between one guard row on each side."""
    return torch.full((T + 2, N), sentinel, dtype=dtype, device=DEV)


@pytest.mark.parametrize("case", CASES, ids=[_case_id(c) for c in CASES])
def test_policy_step_instance_env_half_and_sampler_half(pools, case):
    N = case.n(_sms())
    T = 24 if N <= 5000 else (12 if N <= 20000 else 8)
    every = 1 if N <= 5000 else 3
    rng = np.random.default_rng(N)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        # ---- sampled run on the MERLIN pool, outputs landing in rollout rows, first-episode record bound ----------
        run = _Run(case, pools["merlin"], N, max_steps=7)
        env = run.env
        acts, lps, vals = _rows(T, N, torch.int64, SENT_ACT), _rows(T, N, torch.float32, SENT_F), _rows(T, N, torch.float32, SENT_F)
        ios = [env.make_policy_io(run.logits, run.value, action=acts[t + 1], logprob=lps[t + 1], value_out=vals[t + 1],
                                  record=run.rec) for t in range(T)]
        env.seed_sampler(SEED)
        kept = []
        n_done = 0
        for t in range(T):
            L, finite, V = run.load(rng)
            a = run.step(ios[t], frames_now=t % every == 0 or t == T - 1)
            n_done += int(_np(env.done).sum())
            lp, v = _np(lps[t + 1]), _np(vals[t + 1])
            _check_sampler(L, finite, a, lp, SEED, draw=t)
            assert np.array_equal(v, V), t                      # value_out = value[e * stride], bit for bit
            kept.append((a.copy(), lp.copy(), v.copy()))
            assert bool((acts[t + 2:] == SENT_ACT).all()) and bool((acts[0] == SENT_ACT).all()), t
            assert bool((lps[t + 2:] == SENT_F).all()) and bool((lps[0] == SENT_F).all()), t
            assert bool((vals[t + 2:] == SENT_F).all()) and bool((vals[0] == SENT_F).all()), t
        for t, (a, lp, v) in enumerate(kept):                   # no later step wrote into an earlier row
            assert np.array_equal(_np(acts[t + 1]), a) and np.array_equal(_np(lps[t + 1]), lp, equal_nan=True)
            assert np.array_equal(_np(vals[t + 1]), v), t
        assert n_done > 0
        run.check_record()
        run.check_end()
        n_steps = T
        del run, acts, lps, vals, ios

        # ---- greedy run with the record on an object pool (lava ends episodes without a goal) ----------------------
        run = _Run(case, pools["objects"], N, max_steps=9)
        env = run.env
        env.seed_sampler(SEED)
        gio = env.make_policy_io(run.logits, run.value, greedy=True, record=run.rec)
        for t in range(12):
            L, finite, V = run.load(rng)
            a = run.step(gio, frames_now=t % every == 0)
            assert np.array_equal(a[finite], np.argmax(L[finite], axis=1)), t   # first maximum, ties included
            u0 = np.zeros(int(finite.sum()))
            _, logp64, _ = sampler.reference_f64(L[finite], u0)
            _check_logp(L[finite], a[finite], _np(gio.logprob)[finite], logp64)
            assert np.array_equal(_np(gio.value_out), V), t
            if t == 1:  # a masked reset (the STEP = 0 kernel) between policy steps
                mask = np.arange(N) % 5 == 0
                env.reset(torch.as_tensor(mask, device=DEV), frames=case.rgb)
                _, rsym = run.ref.reset(mask)
                assert np.array_equal(_np(env.obs_symbolic), rsym)
        assert run.book["finished"].all()
        run.check_record()
        lava = run.book["finished"] & ~run.book["first_goal"] & (run.book["first_length"] < 9)
        assert lava.any()   # first episodes that terminated without reaching the goal (lava): the goal flag is read

        # ---- draw counter: greedy steps, masked and automatic resets did not advance it; seed_sampler restarts it ----
        sio = env.make_policy_io(run.logits, run.value)

        def sampled(seed, draw):
            L, finite, _ = run.load(rng)
            a = run.step(sio, frames_now=False)
            _check_sampler(L, finite, a, _np(sio.logprob), seed, draw)
            return L, finite, a

        sampled(SEED, 0)
        sampled(SEED, 1)
        env.seed_sampler(SEED)
        sampled(SEED, 0)
        env.seed_sampler(SEED_HI)
        L, finite, a = sampled(SEED_HI, 0)
        ract, _, _ = sampler.sample_batch(L, SEED, np.zeros(N))
        assert not np.array_equal(a[finite], ract[finite])   # the high word of the key selects the stream
        run.check_end()
        n_steps += 12 + 4
        torch.cuda.synchronize()
    _assert_policy_steps_launched(prof, case, n_steps)


GRAPH_CASES = [c for c in CASES if c.kernel in ("env_kernel_warp", "env_kernel_quad") and c.args[1] == "true"
               and c.cfg == "lean"]


@pytest.mark.parametrize("case", GRAPH_CASES, ids=[_case_id(c) for c in GRAPH_CASES])
def test_policy_step_graph_replay_at_pdl_sizes(pools, case):
    """Four policy steps of a PDL instance captured in a CUDA graph and replayed three times: each replay draws fresh
    actions (draw number 4 x replay + step) and steps the envs bit-exactly.  The case is a row of CASES: the batch size
    and flags that test_policy_step_instance_env_half_and_sampler_half proves launch the PDL instance."""
    N = case.n(_sms())
    run = _Run(case, pools["merlin"], N, max_steps=7)
    env = run.env
    acts, lps, vals = _rows(4, N, torch.int64, SENT_ACT), _rows(4, N, torch.float32, SENT_F), _rows(4, N, torch.float32, SENT_F)
    ios = [env.make_policy_io(run.logits, run.value, action=acts[t + 1], logprob=lps[t + 1], value_out=vals[t + 1])
           for t in range(4)]
    bufs = [env.make_step_buffers() for _ in range(4)]
    obs = torch.empty((4, N, 56, 56, 3), dtype=torch.uint8, device=DEV)
    sym = torch.empty((4, N, 7, 7, 3), dtype=torch.uint8, device=DEV)
    # warm-up outside the capture: shared-memory attribute and occupancy of the instance
    env.policy_step(ios[0], out_obs=obs[0], out_symbolic=sym[0], out=bufs[0])
    torch.cuda.synchronize()
    env.set_cursors(None)   # the envs start over exactly as the fresh oracle does
    env.reset()
    ref = fast.OracleVecEnv(N, *pools["merlin"], max_steps=7)
    ref.reset()
    env.seed_sampler(SEED)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for t in range(4):
            env.policy_step(ios[t], out_obs=obs[t], out_symbolic=sym[t], out=bufs[t])
    rng = np.random.default_rng(N)
    for rep in range(3):
        L, finite, V = run.load(rng)
        acts.fill_(SENT_ACT); lps.fill_(SENT_F); vals.fill_(SENT_F)
        g.replay()
        torch.cuda.synchronize()
        for t in range(4):
            a = _np(acts[t + 1])
            _check_sampler(L, finite, a, _np(lps[t + 1]), SEED, draw=4 * rep + t)
            assert np.array_equal(_np(vals[t + 1]), V)
            robs, rr, rte, rtr, rinfo = ref.step(a)
            b = bufs[t]
            assert np.array_equal(_np(b.reward), rr) and np.array_equal(_np(b.terminated), rte), (rep, t)
            assert np.array_equal(_np(b.truncated), rtr) and np.array_equal(_np(b.done), (rte | rtr).astype(np.float32))
            assert np.array_equal(_np(b.episode_return), rinfo["episode_return"]), (rep, t)
            assert np.array_equal(_np(b.episode_length), rinfo["episode_length"]), (rep, t)
            assert np.array_equal(_np(sym[t]), rinfo["obs_symbolic"]), (rep, t)
            assert np.array_equal(_np(obs[t]), robs), (rep, t)
        for x, sent in ((acts, SENT_ACT), (lps, SENT_F), (vals, SENT_F)):
            assert bool((x[0] == sent).all()) and bool((x[5] == sent).all())
    assert np.array_equal(env.pose_numpy(), helpers.get_pose(ref))
    assert env.bad_actions() == 0
