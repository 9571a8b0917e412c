"""GPU tests of final observations (run with -m gpu on a B200): `step(..., final_obs=...)` /
`policy_step(..., final_obs=...)` run the STEP = 3 / 4 instance of the step-kernel mapping a handle selects.

Every instance is driven at a batch size that selects it, proven launched from the profiler with all its template
arguments, and checked three ways each step:
  * side by side: a second handle steps the same pool with the same actions (or the same logits and sampler seed)
    WITHOUT final_sym; every output, the env state and the draw counters are bit-identical between the two;
  * final rows: the rows of the envs whose episode ended equal the oracle's terminal images (tests/final_obs_oracle.py, replaying
    the kernel's actions) bit for bit; every other row keeps its sentinel bytes, and guard rows surround the buffer;
  * the label `merlin_env_final_step_kernel` gives names the launched mapping."""
from __future__ import annotations

from collections import namedtuple

import numpy as np
import pytest
import torch
from torch.autograd import DeviceType
from torch.profiler import ProfilerActivity, profile

from final_obs_oracle import FinalObsOracle
from test_gpu_parity import _object_layouts
from test_gpu_policy_step_instances import _launched_key

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SENT = 0xA5        # sentinel byte of final_sym rows that must not be written
SEED = 0x9E3779B97F4A7C15

CONFIGS = {
    "lean": dict(n_actions=3),
    "lean_same": dict(n_actions=3, reset_mode="same"),
    "lean_manual": dict(n_actions=3, auto_reset=False),
    "seven": dict(n_actions=7),
    "seven_manual": dict(n_actions=7, auto_reset=False),
    "stuck": dict(n_actions=3, stuck_penalty=True),
    "explore": dict(n_actions=3, exploration_bonus=0.02),
    "seven_stuck_explore": dict(n_actions=7, stuck_penalty=True, stuck_max_stay=2, stuck_penalty_value=-0.25,
                                exploration_bonus=0.01, reset_mode="same"),
}

# One row per final-observation mapping: the launched kernel (base name, template arguments with "S" for STEP), kernel
# choice, observation path, RGB frames or symbolic only, configuration, batch size as a function of the SM count, and
# the label merlin_env_final_step_kernel gives.  Thresholds as in test_gpu_policy_step_instances.py; kernel choice 7
# (the quad kernel) runs the warp kernel for these steps.
Row = namedtuple("Row", "kernel args choice path rgb cfg n label")
ROWS = [
    Row("env_kernel", ("4", "S"), 1, 0, True, "seven", lambda s: 1000, "env_kernel<4,true>"),
    Row("env_kernel", ("8", "S"), 1, 0, True, "lean", lambda s: 64 * s + 5, "env_kernel<8,true>"),
    Row("env_kernel", ("16", "S"), 1, 0, True, "stuck", lambda s: 128 * s + 3, "env_kernel<16,true>"),
    Row("env_kernel", ("32", "S"), 1, 0, True, "lean_same", lambda s: 256 * s + 7, "env_kernel<32,true>"),
    Row("env_kernel_tile", ("8", "S", "false"), 3, 1, True, "explore", lambda s: 2000, "env_kernel_tile<8,true>"),
    Row("env_kernel_tile", ("8", "S", "true"), 3, 2, True, "seven", lambda s: 1500, "env_kernel_tile<8,true>"),
    Row("env_kernel_tile", ("16", "S", "false"), 3, 0, True, "lean_manual", lambda s: 64 * s + 1,
        "env_kernel_tile<16,true>"),
    Row("env_kernel_tile", ("16", "S", "true"), 3, 2, True, "seven_stuck_explore", lambda s: 64 * s + 100,
        "env_kernel_tile<16,true>"),
    Row("env_kernel_tile_tma", ("S",), 4, 0, True, "seven", lambda s: 3000, "env_kernel_tile_tma<true>"),
    Row("env_kernel_ordered", ("S", "false"), 6, 0, True, "lean_same", lambda s: 2500, "env_kernel_ordered<true>"),
    Row("env_kernel_ordered", ("S", "true"), 6, 2, True, "explore", lambda s: 2600, "env_kernel_ordered<true>"),
    Row("env_kernel_sym", ("S", "false"), 5, 1, False, "seven_manual", lambda s: 5000, "env_kernel_sym<true>"),
    Row("env_kernel_sym", ("S", "true"), 5, 0, False, "lean", lambda s: 20000, "env_kernel_sym<true>"),
    Row("env_kernel_warp", ("S", "false", "false"), 2, 0, True, "seven_manual", lambda s: 1000, "env_kernel_warp<true>"),
    Row("env_kernel_warp", ("S", "false", "true"), 2, 0, False, "lean", lambda s: 3000, "env_kernel_warp<true>"),
    Row("env_kernel_warp", ("S", "true", "true"), 2, 0, True, "lean", lambda s: 6000, "env_kernel_warp<true>"),
    Row("env_kernel_warp", ("S", "true", "false"), 2, 0, True, "stuck", lambda s: 4500, "env_kernel_warp<true>"),
    Row("env_kernel_warp", ("S", "false", "true"), 7, 0, True, "lean_manual", lambda s: 3001, "env_kernel_warp<true>"),
]
Case = namedtuple("Case", "row step")
CASES = [Case(r, s) for r in ROWS for s in (3, 4)]


def _case_id(c):
    name = c.row.kernel[len("env_kernel"):].lstrip("_") or "group"
    return f"{name}<{','.join(str(c.step) if a == 'S' else a for a in c.row.args)}>-choice{c.row.choice}"


def _key(c):
    return c.row.kernel, tuple(str(c.step) if a == "S" else a for a in c.row.args)


def _np(x):
    return x.detach().cpu().numpy()


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def pools():
    from merlin_b200 import codes, layouts
    cells, agent = layouts.generate("mediumhard", 16, range(4200, 4264))
    objects = _object_layouts(np.random.default_rng(3), 96, 11)   # lava, doors, keys, balls, boxes
    return {"merlin": (codes.unpack_to_encoding(cells, 16, 16), agent), "objects": objects}


def _final_rows(N, T=1):
    """[T + 2, N, 7, 7, 3] sentinel buffer: rows 1..T are handed to the kernel, rows 0 and T + 1 are guard bands."""
    return torch.full((T + 2, N, 7, 7, 3), SENT, dtype=torch.uint8, device=DEV)


class _Pair:
    """Two handles on one pool, `a` stepping with final_sym and `b` without, and the oracle replaying a's actions."""

    def __init__(self, pool, N, cfg, rgb, choice=0, path=0, max_steps=7, stagger=True):
        from merlin_b200 import BatchedMerlinEnv
        enc, agent = pool
        kw = dict(CONFIGS[cfg])
        self.N, self.A, self.rgb = N, kw["n_actions"], rgb
        self.manual = not kw.get("auto_reset", True)
        self.a, self.b = (BatchedMerlinEnv(N, enc=enc, agent=agent, max_steps=max_steps, device=DEV, want_rgb=rgb,
                                           **kw) for _ in range(2))
        for env in (self.a, self.b):
            env.set_kernel_choice(choice)
            env.set_observation_path(path)
            env.reset(frames=rgb)
            env.seed_sampler(SEED)
        self.ref = FinalObsOracle(N, enc, agent, max_steps=max_steps, want_rgb=False, **kw)
        self.ref.reset()
        if stagger:   # every step ends about N / max_steps episodes by truncation
            for env in (self.a, self.b):
                env.stagger_episode_clocks(seed=N)
            self.ref.stepc[:] = self.a.state_raw()[0][:, 1]
        self.heads = torch.zeros((2, N, self.A), device=DEV)
        z = lambda dt: torch.zeros(N, dtype=dt, device=DEV)
        self.recs = [{"finished": z(torch.bool), "first_return": z(torch.float32), "first_length": z(torch.int32),
                      "first_goal": z(torch.bool)} for _ in range(2)]
        self.ios = [env.make_policy_io(self.heads[0], self.heads[1, :, 0], record=rec)
                    for env, rec in zip((self.a, self.b), self.recs)]
        self.bufs = [env.make_step_buffers() for env in (self.a, self.b)]

    def step(self, policy, rng, final):
        """One step of both handles; returns (actions, done mask, oracle info)."""
        if policy:
            self.heads.copy_(torch.from_numpy(rng.standard_normal((2, self.N, self.A)).astype(np.float32) * 2))
            ra = self.a.policy_step(self.ios[0], out=self.bufs[0], frames=self.rgb, final_obs=final)
            rb = self.b.policy_step(self.ios[1], out=self.bufs[1], frames=self.rgb)
            acts = _np(self.ios[0].action)
            assert torch.equal(self.ios[0].action, self.ios[1].action)
            assert torch.equal(self.ios[0].logprob, self.ios[1].logprob)
            assert torch.equal(self.ios[0].value_out, self.ios[1].value_out)
        else:
            acts = rng.integers(0, self.A, self.N)
            t = torch.as_tensor(acts, device=DEV)
            ra = self.a.step(t, out=self.bufs[0], frames=self.rgb, final_obs=final)
            rb = self.b.step(t, out=self.bufs[1], frames=self.rgb)
        assert ra[4]["final_obs_symbolic"] is final and "final_obs_symbolic" not in rb[4]
        if self.rgb:
            assert torch.equal(ra[0], rb[0])
        for k in ("obs_symbolic", "episode_return", "episode_length", "stuck", "done"):
            assert torch.equal(ra[4][k], rb[4][k]), k
        for x, y in zip(ra[1:4], rb[1:4]):
            assert torch.equal(x, y)
        _, rr, rte, rtr, rinfo = self.ref.step(acts)
        assert np.array_equal(_np(ra[1]), rr) and np.array_equal(_np(ra[2]), rte) and np.array_equal(_np(ra[3]), rtr)
        assert np.array_equal(_np(ra[4]["obs_symbolic"]), rinfo["obs_symbolic"])
        return acts, rte | rtr, rinfo

    def check_same_state(self):
        sa, ea = self.a.state_raw()
        sb, eb = self.b.state_raw()
        assert np.array_equal(sa, sb) and np.array_equal(ea, eb)
        if self.A == 7:
            assert np.array_equal(self.a.cells_numpy(), self.b.cells_numpy())
        for k in self.recs[0]:
            assert torch.equal(self.recs[0][k], self.recs[1][k]), k
        assert self.a.bad_actions() == 0 and self.b.bad_actions() == 0


def _check_final(buf, t, done, rinfo, manual, obs_sym):
    """Row t of the final-observation buffer after one step; guard rows and the rows of envs still running untouched."""
    got = _np(buf[t + 1])
    assert np.array_equal(got[done], rinfo["final_obs_symbolic"][done]), np.nonzero(~(got[done] == rinfo["final_obs_symbolic"][done]).all(axis=(1, 2, 3)))[0][:8]
    assert (got[~done] == SENT).all()
    if manual:   # without auto-reset the final row is the step's own observation
        assert np.array_equal(got[done], _np(obs_sym)[done])


@pytest.mark.parametrize("case", CASES, ids=[_case_id(c) for c in CASES])
def test_final_obs_instance(pools, case):
    row = case.row
    N = row.n(_sms())
    T = 10 if N <= 5000 else 5
    pool = pools["objects" if CONFIGS[row.cfg]["n_actions"] == 7 else "merlin"]
    rng = np.random.default_rng(N + case.step)
    pair = _Pair(pool, N, row.cfg, row.rgb, row.choice, row.path)
    assert pair.a.step_kernel(final=True) == "merlin::" + row.label
    buf = _final_rows(N, T)
    torch.cuda.synchronize()
    n_done = 0
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for t in range(T):
            _, done, rinfo = pair.step(case.step == 4, rng, buf[t + 1])
            torch.cuda.synchronize()
            _check_final(buf, t, done, rinfo, pair.manual, pair.a.obs_symbolic)
            n_done += int(done.sum())
            assert done.any(), t
        torch.cuda.synchronize()
    assert (_np(buf[0]) == SENT).all() and (_np(buf[T + 1]) == SENT).all()
    pair.check_same_state()
    keys = [_launched_key(e.name) for e in prof.events() if e.device_type == DeviceType.CUDA and "env_kernel" in e.name]
    final = [k for k in keys if k == _key(case)]
    assert len(final) == T, (keys[:6], _key(case))
    assert len(keys) == 2 * T, keys[:6]   # the other T launches: the same mapping without final observations


def _goal_room(size=16):
    """One layout: an empty walled room, the agent at (1, 1) facing the goal at (2, 1)."""
    enc = np.zeros((1, size, size, 3), np.uint8)
    enc[..., 0] = 1
    enc[0, 0, :] = enc[0, -1, :] = enc[0, :, 0] = enc[0, :, -1] = (2, 5, 0)
    enc[0, 2, 1] = (8, 1, 0)
    enc[0, 5, 5] = (9, 0, 0)
    return enc, np.array([[1, 1, 0]], np.int32)


@pytest.mark.parametrize("choice,N", [(2, 64), (3, 3000), (5, 5000)])
@pytest.mark.parametrize("policy", [False, True])
def test_goal_on_the_last_step_is_terminated_and_truncated(choice, N, policy):
    """An env whose clock stands at max_steps - 1 walks into the goal: terminated and truncated at once; its final row
    is the terminal image (the agent on the goal), the same as the oracle's."""
    pair = _Pair(_goal_room(), N, "lean", choice != 5, choice=choice, max_steps=9, stagger=False)
    st, epr = pair.a.state_raw()
    st[:, 1] = np.arange(N) % 9              # env e has run e % 9 steps: e % 9 == 8 ends on this step either way
    for env in (pair.a, pair.b):
        env.load_state_raw(st, epr)
    pair.ref.stepc[:] = st[:, 1]
    buf = _final_rows(N)
    if policy:   # every env moves forward: logits favour action 2
        pair.heads[0].copy_(torch.tensor([-50.0, -50.0, 50.0], device=DEV).expand(N, 3))
        pair.heads[1].zero_()
        ra = pair.a.policy_step(pair.ios[0], out=pair.bufs[0], frames=pair.rgb, final_obs=buf[1])
        pair.b.policy_step(pair.ios[1], out=pair.bufs[1], frames=pair.rgb)
        acts = _np(pair.ios[0].action)
        assert (acts == 2).all()
        _, rr, rte, rtr, rinfo = pair.ref.step(acts)
    else:
        acts = np.full(N, 2)
        ra = pair.a.step(torch.as_tensor(acts, device=DEV), out=pair.bufs[0], frames=pair.rgb, final_obs=buf[1])
        pair.b.step(torch.as_tensor(acts, device=DEV), out=pair.bufs[1], frames=pair.rgb)
        _, rr, rte, rtr, rinfo = pair.ref.step(acts)
    torch.cuda.synchronize()
    te, tr = _np(ra[2]), _np(ra[3])
    both = te & tr
    assert np.array_equal(both, np.arange(N) % 9 == 8) and np.array_equal(te, np.ones(N, bool))
    done = te | tr
    _check_final(buf, 0, done, rinfo, False, None)
    assert np.array_equal(_np(ra[1]), rr) and (rr > 0).all()
    pair.check_same_state()


@pytest.mark.parametrize("choice,N,cfg", [(2, 1000, "lean"), (3, 3000, "seven"), (1, 2000, "stuck")])
def test_rendered_final_rows_are_the_frames_of_a_handle_without_auto_reset(pools, choice, N, cfg):
    """render(final_sym, index=done) equals, bit for bit, the frame a handle with auto_reset=False wrote for the same
    step."""
    from merlin_b200 import BatchedMerlinEnv
    enc, agent = pools["objects" if CONFIGS[cfg]["n_actions"] == 7 else "merlin"]
    kw = dict(CONFIGS[cfg])
    auto = BatchedMerlinEnv(N, enc=enc, agent=agent, max_steps=7, device=DEV, **kw)
    manual = BatchedMerlinEnv(N, enc=enc, agent=agent, max_steps=7, device=DEV, **dict(kw, auto_reset=False))
    rng = np.random.default_rng(N)
    for env in (auto, manual):
        env.set_kernel_choice(choice)
        env.reset()
        env.stagger_episode_clocks(seed=1)
    seen = np.zeros(N, bool)
    for t in range(4):
        acts = torch.as_tensor(rng.integers(0, kw["n_actions"], N), device=DEV)
        _, _, te, tr, info = auto.step(acts, final_obs=True)
        mobs, _, _, _, _ = manual.step(acts)
        done = _np(te | tr)
        fresh = done & ~seen          # the manual handle's episode is the auto one's until the first end
        idx = torch.as_tensor(np.nonzero(fresh)[0], device=DEV)
        assert idx.numel() > 0, t
        assert torch.equal(auto.render(info["final_obs_symbolic"], index=idx), mobs[idx])
        seen |= done


def test_policy_step_final_graph_replay_equals_eager(pools):
    """policy_step_final into the rows of a [T, N, 7, 7, 3] buffer, captured in a CUDA graph and replayed twice, equals
    the same steps run eagerly on a second handle."""
    from merlin_b200 import BatchedMerlinEnv
    enc, agent = pools["merlin"]
    N, T = 4096, 6
    envs = [BatchedMerlinEnv(N, enc=enc, agent=agent, max_steps=9, device=DEV) for _ in range(2)]
    heads = torch.zeros((2, N, 3), device=DEV)
    bufs = [_final_rows(N, T) for _ in range(2)]
    ios, rows = [], []
    for env in envs:
        env.reset()
        # warm-up outside the capture: shared-memory attribute and occupancy of the instance
        env.policy_step(env.make_policy_io(heads[0], heads[1, :, 0]), final_obs=True)
        env.set_cursors(None)
        env.reset()
        env.stagger_episode_clocks(seed=5)
        env.seed_sampler(SEED)
        ios.append([env.make_policy_io(heads[0], heads[1, :, 0]) for _ in range(T)])
        rows.append([env.make_step_buffers() for _ in range(T)])
    g_env, e_env = envs
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for t in range(T):
            g_env.policy_step(ios[0][t], out=rows[0][t], final_obs=bufs[0][t + 1])
    rng = np.random.default_rng(0)
    for rep in range(2):
        heads.copy_(torch.from_numpy(rng.standard_normal((2, N, 3)).astype(np.float32)))
        for b in bufs:
            b.fill_(SENT)
        graph.replay()
        for t in range(T):
            e_env.policy_step(ios[1][t], out=rows[1][t], final_obs=bufs[1][t + 1])
        torch.cuda.synchronize()
        assert torch.equal(bufs[0], bufs[1]), rep
        for t in range(T):
            assert torch.equal(ios[0][t].action, ios[1][t].action), (rep, t)
            for k in ("reward", "terminated", "truncated", "done", "episode_length"):
                assert torch.equal(getattr(rows[0][t], k), getattr(rows[1][t], k)), (rep, t, k)
        done = torch.stack([r.done for r in rows[0]]).bool()
        assert done.any(dim=1).all()
        assert (bufs[0][1:T + 1][~done] == SENT).all()
    assert np.array_equal(g_env.state_raw()[0], e_env.state_raw()[0])


# ---- PPO: bootstrapping truncated episodes -------------------------------------------------------------------------
def _ppo_env(N):
    from merlin_b200 import BatchedMerlinEnv, codes, layouts
    cells, agent = layouts.generate("mediumhard", 16, range(9000, 9064))
    return BatchedMerlinEnv(N, enc=codes.unpack_to_encoding(cells, 16, 16), agent=agent, max_steps=11, device=DEV,
                            want_symbolic=True)


@pytest.mark.parametrize("storage", ["rgb", "symbolic"])
@pytest.mark.parametrize("graph", [False, True])
def test_ppo_bootstrap_truncated(storage, graph):
    """bootstrap_truncated=False rolls out bit for bit what a PPO without the option does.  With True, rewards differ
    only where a step truncated an episode without terminating it, and there by gamma * V, V = the critic's value of
    the frame of the oracle's terminal image (the oracle replays the rollout's actions)."""
    from src.ppo import PPO
    N, T = 512, 24
    runs = {}
    for opt in (None, False, True):
        torch.manual_seed(0)
        env = _ppo_env(N)
        kw = {} if opt is None else dict(bootstrap_truncated=opt)
        agent = PPO(env, batch_size=N * T, minibatch_size=1000, update_epochs=1, use_cuda_graph=graph,
                    obs_storage=storage, **kw)
        env.seed_sampler(123)
        agent.collect_rollouts()
        b = agent.buffer
        runs[opt] = (agent, env, b.rewards.clone(), b.actions.clone(), b.dones.clone(), b.values.clone(),
                     b.logprobs.clone())
    base, off, on = runs[None], runs[False], runs[True]
    for x, y in zip(base[2:], off[2:]):
        assert torch.equal(x, y)
    for x, y in zip(base[3:], on[3:]):
        assert torch.equal(x, y)
    agent, env = on[0], on[1]
    mask = (agent._truncated & ~agent._terminated)
    assert mask.any() and (agent._terminated & agent._truncated).sum() < mask.sum()
    assert torch.equal(on[2][~mask], base[2][~mask])
    # oracle replay of the kernel's actions: its terminal images, rendered and valued by the critic
    from merlin_b200 import codes, layouts
    cells, ag = layouts.generate("mediumhard", 16, range(9000, 9064))
    ref = FinalObsOracle(N, codes.unpack_to_encoding(cells, 16, 16), ag, max_steps=11, want_rgb=False)
    ref.reset()
    acts = _np(on[3])
    finals = np.zeros((T, N, 7, 7, 3), np.uint8)
    for t in range(T):
        _, _, rte, rtr, rinfo = ref.step(acts[t])
        assert np.array_equal(rtr & ~rte, _np(mask[t])), t
        finals[t] = rinfo["final_obs_symbolic"]
    m = _np(mask)
    sym = torch.as_tensor(finals[m], device=DEV)
    with torch.no_grad():
        v = agent.ac(env.render(sym, blocked=True, dtype=torch.float32))[1].float()
    want = base[2][mask] + agent.gamma * v
    got = on[2][mask]
    assert torch.allclose(got, want, rtol=1e-5, atol=1e-6), (got - want).abs().max()
    assert not torch.equal(got, base[2][mask])

