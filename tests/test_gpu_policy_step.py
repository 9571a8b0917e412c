"""GPU tests of merlin_env_policy_step -- the fused "act -> sample -> step -> store" transition -- and of the
multi-handle / multi-stream contract of the C ABI (run with -m gpu on a B200).

Sampling cannot be bit-compared with the reference (torch's generator stream is not reproducible by a fused kernel,
SURVEY section 7), so it is checked four ways: (1) the env half of the launch is replayed through the oracle with the
actions the kernel itself chose -- observations, rewards and flags bit-exact; (2) actions / log-probabilities against
the independent restatement of the specified sampler (oracle/sampler.py: Philox KATs, float32 inverse CDF) and its
float64 reference; (3) statistically against softmax(logits); (4) every kernel mapping draws the same actions.
(1) and (2) run for every kernel instance in test_gpu_policy_step_instances.py."""
from __future__ import annotations

import threading

import numpy as np
import pytest
import torch

from oracle import fast, sampler

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _mods():
    from merlin_b200 import BatchedMerlinEnv, codes, layouts
    return BatchedMerlinEnv, codes, layouts


def _np(x):
    return x.detach().cpu().numpy()


def _pool(n=64, diff="mediumhard", size=16, first=4200):
    _, codes, layouts = _mods()
    cells, agent = layouts.generate(diff, size, range(first, first + n))
    return cells, agent, codes.unpack_to_encoding(cells, size, size)


def test_policy_step_same_draws_under_every_kernel_mapping_and_reseed():
    BatchedMerlinEnv, _, _ = _mods()
    cells, agent, _ = _pool()
    N, T = 777, 12
    gen = torch.Generator(device=DEV).manual_seed(5)
    all_logits = torch.randn((T, N, 3), generator=gen, device=DEV) * 1.5
    runs = {}
    for choice in (1, 2, 3, 4, 6, 7, 5):
        env = BatchedMerlinEnv(N, cells, agent, width=16, height=16, max_steps=9, device=DEV)
        env.set_kernel_choice(choice)
        env.seed_sampler(31337)
        env.reset()
        logits = torch.empty((N, 3), device=DEV)
        io = env.make_policy_io(logits)
        acts, lps, syms = [], [], []
        for t in range(T):
            logits.copy_(all_logits[t])
            _, _, _, _, info = env.policy_step(io)
            acts.append(io.action.clone()); lps.append(io.logprob.clone()); syms.append(info["obs_symbolic"].clone())
        runs[choice] = (torch.stack(acts), torch.stack(lps), torch.stack(syms))
        if choice == 1:  # same seed again -> the same stream; another seed -> another stream
            env.seed_sampler(31337)
            env.reset()
            logits.copy_(all_logits[0])
            env.policy_step(io)
            assert torch.equal(io.action, runs[1][0][0])
            env.seed_sampler(31338)
            env.reset()
            env.policy_step(io)
            assert not torch.equal(io.action, runs[1][0][0])
    for choice in (2, 3, 4, 6, 7, 5):
        for a, b in zip(runs[1], runs[choice]):
            assert torch.equal(a, b), choice
    a = runs[1][0]
    assert not torch.equal(a[0], a[1])  # the draw counter advances


def test_policy_step_frequencies_follow_softmax_and_seven_actions():
    BatchedMerlinEnv, _, _ = _mods()
    cells, agent, _ = _pool()
    N = 65536
    for A, row in ((3, [0.3, -1.2, 1.1]), (7, [0.0, 0.5, -0.5, 1.0, -2.0, 0.2, 0.7])):
        env = BatchedMerlinEnv(N, cells, agent, width=16, height=16, device=DEV, n_actions=A, want_rgb=False)
        env.seed_sampler(A)
        env.reset(frames=False)
        logits = torch.tensor([row], device=DEV).repeat(N, 1).contiguous()
        io = env.make_policy_io(logits)
        counts = np.zeros(A)
        for _ in range(4):
            env.policy_step(io, frames=False)
            counts += np.bincount(_np(io.action), minlength=A)
        p = np.exp(np.asarray(row, np.float64)); p /= p.sum()
        n = counts.sum()
        chi2 = float(((counts - n * p) ** 2 / (n * p)).sum())
        assert chi2 < {3: 18.4, 7: 27.9}[A], (A, counts, chi2)  # p = 1e-4 at 2 / 6 degrees of freedom
        assert env.bad_actions() == 0


def test_policy_step_greedy_and_first_episode_record_match_the_python_bookkeeping():
    """greedy = argmax; the in-kernel first-episode record == the torch bookkeeping src/evaluation.py used to do."""
    BatchedMerlinEnv, _, _ = _mods()
    cells, agent, _ = _pool(48)
    N = 48
    env = BatchedMerlinEnv(N, cells, agent, width=16, height=16, max_steps=40, device=DEV, reset_mode="same", want_rgb=False)
    env.reset(frames=False)
    rec = {"finished": torch.zeros(N, dtype=torch.bool, device=DEV), "first_return": torch.zeros(N, device=DEV),
           "first_length": torch.zeros(N, dtype=torch.int32, device=DEV), "first_goal": torch.zeros(N, dtype=torch.bool, device=DEV)}
    logits = torch.empty((N, 3), device=DEV)
    io = env.make_policy_io(logits, greedy=True, record=rec)
    ret = torch.zeros(N, device=DEV); length = torch.zeros(N, dtype=torch.int32, device=DEV)
    goal = torch.zeros(N, dtype=torch.bool, device=DEV); finished = torch.zeros(N, dtype=torch.bool, device=DEV)
    gen = torch.Generator(device=DEV).manual_seed(3)
    for t in range(90):
        logits.copy_(torch.randn((N, 3), generator=gen, device=DEV) + torch.tensor([0.0, 0.0, 1.0], device=DEV))
        _, r, term, _, info = env.policy_step(io, frames=False)
        assert torch.equal(io.action, logits.argmax(-1))
        first = (info["episode_length"] > 0) & ~finished
        ret = torch.where(first, info["episode_return"], ret)
        length = torch.where(first, info["episode_length"], length)
        goal |= first & term
        finished |= first
    assert bool(finished.all())
    assert torch.equal(rec["finished"], finished) and torch.equal(rec["first_return"], ret)
    assert torch.equal(rec["first_length"], length) and torch.equal(rec["first_goal"], goal)


def test_policy_step_in_cuda_graph_draws_fresh_actions_every_replay():
    BatchedMerlinEnv, _, _ = _mods()
    cells, agent, enc = _pool()
    N = 512
    env = BatchedMerlinEnv(N, cells, agent, width=16, height=16, max_steps=50, device=DEV, want_rgb=False)
    env.seed_sampler(11)
    env.reset(frames=False)
    logits = torch.zeros((N, 3), device=DEV)
    acts = torch.zeros((4, N), dtype=torch.int64, device=DEV)
    lps = torch.zeros((4, N), device=DEV)
    ios = [env.make_policy_io(logits, action=acts[t], logprob=lps[t]) for t in range(4)]
    s = torch.cuda.Stream(DEV)
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        env.policy_step(ios[0], frames=False)  # warm-up outside capture
    torch.cuda.current_stream().wait_stream(s)
    env.seed_sampler(11)
    env.reset(frames=False)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for t in range(4):
            env.policy_step(ios[t], frames=False)
    ref = fast.OracleVecEnv(N, enc, agent, max_steps=50)
    ref.reset()
    ref.reset()  # the device env was reset twice (before the warm-up step and before the capture): one layout further
    seen = []
    for rep in range(3):
        g.replay()
        torch.cuda.synchronize()
        a = _np(acts)
        seen.append(a.copy())
        for t in range(4):
            ract, _, margin = sampler.sample_batch(_np(logits), 11, np.full(N, rep * 4 + t))
            assert np.array_equal(a[t], ract)  # uniform logits: boundaries at 1/3, 2/3 -- margins are wide
            _, _, _, _, rinfo = ref.step(a[t])
        assert np.array_equal(_np(env.obs_symbolic), rinfo["obs_symbolic"])
    assert not np.array_equal(seen[0], seen[1])


# ---- multi-handle / multi-stream contract ------------------------------------------------------------------------
def test_two_handles_two_threads_different_kernel_choices():
    """Per-handle kernel choice / occupancy caches: two handles (on two devices when the box has them, else both on
    device 0) stepped concurrently from two threads with different mappings, each checked against the oracle."""
    BatchedMerlinEnv, _, _ = _mods()
    cells, agent, enc = _pool()
    n_dev = torch.cuda.device_count()
    devs = ["cuda:0", f"cuda:{1 if n_dev > 1 else 0}"]
    N, T = 3000, 30
    errors = []

    def work(dev, choice, seed):
        try:
            torch.cuda.set_device(dev)
            with torch.cuda.stream(torch.cuda.Stream(dev)):
                env = BatchedMerlinEnv(N, cells, agent, width=16, height=16, max_steps=11, device=dev)
                env.set_kernel_choice(choice)
                assert ("tile" if choice == 3 else "warp") in env.step_kernel()
                ref = fast.OracleVecEnv(N, enc, agent, max_steps=11)
                obs, _ = env.reset()
                assert np.array_equal(_np(obs), ref.reset()[0])
                rng = np.random.default_rng(seed)
                for t in range(T):
                    a = rng.integers(0, 3, N)
                    obs, r, te, tr, _ = env.step(torch.as_tensor(a, device=dev))
                    robs, rr, rte, rtr, _ = ref.step(a)
                    assert np.array_equal(_np(obs), robs) and np.array_equal(_np(r), rr), (dev, choice, t)
                    assert np.array_equal(_np(te), rte) and np.array_equal(_np(tr), rtr)
        except Exception as exc:  # noqa: BLE001 -- reported to the main thread
            errors.append((dev, choice, repr(exc)))

    threads = [threading.Thread(target=work, args=(devs[0], 3, 1)), threading.Thread(target=work, args=(devs[1], 2, 2))]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    torch.cuda.set_device(0)
    assert not errors, errors


def test_handle_choice_overrides_the_process_default_and_can_follow_it_again():
    from merlin_b200 import set_kernel_choice
    BatchedMerlinEnv, _, _ = _mods()
    cells, agent, _ = _pool()
    env = BatchedMerlinEnv(100000, cells, agent, width=16, height=16, device=DEV)
    try:
        set_kernel_choice(2)
        assert "warp" in env.step_kernel()
        env.set_kernel_choice(3)
        assert "tile" in env.step_kernel()
        env.set_kernel_choice(-1)
        assert "warp" in env.step_kernel()
    finally:
        set_kernel_choice(0)
    assert "tile" in env.step_kernel()
    with pytest.raises(ValueError):
        env.set_kernel_choice(9)


def test_steps_and_renders_alternating_between_streams_stay_ordered():
    """Calls of one handle hopping between two streams (no user-side events): the library orders them, results stay
    bit-exact; a render on a side stream may overlap the next step (separate ticket counters)."""
    BatchedMerlinEnv, _, _ = _mods()
    cells, agent, enc = _pool()
    N = 50000
    env = BatchedMerlinEnv(N, cells, agent, width=16, height=16, max_steps=11, device=DEV)
    ref = fast.OracleVecEnv(N, enc, agent, max_steps=11)
    streams = [torch.cuda.Stream(DEV), torch.cuda.Stream(DEV)]
    env.reset(); ref.reset()
    rng = np.random.default_rng(0)
    torch.cuda.synchronize()
    acts = [torch.as_tensor(rng.integers(0, 3, N), device=DEV) for _ in range(12)]
    torch.cuda.synchronize()
    frames = []
    for t in range(12):
        with torch.cuda.stream(streams[t & 1]):
            obs, r, te, tr, info = env.step(acts[t])
            if t % 4 == 3:
                sym_copy = info["obs_symbolic"].clone()
                other = streams[1 - (t & 1)]
                other.wait_stream(streams[t & 1])  # the DATA dependency (sym_copy) is the caller's to order
                with torch.cuda.stream(other):     # the render hops streams; ticket counters are the library's
                    frames.append((t, env.render(sym_copy)))
        rref = ref.step(_np(acts[t]))
        if t % 4 == 3:
            frames[-1] += (rref[0].copy(),)
    torch.cuda.synchronize()
    assert np.array_equal(_np(obs), rref[0]) and np.array_equal(_np(r), rref[1])
    for t, got, want in frames:
        assert np.array_equal(_np(got), want), t
    env.rearm()
    obs, *_ = env.step(acts[0])
    assert np.array_equal(_np(obs), ref.step(_np(acts[0]))[0])


# ---- state save / restore (merlin_env_read_state / merlin_env_write_state) ----------------------------------------
def test_write_state_resumes_a_rollout_bit_exactly_and_validates():
    """Save the env state mid-rollout, run on, restore it into a SECOND handle and replay the same actions: identical
    observations, rewards and flags (the state words are the whole state for immutable grids); staggered episode clocks
    make envs truncate at the steady-state rate; bad states are rejected."""
    BatchedMerlinEnv, _, _ = _mods()
    cells, agent, enc = _pool(96)
    N = 4096
    envs = [BatchedMerlinEnv(N, cells, agent, width=16, height=16, max_steps=64, device=DEV) for _ in range(2)]
    rng = np.random.default_rng(3)
    acts = [torch.as_tensor(rng.integers(0, 3, N), device=DEV) for _ in range(24)]
    a, b = envs
    a.reset(); b.reset()
    for t in range(8):
        a.step(acts[t])
    st, epr = a.state_raw()
    tail = [tuple(x.clone() for x in a.step(acts[t])[:4]) for t in range(8, 24)]
    b.load_state_raw(st, epr)
    for t in range(8, 24):
        obs, r, te, tr, info = b.step(acts[t])
        want = tail[t - 8]
        assert torch.equal(obs, want[0]) and torch.equal(r, want[1]) and torch.equal(te, want[2]) and torch.equal(tr, want[3]), t
    assert np.array_equal(a.pose_numpy(), b.pose_numpy())
    # staggered clocks: truncations arrive at ~N / max_steps per step instead of all at step 64
    b.reset()
    b.stagger_episode_clocks(seed=1)
    assert len(np.unique(b.state_numpy()["step_count"])) == 64
    n_trunc = [int(b.step(acts[t])[3].sum()) for t in range(16)]
    assert min(n_trunc) > 0 and max(n_trunc) < 4 * N // 64
    bad = st.copy(); bad[0, 2] = 10_000          # layout index outside the pool
    with pytest.raises(ValueError):
        b.load_state_raw(bad)
    bad = st.copy(); bad[5, 1] = 64               # step_count == max_steps
    with pytest.raises(ValueError):
        b.load_state_raw(bad)
    with pytest.raises(ValueError):
        b.load_state_raw(st[:10])
