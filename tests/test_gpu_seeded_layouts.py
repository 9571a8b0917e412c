"""GPU tier: merlin_env_generate_seeded_layouts -- the reference's per-seed layouts (`env.reset(seed=s)` -> `_gen_grid`)
built on the device from numpy's default_rng stream (csrc/np_random.cuh).  The pools must equal the host generator
(merlin_b200.layouts, pinned to the reference by the golden fixtures) byte for byte, cells and agent poses; the seeds the
host generator cannot build must fail the call.  The counter-based generator beside it (merlin_env_generate_layouts)
shares the layout routines, so its pools are pinned here by digests recorded before the routines were shared."""
from __future__ import annotations

import hashlib

import numpy as np
import pytest
import torch

import helpers
from oracle import fast

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
WHY = f"(host generator under numpy {np.__version__})"

# smallest side the seeded entry accepts, per difficulty
MIN_SIDE = {"easy": 6, "medium": 4, "mediumhard": 4, "hard": 5, "hardest": 8}
SEEDS_16 = (list(range(1024)) + list(range(200_000, 201_024)) + list(range(777_000_000, 777_001_024))
            + list(range(2**32 - 512, 2**32 + 512)) + [2**40 + 3, 2**63, 2**64 - 1])


def _env(N, W, H, **kw):
    from merlin_b200 import BatchedMerlinEnv
    return BatchedMerlinEnv(N, width=W, height=H, device=DEV, **kw)


def _host(difficulty, W, H, seeds):
    """The host generator's layouts of `seeds` on a W x H grid, driving layouts._Builder directly (W may differ from
    H); the index of the first seed it raises on, else None."""
    from merlin_b200 import layouts
    cells = np.empty((len(seeds), W * H), np.uint8)
    agent = np.empty((len(seeds), 3), np.int32)
    for k, s in enumerate(seeds):
        b = layouts._Builder(np.random.default_rng(int(s)), W, H)
        try:
            layouts._GENERATORS[difficulty](b)
        except (ValueError, RecursionError):
            return cells[:k], agent[:k], k
        cells[k], agent[k] = b.g.reshape(-1), (b.agent_pos[0], b.agent_pos[1], b.agent_dir)
    return cells, agent, None


def _assert_same(got, want, what):
    gc, ga = got
    wc, wa = want
    bad = np.flatnonzero((gc != wc).any(1) | (ga != wa).any(1))
    assert bad.size == 0, f"{what}: {bad.size} of {len(wc)} layouts differ, first at slot {bad[0]} {WHY}"


# ---- the pools equal the host generator's ----------------------------------------------------------------------------
CASES = [(d, s) for d in MIN_SIDE for s in sorted({MIN_SIDE[d], 8, 11, 16, 24, 32, 64}) if s >= MIN_SIDE[d]]


@pytest.mark.parametrize("difficulty,size", CASES)
def test_seeded_pool_equals_host_layouts(difficulty, size):
    from merlin_b200 import layouts
    if size == 16:
        seeds = SEEDS_16
    else:
        n = {64: 48, 32: 200}.get(size, 600)
        seeds = list(range(n // 2)) + list(range(777_000_000, 777_000_000 + n // 2)) + [2**32, 2**64 - 1]
    want = layouts.generate(difficulty, size, seeds)
    env = _env(4, size, size, generate_seeded=(difficulty, seeds))
    assert env.n_layouts == len(seeds) and env.difficulty == difficulty
    _assert_same(env.layouts_numpy(), want, f"{difficulty} {size}x{size}")


@pytest.mark.parametrize("difficulty,W,H", [("easy", 7, 12), ("medium", 5, 30), ("mediumhard", 20, 6),
                                            ("hard", 24, 12), ("hard", 16, 7), ("hardest", 9, 13), ("hardest", 40, 8)])
def test_seeded_pool_equals_host_builder_on_rectangular_grids(difficulty, W, H):
    seeds = list(range(400)) + list(range(200_000, 200_200))
    cells, agent, failed = _host(difficulty, W, H, seeds)
    assert failed is None
    env = _env(4, W, H, generate_seeded=(difficulty, seeds))
    _assert_same(env.layouts_numpy(), (cells, agent), f"{difficulty} {W}x{H}")


@pytest.mark.parametrize("name", helpers.layout_names())
def test_seeded_pool_equals_golden_fixtures(name):
    from merlin_b200 import codes
    fx = helpers.load(name + ".npz")
    _, diff, size = name.split("_")
    env = _env(4, int(size), int(size), generate_seeded=(diff, [int(s) for s in fx["seeds"]]))
    _assert_same(env.layouts_numpy(), (codes.pack_encoding(fx["enc"]), fx["agent"]), name)


def test_create_batched_env_device_seeds_equals_host_path():
    from src.scenario_creator.scenario_creator import ScenarioCreator
    sc = ScenarioCreator()
    seeds = range(777_000_000, 777_000_000 + 3000)
    dev = sc.create_batched_env("hard", 64, device=DEV, layouts="device", seeds=seeds)
    host = sc.create_batched_env("hard", 64, device=DEV, layouts=None, seeds=seeds)
    assert dev.n_layouts == host.n_layouts == 3000 and dev.difficulty == host.difficulty
    _assert_same(dev.layouts_numpy(), host.layouts_numpy(), "create_batched_env")
    # an int keeps selecting the counter-based stream
    keyed = sc.create_batched_env("hard", 64, device=DEV, layouts="device", seeds=5, n_layouts=512)
    ref = _env(4, 16, 16, generate=("hard", 5, 512))
    assert keyed.n_layouts == 512
    _assert_same(keyed.layouts_numpy(), ref.layouts_numpy(), "create_batched_env, int seed")


# ---- pool semantics ------------------------------------------------------------------------------------------------
def test_rollout_on_a_seeded_pool_matches_the_oracle():
    """Frames, symbolic observations, rewards and flags bit-exact against the oracle over the HOST layouts of the same
    seeds, with auto-reset moving envs through the pool (the atlas mask of a generated pool must cover every frame)."""
    from merlin_b200 import codes, layouts
    N, T, seeds = 3000, 40, list(range(200_000, 200_777))
    cells, agent = layouts.generate("mediumhard", 16, seeds)
    env = _env(N, 16, 16, generate_seeded=("mediumhard", seeds), max_steps=17)
    ref = fast.OracleVecEnv(N, codes.unpack_to_encoding(cells, 16, 16), agent, max_steps=17)
    obs, sym = env.reset()
    robs, rsym = ref.reset()
    assert np.array_equal(obs.cpu().numpy(), robs) and np.array_equal(sym.cpu().numpy(), rsym)
    rng = np.random.default_rng(3)
    for t in range(T):
        a = rng.integers(0, 3, N)
        obs, r, te, tr, info = env.step(torch.as_tensor(a, device=DEV))
        robs, rr, rte, rtr, rinfo = ref.step(a)
        assert np.array_equal(obs.cpu().numpy(), robs), t
        assert np.array_equal(info["obs_symbolic"].cpu().numpy(), rinfo["obs_symbolic"]), t
        assert np.array_equal(r.cpu().numpy(), rr) and np.array_equal(te.cpu().numpy(), rte), t
        assert np.array_equal(tr.cpu().numpy(), rtr), t


def test_in_place_regeneration_under_a_captured_step():
    """Same-sized regeneration rewrites the pool in place: a CUDA graph captured over step() before it keeps working and
    steps the new layouts."""
    from merlin_b200 import codes, layouts
    N, L = 512, 64
    first, second = list(range(L)), list(range(777_000_000, 777_000_000 + L))
    env = _env(N, 16, 16, generate_seeded=("hard", first), max_steps=9)
    env.reset()
    static_a = torch.zeros(N, dtype=torch.int64, device=DEV)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        env.step(static_a)  # warm-up outside capture
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        env.step(static_a)
    env.generate_seeded_layouts("hard", second)
    cells, agent = layouts.generate("hard", 16, second)
    _assert_same(env.layouts_numpy(), (cells, agent), "regenerated pool")
    ref = fast.OracleVecEnv(N, codes.unpack_to_encoding(cells, 16, 16), agent, max_steps=9)
    obs, _ = env.reset()
    assert np.array_equal(obs.cpu().numpy(), ref.reset()[0])
    rng = np.random.default_rng(4)
    for t in range(20):
        a = rng.integers(0, 3, N)
        static_a.copy_(torch.as_tensor(a, device=DEV))
        graph.replay()
        robs, rr, rte, rtr, _ = ref.step(a)
        assert np.array_equal(env.obs.cpu().numpy(), robs) and np.array_equal(env.reward.cpu().numpy(), rr), t
        assert np.array_equal(env.terminated.cpu().numpy(), rte) and np.array_equal(env.truncated.cpu().numpy(), rtr), t


# ---- errors ------------------------------------------------------------------------------------------------------------
def test_rejected_arguments():
    env = _env(4, 16, 16, generate_seeded=("medium", [1, 2, 3]))
    for bad in ([-1], [2**64], [1.5], ["7"], [], "123", [[1, 2]]):
        with pytest.raises(ValueError):
            env.generate_seeded_layouts("medium", bad)
    with pytest.raises(ValueError):
        env.generate_seeded_layouts("nightmare", [1])
    assert env.n_layouts == 3
    env.reset()  # the pool survived every rejected call
    with pytest.raises(ValueError):
        _env(4, 7, 7, generate_seeded=("hardest", [0]))   # hardest raises below 8 (integers(2, my - 1))
    with pytest.raises(ValueError):
        _env(4, 4, 4, generate_seeded=("hard", [0]))      # hard loops forever or raises below 5
    with pytest.raises(ValueError):
        _env(4, 5, 5, generate_seeded=("easy", [0]))      # rejected by both device generators
    with pytest.raises(ValueError):
        _env(4, 16, 16, generate=("easy", 0, 4), generate_seeded=("easy", [0]))


def test_a_seed_the_host_cannot_build_fails_the_call():
    """hard on a 13x5 grid draws up to 5 gap rows out of 3: numpy's choice raises for those seeds.  The call fails
    naming the first of them; the handle refuses reset (and so step) until the next good generation."""
    fails = {s: _host("hard", 13, 5, [s])[2] is not None for s in range(200)}
    good = [s for s in range(200) if not fails[s]][:40]
    bad = [s for s in range(200) if fails[s]][:2]
    mixed = good[:20] + [bad[0]] + good[20:] + [bad[1]]
    env = _env(8, 13, 5, generate_seeded=("hard", good))
    env.reset()
    with pytest.raises(ValueError, match=f"seed {bad[0]} "):
        env.generate_seeded_layouts("hard", mixed)
    assert env.n_layouts == len(mixed)
    with pytest.raises(RuntimeError):
        env.reset()
    with pytest.raises(RuntimeError):
        env.step(torch.zeros(8, dtype=torch.int64, device=DEV))
    env.generate_seeded_layouts("hard", good)
    cells, agent, _ = _host("hard", 13, 5, good)
    _assert_same(env.layouts_numpy(), (cells, agent), "after recovery")
    env.reset()


# ---- the counter-based generator is unchanged --------------------------------------------------------------------------
# SHA-256 of layouts_numpy() (cells bytes, then agent bytes) for generate=(d, 12345, 2000) regenerated in place with
# first_number=1000, recorded with the layout routines as they were before they became templates on the stream
SPLITMIX_DIGESTS = {
    ("easy", 8, 8): "56c23e1934b50c08cb137ec1802b6741475c0a532a3eded5a3c924e0f8c2df1b",
    ("easy", 16, 16): "ce1f563aa659ec5d06021a6d8a1a85880676ce5f5add9d9cff45b4e66b0aabfd",
    ("medium", 8, 8): "3545179140a7ad41ebf9a593f1b68860b66c499bb447c9d2d139d1a7326aaa7b",
    ("medium", 16, 16): "459e753215c98eb5c1aac077824fe1157720989d249dc2e9efa6a3393d325492",
    ("mediumhard", 8, 8): "c62cba2acf916cf03cf9d9e4bcbccf2501483c89066349ea6702a2bbb9e2f8ee",
    ("mediumhard", 16, 16): "b2cecbd10e95bba49b99fcb0a35d114552cfb4030916e7b2de82e2829bf50292",
    ("hard", 8, 8): "0831438dd96dbd880a72abdf4c54a072bf9e91c3cd55540f4ae575905f2b236e",
    ("hard", 32, 32): "68520c6a840010b85871360b1d5a83151b57b1e5c427a6567d5a3b49ce808eec",
    ("hardest", 8, 8): "e4dda166dbfdf01065cb70b865c56dfe1f347bdd82c771fd4429597a1796e6f8",
    ("hardest", 16, 16): "687d5de849b1ed19fc58c82ffc3299bcbf9c0a680dd9203fbbf3f65c0b561a3c",
    ("hard", 24, 12): "a060b24682a7d04f100febabfae6e43ab6fa05d0729dff034ce4392692f940c8",
    ("hardest", 9, 13): "f94cdd6837f0ae93bbac836ffc5e75d6aa9e85755fcc407700a73cae70356453",
    ("mediumhard", 4, 4): "76457d85c8375ffc8433a2afa73601db050f48eae1b216cba05063c24e601858",
}


@pytest.mark.parametrize("difficulty,W,H", list(SPLITMIX_DIGESTS))
def test_counter_based_pools_unchanged(difficulty, W, H):
    env = _env(4, W, H, generate=(difficulty, 12345, 2000))
    env.generate_layouts(difficulty, 12345, 2000, first_number=1000)
    c, a = env.layouts_numpy()
    assert hashlib.sha256(c.tobytes() + a.tobytes()).hexdigest() == SPLITMIX_DIGESTS[(difficulty, W, H)]
