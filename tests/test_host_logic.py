"""CPU tests of the PRODUCT's host-side logic (no GPU):
  * merlin_b200.layouts vs the fixtures made by the reference's own _gen_grid (same seeds -> same layouts)
  * merlin_b200.tiles (array renderer) vs the literal per-pixel renderer of the oracle
  * merlin_b200.codes round trips
  * ppo-2dgrid_b200/csrc/env_logic.cuh -- the per-env functions the CUDA kernels call -- compiled for the host
    (tests/csrc/host_model.cpp) and compared with the oracle on random grids, incl. doors/keys/boxes/lava.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np
import pytest

import helpers
from merlin_b200 import codes, layouts, tiles
from oracle import fast

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


# ---- layouts ------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", helpers.layout_names())
def test_product_layouts_match_reference_fixtures(name):
    fx = helpers.load(name + ".npz")
    _, diff, size = name.split("_")
    cells, agent = layouts.generate(diff, int(size), fx["seeds"])
    assert np.array_equal(cells, codes.pack_encoding(fx["enc"]))
    assert np.array_equal(agent, fx["agent"])


@pytest.mark.parametrize("name", ["mediumhard_goal", "hard_goal", "hardest_goal", "medium_goal"])
def test_product_layout_stream_matches_unseeded_resets(name):
    tr = helpers.load(f"trace_{name}.npz")
    n = tr["ep_enc"].shape[0]
    cells, agent = layouts.generate_stream(str(tr["difficulty"]), int(tr["size"]), int(tr["seed"]), n)
    assert np.array_equal(cells, codes.pack_encoding(tr["ep_enc"]))
    assert np.array_equal(agent, tr["ep_agent"])


def test_unknown_difficulty_raises_value_error():
    with pytest.raises(ValueError):
        layouts.generate("impossible", 16, [0])


# ---- codes / tiles ------------------------------------------------------------------------------
def test_codes_round_trip():
    fx = helpers.load("layouts_hardest_16.npz")
    packed = codes.pack_encoding(fx["enc"])
    assert np.array_equal(codes.unpack_to_encoding(packed, 16, 16), fx["enc"])
    assert codes.pack(4, 3, 1) == (codes.DOOR_CLOSED | (3 << 4)) and codes.pack(4, 3, 2) == (codes.DOOR_LOCKED | (3 << 4))
    assert codes.pack(8, 5, 0) == codes.CODE_GOAL and codes.pack(0, 0, 0) == codes.CODE_EMPTY


def test_atlas_matches_literal_renderer():
    at = tiles.build_atlas()
    oa = fast.TileAtlas(8)
    assert np.array_equal(at[0], oa.tiles[fast.tile_slot(1, 0, 0, 0, 0)])
    assert np.array_equal(at[1], oa.tiles[fast.tile_slot(1, 0, 0, 0, 1)])
    assert np.array_equal(at[10], oa.tiles[fast.tile_slot(1, 0, 0, 1, 1)])
    for color in range(6):
        for t in codes.VALID_TYPES:
            if t == codes.EMPTY:
                continue
            mt, st = (4, {4: 0, 11: 1, 12: 2}[t]) if t in (4, 11, 12) else (t, 0)
            oa.ensure([(mt, color, st)])
            assert np.array_equal(at[t | (color << 4)], oa.tiles[fast.tile_slot(mt, color, st, 0, 1)]), (t, color)
            if t in (codes.KEY, codes.BALL, codes.BOX):
                assert np.array_equal(at[(t + 8) | (color << 4)], oa.tiles[fast.tile_slot(mt, color, st, 1, 1)])


# ---- env_logic.cuh on the host ----------------------------------------------------------------
def _host_model():
    src = os.path.join(ROOT, "tests", "csrc", "host_model.cpp")
    hdr = os.path.join(ROOT, "ppo-2dgrid_b200", "csrc", "env_logic.cuh")
    hdr2 = os.path.join(ROOT, "ppo-2dgrid_b200", "csrc", "obs_swar.cuh")
    out = os.path.join(ROOT, "tests", "csrc", "_build", "libhost_model.so")
    if not os.path.exists(out) or os.path.getmtime(out) < max(os.path.getmtime(f) for f in (src, hdr, hdr2)):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-Wno-unknown-pragmas",
                               "-I" + os.path.dirname(hdr), src, "-o", out])
    lib = ctypes.CDLL(out)
    lib.hm_step.restype = ctypes.c_int
    return lib


class HostModelEnv:
    """The kernel's per-env logic driven from numpy (auto-reset off), for comparison with OracleVecEnv."""

    def __init__(self, cells, agent, W, H, max_steps, n_actions=3, stuck=False, bonus=0.0):
        self.lib = _host_model()
        self.N, self.W, self.H, self.max_steps, self.n_actions = cells.shape[0], W, H, max_steps, n_actions
        self.stride = (W * H + 15) & ~15
        self.cells = np.full((self.N, self.stride), codes.CODE_EMPTY, np.uint8)
        self.cells[:, : W * H] = cells
        self.state = np.zeros((self.N, 4), np.int32)
        self.state[:, 0] = agent[:, 0] | (agent[:, 1] << 8) | (agent[:, 2] << 16)
        self.state[:, 3] = (agent[:, 0] << 16) | (agent[:, 1] << 24)
        self.stuck_on, self.bonus = stuck, bonus
        self.vw = (W * H + 31) // 32
        self.visited = np.zeros((self.N, self.vw), np.uint32)
        cell = agent[:, 1] * W + agent[:, 0]
        self.visited[np.arange(self.N), cell >> 5] = (1 << (cell & 31)).astype(np.uint32)
        self.atlas = np.ascontiguousarray(tiles.build_atlas())

    def call(self, actions, do_step):
        N = self.N
        rgb = np.zeros((N, 56, 56, 3), np.uint8)
        sym = np.zeros((N, 7, 7, 3), np.uint8)
        rew = np.zeros(N, np.float32)
        te, tr, sk = np.zeros(N, np.uint8), np.zeros(N, np.uint8), np.zeros(N, np.uint8)
        actions = np.ascontiguousarray(actions, np.int64)
        p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        self.lib.hm_step(N, self.W, self.H, self.max_steps, self.stride, self.n_actions, int(do_step), int(self.stuck_on),
                         3, ctypes.c_double(-0.1), int(self.bonus != 0), ctypes.c_double(self.bonus), self.vw,
                         p(self.state), p(self.cells), p(self.visited), p(actions), p(self.atlas), p(rgb), p(sym),
                         p(rew), p(te), p(tr), p(sk))
        # the row-parallel observation (obs_swar.cuh) must agree with the per-cell form on every call
        if self.W >= 7:
            rgb2, sym2 = np.zeros_like(rgb), np.zeros_like(sym)
            padded = np.concatenate([self.cells.reshape(-1), np.zeros(8, np.uint8)])
            # grids without closed / locked doors also go through the short path the kernels take for door-free pools
            has_doors = bool(np.isin(self.cells & 0xF, (11, 12)).any())
            for doors in ((1,) if has_doors else (1, 0)):
                rgb2.fill(0); sym2.fill(0)
                self.lib.hm_observe_swar(N, self.W, self.H, self.stride, p(self.state), p(padded), p(self.atlas), p(rgb2),
                                         p(sym2), doors)
                assert np.array_equal(sym2, sym), f"obs_swar symbolic image differs from the per-cell form (doors={doors})"
                assert np.array_equal(rgb2, rgb), f"obs_swar tile kinds differ from the per-cell form (doors={doors})"
        return rgb, sym, rew, te.astype(bool), tr.astype(bool), sk.astype(bool)


def _random_object_layouts(rng, L, size):
    enc = np.zeros((L, size, size, 3), np.uint8)
    enc[..., 0] = 1
    enc[:, 0, :, :] = enc[:, -1, :, :] = enc[:, :, 0, :] = enc[:, :, -1, :] = (2, 5, 0)
    agent = np.zeros((L, 3), np.int32)
    objs = [(2, 5, 0), (2, 5, 0), (2, 5, 0), (8, 1, 0), (9, 0, 0), (3, 2, 0), (4, 4, 0), (4, 4, 1), (4, 4, 2),
            (5, 4, 0), (6, 0, 0), (7, 3, 0), (4, 2, 1), (5, 2, 0)]
    for l in range(L):
        for _ in range(int(rng.integers(5, 30))):
            x, y = rng.integers(1, size - 1, 2)
            enc[l, x, y] = objs[int(rng.integers(0, len(objs)))]
        while True:
            x, y = rng.integers(1, size - 1, 2)
            if enc[l, x, y, 0] == 1:
                break
        agent[l] = (x, y, rng.integers(0, 4))
    return enc, agent


@pytest.mark.parametrize("n_actions,stuck,bonus,size", [(3, False, 0.0, 16), (7, True, 0.0, 9), (7, False, 0.05, 12),
                                                       (3, True, 0.01, 16)])
def test_kernel_logic_on_host_matches_oracle(n_actions, stuck, bonus, size):
    rng = np.random.default_rng(n_actions * 100 + size)
    L = 64
    if n_actions == 3:
        cells, agent = layouts.generate("mediumhard", size, range(1000, 1000 + L))
        enc = codes.unpack_to_encoding(cells, size, size)
    else:
        enc, agent = _random_object_layouts(rng, L, size)
        cells = codes.pack_encoding(enc)
    max_steps = 50
    ref = fast.OracleVecEnv(L, enc, agent, max_steps=max_steps, n_actions=n_actions, auto_reset=False,
                            stuck_penalty=stuck, exploration_bonus=bonus)
    hm = HostModelEnv(cells, agent, size, size, max_steps, n_actions, stuck, bonus)
    rgb0, sym0 = ref.reset()
    rgb, sym, *_ = hm.call(np.zeros(L, np.int64), do_step=False)
    assert np.array_equal(sym, sym0) and np.array_equal(rgb, rgb0)
    for t in range(80):
        a = rng.integers(0, n_actions, L)
        if n_actions == 7:  # bias towards moving so objects get reached
            a = np.where(rng.random(L) < 0.4, 2, a)
        rgb0, r0, te0, tr0, info = ref.step(a)
        rgb, sym, r, te, tr, sk = hm.call(a, do_step=True)
        assert np.array_equal(r, r0), t
        assert np.array_equal(te, te0) and np.array_equal(tr, tr0), t
        assert np.array_equal(sk, info["stuck"]), t
        assert np.array_equal(sym, info["obs_symbolic"]), t
        assert np.array_equal(rgb, rgb0), t
        pose = hm.state[:, 0]
        assert np.array_equal(pose & 0xFF, ref.ax) and np.array_equal((pose >> 8) & 0xFF, ref.ay)
        assert np.array_equal((pose >> 16) & 3, ref.adir) and np.array_equal(hm.state[:, 1], ref.stepc)


@pytest.mark.parametrize("W,H", [(7, 7), (7, 30), (8, 9), (9, 8), (13, 11), (16, 16), (17, 23), (31, 7), (40, 33), (255, 9)])
def test_row_parallel_observation_equals_per_cell_form(W, H):
    """obs_swar.cuh against gather_view + visibility + sym_of_code on grids WITHOUT a border wall: agents on every edge
    and corner (windows hanging out of the grid on any side), every heading, every object type, carried objects."""
    rng = np.random.default_rng(W * 1000 + H)
    L = 400
    objs = [(1, 0, 0)] * 6 + [(2, 5, 0)] * 4 + [(8, 1, 0), (9, 0, 0), (3, 2, 0), (4, 4, 0), (4, 4, 1), (4, 4, 2), (5, 4, 0),
                                             (6, 0, 0), (7, 3, 0), (4, 2, 1), (5, 2, 0), (4, 0, 2), (6, 5, 0)]
    pick = rng.integers(0, len(objs), (L, W, H))
    enc = np.asarray(objs, np.uint8)[pick]
    agent = np.stack([rng.integers(0, W, L), rng.integers(0, H, L), rng.integers(0, 4, L)], axis=1).astype(np.int32)
    edge = rng.random(L) < 0.5  # half of the agents sit on an edge or in a corner
    agent[edge, 0] = np.where(rng.random(edge.sum()) < 0.5, rng.choice([0, W - 1], edge.sum()), agent[edge, 0])
    agent[edge, 1] = np.where(rng.random(edge.sum()) < 0.5, rng.choice([0, H - 1], edge.sum()), agent[edge, 1])
    hm = HostModelEnv(codes.pack_encoding(enc), agent, W, H, 100, n_actions=7)
    carried = np.asarray([0, 0, codes.pack(5, 4, 0), codes.pack(6, 0, 0), codes.pack(7, 3, 0)], np.int32)[rng.integers(0, 5, L)]
    hm.state[:, 0] |= carried << 24
    rgb, sym, *_ = hm.call(np.zeros(L, np.int64), do_step=False)  # asserts the two forms agree
    assert (sym[:, 3, 6, 0] != 0).all()  # the agent's own cell is always visible
    assert len(np.unique(sym[..., 0])) >= 9


def test_visibility_bitmask_exhaustive_rows():
    """Bitmask process_vis vs the literal sweeps on 20k random 7x7 transparency patterns (via full envs)."""
    rng = np.random.default_rng(99)
    L, size = 512, 9
    enc = np.zeros((L, size, size, 3), np.uint8)
    enc[..., 0] = 1
    walls = rng.random((L, size, size)) < rng.uniform(0.1, 0.6, (L, 1, 1))
    enc[walls] = (2, 5, 0)
    enc[:, 4, 4] = (1, 0, 0)
    agent = np.tile(np.array([[4, 4, 0]], np.int32), (L, 1))
    agent[:, 2] = rng.integers(0, 4, L)
    ref = fast.OracleVecEnv(L, enc, agent, auto_reset=False)
    hm = HostModelEnv(codes.pack_encoding(enc), agent, size, size, 100)
    ref.reset()
    for _ in range(40):
        a = rng.integers(0, 2, L)  # spin in place: new headings over the same random walls
        rgb0, _, _, _, info = ref.step(a)
        rgb, sym, *_ = hm.call(a, do_step=True)
        assert np.array_equal(sym, info["obs_symbolic"])
        assert np.array_equal(rgb, rgb0)


def test_visibility_row_carry_chain_form_equals_literal_sweeps_exhaustively():
    """vis_row (one addition per sweep) == vis_row_literal (six propagation steps per sweep, the upstream loops) for
    ALL 128 x 128 (lit-from-below, transparency) rows, and visibility == visibility_literal on random 49-bit masks."""
    lib = _host_model()
    lib.hm_vis_row.restype = ctypes.c_uint32
    lib.hm_vis_row.argtypes = [ctypes.c_uint32, ctypes.c_uint32, ctypes.c_int]
    for seed in range(128):
        for T in range(128):
            assert lib.hm_vis_row(seed, T, 0) == lib.hm_vis_row(seed, T, 1), (seed, T)
    lib.hm_visibility.restype = lib.hm_visibility_literal.restype = ctypes.c_uint64
    lib.hm_visibility.argtypes = lib.hm_visibility_literal.argtypes = [ctypes.c_uint64]
    rng = np.random.default_rng(7)
    for dens in (0.2, 0.5, 0.8, 0.95):
        for _ in range(5000):
            m = int(sum(1 << i for i in np.nonzero(rng.random(49) < dens)[0]))
            assert lib.hm_visibility(m) == lib.hm_visibility_literal(m), m
    # the byte-per-row form (env_kernel_quad): same rows in, same rows out
    lib.hm_visibility_rows.restype = ctypes.c_uint64
    lib.hm_visibility_rows.argtypes = [ctypes.c_uint64]
    spread = lambda m: sum(((m >> (7 * vj)) & 0x7f) << (8 * vj) for vj in range(7))
    for _ in range(5000):
        m = int(sum(1 << i for i in np.nonzero(rng.random(49) < 0.7)[0]))
        assert lib.hm_visibility_rows(spread(m)) == spread(lib.hm_visibility(m)), m


# ---- in-kernel action sampler (env_logic.cuh: Philox4x32-10, inverse CDF) -------------------------------------
PHILOX_KAT = [  # Random123 known-answer vectors for philox4x32-10: (counter, key, output)
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0), (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
]


def test_philox_known_answers_oracle_and_kernel_header():
    from oracle import sampler
    lib = _host_model()
    for ctr, key, want in PHILOX_KAT:
        assert sampler.philox4x32_10(ctr, key) == want
        c, k, o = (ctypes.c_uint32 * 4)(*ctr), (ctypes.c_uint32 * 2)(*key), (ctypes.c_uint32 * 4)()
        lib.hm_philox(c, k, o)
        assert tuple(o) == want


def _hm_sample(logits, seed, draws, greedy=False):
    lib = _host_model()
    N, A = logits.shape
    lib.hm_sample.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_int,
                              ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    logits = np.ascontiguousarray(logits, np.float32)
    draws = np.ascontiguousarray(draws, np.uint32)
    act, lp, u = np.zeros(N, np.int64), np.zeros(N, np.float32), np.zeros(N, np.float32)
    lib.hm_sample(N, A, logits.ctypes.data, seed, draws.ctypes.data, int(greedy), act.ctypes.data, lp.ctypes.data, u.ctypes.data)
    return act, lp, u


@pytest.mark.parametrize("A", [3, 7])
def test_sampler_header_matches_oracle_restatement(A):
    """sample_policy / sampler_uniform as the kernels compile them (host build) vs the independent numpy restatement:
    identical uniforms, identical actions (away from CDF boundaries), log-probabilities to float32 rounding."""
    from oracle import sampler
    rng = np.random.default_rng(A)
    N, seed = 4000, 0x1234_5678_9ABC_DEF0
    logits = (rng.standard_normal((N, A)) * rng.choice([0.01, 1.0, 5.0], (N, 1))).astype(np.float32)
    draws = rng.integers(0, 1 << 20, N)
    act, lp, u = _hm_sample(logits, seed, draws)
    assert np.array_equal(u, np.array([sampler.uniform(seed, e, int(draws[e])) for e in range(N)], np.float32))
    assert (u >= 0).all() and (u < 1).all()
    ract, rlp, margin = sampler.sample_batch(logits, seed, draws)
    safe = margin > 1e-5
    assert safe.mean() > 0.99
    assert np.array_equal(act[safe], ract[safe])
    same = act == ract
    assert np.allclose(lp[same], rlp[same], rtol=0, atol=2e-6)
    ref_lp = logits - logits.max(1, keepdims=True)
    ref_lp = ref_lp - np.log(np.exp(ref_lp.astype(np.float64)).sum(1, keepdims=True))
    assert np.allclose(lp, ref_lp[np.arange(N), act], atol=3e-6)
    g_act, g_lp, _ = _hm_sample(logits, seed, draws, greedy=True)
    assert np.array_equal(g_act, logits.argmax(1))
    assert np.allclose(g_lp, ref_lp[np.arange(N), g_act], atol=3e-6)


def test_sampler_frequencies_follow_softmax():
    """Chi-square of the sampled action counts against softmax(logits): one fixed logit row, 60k independent draws
    (env index and draw number both vary)."""
    logits = np.tile(np.array([[0.3, -1.2, 1.1]], np.float32), (60000, 1))
    p = np.exp(logits[0].astype(np.float64)); p /= p.sum()
    draws = np.arange(60000) % 7
    act, _, _ = _hm_sample(logits, 99, draws)
    counts = np.bincount(act, minlength=3)
    chi2 = float(((counts - 60000 * p) ** 2 / (60000 * p)).sum())
    assert chi2 < 18.4  # chi-square, 2 degrees of freedom: p = 1e-4
    # degenerate rows never leave the action range
    weird = np.array([[np.inf, 0, 0], [-np.inf, -np.inf, -np.inf], [np.nan, 0, 0], [1e30, -1e30, 0]], np.float32)
    a, _, _ = _hm_sample(weird, 1, np.zeros(4))
    assert ((a >= 0) & (a < 3)).all()


def test_vectorised_uniforms_equal_the_scalar_restatement_and_known_answers():
    """uniform_batch (uint64 numpy Philox) == the pinned scalar restatement and the header, on keys whose high word
    matters, draw numbers past 2^31 and env indices up to 2^20; philox4x32_10_batch reproduces the Random123 vectors."""
    from oracle import sampler
    for ctr, key, want in PHILOX_KAT:
        got = sampler.philox4x32_10_batch([np.full(3, c) for c in ctr], key)
        assert all((w == np.uint64(x)).all() for w, x in zip(got, want))
    rng = np.random.default_rng(11)
    envs = np.concatenate([[0, 1, (1 << 20) - 1, 1 << 20], rng.integers(0, (1 << 20) + 1, 600)])
    draws = np.concatenate([[0, (1 << 31) - 1, 1 << 31, (1 << 32) - 1], rng.integers(0, 1 << 32, 600)])
    for seed in (0x9E3779B97F4A7C15, 0xFFFFFFFF00000000, 1 << 32, 0x1234_5678_9ABC_DEF0, 7):
        u = sampler.uniform_batch(seed, envs, draws)
        want = np.array([sampler.uniform(seed, int(e), int(d)) for e, d in zip(envs, draws)], np.float32)
        assert u.dtype == np.float32 and np.array_equal(u, want), hex(seed)
    # the header draws the same uniforms (hm_sample takes env = row index: the first 2^12 envs, draws past 2^31)
    seed = 0x9E3779B97F4A7C15
    d = rng.integers(1 << 31, 1 << 32, 4096)
    _, _, u_hdr = _hm_sample(np.zeros((4096, 3), np.float32), seed, d)
    assert np.array_equal(u_hdr, sampler.uniform_batch(seed, np.arange(4096), d))
    # the high word of the key changes the stream
    assert not np.array_equal(sampler.uniform_batch(seed, np.arange(64), 0),
                              sampler.uniform_batch(seed & 0xFFFFFFFF, np.arange(64), 0))


def _edge_rows(A):
    """Finite edge rows (ties, spreads from 100 to 6e38 = 3e38 - -3e38, -inf logits) with `A` actions."""
    rows = [[1.0] * A, [2.0] + [5.0] * (A - 1), [5.0] * (A - 1) + [2.0], [0.0] * (A - 1) + [3.0]]
    for s in (100.0, 1e3, 1e5, 1e10, 1e20, 3e38):
        rows += [[s] + [0.0] * (A - 2) + [-s], [-s] + [0.0] * (A - 2) + [s], [0.0] * (A - 1) + [-s],
                 [0.0, -s] + [0.0] * (A - 2)]
    ninf = -np.inf
    rows += [[ninf] + [0.0] * (A - 1), [0.0, ninf] + [1.0] * (A - 2), [1.0] * (A - 1) + [ninf],
             [ninf] * (A - 1) + [0.5], [2.0, ninf] + [2.0] * (A - 2), [ninf, 1e30] + [-1e30] * (A - 2)]
    return np.asarray(rows, np.float32)


@pytest.mark.parametrize("A", [3, 7])
def test_sampler_header_obeys_the_float64_reference_on_edge_rows(A):
    """sample_policy (host build of the header) on edge rows, every row drawn with 2000 draw numbers: the action is one
    reference_f64 allows for the header's own uniform (a -inf logit is never drawn), the log-probability is finite and
    within float32 rounding of log_softmax in float64, and greedy picks the first maximum."""
    from oracle import sampler
    rows = _edge_rows(A)
    R, D = len(rows), 2000
    logits = np.repeat(rows, D, axis=0)
    draws = np.tile(np.arange(D), R) * 7919
    act, lp, u = _hm_sample(logits, 0x9E3779B97F4A7C15, draws)
    _, logp64, allowed = sampler.reference_f64(logits, u)
    n = np.arange(len(logits))
    assert allowed[n, act].all(), np.unique(np.nonzero(~allowed[n, act])[0] // D)
    assert not np.isneginf(logits[n, act]).any()
    assert np.isfinite(lp).all()
    l64 = logits.astype(np.float64)
    z = l64[n, act] - l64.max(axis=1)
    lse = np.log(np.exp(l64 - l64.max(axis=1, keepdims=True)).sum(axis=1))
    assert (np.abs(lp - logp64[n, act]) <= 2e-6 + 4 * 2.0 ** -24 * (np.abs(z) + np.abs(lse))).all()
    g_act, g_lp, _ = _hm_sample(rows, 1, np.zeros(R), greedy=True)
    assert np.array_equal(g_act, np.argmax(rows, axis=1))   # first maximum, ties included
    assert np.isfinite(g_lp).all()


@pytest.mark.parametrize("A", [3, 7])
def test_sampler_header_non_finite_rows_stay_in_range(A):
    """NaN, +inf and all -inf rows: what is specified is an action in [0, A).  The header falls back to the last action
    with logp = NaN when sampling; greedy skips a NaN after the first logit, and a NaN first logit wins."""
    nan, inf = np.nan, np.inf
    rows = np.asarray([[nan] + [0.0] * (A - 1), [0.0, nan] + [1.0] * (A - 2), [0.0] * (A - 1) + [nan],
                       [0.0, inf] + [0.0] * (A - 2), [inf] * A, [-inf] * A, [inf, -inf] + [nan] * (A - 2),
                       [-inf] * (A - 1) + [inf]], np.float32)
    R = len(rows)
    logits = np.repeat(rows, 500, axis=0)
    act, lp, _ = _hm_sample(logits, 0x9E3779B97F4A7C15, np.arange(len(logits)))
    assert ((act >= 0) & (act < A)).all()
    assert (act == A - 1).all() and np.isnan(lp).all()
    g_act, _, _ = _hm_sample(rows, 0, np.zeros(R), greedy=True)
    assert ((g_act >= 0) & (g_act < A)).all()
    assert g_act[0] == 0 and g_act[1] == 2 and g_act[3] == 1 and g_act[4] == 0 and g_act[7] == A - 1


# ---- property tests (hypothesis): arbitrary W x H rooms, full object set, arbitrary action strings ----------------
from hypothesis import HealthCheck, given, settings, strategies as st  # noqa: E402

_OBJS = [(2, 5, 0), (8, 1, 0), (9, 0, 0), (3, 2, 0), (4, 4, 0), (4, 4, 1), (4, 4, 2), (5, 4, 0), (6, 0, 0), (7, 3, 0),
         (4, 2, 1), (5, 2, 0), (5, 4, 0)]


@st.composite
def _rooms(draw):
    W, H = draw(st.integers(3, 14)), draw(st.integers(3, 14))
    enc = np.zeros((1, W, H, 3), np.uint8)
    enc[..., 0] = 1
    enc[:, 0, :, :] = enc[:, -1, :, :] = enc[:, :, 0, :] = enc[:, :, -1, :] = (2, 5, 0)
    interior = [(x, y) for x in range(1, W - 1) for y in range(1, H - 1)]
    ax, ay = draw(st.sampled_from(interior))
    n_obj = draw(st.integers(0, min(12, len(interior) - 1)))
    for _ in range(n_obj):
        x, y = draw(st.sampled_from(interior))
        if (x, y) != (ax, ay):
            enc[0, x, y] = draw(st.sampled_from(_OBJS))
    agent = np.array([[ax, ay, draw(st.integers(0, 3))]], np.int32)
    seven = draw(st.booleans())
    actions = draw(st.lists(st.integers(0, 6 if seven else 2), min_size=1, max_size=40))
    return W, H, enc, agent, seven, actions, draw(st.booleans()), draw(st.sampled_from([0.0, 0.03]))


@settings(max_examples=60, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.data_too_large])
@given(_rooms())
def test_property_kernel_logic_equals_oracle_on_arbitrary_rooms(case):
    """The kernel's per-env arithmetic (env_logic.cuh, compiled for the host) == the oracle for any room shape,
    object placement, wrapper setting and action string; frames, symbolic images, rewards, flags and poses bit-exact."""
    W, H, enc, agent, seven, actions, stuck, bonus = case
    n_actions = 7 if seven else 3
    ref = fast.OracleVecEnv(1, enc, agent, max_steps=25, n_actions=n_actions, auto_reset=False, stuck_penalty=stuck,
                            exploration_bonus=bonus)
    hm = HostModelEnv(codes.pack_encoding(enc), agent, W, H, 25, n_actions, stuck, bonus)
    rgb0, sym0 = ref.reset()
    rgb, sym, *_ = hm.call(np.zeros(1, np.int64), do_step=False)
    assert np.array_equal(sym, sym0) and np.array_equal(rgb, rgb0)
    for a in actions:
        rgb0, r0, te0, tr0, info = ref.step(np.array([a]))
        rgb, sym, r, te, tr, sk = hm.call(np.array([a]), do_step=True)
        assert np.array_equal(r, r0) and np.array_equal(te, te0) and np.array_equal(tr, tr0)
        assert np.array_equal(sk, info["stuck"]) and np.array_equal(sym, info["obs_symbolic"]) and np.array_equal(rgb, rgb0)
        assert (hm.state[0, 0] & 0xFF, (hm.state[0, 0] >> 8) & 0xFF, (hm.state[0, 0] >> 16) & 3) == (ref.ax[0], ref.ay[0], ref.adir[0])
        if te0[0] or tr0[0]:
            break


@settings(max_examples=200, deadline=None)
@given(st.integers(0, (1 << 49) - 1))
def test_property_visibility_invariants(transp):
    """process_vis invariants on any 49-bit transparency pattern: the agent cell is always visible, the row in front of
    it is reachable only through transparent cells, visibility is monotone in transparency, and an all-opaque row
    hides everything behind it."""
    lib = _host_model()
    lib.hm_visibility.restype = ctypes.c_uint64
    lib.hm_visibility.argtypes = [ctypes.c_uint64]
    vis = lib.hm_visibility(transp)
    agent_bit = 1 << (6 * 7 + 3)
    assert vis & agent_bit
    more = lib.hm_visibility(transp | (1 << 20) | (1 << 45))
    assert more & vis == vis  # monotone: making cells transparent never hides anything
    for row in range(6):  # rows are vj = 0 (far) .. 6 (agent row)
        if (transp >> (row * 7)) & 0x7F == 0 and row < 6:
            hidden_above = (1 << (row * 7)) - 1
            lit_row = (vis >> (row * 7)) & 0x7F
            if lit_row == 0:
                assert vis & hidden_above == 0
    if not (transp & agent_bit):  # the agent stands on an opaque cell (closed door): it sees only its own cell
        assert vis == agent_bit
