"""Render kernels against an independent reference (run with -m gpu on a B200): merlin_env_render (u8 frames, both
layouts) and merlin_env_render_f32 (the first layer's float32 input, three roundings) in every launch mode, compared bit
for bit with the literal tile renderer of tests/test_render_reference.py -- not with frames the step kernels wrote, which
share the product's atlas and kind mapping with the render kernels.

Inputs: a catalogue that puts every triple Grid.encode can produce at every non-agent cell and shows all 19 agent-cell
contents, random images over that set, and symbolic rollouts stepped on MERLIN pools.  Every output sits between 4 KB
guard bands and starts out as a sentinel (u8 0xA5, f32 -7.0): each test checks that every frame was written and that
nothing outside the output changed.

The tests of images that show tile kinds the handle's current pool cannot come first: a CTA that reads a tile it never
staged would find whatever an earlier launch left in shared memory there, and a launch that staged the whole atlas can
make such a frame look right.  They also install an inverted atlas (255 - every byte) after any step ran on the handle,
so no stale copy of a tile can hold the bytes the frame needs."""
from __future__ import annotations

import numpy as np
import pytest
import torch

from oracle import fast
from test_gpu_parity import _object_layouts
from test_render_reference import (blocked_of, catalogue, f32_table, frames_from_slots, random_images,
                                   reference_atlas, reference_slots)

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
FRAME = 56 * 56 * 3
GUARD = 4096                        # bytes of sentinel before and after every output
U8_SENTINEL, F32_SENTINEL = 0xA5, -7.0
NORMALISE = {0: False, 1: "divide", 2: "reciprocal"}
CHUNK = 8192                        # frames compared per slice (bounds the reference's device memory)


def _merlin_pool(size=11, n=64, first=0):
    from merlin_b200 import codes, layouts
    cells, agent = layouts.generate("mediumhard", size, range(first, first + n))
    return codes.unpack_to_encoding(cells, size, size), agent


def _env(num_envs, enc, agent, n_actions=3, **kw):
    from merlin_b200 import BatchedMerlinEnv
    return BatchedMerlinEnv(num_envs, enc=enc, agent=agent, n_actions=n_actions, device=DEV, **kw)


def _set_atlas(env, tiles):
    from merlin_b200 import _lib
    tiles = np.ascontiguousarray(tiles, dtype=np.uint8)
    _lib.check(env._lib.merlin_env_set_tile_atlas(env._h, tiles.ctypes.data, tiles.shape[0]))


def _invert_atlas(env):
    from merlin_b200 import tiles
    _set_atlas(env, 255 - tiles.build_atlas())


class Reference:
    """Reference frames u8[R, 56, 56, 3] of stored rows, expanded on the device from the literal tile atlas."""

    def __init__(self, sym, inverted=False):
        sym = np.asarray(sym.cpu() if torch.is_tensor(sym) else sym).reshape(-1, 7, 7, 3)
        tiles = torch.as_tensor(reference_atlas().tiles, device=DEV)
        if inverted:
            tiles = 255 - tiles
        self.tiles = tiles
        self.slots = torch.as_tensor(reference_slots(sym), device=DEV)
        self.n_rows = sym.shape[0]

    def frames(self, rows, blocked=False):
        rgb = frames_from_slots(self.tiles, self.slots[rows])
        return blocked_of(rgb) if blocked else rgb


def _render(env, sym, m, index=None, blocked=False, normalise=None, stream=None):
    """Render into a sentinel-filled output between guard bands; returns (whole buffer, output view)."""
    f32 = normalise is not None
    shape = (m, 14, 14, 48) if blocked else (m, 56, 56, 3)
    if f32:
        g = GUARD // 4
        buf = torch.full((g + m * FRAME + g,), F32_SENTINEL, dtype=torch.float32, device=DEV)
    else:
        g = GUARD
        buf = torch.full((g + m * FRAME + g,), U8_SENTINEL, dtype=torch.uint8, device=DEV)
    out = buf[g:g + m * FRAME].view(shape)
    if stream is not None:
        stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(stream):
            got = env.render(sym, index, out=out, blocked=blocked, dtype=torch.float32 if f32 else torch.uint8,
                             normalise=NORMALISE[normalise] if f32 else False)
    else:
        got = env.render(sym, index, out=out, blocked=blocked, dtype=torch.float32 if f32 else torch.uint8,
                         normalise=NORMALISE[normalise] if f32 else False)
    assert got.data_ptr() == out.data_ptr()
    return buf, out


def _check(buf, out, ref, rows, blocked=False, normalise=None, what=""):
    """`out` == the reference frames of `rows` bit for bit, every frame written, both guard bands untouched."""
    f32 = normalise is not None
    sentinel = F32_SENTINEL if f32 else U8_SENTINEL
    g = GUARD // 4 if f32 else GUARD
    m = out.shape[0]
    assert bool((buf[:g] == sentinel).all()) and bool((buf[-g:] == sentinel).all()), f"{what}: wrote outside its output"
    assert not bool((out.view(m, -1) == sentinel).all(dim=1).any()), f"{what}: a frame was not written"
    rows = torch.as_tensor(rows, device=DEV)
    table = torch.as_tensor(f32_table(normalise), device=DEV) if f32 else None
    for lo in range(0, m, CHUNK):
        want = ref.frames(rows[lo:lo + CHUNK], blocked)
        if f32:
            want = table[want.long()]
        got = out[lo:lo + CHUNK]
        if not torch.equal(got, want):
            bad = (got != want).reshape(got.shape[0], -1).any(dim=1).nonzero()[:, 0]
            raise AssertionError(f"{what}: {bad.numel()} frames differ from the reference, first at frame {lo + int(bad[0])}")


def _check_all_modes(env, ref, sym, rows_m, index=None, rows=None, what=""):
    """u8 in both layouts and f32 in all three roundings."""
    rows = torch.arange(rows_m, device=DEV) if rows is None else rows
    for blocked in (False, True):
        buf, out = _render(env, sym, rows_m, index, blocked=blocked)
        _check(buf, out, ref, rows, blocked, what=f"{what} u8 blocked={blocked}")
    for nm in (0, 1, 2):
        buf, out = _render(env, sym, rows_m, index, blocked=True, normalise=nm)
        _check(buf, out, ref, rows, True, nm, what=f"{what} f32 normalise={nm}")


# ---- tile kinds the current layout pool cannot show (first: see the module docstring) ---------------------------------
@pytest.mark.parametrize("m", [52, 9, 8193, 65536])
def test_catalogue_on_a_fresh_merlin_handle(m):
    """Every producible image on a 3-action handle whose pool shows 5 tile kinds: u8 with groups of 8 and of 32, f32
    one CTA per frame and in ticket mode."""
    enc, agent = _merlin_pool()
    env = _env(64, enc, agent)
    _invert_atlas(env)
    cat = catalogue()
    ref = Reference(cat, inverted=True)
    sym = torch.as_tensor(cat, device=DEV)
    if m == len(cat):
        _check_all_modes(env, ref, sym, m, what=f"catalogue M={m}")
    else:
        idx = torch.arange(m, device=DEV) % len(cat)
        _check_all_modes(env, ref, sym, m, index=idx, rows=idx, what=f"catalogue M={m}")


@pytest.mark.parametrize("new_pool", ["same_size", "other_size"])
def test_stored_images_rendered_after_the_pool_changed(new_pool):
    """Observations stepped on an object pool (doors, lava, floor, keys, balls, boxes), rendered after upload_layouts
    replaced it by a MERLIN pool: the reference, and the frames the step wrote."""
    from merlin_b200 import codes
    rng = np.random.default_rng(21)
    enc, agent = _object_layouts(rng, 48, 11)
    N, T = 512, 12
    env = _env(N, enc, agent, max_steps=9)
    sym = torch.empty((T + 1, N, 7, 7, 3), dtype=torch.uint8, device=DEV)
    rgb = torch.empty((T + 1, N, 56, 56, 3), dtype=torch.uint8, device=DEV)
    env.reset(out_obs=rgb[0], out_symbolic=sym[0])
    for t in range(T):
        env.step(torch.as_tensor(rng.integers(0, 3, N), device=DEV), out_obs=rgb[t + 1], out_symbolic=sym[t + 1])
    types = set(np.unique(sym[..., 0].cpu().numpy()).tolist())
    assert {3, 4, 5, 6, 7, 9} <= types   # floor, doors, key, ball, box, lava are all on view
    menc, magent = _merlin_pool(11, 48 if new_pool == "same_size" else 20, first=500)
    env.upload_layouts(codes.pack_encoding(menc), magent)
    _invert_atlas(env)   # after the steps: no stale copy of a tile in shared memory holds what the frames need
    flat_sym, flat_rgb = sym.reshape(-1, 7, 7, 3), rgb.reshape(-1, 56, 56, 3)
    R = flat_sym.shape[0]
    ref = Reference(flat_sym, inverted=True)
    assert torch.equal(ref.frames(torch.arange(R, device=DEV)), 255 - flat_rgb)   # reference == the step's frames
    _check_all_modes(env, ref, flat_sym, R, what="all stored rows")
    idx = torch.as_tensor(rng.integers(0, R, 65537), device=DEV)
    buf, out = _render(env, flat_sym, idx.numel(), idx)
    _check(buf, out, ref, idx, what="65 537 gathered rows, groups of 32")
    assert torch.equal(out, 255 - flat_rgb[idx])
    buf, out = _render(env, flat_sym, 16385, idx[:16385], blocked=True, normalise=1)
    _check(buf, out, ref, idx[:16385], True, 1, what="16 385 gathered rows, f32 ticket mode")


# ---- every launch mode, both handle kinds -------------------------------------------------------------------------
@pytest.fixture(scope="module")
def source():
    """Stored rows: the catalogue, 100 000 random images and 163 840 observations of 3-action MERLIN rollouts (4096 envs
    x 40 steps), on the device; with their reference."""
    rng = np.random.default_rng(7)
    enc, agent = _merlin_pool(16, 256, first=1000)
    env = _env(4096, enc, agent, max_steps=30)
    roll = torch.empty((40, 4096, 7, 7, 3), dtype=torch.uint8, device=DEV)
    env.reset()
    for t in range(40):
        env.step(torch.as_tensor(rng.integers(0, 3, 4096), device=DEV), out_symbolic=roll[t], frames=False)
    env.close()
    sym = torch.cat([torch.as_tensor(catalogue(), device=DEV), torch.as_tensor(random_images(rng, 100_000), device=DEV),
                     roll.reshape(-1, 7, 7, 3)]).contiguous()
    return sym, Reference(sym), roll.reshape(-1, 7, 7, 3).contiguous()


@pytest.fixture(scope="module")
def handles():
    """A 3-action MERLIN handle (5 tile kinds: render_f32 stages cap_tiles = 8) and a 7-action handle (mutable grids:
    every atlas slot staged, render_f32 opts in to more than 48 KB of shared memory)."""
    enc, agent = _merlin_pool()
    oenc, oagent = _object_layouts(np.random.default_rng(4), 32, 11)
    return {3: _env(64, enc, agent), 7: _env(64, oenc, oagent, n_actions=7)}


U8_SIZES = [1, 7, 8, 9, 8191, 65535, 65536, 65537, 262147]   # straddle the 8/32 group switch, ragged last groups, > 2^31 B
F32_SIZES = [1, 445, 8191, 8192, 8193, 16384, 16385, 40000]  # one CTA per frame (445: the grid strides) / ticket mode


@pytest.mark.parametrize("n_actions,m", [(a, m) for a in (3, 7) for m in U8_SIZES])
def test_render_u8_every_size(source, handles, n_actions, m):
    sym, ref, _ = source
    env = handles[n_actions]
    R = sym.shape[0]
    gather = torch.as_tensor(np.random.default_rng(m).integers(0, R, m), device=DEV)
    for blocked in (False, True):
        buf, out = _render(env, sym[:m], m, blocked=blocked)
        _check(buf, out, ref, torch.arange(m, device=DEV), blocked, what=f"M={m} rows 0..M-1 blocked={blocked}")
        del buf, out
        buf, out = _render(env, sym, m, gather, blocked=blocked)
        _check(buf, out, ref, gather, blocked, what=f"M={m} gathered blocked={blocked}")
        del buf, out


@pytest.mark.parametrize("n_actions,m", [(a, m) for a in (3, 7) for m in F32_SIZES])
def test_render_f32_every_size(source, handles, n_actions, m):
    sym, ref, _ = source
    env = handles[n_actions]
    R = sym.shape[0]
    gather = torch.as_tensor(np.random.default_rng(m + 1).integers(0, R, m), device=DEV)
    for nm in (0, 1, 2):
        buf, out = _render(env, sym[:m], m, blocked=True, normalise=nm)
        _check(buf, out, ref, torch.arange(m, device=DEV), True, nm, what=f"M={m} rows 0..M-1 normalise={nm}")
        buf, out = _render(env, sym, m, gather, blocked=True, normalise=nm)
        _check(buf, out, ref, gather, True, nm, what=f"M={m} gathered normalise={nm}")


@pytest.mark.parametrize("n_actions", [3, 7])
def test_gather_edge_cases(source, handles, n_actions):
    sym, ref, _ = source
    env = handles[n_actions]
    R = sym.shape[0]
    cases = {
        "repeated rows": torch.tensor([5, 5, 5, 0, 0, 51, 51, 5, 17], device=DEV),
        "reversed": torch.arange(R - 1, R - 1 - 9000, -1, device=DEV),
        # rows outside [0, n_rows) render row 0: the library never reads outside the buffer it was given
        "out of range": torch.tensor([-1, R, 2 ** 40, 3, -(2 ** 40), R - 1, 2 ** 63 - 1, -(2 ** 63)], device=DEV),
    }
    for name, idx in cases.items():
        rows = torch.where((idx < 0) | (idx >= R), torch.zeros_like(idx), idx)
        _check_all_modes(env, ref, sym, idx.numel(), index=idx, rows=rows, what=name)
    # more frames than rows: 20 000 frames from the 52 catalogue rows (u8 with groups of 8, f32 in ticket mode)
    idx = torch.as_tensor(np.random.default_rng(3).integers(0, 52, 20000), device=DEV)
    _check_all_modes(env, ref, sym[:52], idx.numel(), index=idx, rows=idx, what="more frames than rows")
    # a non-contiguous index tensor
    wide = torch.as_tensor(np.random.default_rng(5).integers(0, R, 3 * 700), device=DEV)
    idx = wide[::3]
    assert not idx.is_contiguous()
    _check_all_modes(env, ref, sym, idx.numel(), index=idx, rows=idx.contiguous(), what="non-contiguous index")


# ---- the self-rearming ticket counters ------------------------------------------------------------------------------
def test_forty_renders_on_two_streams_between_steps(source):
    """40 renders on one handle cycle through u8 with groups of 32 and of 8, f32 in ticket mode and one CTA per frame,
    alternating two streams, with a step after every pair: every render is complete and exact, every step bit-exact
    against the oracle.  A counter pair left armed would make a later render on it skip groups silently."""
    _, _, roll = source
    ref_roll = Reference(roll)
    enc, agent = _merlin_pool(16, 64, first=3000)
    N = 256
    env = _env(N, enc, agent, max_steps=13)
    oracle = fast.OracleVecEnv(N, enc, agent, max_steps=13)
    obs, _ = env.reset()
    assert np.array_equal(obs.cpu().numpy(), oracle.reset()[0])
    streams = [torch.cuda.Stream(DEV), torch.cuda.Stream(DEV)]
    rng = np.random.default_rng(40)
    modes = [(65537, False, None), (8193, True, None), (16385, True, 2), (445, True, 1)]
    for i in range(0, 40, 2):
        done = []
        for j in (i, i + 1):
            m, blocked, nm = modes[j % 4]
            idx = torch.as_tensor(rng.integers(0, roll.shape[0], m), device=DEV)
            buf, out = _render(env, roll, m, idx, blocked=blocked, normalise=nm, stream=streams[j % 2])
            done.append((buf, out, idx, blocked, nm, j))
        a = rng.integers(0, 3, N)
        obs, *_ = env.step(torch.as_tensor(a, device=DEV))
        robs, *_ = oracle.step(a)
        torch.cuda.synchronize()
        for buf, out, idx, blocked, nm, j in done:
            _check(buf, out, ref_roll, idx, blocked, nm, what=f"render {j}")
        assert np.array_equal(obs.cpu().numpy(), robs), f"step after render {i + 1}"
    a = rng.integers(0, 3, N)
    obs, *_ = env.step(torch.as_tensor(a, device=DEV))
    assert np.array_equal(obs.cpu().numpy(), oracle.step(a)[0])


def test_ticket_renders_replayed_from_a_cuda_graph(source):
    """One u8 render with groups of 32 and one f32 ticket-mode render captured in a CUDA graph, replayed 20 times with
    the sentinels refilled in between: every replay writes every frame."""
    _, _, roll = source
    ref_roll = Reference(roll)
    enc, agent = _merlin_pool()
    env = _env(64, enc, agent)
    rng = np.random.default_rng(20)
    idx_u8 = torch.as_tensor(rng.integers(0, roll.shape[0], 65537), device=DEV)
    idx_f32 = torch.as_tensor(rng.integers(0, roll.shape[0], 8200), device=DEV)
    buf_u8 = torch.full((GUARD + 65537 * FRAME + GUARD,), U8_SENTINEL, dtype=torch.uint8, device=DEV)
    buf_f32 = torch.full((GUARD // 4 + 8200 * FRAME + GUARD // 4,), F32_SENTINEL, dtype=torch.float32, device=DEV)
    out_u8 = buf_u8[GUARD:GUARD + 65537 * FRAME].view(65537, 14, 14, 48)
    out_f32 = buf_f32[GUARD // 4:GUARD // 4 + 8200 * FRAME].view(8200, 14, 14, 48)

    def renders():
        env.render(roll, idx_u8, out=out_u8, blocked=True)
        env.render(roll, idx_f32, out=out_f32, blocked=True, dtype=torch.float32, normalise="divide")

    side = torch.cuda.Stream(DEV)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        renders()   # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        renders()
    for rep in range(20):
        buf_u8.fill_(U8_SENTINEL)
        buf_f32.fill_(F32_SENTINEL)
        graph.replay()
        torch.cuda.synchronize()
        _check(buf_u8, out_u8, ref_roll, idx_u8, True, what=f"replay {rep} u8")
        _check(buf_f32, out_f32, ref_roll, idx_f32, True, 1, what=f"replay {rep} f32")
