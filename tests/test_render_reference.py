"""A reference for frames rendered from symbolic observations that uses no product code, and its CPU anchor.

RGBImgPartialObsWrapper.observation, restated from the stored `Grid.encode` image alone: every cell's tile is the
literal `Grid.render_tile` (oracle.fast.TileAtlas over minigrid_restated), chosen by (type, colour, state, agent,
highlight) -- an unseen cell is the plain empty tile, the agent's cell (vi, vj) = (3, 6) shows the agent over what it
carries, every other cell is highlighted.  tests/test_gpu_render.py holds the render kernels to this reference bit for bit;
the tests here pin the reference itself to the oracle's own frames."""
from __future__ import annotations

import numpy as np

from oracle import fast
from oracle import minigrid_restated as mg

VIEW, TILE = 7, 8
AGENT_CELL = (VIEW // 2, VIEW - 1)   # [vi][vj] of the agent in the stored image
AGENT_FLAT = AGENT_CELL[0] * VIEW + AGENT_CELL[1]


def _producible():
    """(type, colour, state) triples Grid.encode can store: unseen, empty, and every object that decodes and re-encodes
    to itself (a goal is always green, lava always red, only doors have a state)."""
    out = [(0, 0, 0), (1, 0, 0)]
    for t in range(2, 10):
        for c in range(6):
            for s in range(3):
                obj = mg.WorldObj.decode(t, c, s)
                if obj is not None and tuple(int(v) for v in obj.encode()) == (t, c, s):
                    out.append((t, c, s))
    return out


PRODUCIBLE = _producible()                                                   # 52 triples
AGENT_CASES = [(1, 0, 0)] + [(t, c, 0) for t in (5, 6, 7) for c in range(6)]  # carrying nothing, a key, ball or box: 19

_ATLAS = None


def reference_atlas():
    """TileAtlas with every tile a producible image can show (agent and highlight variants included)."""
    global _ATLAS
    if _ATLAS is None:
        atlas = fast.TileAtlas(TILE)
        atlas.ensure([t for t in PRODUCIBLE if t[0] != 0])
        _ATLAS = atlas
    return _ATLAS


def reference_slots(sym):
    """u8[M, 7, 7, 3] stored images -> int64[M, 7, 7] TileAtlas slots (fast.tile_slot), for numpy input."""
    sym = np.asarray(sym)
    t, c, s = (sym[..., k].astype(np.int64) for k in range(3))
    agent = np.zeros(sym.shape[:-1], np.int64)
    agent[:, AGENT_CELL[0], AGENT_CELL[1]] = 1
    unseen = t == 0
    slots = fast.tile_slot(np.where(unseen, 1, t), np.where(unseen, 0, c), np.where(unseen, 0, s), agent,
                           np.where(unseen, 0, 1))
    if not reference_atlas().present[slots].all():
        raise ValueError("image holds a triple Grid.encode cannot produce")
    return slots


def _permute(x, axes):
    return x.permute(*axes) if hasattr(x, "permute") else x.transpose(axes)


def frames_from_slots(tiles, slots):
    """Gather tiles [S, 8, 8, 3] by slots [M, 7(vi), 7(vj)] into frames [M, 56, 56, 3]: pixel row vj*8 + py, column
    vi*8 + px.  Works on numpy arrays and on torch tensors alike (the GPU tests expand on the device)."""
    m = slots.shape[0]
    g = tiles[slots.reshape(-1)].reshape(m, VIEW, VIEW, TILE, TILE, 3)
    return _permute(g, (0, 2, 3, 1, 4, 5)).reshape(m, VIEW * TILE, VIEW * TILE, 3)


def blocked_of(rgb):
    """u8[M, 56, 56, 3] -> u8[M, 14, 14, 48]: every 4x4 pixel block contiguous, channel index c*16 + dy*4 + dx."""
    m = rgb.shape[0]
    return _permute(rgb.reshape(m, 14, 4, 14, 4, 3), (0, 1, 3, 5, 2, 4)).reshape(m, 14, 14, 48)


def reference_frames(sym):
    return frames_from_slots(reference_atlas().tiles, reference_slots(sym))


def f32_table(normalise):
    """float32 value of each pixel byte: 0 the byte itself, 1 torch's CPU `x / 255.0` (IEEE division), 2 torch's CUDA
    `x / 255.0` (multiplication by the float32 reciprocal)."""
    px = np.arange(256, dtype=np.float32)
    if normalise == 0:
        return px
    if normalise == 1:
        return px / np.float32(255)
    return px * (np.float32(1) / np.float32(255))


def catalogue():
    """u8[52, 7, 7, 3]: image k holds producible triple (k + p) mod 52 at non-agent position p, so every triple sits at
    each of the 48 non-agent positions once; its agent cell holds case k mod 19."""
    n = len(PRODUCIBLE)
    trip = np.asarray(PRODUCIBLE, np.uint8)
    sym = np.zeros((n, VIEW * VIEW, 3), np.uint8)
    others = [p for p in range(VIEW * VIEW) if p != AGENT_FLAT]
    for k in range(n):
        for j, p in enumerate(others):
            sym[k, p] = trip[(k + j) % n]
        sym[k, AGENT_FLAT] = AGENT_CASES[k % len(AGENT_CASES)]
    return sym.reshape(n, VIEW, VIEW, 3)


def random_images(rng, m):
    """u8[m, 7, 7, 3]: every non-agent cell a uniform producible triple, the agent cell a uniform agent case."""
    trip = np.asarray(PRODUCIBLE, np.uint8)
    sym = trip[rng.integers(0, len(trip), (m, VIEW * VIEW))]
    sym[:, AGENT_FLAT] = np.asarray(AGENT_CASES, np.uint8)[rng.integers(0, len(AGENT_CASES), m)]
    return sym.reshape(m, VIEW, VIEW, 3)


# ---- the CPU anchor: the reference against the oracle's own frames ------------------------------------------------
def _rollout_matches_oracle(enc, agent, n_actions, n_envs, steps, seed):
    ref = fast.OracleVecEnv(n_envs, enc, agent, n_actions=n_actions, max_steps=19)
    rgb, sym = ref.reset()
    rng = np.random.default_rng(seed)
    frames = carried = 0
    for _ in range(steps + 1):
        assert np.array_equal(reference_frames(sym), rgb)
        assert np.array_equal(blocked_of(reference_frames(sym)), blocked_of(rgb))
        frames += sym.shape[0]
        carried += int((sym[:, AGENT_CELL[0], AGENT_CELL[1], 0] != 1).sum())
        a = rng.integers(0, n_actions, n_envs)
        if n_actions == 7:
            a = np.where(rng.random(n_envs) < 0.3, 3, a)   # many pickups: carried objects under the agent
        rgb, _, _, _, info = ref.step(a)
        sym = info["obs_symbolic"]
    return frames, carried


def test_reference_equals_oracle_frames_on_merlin_pools():
    from merlin_b200 import codes, layouts
    for diff, size in (("mediumhard", 16), ("hardest", 16), ("easy", 8)):
        cells, agent = layouts.generate(diff, size, range(300, 340))
        frames, _ = _rollout_matches_oracle(codes.unpack_to_encoding(cells, size, size), agent, 3, 500, 7, seed=size)
        assert frames == 4000


def test_reference_equals_oracle_frames_with_objects_and_pickups():
    from test_gpu_parity import _object_layouts
    enc, agent = _object_layouts(np.random.default_rng(9), 64, 11)
    frames, carried = _rollout_matches_oracle(enc, agent, 7, 500, 23, seed=9)
    assert frames == 12000 and carried > 100


def test_catalogue_and_random_images_cover_the_producible_set():
    assert len(PRODUCIBLE) == 52 and len(set(PRODUCIBLE)) == 52 and len(set(AGENT_CASES)) == 19
    cat = catalogue().reshape(-1, VIEW * VIEW, 3)
    others = [p for p in range(VIEW * VIEW) if p != AGENT_FLAT]
    for p in others:
        assert {tuple(v) for v in cat[:, p].tolist()} == set(PRODUCIBLE)
    assert {tuple(v) for v in cat[:, AGENT_FLAT].tolist()} == set(AGENT_CASES)
    rnd = random_images(np.random.default_rng(0), 4000).reshape(-1, VIEW * VIEW, 3)
    assert {tuple(v) for v in rnd[:, others].reshape(-1, 3).tolist()} == set(PRODUCIBLE)
    reference_slots(catalogue())   # every tile is in the atlas
    bad = catalogue()
    bad[0, 0, 0] = (8, 2, 0)       # a blue goal: no object encodes to it
    try:
        reference_slots(bad)
    except ValueError:
        pass
    else:
        raise AssertionError("a triple outside the producible set was accepted")


def test_reference_tiles_are_distinct_where_the_kernels_could_confuse_them():
    """Every producible cell content draws a tile of its own -- except a green wall, which Grid.render_tile fills
    exactly like the (always green) goal -- so a kernel that picks the wrong tile for a cell cannot match the reference
    by accident; the f32 tables differ where torch's two roundings differ."""
    atlas = reference_atlas()
    cases = [((1, 0, 0), 0, 0)] + [(t, 0, 1) for t in PRODUCIBLE[1:]] + [(t, 1, 1) for t in AGENT_CASES]
    first, same = {}, []
    for (t, c, s), agent, hl in cases:
        key = atlas.tiles[fast.tile_slot(t, c, s, agent, hl)].tobytes()
        if key in first:
            same.append((first[key], (t, c, s)))
        first.setdefault(key, (t, c, s))
    assert same == [((2, 1, 0), (8, 1, 0))]
    t1, t2 = f32_table(1), f32_table(2)
    assert (t1 != t2).any() and np.array_equal(f32_table(0), np.arange(256, dtype=np.float32))
    assert t1[255] == np.float32(1) and t1.dtype == t2.dtype == np.float32
