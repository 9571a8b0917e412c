"""CPU tier: ppo-2dgrid_b200/csrc/np_random.cuh -- the restatement of numpy's `default_rng(seed)` stream that the seeded
layout kernel runs -- compiled for the host (tests/csrc/np_random_model.cpp) and compared with numpy itself: the
SeedSequence state, PCG64's raw outputs, `integers` over degenerate to 2^32-wide ranges, and `choice(replace=False)`
interleaved with `integers`, each for 2 000+ seeds including the ends of the 32- and 64-bit seed ranges."""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
SEEDS = np.array(list(range(1800)) + list(range(200_000, 200_050)) + list(range(777_000_000, 777_000_050))
                 + [2**32 - 2, 2**32 - 1, 2**32, 2**32 + 1, 2**40 + 3, 2**63 - 1, 2**63, 2**63 + 5, 2**64 - 2, 2**64 - 1]
                 + [int(s) for s in np.random.default_rng(5).integers(0, 2**64, 90, dtype=np.uint64)], dtype=np.uint64)
WHY = f"(numpy {np.__version__}; np_random.cuh restates numpy 2.3.5)"


@pytest.fixture(scope="module")
def lib():
    src = os.path.join(ROOT, "tests", "csrc", "np_random_model.cpp")
    hdr = os.path.join(ROOT, "ppo-2dgrid_b200", "csrc", "np_random.cuh")
    out = os.path.join(ROOT, "tests", "csrc", "_build", "libnp_random_model.so")
    if not os.path.exists(out) or os.path.getmtime(out) < max(os.path.getmtime(f) for f in (src, hdr)):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I" + os.path.dirname(hdr),
                               src, "-o", out])
    return ctypes.CDLL(out)


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _run_script(lib, seeds, ops):
    ops = np.ascontiguousarray(ops, dtype=np.int64).reshape(-1, 3)
    n_out = int(sum(1 if kind == 0 else b for kind, _, b in ops))
    seeds = np.ascontiguousarray(seeds, dtype=np.uint64)
    out = np.zeros((len(seeds), n_out), dtype=np.int64)
    lib.nr_script(_p(seeds), ctypes.c_int(len(seeds)), _p(ops), ctypes.c_int(len(ops)), ctypes.c_int(n_out), _p(out))
    return out


def _numpy_script(seed, ops):
    g = np.random.default_rng(int(seed))
    vals = []
    for kind, a, b in ops:
        if kind == 0:
            vals.append(int(g.integers(a, b)))
        else:
            vals.extend(int(v) for v in g.choice(a, size=b, replace=False))
    return vals


def test_seed_count():
    assert len(SEEDS) >= 2000 and len(set(SEEDS.tolist())) == len(SEEDS)
    assert {0, 2**32 - 1, 2**32, 2**63, 2**64 - 1} <= set(int(s) for s in SEEDS)


def test_seed_sequence_state(lib):
    out = np.zeros((len(SEEDS), 4), dtype=np.uint64)
    lib.nr_seed_state(_p(SEEDS), ctypes.c_int(len(SEEDS)), _p(out))
    ref = np.stack([np.random.SeedSequence(int(s)).generate_state(4, np.uint64) for s in SEEDS])
    bad = np.flatnonzero((out != ref).any(1))
    assert bad.size == 0, f"SeedSequence state differs for seeds {SEEDS[bad[:5]].tolist()} {WHY}"


def test_pcg64_raw_outputs(lib):
    count = 24
    out = np.zeros((len(SEEDS), count), dtype=np.uint64)
    lib.nr_raw(_p(SEEDS), ctypes.c_int(len(SEEDS)), ctypes.c_int(count), _p(out))
    ref = np.stack([np.random.PCG64(int(s)).random_raw(count) for s in SEEDS])
    bad = np.flatnonzero((out != ref).any(1))
    assert bad.size == 0, f"PCG64 raw outputs differ for seeds {SEEDS[bad[:5]].tolist()} {WHY}"


# degenerate (one value: no draw), narrow, the layout routines' ranges, and widths up to 2^32 (one whole next_uint32)
RANGES = [(0, 1), (7, 8), (0, 2), (1, 15), (2, 6), (0, 4), (19, 40), (6, 13), (3, 4), (1, 2), (-5, 5), (0, 3),
          (0, 2**16 + 1), (0, 2**31 - 1), (0, 2**31), (10**9, 10**9 + 2**31), (-(2**31), 1), (0, 2**32), (5, 6), (0, 253)]


def test_integers(lib):
    ops = [(0, lo, hi) for _ in range(2) for lo, hi in RANGES]  # 40 calls: the buffered half-word spans calls
    out = _run_script(lib, SEEDS, ops)
    for i, s in enumerate(SEEDS):
        ref = _numpy_script(s, ops)
        assert out[i].tolist() == ref, f"integers differ for seed {int(s)}: {out[i].tolist()} vs {ref} {WHY}"


def _choice_scripts():
    """Four scripts of interleaved choice(pop, k, replace=False) and integers calls, as hard's `_gen_grid` makes them
    (pop = H - 2 gap rows, k = 1..5) plus the edges k == pop and pop == 1."""
    r = np.random.default_rng(11)
    scripts = []
    for _ in range(4):
        ops = [(1, 1, 1), (1, 3, 3), (0, 2, 6)]
        for _ in range(14):
            pop = int(r.choice([3, 6, 9, 14, 22, 30, 62, 253]))
            ops.append((1, pop, int(r.integers(1, min(pop, 5) + 1))))
            ops.extend((0, int(lo), int(lo) + int(w)) for lo, w in zip(r.integers(0, 20, 2), r.integers(1, 40, 2)))
        scripts.append(ops)
    return scripts


def test_choice_interleaved_with_integers(lib):
    for k, ops in enumerate(_choice_scripts()):
        seeds = SEEDS[k::4]
        out = _run_script(lib, seeds, ops)
        for i, s in enumerate(seeds):
            ref = _numpy_script(s, ops)
            assert out[i].tolist() == ref, f"script {k}, seed {int(s)}: {out[i].tolist()} vs {ref} {WHY}"
