"""GPU tier: the C ABI driven from plain C (tests/csrc/cabi_smoke.c: gcc + libcudart only, no Python in the loop), and a
loose throughput floor for the step kernel so that a mapping regression cannot pass silently."""
from __future__ import annotations

import json
import os
import subprocess

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def test_c_program_links_and_runs_against_the_shared_library(tmp_path):
    from merlin_b200 import _lib
    _lib.load()
    out = str(tmp_path / "cabi_smoke")   # built outside the repository tree, which may be read-only
    libdir = os.path.dirname(_lib.LIB_PATH)
    subprocess.check_call(["gcc", os.path.join(ROOT, "tests", "csrc", "cabi_smoke.c"), "-I" + os.path.join(ROOT, "include"),
                           "-I/usr/local/cuda/include", "-L" + libdir, "-lmerlin_b200", "-L/usr/local/cuda/lib64", "-lcudart",
                           "-lm", "-Wl,-rpath," + libdir, "-o", out])
    res = subprocess.run([out], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr
    assert "cabi_smoke ok" in res.stdout


def test_step_kernel_throughput_floor():
    """262 144 mediumhard envs, RGB: the measured figure is ~1.07 of the HBM copy peak; fail below 0.8."""
    from merlin_b200 import BatchedMerlinEnv, layouts
    try:
        peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        peak = 6650.0
    N = 262144
    cells, agent = layouts.generate("mediumhard", 16, range(777_000_000, 777_000_000 + 1024))
    env = BatchedMerlinEnv(N, cells, agent, width=16, height=16, device="cuda:0", want_symbolic=False)
    env.reset()
    acts = torch.randint(0, 3, (8, N), device="cuda:0")
    for i in range(8):
        env.step(acts[i % 8])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(64):
        env.step(acts[i % 8])
    e1.record()
    torch.cuda.synchronize()
    gbs = 9710 * N * 64 / e0.elapsed_time(e1) / 1e6
    assert "tile" in env.step_kernel()
    assert gbs > 0.8 * peak, f"{gbs:.0f} GB/s of algorithmic traffic = {gbs / peak:.2f} of the HBM peak"
