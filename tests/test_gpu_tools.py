"""GPU tier: the measurement tools run end to end on tiny configurations and print the JSON they promise."""
from __future__ import annotations

import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def _run(args, timeout=600):
    res = subprocess.run([sys.executable] + args, cwd=ROOT, capture_output=True, text=True, timeout=timeout)
    assert res.returncode == 0, res.stderr[-2000:]
    return res.stdout.strip().splitlines()


def test_train_ppo_tool_tiny(tmp_path):
    ckpt = str(tmp_path / "ppo.pth")
    lines = _run(["tools/train_ppo.py", "--envs", "64", "--horizon", "8", "--minibatch", "128", "--update-epochs", "1",
                  "--total-steps", "1024", "--layouts", "256", "--eval-tasks", "4", "--save", ckpt])
    out = json.loads(lines[-1])
    assert out["unit"] == "env-steps/s" and out["total_steps"] == 1024 and out["value"] > 0
    assert out["config"]["obs_storage"] == "symbolic" and os.path.exists(ckpt)
    lines = _run(["tools/eval_sweep.py", "--ckpt", ckpt, "--difficulty", "medium", "--sizes", "8", "--tasks", "6"])
    row = json.loads(lines[-1])
    assert row["tasks"] == 6 and 1 <= row["mean_steps"] <= 256


def test_train_fomaml_tool_tiny(tmp_path):
    lines = _run(["tools/train_fomaml.py", "--iterations", "2", "--tasks-per-batch", "4", "--k-steps", "16", "--warmup", "1"])
    out = json.loads(lines[-1])
    assert out["iterations"] == 2 and out["value"] > 0 and len(out["history"]) >= 2


def test_bench_tool_small_batch():
    lines = _run(["bench.py", "--envs", "32768", "--steps", "16", "--warmup", "3", "--layouts", "256", "--skip-cpu-baseline",
                  "--ppo-envs", "64", "--ppo-horizon", "8", "--ppo-iters", "1", "--fomaml-tasks", "4", "--fomaml-k", "16",
                  "--fomaml-iters", "1"])
    assert len(lines) == 1  # ONE JSON line on stdout
    out = json.loads(lines[0])
    # the learner sections (BASELINE metric's second half; configs 3 and 4), every N
    assert out["ppo"]["value"] > 0 and out["ppo"]["unit"] == "env-steps/s" and out["ppo"]["allreduce_bytes"] == 744772 * 4
    assert {"rollout_s", "update_s", "allreduce_s"} <= set(out["ppo"])
    assert out["fomaml"]["strong"]["s_per_iteration"] > 0 and out["fomaml"]["strong"]["tasks_per_gpu"] == 4
    # clocks are sampled in-process: a 16-step timed region still holds samples
    assert out["clocks"]["samples"] >= 1 and out["clocks"]["sm_mhz"] > 0
    assert out["config"]["layout_pool"] == 256 and out["config"]["envs_restarted_on_a_new_layout_in_timed_region_rank0"] > 0
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "dtype", "data", "config", "clocks", "gpu_launches", "roofline", "e2e"):
        assert key in out, key
    assert out["gpu_launches"] == 16 and out["roofline"]["bound"] == "hbm" and out["e2e"]["h2d_bytes_per_step"] == 32768 * 8
    assert "sym" in out["symbolic_only"]["kernel"] and out["symbolic_only"]["value_per_gpu"] > out["value"]


def test_bench_dump_outputs_repeat_exactly(tmp_path):
    """--dump-outputs: the last timed step's outputs as float .npy files, identical for two runs with the same arguments."""
    import numpy as np
    names = {"obs", "obs_env_index", "env_index", "reward", "terminated", "truncated", "episode_return", "episode_length",
             "stuck", "done"}
    N, K = 4096, 37
    dumps = []
    for run in range(2):
        d = tmp_path / f"run{run}"
        lines = _run(["bench.py", "--envs", str(N), "--steps", str(K), "--warmup", "3", "--layouts", "256", "--skip-cpu-baseline",
                      "--skip-e2e", "--skip-learners", "--dump-outputs", str(d)])
        out = json.loads(lines[-1])
        assert out["steps"] == K and out["gpu_launches"] == K
        assert {p.name for p in d.iterdir()} == {n + ".npy" for n in names}
        dumps.append({n: np.load(d / (n + ".npy")) for n in names})
        assert sum(p.stat().st_size for p in d.iterdir()) <= 64 << 20
    a, b = dumps
    for n in names:
        assert a[n].dtype in (np.float32, np.float64), n
        assert np.array_equal(a[n], b[n]), n
    assert a["obs"].shape == (512, 56, 56, 3) and a["reward"].shape == (N,)
    assert np.array_equal(a["env_index"], np.arange(N)) and np.all(np.diff(a["obs_env_index"]) > 0)
    assert np.array_equal(a["done"], np.maximum(a["terminated"], a["truncated"]))
    assert np.all((a["episode_length"] > 0) == (a["done"] > 0))
