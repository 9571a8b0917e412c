#!/usr/bin/env python
"""Time on-device layout generation against the host generator, on the two pools the project builds most:
  - 65 536 mediumhard 16x16 layouts of seeds 777 000 000.. (bench.py's pool),
  - 100 hard 64x64 layouts of seeds 200 000.. (config 5's largest grid).
For each: merlin_env_generate_seeded_layouts (the reference's per-seed layouts, numpy's stream restated on the GPU),
merlin_env_generate_layouts (the counter-based stream, same shape) and single-process merlin_b200.layouts.generate.
Device times are CUDA events on the calling stream around the whole synchronous call (seed upload, kernel, failure
flag read-back; medians of --reps calls after two warm-up calls); `call_ms` is the host wall clock of the same calls.
The seeded pool is checked equal to the host generator's before anything is reported.  Prints one JSON line with the
GPU name and power limit read in the same run."""
import argparse, json, os, statistics, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "ppo-2dgrid_b200"))
import numpy as np
import torch
from merlin_b200 import BatchedMerlinEnv, layouts

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=None)
ap.add_argument("--reps", type=int, default=10)
a = ap.parse_args()
dev = "cuda:0"


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        return float(out.splitlines()[0])
    except Exception:
        return None


def timed(fn):
    fn(); fn()  # warm-up: module load, first-touch of the pool
    dev_ms, call_ms = [], []
    for _ in range(a.reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        call_ms.append((time.perf_counter() - t0) * 1e3)
        dev_ms.append(e0.elapsed_time(e1))
    return statistics.median(dev_ms), statistics.median(call_ms)


rows = []
for difficulty, size, first, n in (("mediumhard", 16, 777_000_000, 65536), ("hard", 64, 200_000, 100)):
    seeds = list(range(first, first + n))
    env = BatchedMerlinEnv(4, width=size, height=size, device=dev, generate_seeded=(difficulty, seeds))
    seeded_dev, seeded_call = timed(lambda: env.generate_seeded_layouts(difficulty, seeds))
    keyed_dev, keyed_call = timed(lambda: env.generate_layouts(difficulty, first, n))
    env.generate_seeded_layouts(difficulty, seeds)
    got = env.layouts_numpy()
    t0 = time.perf_counter()
    want = layouts.generate(difficulty, size, seeds)
    host_ms = (time.perf_counter() - t0) * 1e3
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), f"{difficulty} {size}: pools differ"
    rows.append({"difficulty": difficulty, "size": size, "layouts": n, "first_seed": first,
                 "seeded_device_ms": round(seeded_dev, 4), "seeded_call_ms": round(seeded_call, 4),
                 "keyed_device_ms": round(keyed_dev, 4), "keyed_call_ms": round(keyed_call, 4),
                 "host_single_process_ms": round(host_ms, 1),
                 "host_over_seeded_call": round(host_ms / seeded_call, 1)})

res = {"gpu": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w(), "numpy": np.__version__,
       "reps": a.reps, "rows": rows}
print(json.dumps(res))
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
