"""Cost of final observations: the same step with and without `final_obs`, alternated inside one run.

    python tools/bench_final_obs.py [--rounds 7] [--steps 20] [--out FILE]

mediumhard 16x16, episode clocks staggered (about N / max_steps episodes end per step, the steady state), random
actions already in HBM.  Cases: 4096 and 16 384 envs with RGB frames under CUDA-graph replay (the warp kernel),
1 048 576 envs with RGB (the tile kernel) and symbolic-only (the symbolic kernel), eager; each once at max_steps 1024
and once at max_steps 16 (high turnover, the worst case).  Every round times `--steps` steps of each variant with CUDA
events, plain first or final first in turn; the median per-step time of each variant and their ratio are printed, with
the card's name and power limit read in the same run.  Prints one JSON line per case.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "ppo-2dgrid_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


def run_case(N, rgb, graph, max_steps, steps, rounds, pool):
    from merlin_b200 import BatchedMerlinEnv
    cells, agent = pool
    env = BatchedMerlinEnv(N, cells, agent, width=16, height=16, max_steps=max_steps, device="cuda:0", want_rgb=rgb,
                           want_symbolic=True, episode_stats=False)
    env.reset(frames=rgb)
    env.stagger_episode_clocks(seed=N + max_steps)
    final = torch.empty((N, 7, 7, 3), dtype=torch.uint8, device="cuda:0")
    acts = torch.randint(0, 3, (steps, N), dtype=torch.int64, device="cuda:0")

    def run(with_final):
        for k in range(steps):
            env.step(acts[k], frames=rgb, final_obs=final if with_final else None)

    run(False)
    run(True)   # warm-up: occupancy and shared-memory attributes of both instances
    torch.cuda.synchronize()
    fns = {False: lambda: run(False), True: lambda: run(True)}
    if graph:
        for v in (False, True):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                run(v)
            fns[v] = g.replay
        fns[False]()
        fns[True]()
    torch.cuda.synchronize()
    times = {False: [], True: []}
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for r in range(rounds):
        for v in ((False, True) if r % 2 == 0 else (True, False)):
            start.record()
            fns[v]()
            stop.record()
            stop.synchronize()
            times[v].append(start.elapsed_time(stop) * 1e3 / steps)
    plain, fin = float(np.median(times[False])), float(np.median(times[True]))
    kernel = env.step_kernel(final=False), env.step_kernel(final=True)
    del env, final, acts
    torch.cuda.empty_cache()
    return {"envs": N, "rgb": rgb, "graph": graph, "max_steps": max_steps, "kernel": kernel[0],
            "final_kernel": kernel[1], "us_per_step": plain, "us_per_step_final": fin, "ratio": fin / plain,
            "spread_us": [float(np.min(times[False])), float(np.max(times[False])), float(np.min(times[True])),
                          float(np.max(times[True]))]}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_final_obs needs a CUDA device"
    from merlin_b200 import layouts
    pool = layouts.generate("mediumhard", 16, range(777_000_000, 777_000_000 + 4096))
    device = card()
    cases = [(4096, True, True), (16384, True, True), (1 << 20, True, False), (1 << 20, False, False)]
    lines = []
    for max_steps in (1024, 16):
        for N, rgb, graph in cases:
            res = run_case(N, rgb, graph, max_steps, a.steps, a.rounds, pool)
            res["device"] = device
            line = json.dumps(res)
            print(line, flush=True)
            lines.append(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
