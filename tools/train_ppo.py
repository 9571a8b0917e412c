#!/usr/bin/env python
"""End-to-end PPO on device-resident rollouts (BASELINE config 3: mediumhard 16x16, 5M total steps, 4096 envs on one
B200; with torchrun: the same per GPU, gradients all-reduced over NCCL).  Mirrors ppo/ppo_train.py's loop
(collect -> update -> periodic deterministic eval) with the reference's hyper-parameters where they carry over
(lr 3e-4, gamma .99, lambda .95, clip .2, 10 epochs, ent .05, vf .5); the batched regime's own choices (envs, horizon,
minibatch) are flags and are recorded in the output.

    python tools/train_ppo.py --envs 4096 --horizon 128 --minibatch 16384 --total-steps 5000000 --out profiles/r01_ppo.json
    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 tools/train_ppo.py ...

Prints one JSON line: wall-clock, SPS (env-steps/s including policy forward, env, GAE, update, all-reduce), the
rollout/update split, and the greedy evaluation on unseen seeds 200000.. (src/sweep_checkpoints.py:90).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "ppo-2dgrid_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--difficulty", default="mediumhard")
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--horizon", type=int, default=128)
    ap.add_argument("--minibatch", type=int, default=16384)
    ap.add_argument("--update-epochs", type=int, default=10)
    ap.add_argument("--total-steps", type=int, default=5_000_000)
    ap.add_argument("--lr", type=float, default=3e-4)
    ap.add_argument("--ent-coef", type=float, default=0.05)
    ap.add_argument("--seed", type=int, default=777)
    ap.add_argument("--layouts", type=int, default=65536)
    ap.add_argument("--eval-tasks", type=int, default=100)
    ap.add_argument("--device-layouts", action="store_true",
                    help="generate the layout pool on the GPU (fresh layouts, not the reference's per-seed ones)")
    ap.add_argument("--tf32-matmul", action="store_true",
                    help="allow TF32 in the linear layers too (PyTorch's default keeps them in fp32; cuDNN convolutions "
                         "already run TF32 by default)")
    ap.add_argument("--amp", choices=["none", "bf16"], default="none",
                    help="bf16 autocast for the policy evaluation in the update (reduced precision: not the headline setting)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--bootstrap-truncated", action="store_true",
                    help="add gamma * V(final observation) to the reward of steps cut by the episode step limit")
    ap.add_argument("--obs-storage", choices=["rgb", "symbolic"], default="symbolic",
                    help="rollout keeps 56x56x3 frames, or the 7x7x3 symbolic image rendered on read (64x smaller)")
    ap.add_argument("--mb-frames", choices=["f32", "u8"], default="f32",
                    help="symbolic storage: the render kernel writes minibatches as the normalised float32 first-layer input "
                         "(default) or as blocked uint8 pixels that PyTorch casts afterwards")
    ap.add_argument("--cpu-baseline", action="store_true",
                    help="also time one reference-style PPO iteration (N=1, 2048 steps) on the host cores (oracle port)")
    ap.add_argument("--out", default=None)
    ap.add_argument("--save", default=None, help="path for the final state_dict (.pth, reference format)")
    a = ap.parse_args()

    import numpy as np
    import torch
    import torch.distributed as dist

    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from merlin_b200 import layouts
    from src.evaluation import evaluate_seeds
    from src.ppo import PPO
    from src.scenario_creator.scenario_creator import ScenarioCreator
    from src.utils.utils import set_seed

    set_seed(a.seed + rank)
    torch.backends.cudnn.benchmark = True
    if a.tf32_matmul:
        torch.backends.cuda.matmul.allow_tf32 = True
    sc = ScenarioCreator()
    t_lay = time.perf_counter()
    per_rank = a.layouts // world
    base = a.seed * 1_000_000 + rank * per_rank
    if a.device_layouts:
        env = sc.create_batched_env(a.difficulty, a.envs, device=dev, layouts="device", seeds=a.seed * 1000 + rank,
                                    n_layouts=per_rank, want_symbolic=a.obs_storage == "symbolic")
        torch.cuda.synchronize(dev)
    else:
        from multiprocessing import Pool
        chunks = [range(base + i, min(base + i + 2048, base + per_rank)) for i in range(0, per_rank, 2048)]
        with Pool(min(len(chunks), len(os.sched_getaffinity(0)))) as pool:
            parts = pool.starmap(layouts.generate, [(a.difficulty, 16, c) for c in chunks])
        cells = np.concatenate([p[0] for p in parts])
        agent_xyd = np.concatenate([p[1] for p in parts])
        env = sc.create_batched_env(a.difficulty, a.envs, device=dev, layouts=(cells, agent_xyd),
                                    want_symbolic=a.obs_storage == "symbolic")
    t_lay = time.perf_counter() - t_lay
    agent = PPO(env, lr=a.lr, gamma=0.99, lam=0.95, clip_eps=0.2, update_epochs=a.update_epochs,
                batch_size=a.envs * a.horizon, minibatch_size=a.minibatch, vf_coef=0.5, ent_coef=a.ent_coef,
                use_cuda_graph=not a.no_graph, obs_storage=a.obs_storage,
                amp_dtype=torch.bfloat16 if a.amp == "bf16" else None,
                minibatch_frames=torch.float32 if a.mb_frames == "f32" else torch.uint8,
                bootstrap_truncated=a.bootstrap_truncated)

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # warm-up iteration (cuDNN autotune, graph capture) -- not counted in steps or time
    agent.update(agent.collect_rollouts())
    sync()
    steps_per_iter = a.envs * a.horizon * world
    iters = max(1, -(-a.total_steps // steps_per_iter))
    t_roll = t_upd = 0.0
    log = []
    t0 = time.perf_counter()
    for it in range(iters):
        ta = time.perf_counter()
        lv = agent.collect_rollouts()
        torch.cuda.synchronize(dev)
        tb = time.perf_counter()
        m = agent.update(lv)
        tc = time.perf_counter()
        t_roll += tb - ta
        t_upd += tc - tb
        rets = agent.episode_returns[-2000:]
        log.append({"iter": it, "steps": (it + 1) * steps_per_iter, "mean_return": float(np.mean(rets)) if rets else 0.0,
                    "kl": m["kl"], "entropy": m["entropy"], "v_loss": m["v_loss"]})
        agent.episode_returns.clear()
        agent.episode_lengths.clear()
    sync()
    wall = time.perf_counter() - t0

    if rank == 0:
        te = time.perf_counter()
        r, n, g = evaluate_seeds(agent.ac, a.difficulty, 16, range(200000, 200000 + a.eval_tasks), device=dev)
        torch.cuda.synchronize(dev)
        te = time.perf_counter() - te
        if a.save:
            torch.save(agent.ac.state_dict(), a.save)
        out = {"metric": "end-to-end PPO env-steps/s (policy fwd + env + GAE + update)", "value": iters * steps_per_iter / wall,
               "unit": "env-steps/s", "n_gpus": world, "wall_s": wall, "total_steps": iters * steps_per_iter,
               "iterations": iters, "rollout_s": t_roll, "update_s": t_upd,
               "config": {"workload": f"configs[2]: PPO {a.difficulty} 16x16, {a.envs} envs/GPU x horizon {a.horizon}",
                          "minibatch": a.minibatch, "update_epochs": a.update_epochs, "lr": a.lr, "ent_coef": a.ent_coef,
                          "cuda_graph_rollout": not a.no_graph, "obs_storage": a.obs_storage,
                          "minibatch_frames": a.mb_frames if a.obs_storage == "symbolic" else None,
                          "rollout_obs_bytes": int(agent.buffer.states.numel() * agent.buffer.states.element_size()),
                          "peak_device_memory_gb": torch.cuda.max_memory_allocated(dev) / 1e9, "layout_pool_per_gpu": per_rank,
                          "layout_source": "device" if a.device_layouts else "host (reference seeds)", "layout_setup_s": t_lay, "dtype": "fp32 policy (PyTorch defaults: TF32 convolutions" + (", TF32 linear layers" if a.tf32_matmul else ", fp32 linear layers") + ")" + (", bf16 autocast in the update" if a.amp == "bf16" else "") + ", u8 frames", "seed": a.seed},
               "eval": {"tasks": a.eval_tasks, "seeds": "200000..", "mean_return": float(np.mean(r)),
                        "mean_steps": float(np.mean(n)), "success_rate": float(np.mean(g)), "eval_s": te},
               "train_log": log[:: max(1, len(log) // 20)] + log[-1:]}
        if a.cpu_baseline:
            from oracle import ppo_ref
            cb = ppo_ref.cpu_ppo_sps(a.difficulty, 16, a.seed, update_budget_s=30.0)
            out["cpu_baseline"] = {
                "value": cb["steps_per_s"], "unit": "env-steps/s", "cores": cb["torch_threads"], "kind": "port",
                "sample": f"one PPO iteration of the reference regime (1 env x 2048 steps, batch-1 inference, 10 epochs x 8 "
                          f"minibatches of 256): rollout {cb['rollout_s']:.1f} s + update {cb['update_s']:.1f} s "
                          f"({cb['minibatches_run']}/{cb['minibatches_total']} minibatch steps measured); literal minigrid "
                          "restatement + reference wrapper stack, torch CPU",
                "projected_wall_s_for_total_steps": iters * steps_per_iter / cb["steps_per_s"]}
        print(json.dumps(out), flush=True)
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "w") as f:
                json.dump(out, f, indent=1)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
