#!/usr/bin/env python
"""bench.py -- batched env-steps/s of the fused MERLIN step kernel (step + gen_obs/process_vis + RGB render).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--envs E] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One "step" = one pass of the hot path over one batch: every env of the batch takes one action and gets its
56x56x3 observation, reward and flags (BASELINE.json configs[1]: mediumhard 16x16, random actions, synthetic
seeded layouts).  Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.

  value      env-steps/s over all GPUs, inputs (actions) already in HBM, device-timed with CUDA events
  e2e        same metric through the public host API with HOST action buffers: per step a pinned H2D copy of the
             actions and a D2H read of reward/terminated/truncated; observations stay in HBM where the policy
             consumes them (e2e.value_obs_to_host additionally copies every observation to the host: PCIe-bound)
  roofline   algorithmic bytes per launch (9710 B x envs) / mean kernel time, against the measured HBM copy peak
  cpu_baseline  the reference-style CPU path (oracle port: literal minigrid-3.0.0 restatement + wrapper stack),
             one env per host core, bounded sample; plus the optimised C oracle as a second data point
  ppo        BASELINE's second metric half, every N: end-to-end PPO env-steps/s in the config-3 regime (4096 envs per
             GPU x horizon 128, minibatch 16384, 10 epochs; fused rollouts replayed from a CUDA graph; the flattened
             gradient all-reduced over NCCL once per minibatch step), with the rollout / update / all-reduce split
  fomaml     config 4: seconds per FOMAML meta-iteration, 32 tasks x (256 support + 256 query) steps, tasks sharded
             over the N GPUs (strong scaling) and 32 tasks PER GPU (weak scaling); one gradient all-reduce per iteration
  --impl reference : only the CPU path, same metric/config, all host cores
  --dump-outputs DIR : after the timed steps, write what the last one returned to DIR/<name>.npy (see dump_outputs)
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "ppo-2dgrid_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "batched env-steps/sec (mediumhard 16x16, step+gen_obs+RGB render)"
UNIT = "env-steps/s"
SIZE = 16
ALGO_BYTES_PER_STEP = 56 * 56 * 3 + SIZE * SIZE + 32 + 8 + 6  # 9710, SURVEY 8d / DESIGN.md
FALLBACK_HBM_GBS = 6650.0


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2048)
    ap.add_argument("--warmup", type=int, default=64)
    ap.add_argument("--envs", type=int, default=1 << 20, help="envs per GPU (weak scaling)")
    ap.add_argument("--layouts", type=int, default=65536, help="layout pool size per GPU (SURVEY 8d: 65 536)")
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU-baseline sample budget")
    ap.add_argument("--skip-learners", action="store_true", help="no PPO / FOMAML sections")
    ap.add_argument("--ppo-iters", type=int, default=3, help="timed PPO iterations (after one warm-up iteration)")
    ap.add_argument("--ppo-envs", type=int, default=4096, help="PPO envs per GPU (config 3)")
    ap.add_argument("--ppo-horizon", type=int, default=128)
    ap.add_argument("--fomaml-iters", type=int, default=5, help="timed FOMAML meta-iterations (after two warm-up ones)")
    ap.add_argument("--fomaml-tasks", type=int, default=32, help="tasks per meta-batch (config 4)")
    ap.add_argument("--fomaml-k", type=int, default=256, help="support and query steps per task (config 4)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs (rank 0) as DIR/<name>.npy, to compare two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs: not with --impl reference")
    return args


# ----------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock / power / throttle reasons sampled IN-PROCESS through NVML on a background thread (every 10 ms), so even a
    30 ms timed region holds samples; falls back to an `nvidia-smi -lms` child when NVML cannot be loaded."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index=0, uuid=None):
        self.index, self.uuid = index, uuid
        self.proc = self.thread = self.nvml = None
        self.samples, self.marks = [], {}

    def start(self):
        import threading
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            if self.uuid:
                try:
                    h = pynvml.nvmlDeviceGetHandleByUUID(self.uuid if self.uuid.startswith("GPU-") else "GPU-" + self.uuid)
                except Exception:  # noqa: BLE001
                    h = None
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.nvml, self.handle = pynvml, h
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self.stop_flag = False
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            while not self.samples:  # the first sample exists before any timed region can start
                time.sleep(0.001)
            return
        except Exception:  # noqa: BLE001 -- no NVML: fall back to the CLI
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                sm = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                pw = n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
                rs = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                self.samples.append((time.perf_counter(), sm, pw, rs))
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.01)

    def mark(self, name):
        """Remember `now` under `name` ("<region>_start" / "<region>_end"): samples are attributed to regions afterwards."""
        self.marks[name] = time.perf_counter()

    def region(self, name):
        t0, t1 = self.marks.get(name + "_start"), self.marks.get(name + "_end")
        if self.nvml is None or t0 is None or t1 is None:
            return None
        # a region shorter than the polling period still owns the sample taken just after it started
        inside = [x for x in self.samples if t0 <= x[0] <= t1]
        nearest_ms = None
        if not inside and self.samples:
            # a region shorter than one polling period: the sample closest to it in time stands in (and says so)
            x = min(self.samples, key=lambda x: min(abs(x[0] - t0), abs(x[0] - t1)))
            nearest_ms = 1e3 * min(abs(x[0] - t0), abs(x[0] - t1))
            inside = [x]
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": self.max_sm, "samples": 0, "reasons": ["no samples"]}
        bits = 0
        for x in inside:
            bits |= x[3]
        out = {"sm_mhz": statistics.median(x[1] for x in inside), "sm_max_mhz": self.max_sm,
               "power_w_max": max(x[2] for x in inside), "samples": len(inside),
               "reasons": sorted(v for k, v in self.REASONS.items() if bits & k)}
        if nearest_ms is not None:
            out["nearest_sample_ms_from_region"] = nearest_ms
        return out

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.thread.join(timeout=1.0)
            out = self.region("timed") or {"sm_mhz": None, "sm_max_mhz": self.max_sm, "reasons": ["no samples"]}
            out["source"] = "NVML in-process (one sample per ~10 ms), samples inside the device-timed region"
            if self.region("timed"):
                out["region_ms"] = 1e3 * (self.marks["timed_end"] - self.marks["timed_start"])
            for extra in ("ppo", "fomaml"):
                r = self.region(extra)
                if r:
                    out[extra] = {k: r[k] for k in ("sm_mhz", "power_w_max", "samples", "reasons") if k in r}
            return out
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        # samples under load = upper half by power draw (the CLI sampler also sees setup / idle time)
        order = sorted(range(len(sm)), key=lambda i: pw[i])
        loaded = [sm[i] for i in order[len(order) // 2:]]
        return {"sm_mhz": statistics.median(loaded), "sm_max_mhz": max(mx), "power_w_max": max(pw),
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi -lms 100 (NVML unavailable)"}


# ----------------------------------------------------------------------------------------- CPU paths
_W = {}


def _cpu_worker_init(seed):
    from oracle import merlin_ref as mr
    env = mr.make_env("mediumhard", size=SIZE)
    env.reset(seed=777_000_000 + seed)
    import numpy as np
    _W["env"], _W["rng"] = env, np.random.default_rng(seed)


def _cpu_worker_run(n):
    """n env-steps of the reference-style path (literal minigrid restatement + RGB/Img/ThreeAction wrappers),
    random actions, reset on done -- what src/ppo.py:70-98 does per step minus the policy."""
    if "env" not in _W:
        _cpu_worker_init(os.getpid() % 100000)
    env, rng = _W["env"], _W["rng"]
    t0 = time.perf_counter()
    for _ in range(n):
        _, _, te, tr, _ = env.step(int(rng.integers(0, 3)))
        if te or tr:
            env.reset()
    return time.perf_counter() - t0


class CpuReference:
    """All host cores, one env per process (the reference has no vector env)."""

    def __init__(self, cores=None):
        import multiprocessing as mp
        self.cores = cores or len(os.sched_getaffinity(0))
        self.pool = mp.get_context("spawn").Pool(self.cores)
        self.pool.map(_cpu_worker_run, [20] * self.cores)  # build envs + tile cache

    def run(self, steps_per_proc):
        t0 = time.perf_counter()
        self.pool.map(_cpu_worker_run, [steps_per_proc] * self.cores, chunksize=1)
        dt = time.perf_counter() - t0
        return self.cores * steps_per_proc, dt

    def close(self):
        self.pool.terminate()


def c_oracle_rate(seconds=3.0):
    """Optimised C oracle (OpenMP over envs), NOT the reference: a second CPU data point."""
    import numpy as np
    from merlin_b200 import codes, layouts
    from oracle import fast
    cells, agent = layouts.generate("mediumhard", SIZE, range(777_000_000, 777_000_000 + 256))
    N = 8192
    env = fast.OracleVecEnv(N, codes.unpack_to_encoding(cells, SIZE, SIZE), agent)
    env.reset()
    rng = np.random.default_rng(0)
    acts = rng.integers(0, 3, (8, N))
    env.step(acts[0])
    t0, n = time.perf_counter(), 0
    while time.perf_counter() - t0 < seconds:
        env.step(acts[n % 8]); n += 1
    return N * n / (time.perf_counter() - t0), fast.set_threads(0)


def run_reference(args):
    """--impl reference: the CPU path only, same metric/config; under torchrun rank 0 alone works."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    ref = CpuReference()
    n, dt = ref.run(200)  # calibrate
    rate = n / dt
    budget = 90.0  # seconds for warmup + steps
    per_proc = max(5, int(rate * budget / max(1, args.steps + args.warmup) / ref.cores))
    for _ in range(args.warmup):
        ref.run(per_proc)
    total, t = 0, 0.0
    for _ in range(args.steps):
        n, dt = ref.run(per_proc)
        total += n; t += dt
    ref.close()
    value = total / t
    sample = (f"{args.steps} steps x {ref.cores} procs x {per_proc} env-steps each "
              f"({total} env-steps, {t:.1f} s) of mediumhard 16x16 random-action stepping with reset on done")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t / max(1, args.steps), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "mediumhard 16x16, random actions, one env per host process (reference has no vector env)",
                   "grid": SIZE, "obs": "u8[56,56,3] RGB POV", "actions": 3,
                   "note": "upstream minigrid/gymnasium not installable: literal restatement (oracle port) + reference wrapper stack"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": ref.cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------- GPU path
def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy read+write)"
    except (OSError, KeyError, ValueError):
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def ncu_traffic(envs, kernel=None):
    """DRAM bytes per launch of the step kernel from the committed ncu --set full capture, if it matches."""
    try:
        with open(os.path.join(ROOT, "profiles", "step_kernel_traffic.json")) as f:
            t = json.load(f)
        if int(t.get("envs", -1)) == envs and (kernel is None or t.get("kernel") == kernel):
            return float(t["dram_bytes_read"]) + float(t["dram_bytes_write"])
    except (OSError, KeyError, ValueError):
        pass
    return None


DUMP_ENVS = 1 << 20     # per-env outputs of at most this many envs: 7 float32 arrays (29.4 MB) + a float64 index (8.4 MB)
DUMP_OBS_ENVS = 512     # observation frames of this many envs: 512 x 56 x 56 x 3 float32 = 19.3 MB


def dump_outputs(out_dir, step_out):
    """Write what one `env.step` returned -- the gymnasium 5-tuple and the info tensors -- to out_dir/<name>.npy as float32,
    57.1 MB at most.  Per-env outputs are written for every env up to DUMP_ENVS envs, observation frames for DUMP_OBS_ENVS
    envs; larger batches are sampled with a fixed seed, and the sampled env indices are written as env_index.npy and
    obs_env_index.npy (float64).  With the same arguments two runs step the same envs with the same actions, so the files
    of two builds can be compared array for array."""
    import numpy as np
    import torch
    obs, reward, terminated, truncated, info = step_out
    n = reward.numel()
    rng = np.random.default_rng(20240611)

    def sample(k):
        return np.arange(n) if n <= k else np.sort(rng.choice(n, k, replace=False))

    env_index, obs_index = sample(DUMP_ENVS), sample(DUMP_OBS_ENVS)
    rows = torch.as_tensor(env_index, device=reward.device)
    arrays = {"env_index": env_index.astype(np.float64), "obs_env_index": obs_index.astype(np.float64),
              "obs": obs[torch.as_tensor(obs_index, device=obs.device)].float().cpu().numpy()}
    for name, t in (("reward", reward), ("terminated", terminated), ("truncated", truncated),
                    ("episode_return", info["episode_return"]), ("episode_length", info["episode_length"]),
                    ("stuck", info["stuck"]), ("done", info["done"])):
        arrays[name] = t[rows].float().cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def bench_ppo(args, dev, rank, world, cells, agent, sampler, barrier):
    """End-to-end PPO env-steps/s in the config-3 regime on every GPU (weak scaling: the per-GPU batch is fixed), the
    reference's loop (ppo/ppo_train.py:145-190: collect -> update) and hyper-parameters (lr 3e-4, gamma .99, lambda
    .95, clip .2, 10 epochs, ent .05, vf .5); per-minibatch gradient all-reduce as in src/ppo.py:154-156."""
    import torch
    from src.ppo import PPO
    from src.scenario_creator.scenario_creator import ScenarioCreator
    from src.utils.utils import set_seed

    set_seed(777 + rank)
    torch.backends.cudnn.benchmark = True
    N, T = args.ppo_envs, args.ppo_horizon
    env = ScenarioCreator().create_batched_env("mediumhard", N, device=dev, layouts=(cells, agent), want_symbolic=True)
    ppo = PPO(env, lr=3e-4, gamma=0.99, lam=0.95, clip_eps=0.2, update_epochs=10, batch_size=N * T,
              minibatch_size=min(16384, N * T), vf_coef=0.5, ent_coef=0.05, use_cuda_graph=True, obs_storage="symbolic")
    if ppo._grads is not None:
        ppo._grads.enable_timing()
    ppo.update(ppo.collect_rollouts())      # warm-up iteration: cuDNN autotune, graph capture (fresh-reset graph)
    ppo.update(ppo.collect_rollouts())      # ... and the steady-state graph (episodes carried over)
    if ppo._grads is not None:
        ppo._grads.collective_seconds()
    barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.ppo_iters + 1)]
    sampler.mark("ppo_start")
    t0 = time.perf_counter()
    ev[0].record()
    for it in range(args.ppo_iters):
        lv = ppo.collect_rollouts()
        ev[2 * it + 1].record()
        metrics = ppo.update(lv)
        ev[2 * it + 2].record()
    barrier()
    wall = time.perf_counter() - t0
    sampler.mark("ppo_end")
    roll = sum(ev[2 * i].elapsed_time(ev[2 * i + 1]) for i in range(args.ppo_iters)) * 1e-3
    upd = sum(ev[2 * i + 1].elapsed_time(ev[2 * i + 2]) for i in range(args.ppo_iters)) * 1e-3
    ar = ppo._grads.collective_seconds() if ppo._grads is not None else 0.0
    n_ar = args.ppo_iters * 10 * ((N * T + ppo.minibatch_size - 1) // ppo.minibatch_size) if world > 1 else 0
    t = torch.tensor([wall, roll, upd, ar], dtype=torch.float64, device=dev)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    wall, roll, upd, ar = [float(x) for x in t.tolist()]
    steps = world * N * T * args.ppo_iters
    out = {"metric": "end-to-end PPO env-steps/s (policy fwd + env + GAE + update + gradient all-reduce)",
           "value": steps / wall, "unit": "env-steps/s", "n_gpus": world, "iterations": args.ppo_iters, "seconds": wall,
           "rollout_s": roll, "update_s": upd, "allreduce_s": ar, "allreduce_calls": n_ar,
           "allreduce_bytes": ppo._grads.nbytes() if ppo._grads is not None else sum(p.numel() for p in ppo.ac.parameters()) * 4,
           "allreduce_us_per_call": 1e6 * ar / n_ar if n_ar else None,
           "config": {"workload": f"configs[2] regime: PPO mediumhard 16x16, {N} envs/GPU x horizon {T}, minibatch "
                                  f"{ppo.minibatch_size}, 10 epochs, lr 3e-4, ent 0.05; fused rollouts (CUDA graph), symbolic "
                                  "rollout storage, float32 minibatch frames from the render kernel",
                      "dtype": "fp32 policy (PyTorch defaults: TF32 cuDNN convolutions, fp32 linear layers)",
                      "scaling": "weak (per-GPU batch fixed)", "episodes_carried_across_rollouts": ppo.carry_episodes},
           "last_update": {k: float(v) for k, v in metrics.items()}}
    env.close()
    return out


def bench_fomaml(args, dev, rank, world, sampler, barrier):
    """Seconds per FOMAML meta-iteration (fomaml/fomaml_train.py:100-121: seed 777, task seeds drawn from range(100000),
    lr_inner 0.01, lr_outer 3e-4; k support + k query steps per task).  `strong`: the config-4 meta-batch (32 tasks)
    sharded over the ranks; `weak`: 32 tasks on EVERY rank (256 on 8 GPUs).  One gradient all-reduce per iteration."""
    import numpy as np
    import torch
    from src.fomaml import FOMAML
    from src.scenario_creator.scenario_creator import ScenarioCreator
    from src.utils.utils import set_seed

    set_seed(777)  # identical numpy stream on every rank -> identical task batches
    torch.backends.cudnn.benchmark = True
    fo = FOMAML(ScenarioCreator(), lr_inner=0.01, lr_outer=3e-4, difficulty="mediumhard", device=dev)
    torch.manual_seed(777 + 1000 * rank)
    k = args.fomaml_k
    out = {"metric": "seconds per FOMAML meta-iteration (support + query rollouts, inner SGD, meta update)",
           "unit": "s/iteration", "n_gpus": world, "k_support": k, "k_query": k, "iterations": args.fomaml_iters}
    sampler.mark("fomaml_start")
    for mode, tasks in (("strong", args.fomaml_tasks), ("weak", args.fomaml_tasks * world)):
        if mode == "weak" and world == 1:
            out["weak"] = dict(out["strong"], note="one GPU: the same run as `strong`")
            continue

        def batch():
            return [int(x) for x in np.random.choice(range(100000), size=tasks, replace=False)]
        for _ in range(2):
            fo.meta_train_step(batch(), k_support=k, k_query=k)
        barrier()
        t0 = time.perf_counter()
        nxt = batch()
        for _ in range(args.fomaml_iters):
            cur, nxt = nxt, batch()
            fo.prefetch_tasks(nxt)  # next meta-batch's layouts: host thread, overlapped with this iteration's GPU work
            fo.meta_train_step(cur, k_support=k, k_query=k)
        barrier()
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        dt = float(t.item())
        out[mode] = {"s_per_iteration": dt / args.fomaml_iters, "tasks_per_batch": tasks,
                     "tasks_per_gpu": -(-tasks // world), "env_steps_per_s": tasks * 2 * k * args.fomaml_iters / dt}
    sampler.mark("fomaml_end")
    out["value"] = out["strong"]["s_per_iteration"]
    out["config"] = {"workload": f"configs[3] regime: FOMAML mediumhard 16x16, {args.fomaml_tasks} tasks x (k = {k} support "
                                 f"+ {k} query) per meta-iteration; task-batched fused rollouts replayed from CUDA graphs",
                     "allreduce_bytes_per_iteration": sum(p.numel() for p in fo.meta_policy.parameters()) * 4 + 4,
                     "dtype": "fp32 policy (PyTorch; stacked per-task weights), symbolic rollout storage"}
    return out


def _generate_layouts(base, count, world):
    """`count` host-generated mediumhard layouts for seeds base.. (np.random.default_rng(seed), the reference's
    `reset(seed=s)` layouts), in worker processes: a few seconds instead of ~10 s on one core."""
    import numpy as np
    from merlin_b200 import layouts
    procs = max(1, min(16, len(os.sched_getaffinity(0)) // max(1, world)))
    chunk = 2048
    jobs = [("mediumhard", SIZE, range(base + i, min(base + i + chunk, base + count))) for i in range(0, count, chunk)]
    if procs == 1 or len(jobs) == 1:
        parts = [layouts.generate(*j) for j in jobs]
    else:
        import multiprocessing as mp
        with mp.get_context("spawn").Pool(min(procs, len(jobs))) as pool:
            parts = pool.starmap(layouts.generate, jobs)
    return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback (use --impl reference for the CPU path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from merlin_b200 import BatchedMerlinEnv

    # clocks: sampled in-process from before the env exists until the last learner section ended
    try:
        uuid = str(torch.cuda.get_device_properties(local).uuid)
    except Exception:  # noqa: BLE001
        uuid = None
    sampler = ClockSampler(local, uuid)
    if rank == 0:
        sampler.start()

    N, K, W = args.envs, args.steps, max(3, args.warmup)
    # synthetic seeded layouts, a distinct slice of seeds per rank (SURVEY 8d: seeds 777e6 + l, L = 65 536)
    base = 777_000_000 + rank * args.layouts
    cells, agent = _generate_layouts(base, args.layouts, world)
    env = BatchedMerlinEnv(N, cells, agent, width=SIZE, height=SIZE, device=dev, want_symbolic=False)
    env.reset()
    g = torch.Generator(device=dev).manual_seed(777 + rank)
    ring = 64
    acts = torch.randint(0, 3, (ring, N), generator=g, device=dev)  # outside the timed region

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ageing, untimed: every env gets a random episode clock in [0, max_steps), so the batch truncates and auto-resets
    # at the steady-state rate (N / 1024 envs per step, each onto a NEW layout of the pool) from the first timed step on
    # -- what a >= 2048-step run settles into -- instead of all envs reaching max_steps together at step 1024
    env.stagger_episode_clocks(seed=777 + rank)
    for i in range(W):
        env.step(acts[i % ring])
    barrier()
    lay0 = env.state_numpy()["layout"].copy()
    launches0 = env.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.mark("timed_start")
    e0.record()
    for i in range(K):
        last = env.step(acts[i % ring])
    e1.record()
    barrier()
    sampler.mark("timed_end")
    ms = e0.elapsed_time(e1)
    launches = env.launch_count() - launches0
    restarted = int((env.state_numpy()["layout"] != lay0).sum())  # envs that auto-reset onto another layout while timed
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)  # before the e2e steps below overwrite the env's output buffers
    del last

    # ---- e2e: host action buffers -> step -> host reward/flags (observations stay in HBM) -------------------
    e2e = None
    if not args.skip_e2e:
        Ke = min(K, 256)
        h_ring = 8
        h_act = torch.randint(0, 3, (h_ring, N), dtype=torch.int64).pin_memory()
        d_act = torch.empty(N, dtype=torch.int64, device=dev)
        # Two steps in flight: the H2D copy of step i+1's actions and the D2H copy of step i-1's results run on their
        # own streams beside step i's kernel; the host blocks on step i-1's results before it submits step i+1, so
        # every step's reward/flags are owned by the host one step later (what an asynchronous actor loop does).
        s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        main = torch.cuda.current_stream(dev)
        d_act2 = [torch.empty(N, dtype=torch.int64, device=dev) for _ in range(2)]
        bufs = [env.make_step_buffers() for _ in range(2)]
        h_out = [(torch.empty(N, dtype=torch.float32).pin_memory(), torch.empty(N, dtype=torch.bool).pin_memory(),
                  torch.empty(N, dtype=torch.bool).pin_memory()) for _ in range(2)]
        ev_in = [torch.cuda.Event() for _ in range(2)]
        ev_k = [torch.cuda.Event() for _ in range(2)]
        ev_out = [torch.cuda.Event() for _ in range(2)]

        def e2e_run(n):
            for b in range(2):
                ev_k[b].record(main)
                ev_out[b].record(s_out)
            for i in range(n):
                b = i & 1
                with torch.cuda.stream(s_in):
                    s_in.wait_event(ev_k[b])              # step i-2 has consumed this action buffer
                    d_act2[b].copy_(h_act[i % h_ring], non_blocking=True)
                    ev_in[b].record(s_in)
                main.wait_event(ev_in[b])
                main.wait_event(ev_out[b])                # step i-2's results have left this output buffer
                env.step(d_act2[b], out=bufs[b])
                ev_k[b].record(main)
                with torch.cuda.stream(s_out):
                    s_out.wait_event(ev_k[b])
                    h_out[b][0].copy_(bufs[b].reward, non_blocking=True)
                    h_out[b][1].copy_(bufs[b].terminated, non_blocking=True)
                    h_out[b][2].copy_(bufs[b].truncated, non_blocking=True)
                    ev_out[b].record(s_out)
                if i > 0:
                    ev_out[1 - b].synchronize()           # host now owns step i-1's reward / flags
            ev_out[(n - 1) & 1].synchronize()

        e2e_run(4)
        barrier()
        t0 = time.perf_counter()
        e2e_run(Ke)
        barrier()
        dt = time.perf_counter() - t0
        # serial variant (copy in, step, copy out, synchronise -- one step at a time)
        h_rew, h_te, h_tr = h_out[0]

        def e2e_step(i):
            d_act.copy_(h_act[i % h_ring], non_blocking=True)
            obs, r, te, tr, _ = env.step(d_act)
            h_rew.copy_(r, non_blocking=True); h_te.copy_(te, non_blocking=True); h_tr.copy_(tr, non_blocking=True)
            torch.cuda.current_stream().synchronize()

        for i in range(3):
            e2e_step(i)
        barrier()
        t2 = time.perf_counter()
        for i in range(Ke):
            e2e_step(i)
        barrier()
        dt_serial = time.perf_counter() - t2
        # variant with every observation copied to the host as well (what a host-side consumer would need)
        Ko = min(K, 4)
        n_host = min(N, 1 << 17)  # bound pinned memory: copy the first 131072 frames (1.2 GB) and scale
        h_obs = torch.empty((n_host, 56, 56, 3), dtype=torch.uint8).pin_memory()
        barrier()
        t1 = time.perf_counter()
        for i in range(Ko):
            d_act.copy_(h_act[i % h_ring], non_blocking=True)
            obs, r, te, tr, _ = env.step(d_act)
            h_rew.copy_(r, non_blocking=True)
            for lo in range(0, N, n_host):
                h_obs[: min(n_host, N - lo)].copy_(obs[lo:lo + n_host], non_blocking=True)
            torch.cuda.current_stream().synchronize()
        barrier()
        dt_obs = time.perf_counter() - t1
        e2e = {"seconds": dt, "steps": Ke, "seconds_obs": dt_obs, "steps_obs": Ko, "seconds_serial": dt_serial}

    # ---- reduce over ranks: max time, rank 0 prints -----------------------------------------------------------
    times = torch.tensor([ms, e2e["seconds"] if e2e else 0.0, e2e["seconds_obs"] if e2e else 0.0,
                          e2e["seconds_serial"] if e2e else 0.0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    ms_max, e2e_s, e2e_obs_s, e2e_serial_s = [float(x) for x in times.tolist()]
    step_kernel = env.step_kernel()
    # ---- learners (every rank takes part: gradient all-reduce over NCCL) ----------------------------------------
    env.close()
    del env, acts
    if e2e:
        del bufs, d_act2, h_out, h_obs
    torch.cuda.empty_cache()
    learners = {}
    if not args.skip_learners:
        learners["ppo"] = bench_ppo(args, dev, rank, world, cells, agent, sampler, barrier)
        torch.cuda.empty_cache()
        learners["fomaml"] = bench_fomaml(args, dev, rank, world, sampler, barrier)
        torch.cuda.empty_cache()
    clocks = sampler.stop() if rank == 0 else None
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    total_steps = world * N * K
    value = total_steps / (ms_max * 1e-3)
    peak, peak_src = hbm_peak()
    kernel_ms = ms_max / K
    achieved = ALGO_BYTES_PER_STEP * N / (kernel_ms * 1e-3) / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": kernel_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": f"configs[1]: mediumhard {SIZE}x{SIZE}, {N} envs per GPU, uniform random actions over "
                               "{left,right,forward}, auto-reset, RGB obs u8[N,56,56,3]",
                   "envs_per_gpu": N, "grid": SIZE, "max_steps": 4 * SIZE * SIZE, "layout_pool": args.layouts,
                   "episode_clocks": "staggered uniformly over [0, max_steps) before the warm-up (untimed ageing): the timed "
                                     "steps truncate / auto-reset envs at the steady-state rate of a long run",
                   "envs_restarted_on_a_new_layout_in_timed_region_rank0": restarted,
                   "layout_seeds": f"{base}..{base + args.layouts - 1} (np.random.default_rng, host-generated, uploaded)",
                   "parallelism": f"env-sharded x{world}, no data-path collective",
                   "l2": f"per-step working set {N * ALGO_BYTES_PER_STEP / 1e9:.2f} GB written/read >> 126 MB L2 (inputs larger than L2)"},
        "clocks": clocks,
        "gpu_launches": int(launches) * world,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": ncu_traffic(N, step_kernel), "peak_source": peak_src, "kernel": step_kernel,
                     "algorithmic_bytes_per_env_step": ALGO_BYTES_PER_STEP, "env_steps_per_launch": N,
                     "launch_ms": kernel_ms,
                     "note": "peak = measured COPY bandwidth (half reads, half writes); this kernel is 97% writes and a "
                             "write-only stream reaches 7.4-7.6 TB/s on this part (tools/fill_peak.py, "
                             "tools/cuda/write_pattern_bench.cu), so frac can exceed 1; ncu: 85% of nominal DRAM bandwidth"},
    }
    if e2e:
        h2d = N * 8
        d2h = N * (4 + 1 + 1)
        line["e2e"] = {"value": world * N * e2e["steps"] / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d,
                       "d2h_bytes_per_step": d2h, "obs_resident_in_hbm": True, "steps": e2e["steps"],
                       "pipelining": "two steps in flight (copies on side streams); host owns step i's results before "
                                     "submitting step i+2",
                       "note": "wall-clock over %d steps incl. both copies per step; the kernel runs back to back exactly as "
                               "in the device-timed loop (copies ride on side streams), and this shorter loop is less "
                               "power-capped than the %d-step one, so the two values agree within run-to-run spread" % (e2e["steps"], K),
                       "value_serial": world * N * e2e["steps"] / e2e_serial_s,
                       "value_obs_to_host": world * N * e2e["steps_obs"] / e2e_obs_s,
                       "d2h_bytes_per_step_obs_to_host": N * (56 * 56 * 3 + 4)}
    line.update(learners)
    if not args.skip_e2e:
        # second data point, this rank's GPU only: the same path with gen_obs's own observation (7x7x3 symbolic image,
        # 449 algorithmic B/step) instead of the wrapper's RGB frame -- the instruction-bound end of the path
        senv = BatchedMerlinEnv(N, cells, agent, width=SIZE, height=SIZE, device=dev, want_rgb=False, want_symbolic=True)
        senv.reset()
        senv.stagger_episode_clocks(seed=778)
        acts = torch.randint(0, 3, (ring, N), generator=g, device=dev)
        for i in range(W):
            senv.step(acts[i % ring])
        torch.cuda.synchronize(dev)
        Ks = min(K, 512)
        e0.record()
        for i in range(Ks):
            senv.step(acts[i % ring])
        e1.record()
        torch.cuda.synchronize(dev)
        sms = e0.elapsed_time(e1) / Ks
        sym_bytes = 147 + SIZE * SIZE + 32 + 8 + 6
        line["symbolic_only"] = {"value_per_gpu": N / (sms * 1e-3), "unit": UNIT, "ms_per_step": sms, "steps": Ks,
                                 "kernel": senv.step_kernel(), "algorithmic_bytes_per_env_step": sym_bytes,
                                 "roofline_frac": sym_bytes * N / (sms * 1e-3) / 1e9 / peak,
                                 "note": "ALU-bound (ncu: IPC 2.15, 20 % DRAM): the layout pool is L2-resident, ~160 B/step reach DRAM"}
        del senv
    if not args.skip_cpu_baseline:
        ref = CpuReference()
        n, dt = ref.run(200)
        per_proc = max(50, int(n / dt * args.cpu_seconds / ref.cores))
        n, dt = ref.run(per_proc)
        ref.close()
        c_rate, c_threads = c_oracle_rate()
        line["cpu_baseline"] = {
            "value": n / dt, "unit": UNIT, "cores": ref.cores, "kind": "port",
            "sample": f"{n} env-steps ({ref.cores} procs x {per_proc}) in {dt:.1f} s, mediumhard 16x16 random actions, "
                      "literal minigrid-3.0.0 restatement + reference wrapper stack (upstream not installable)",
            "per_process_value": per_proc / dt,  # one env in one process, the way the reference itself runs
            "c_oracle_value": c_rate, "c_oracle_threads": c_threads,
            "c_oracle_note": "optimised C restatement (OpenMP), not the reference"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def _claim_stdout():
    """Keep fd 1 for the ONE JSON line: everything else that writes to stdout while the bench runs (NCCL's version
    banner, library chatter of child processes) is sent to stderr; the JSON line goes to the saved descriptor."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(saved, "w", buffering=1)


if __name__ == "__main__":
    _claim_stdout()
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
