#!/usr/bin/env python
"""bench.py -- fixed-wing env-steps/sec on B200 (BASELINE.json metric) + PPO SPS, one JSON line on stdout.

Our arm (default)
  step      ONE launch of the fused env-step kernel over one batch of `--envs` environments per GPU (default 65,536 =
            BASELINE configs[1], "batched fixed-wing physics step only, random actions"): 8 physics substeps at 240 Hz per
            env, actions drawn in-kernel from Philox, motor noise on, auto-reset on ground/dome.
  value     envs * n_gpus / (device time of one step).  The timed region is exactly `--steps` launches (a CUDA graph
            sequence), after `--warmup` untimed ones and one untimed call that builds the graphs of the timed call; its CUDA
            events are recorded in the enqueue order behind a warm launch, so host launch latency is outside the region;
            MAX over ranks.  Ask for enough steps that the region lasts tens of milliseconds (`ms_per_step` shows the
            length of one): a shorter window measures the clock as much as the kernel.
  L2        the per-batch state (~7 MB) would sit in the 126 MB L2 between launches, so the loop rotates over enough
            independent env batches that the working set exceeds 2x L2 ("l2" in config).  The launches of the graph are
            chained by programmatic dependent launch edges: consecutive launches step different batches, so the next one
            places its blocks while the previous one drains (its tail otherwise idles 54 % of the schedulers).
  e2e       the same metric through the reference-facing host call FixedwingVecEnv.step_arrays(actions) (VecEnv.step seam;
            C ABI fw_step_host) on the Fixedwing-Waypoints-v3 task with HOST buffers: H2D of the actions and D2H of
            obs/reward/flags inside the timed region (wall clock over `--steps` steps after `--warmup` untimed ones).
  roofline  dominant kernel fw_step_kernel.  `bound` names the pipe that binds it -- FP32 issue (SURVEY 8d: 6,400 flop per
            physics env-step against an FMA-chain peak measured in the same run); the HBM view (152 algorithmic bytes per
            env-step against MEASURED_PEAKS.json) rides along as `roofline.hbm`.
  ppo       PPO SPS (the second half of BASELINE's metric), rank-parallel with the NCCL gradient all-reduce INSIDE the timed
            region: configs[2] at 4,096 envs/GPU -- variant B (n_steps 128, 4 minibatches/epoch) and the SB3-faithful variant
            A (n_steps 2048, batch 128: 65,536 optimiser steps per epoch) -- and configs[3], Waypoint-ObjLock at 65,536
            envs/GPU, n_steps 64.
  cpu_baseline  the fp64 oracle (kind "port") on the host cores, bounded sample, rank 0 at N=1 only.
  --dump-outputs DIR  what the timed steps computed, rank 0's, as DIR/<name>.npy (float32; float64 and integer data as float64):
            step_<field> = state of the env batch the last timed launch stepped, e2e_obs / e2e_reward / e2e_flags = what the
            last e2e step returned, ppo_<workload>_theta / _obs_rms = policy parameters and observation moments after each
            PPO measurement.  Per-env rows are a seeded sample (env_index.npy) when all of them would pass 64 MB.  Every
            input is seeded and every step count fixed by the command line, so two builds run with the same arguments can
            be compared output for output.

Reference arm (--impl reference): the reference's CPU path.  PyFlyt/pybullet/SB3 cannot be installed offline and the
reference has no compilable sources, so this times the oracle port (all host threads) on the workload of our arm's `e2e`
-- Fixedwing-Waypoints-v3 stepped through host buffers -- plus the physics-only rate and a CPU PPO (oracle VecEnv + fp32
torch-CPU PPO, same hyper-parameters, bounded samples); rank 0 only under torchrun.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "fixedwing_env_steps_per_sec"
UNIT = "env-steps/s"
# SURVEY.md section 8(d); lowlevel (2 substeps per env-step): state 76 in + 76 out, action 24, target 12, obs 84, reward 4
# objlock_duck: state 76 + 76, action 16, wind 32, duck/vision planes 80 + 80, vision history 124 + 124, obs 224, reward 4
BYTES_PER_STEP = {"physics_only": 152, "waypoints_v3": 332, "waypoint_objlock": 400, "lowlevel": 276, "objlock_duck": 836}
FLOPS_PER_STEP = {"physics_only": 6400, "waypoints_v3": 7000, "waypoint_objlock": 7000, "lowlevel": 1750, "objlock_duck": 7000}
L2_BYTES = 126 * 1024 * 1024
DUMP_BYTES = 63 * 10**6   # --dump-outputs: array bytes, leaving room for the .npy headers under 64 MB
E2E_WORKLOAD = "waypoints_v3"
# reference's PPO hyper-parameters (train_Fixedwing_Waypoints_v3.py:27-55, train_Fixedwing_Waypoints_ObjLock.py:35-57)
PPO_HP = dict(learning_rate=3e-4, gamma=0.99, gae_lambda=0.95, clip_range=0.2, ent_coef=0.001, vf_coef=0.5, max_grad_norm=0.5)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--envs", type=int, default=65536, help="environments per GPU per launch")
    ap.add_argument("--workload", choices=["physics_only", "waypoints_v3", "waypoint_objlock", "lowlevel", "objlock_duck", "ppo"],
                    default="physics_only",
                    help="ppo = only the PPO measurements (a step is one PPO iteration), as its own JSON line")
    ap.add_argument("--ppo-preset", choices=["waypoints_v3", "waypoint_objlock", "lowlevel", "objlock_duck"], default="waypoints_v3")
    ap.add_argument("--ppo-envs", type=int, default=4096)
    ap.add_argument("--ppo-n-steps", type=int, default=128)
    ap.add_argument("--ppo-minibatches", type=int, default=4)
    ap.add_argument("--ppo-batch-size", type=int, default=0, help="overrides --ppo-minibatches (SB3-faithful: 128)")
    ap.add_argument("--ppo-epochs", type=int, default=20)
    ap.add_argument("--ppo-a-epochs", type=int, default=1,
                    help="variant A (batch 128): epochs of the 20 actually run per timed iteration in the default line; the "
                         "full-iteration SPS is then projected from the measured epoch time and labelled so")
    ap.add_argument("--ppo-a-full", action="store_true", help="variant A: run all 20 epochs (about half a minute per iteration)")
    ap.add_argument("--no-ppo", action="store_true", help="skip the ppo object of the default line")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target duration of the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--steps-per-launch", type=int, default=1,
                    help="env-steps fused into one launch (state kept in registers); a bench step is one launch")
    ap.add_argument("--no-graph", action="store_true", help="issue launches from the host loop instead of a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed steps computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what our arm's timed steps computed; the reference arm has none to write")
    return args


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            with open(path) as f:
                d = json.load(f)
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """SM clocks / throttle reasons during the timed regions (the quantities of the B200_PROFILING.md nvidia-smi recipe,
    read through NVML when nvidia_ml_py is importable, else by polling nvidia-smi)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self._stop_evt = index, [], threading.Event()

    def _nvml(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            bits = (("hw_slowdown", nv.nvmlClocksThrottleReasonHwSlowdown),
                    ("hw_thermal_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown),
                    ("sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwThermalSlowdown),
                    ("sw_power_cap", nv.nvmlClocksThrottleReasonSwPowerCap))

            def sample():
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                return [str(sm), str(mx), "0"] + ["Active" if (r & b) else "Not Active" for _, b in bits]
            sample()
            return sample
        except Exception:
            return None

    def run(self):
        sample = self._nvml()
        while not self._stop_evt.is_set():
            if sample is not None:
                try:
                    self.samples.append(sample())
                except Exception:
                    pass
                self._stop_evt.wait(0.002)
                continue
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 7:
                    self.samples.append(parts)
            except Exception:
                pass
            self._stop_evt.wait(0.1)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        sm, mx, reasons = [], [], set()
        for p in self.samples:
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_model() -> str:
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def bench_config(args) -> dict:
    """`config` of the JSON line: a function of the command line only, so that both arms print the same object."""
    n = args.envs
    if args.workload == "physics_only":
        wl = (f"physics_only: BASELINE configs[1] batched fixed-wing physics step, {n} envs/GPU, in-kernel Philox random "
              f"actions, motor noise on")
    else:
        wl = f"{args.workload}: {n} envs/GPU, random actions"
    return {"workload": wl, "envs_per_gpu": n, "substeps_per_env_step": 2 if args.workload == "lowlevel" else 8,
            "env_steps_per_launch": max(1, args.steps_per_launch),
            "e2e_workload": f"{E2E_WORKLOAD}: Fixedwing-Waypoints-v3 stepped through the host-buffer VecEnv.step seam "
                            f"(actions in host arrays; obs, reward, flags back in host memory), {n} envs/GPU",
            "reference_workload": "the reference arm times the CPU implementation on e2e_workload (its value and e2e) and "
                                  "reports the physics-only rate beside it",
            "ppo_workloads": ["configs[2] waypoints_v3 4096 envs/GPU: variant B n_steps 128 x 4 minibatches, variant A n_steps "
                              "2048 / batch 128", "configs[3] waypoint_objlock 65536 envs/GPU n_steps 64 x 4 minibatches"],
            "timing": f"one region of {args.steps} timed steps after {max(3, args.warmup)} untimed warm-up steps"}


# ----------------------------------------------------------------------------------------------------------- CPU arm
def oracle_rate(workload: str, threads: int, seconds: float, n_envs: int = 4096):
    """Time the fp64 oracle (oracle/) on a bounded sample of the same workload: random actions from the same Philox
    stream, same auto-reset.  Returns (env-steps/s, sample description)."""
    from oracle import fw_oracle as fo
    import pyflyt_drone_b200 as fw
    cfg = fw.make_config(workload)
    env = fo.OracleVecEnv(cfg.as_dict(), n_envs, seed=0, nthreads=threads)
    env.reset()
    t0 = time.perf_counter()
    env.rollout_random(2)
    probe = (time.perf_counter() - t0) / 2
    steps = max(2, min(20000, int(seconds / max(probe, 1e-6))))
    t0 = time.perf_counter()
    done = env.rollout_random(steps)
    dt = time.perf_counter() - t0
    return done / dt, f"{n_envs} envs x {steps} agent steps ({done} env-steps, {dt:.1f} s, {threads} threads, fp64 oracle port)"


def oracle_host_step_rate(workload: str, threads: int, n_envs: int, min_seconds: float, regions: int = 5):
    """The CPU counterpart of our arm's `e2e`: OracleVecEnv.step(actions) with host arrays in and obs/reward/flags/terminal
    obs out (the SubprocVecEnv.step contract), random actions prepared beforehand.  Median of `regions` regions of at
    least `min_seconds` each.  Returns (env-steps/s, steps per region, spread)."""
    import numpy as np
    from oracle import fw_oracle as fo
    import pyflyt_drone_b200 as fw
    cfg = fw.make_config(workload)
    env = fo.OracleVecEnv(cfg.as_dict(), n_envs, seed=0, nthreads=threads)
    env.reset()
    rng = np.random.default_rng(0)
    acts = [rng.uniform(-1, 1, (n_envs, env.act_dim)) for _ in range(8)]
    for s in range(4):                       # page in, spin the thread pool up
        env.step(acts[s % 8])
    t0 = time.perf_counter()
    for s in range(8):
        env.step(acts[s % 8])
    per = (time.perf_counter() - t0) / 8
    steps = max(4, int(np.ceil(min_seconds * 1.1 / max(per, 1e-7))))
    rates = []
    for _ in range(regions):
        t0 = time.perf_counter()
        for s in range(steps):
            env.step(acts[s % 8])
        rates.append(n_envs * steps / (time.perf_counter() - t0))
    rates.sort()
    return rates[len(rates) // 2], steps, (rates[-1] - rates[0]) / rates[len(rates) // 2]


def cpu_ppo(preset: str, n_envs: int, n_steps: int, batch_size: int, n_epochs: int, threads: int, iters: int = 1,
            warm: int = 0, epochs_run: int | None = None) -> dict:
    """CPU PPO SPS on a bounded sample: the fp64 oracle VecEnv on host threads + fp32 torch-CPU PPO with the reference's
    hyper-parameters (oracle/ppo_cpu.py; stable_baselines3 is not installable here).  epochs_run < n_epochs: only that
    many epochs of the update are run and the full iteration is projected (every epoch is the same number of identical
    optimiser steps), exactly as our arm does for variant A."""
    import torch
    import pyflyt_drone_b200 as fw
    from oracle.ppo_cpu import CpuPPO
    # thread counts that are fastest for the sample at hand: a 128-row minibatch through a 64-wide MLP loses time to
    # intra-op thread hand-offs, and an env step of a few dozen envs to thread start-up (measured here: 5.8 ms per
    # optimiser step with 8 torch threads against 3.9 ms with one)
    torch_threads = threads if batch_size >= 2048 else 1
    env_threads = max(1, min(threads, n_envs // 16))
    torch.set_num_threads(torch_threads)
    hp = dict(PPO_HP)
    run_epochs = n_epochs if epochs_run is None else min(epochs_run, n_epochs)
    m = CpuPPO(fw.make_config(preset).as_dict(), n_envs, n_steps, batch_size, run_epochs, lr=hp["learning_rate"], gamma=hp["gamma"],
               gae_lambda=hp["gae_lambda"], clip_range=hp["clip_range"], ent_coef=hp["ent_coef"], vf_coef=hp["vf_coef"],
               max_grad_norm=hp["max_grad_norm"], seed=42, nthreads=env_threads)
    for _ in range(warm):
        m.iteration()
    m.rollout_s = m.update_s = 0.0
    m.samples = 0
    for _ in range(iters):
        m.iteration()
    mb = -(-n_envs * n_steps // batch_size)
    rollout_s, update_s = m.rollout_s / iters, m.update_s / iters
    full = rollout_s + update_s * n_epochs / run_epochs
    out = {"sps": n_envs * n_steps / full, "rollout_s": rollout_s, "update_s": update_s, "envs": n_envs,
           "n_steps": n_steps, "batch_size": batch_size, "n_epochs": n_epochs, "iterations": iters,
           "optimizer_steps_per_iteration": run_epochs * mb, "optimizer_step_us": update_s / (run_epochs * mb) * 1e6,
           "threads": threads, "torch_threads": torch_threads, "env_threads": env_threads,
           "full_iteration": run_epochs == n_epochs,
           "kind": "port", "impl": "fp64 oracle VecEnv + fp32 torch-CPU PPO (oracle/ppo_cpu.py)"}
    if run_epochs < n_epochs:
        out["epochs_timed"] = run_epochs
        out["sps_note"] = (f"update timed for {run_epochs} of {n_epochs} epochs; sps = env-steps of one rollout / (rollout_s + "
                           f"{n_epochs} x epoch_s)")
    return out


def reference_ppo(threads: int) -> dict:
    """Bounded CPU samples of the three PPO workloads of our arm's `ppo` object (same hyper-parameters; fewer envs: the
    per-sample cost is what the rate measures)."""
    out = {}
    out["waypoints_v3_B"] = cpu_ppo("waypoints_v3", 256, 128, 256 * 128 // 4, 20, threads)
    out["waypoints_v3_B"]["sample"] = "256 of 4096 envs, n_steps 128, 4 minibatches x 20 epochs, 1 iteration"
    # the reference's own configuration: 32 envs x 2048 steps, batch 128, 20 epochs (train_Fixedwing_Waypoints_v3.py:28-40)
    out["waypoints_v3_A"] = cpu_ppo("waypoints_v3", 32, 2048, 128, 20, threads, epochs_run=2)
    out["waypoints_v3_A"]["sample"] = "32 envs (the reference's num_envs) of 4096, n_steps 2048, batch 128, 2 of 20 epochs timed"
    out["waypoint_objlock"] = cpu_ppo("waypoint_objlock", 256, 64, 256 * 64 // 4, 20, threads)
    out["waypoint_objlock"]["sample"] = "256 of 65536 envs, n_steps 64, 4 minibatches x 20 epochs, 1 iteration"
    return out


def run_reference(args, rank: int, world: int):
    if rank != 0:
        return
    threads = host_cores()
    n_envs = 16384        # per-step sample: large enough that the per-call thread start-up of the oracle's parallel-for is noise
    wl = E2E_WORKLOAD if args.workload == "physics_only" else args.workload
    v, steps, spread = oracle_host_step_rate(wl, threads, n_envs, 2.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": n_envs / v * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": bench_config(args),
        "timed": {"regions": 5, "steps_per_region": steps, "sample_envs_per_step": n_envs, "region_s": steps * n_envs / v,
                  "spread": spread, "statistic": "median"},
        "note": "reference CPU path restated as the fp64 oracle port (PyFlyt/pybullet/SB3 are not installable offline); each "
                f"step is a bounded sample of the workload: one agent step of a {n_envs}-env slice of the batch through "
                "OracleVecEnv.step (host arrays in and out) on all host threads",
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{wl}: {n_envs} envs per step through host buffers, 5 regions of {steps} steps (>= 2 s each), "
                                   f"median, {threads} host threads, {cpu_model()}"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if args.workload == "physics_only":
        pv, psample = oracle_rate("physics_only", threads, 3.0)
        line["physics_only"] = {"value": pv, "unit": UNIT, "sample": psample,
                                "note": "like-for-like CPU figure for our arm's device-timed `value`"}
    if not args.no_ppo:
        try:
            line["ppo"] = reference_ppo(threads)
        except Exception as e:        # the CPU PPO must never take the env-step line down with it
            line["ppo"] = {"error": f"{type(e).__name__}: {e}"}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------- our arm
def dump_outputs(directory: str, per_env: dict, whole: dict) -> None:
    """Write every array as `directory`/<name>.npy in float32 (float64 for float64 and integer data).  `per_env` arrays
    have the env index as first axis and share one seeded sample of rows (saved as env_index) when all rows would pass
    DUMP_BYTES; `whole` arrays are written in full."""
    import numpy as np

    def wide(a):
        a = np.asarray(a)
        return a if a.dtype in (np.float32, np.float64) else a.astype(np.float64)
    per_env = {k: wide(v) for k, v in per_env.items()}
    whole = {k: wide(v) for k, v in whole.items()}
    os.makedirs(directory, exist_ok=True)
    if per_env:
        n = len(next(iter(per_env.values())))
        row_bytes = sum(v[0].nbytes for v in per_env.values()) + 8
        keep = min(n, (DUMP_BYTES - sum(v.nbytes for v in whole.values())) // row_bytes)
        rows = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        whole["env_index"] = rows.astype(np.float64)
        per_env = {k: v[rows] for k, v in per_env.items()}
    for name, a in {**per_env, **whole}.items():
        np.save(os.path.join(directory, f"{name}.npy"), a)


def _max_over_ranks(x: float, world: int) -> float:
    import torch
    import torch.distributed as dist
    if world == 1:
        return float(x)
    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def ppo_measure(preset: str, n_envs: int, n_steps: int, batch_size: int, n_epochs: int, rank: int, local_rank: int,
                world: int, iters: int = 2, warm: int = 1, epochs_run: int | None = None, outputs: dict | None = None,
                name: str = "") -> dict:
    """One PPO workload: `warm` untimed iterations (the second one captures the rollout CUDA graph), then `iters` timed
    iterations of rollout + update between barriers, device-synchronised on both sides, MAX over ranks.  The NCCL
    all-reduce of the 49 KB gradient runs inside the update of every optimiser step when world > 1.
    epochs_run < n_epochs: the update runs only that many of the n_epochs epochs (variant A's bounded default).
    `outputs`: receives ppo_<name>_theta and ppo_<name>_obs_rms (mean, var, count) as left by the timed iterations."""
    import torch
    import torch.distributed as dist
    from pyflyt_drone_b200.ppo import PPO
    from pyflyt_drone_b200.vec_env import FixedwingVecEnv
    env = FixedwingVecEnv(n_envs, preset=preset, device=local_rank, seed=42, env_id0=rank * n_envs)
    run_epochs = n_epochs if epochs_run is None else min(epochs_run, n_epochs)
    model = PPO("MlpPolicy", env, n_steps=n_steps, batch_size=batch_size, n_epochs=run_epochs, seed=42, **PPO_HP)
    per_iter = n_envs * n_steps * world
    model.learn(max(2, warm + 1) * per_iter)        # eager rollout, then graph capture + replay
    model.stats.__init__()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    model.learn(iters * per_iter)
    torch.cuda.synchronize()
    dt = _max_over_ranks(time.perf_counter() - t0, world)
    if outputs is not None:
        outputs[f"ppo_{name}_theta"] = model.policy.theta.detach().float().cpu().numpy()
        outputs[f"ppo_{name}_obs_rms"] = model.vecnorm.obs_stats.cpu().numpy()
    st = model.stats
    rollout_s = _max_over_ranks(st.rollout_s, world) / iters
    update_s = _max_over_ranks(st.update_s, world) / iters
    mb = -(-n_envs * n_steps // batch_size)
    ar_us = 0.0
    if world > 1:                                    # cost of the path's one collective, measured on its own
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(20):
            dist.all_reduce(model._grad)
        torch.cuda.synchronize(); dist.barrier()
        e0.record()
        for _ in range(200):
            dist.all_reduce(model._grad)
        e1.record(); torch.cuda.synchronize()
        ar_us = _max_over_ranks(e0.elapsed_time(e1) / 200 * 1e3, world)
    in_sync = True
    if world > 1:                                    # every rank must hold the same parameters after the timed updates
        th = model.policy.theta.detach().clone()
        dist.all_reduce(th, op=dist.ReduceOp.MAX)
        in_sync = bool(torch.equal(th, model.policy.theta.detach()))
        flag = torch.tensor([1.0 if in_sync else 0.0], device=th.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        in_sync = bool(flag.item() > 0.5)
    chunk = model._ugraph_key[2] if getattr(model, "_ugraph_key", None) else 0
    # launches of OUR kernels per epoch of the update, by the path PPO._train_kernel took (see pyflyt_drone_b200/ppo.py)
    in_kernel_reduce = world == 1 or getattr(model, "_p2p", None) is not None
    if model.update != "kernel":
        update_launches, update_path = 0, "torch autograd (reference path)"
    elif in_kernel_reduce and batch_size <= model.fused_steps_max_batch and (n_envs * n_steps) % batch_size == 0:
        win = max(c for c in range(1, min(mb, model.update_graph_steps) + 1) if mb % c == 0)
        update_launches = 1 + mb // win                       # permutation + one single-block launch per window of steps
        update_path = f"single-block launches of {win} optimizer steps"
    elif chunk and in_kernel_reduce:
        update_launches = (mb // chunk) * 3 + mb * 2          # per window: permutation window + advance + advantage statistics
        update_path = f"graph windows of {chunk} steps: gradient kernel + reduction with clip/Adam (and the peer exchange) per step"
    elif chunk:
        update_launches = (mb // chunk) * 2 + mb * 4          # adv stats, gradient, reduce, [NCCL], Adam
        update_path = f"graph windows of {chunk} steps with an NCCL all-reduce between reduce and Adam"
    else:
        update_launches, update_path = 1 + mb * 4, "eager optimizer steps"
    out = {"sps": iters * per_iter / dt, "n_gpus": world, "envs_per_gpu": n_envs, "n_steps": n_steps, "batch_size_per_gpu": batch_size,
           "n_epochs": n_epochs, "iterations": iters, "iter_ms": dt / iters * 1e3, "rollout_s": rollout_s, "update_s": update_s,
           "rollout_env_steps_per_sec": per_iter / max(rollout_s, 1e-9),
           "optimizer_steps_per_iteration": run_epochs * mb, "optimizer_step_us": update_s / max(run_epochs * mb, 1) * 1e6,
           "allreduce_us": ar_us, "allreduce_bytes": int(model._grad.numel() * 4),
           "allreduce_in_timed_region": world > 1,
           "update": "fused tcgen05 minibatch gradient kernel + clip/Adam kernel" if model.update == "kernel" else "torch autograd",
           "forward": "tcgen05 kind::tf32 policy/value forward" if model.tensor_core_forward else "CUDA-core fp32 forward",
           # rollout graph per step: policy forward, env step (+ obs moment sums), moments finalize, return moments + reward
           # finalise, bootstrap; per rollout: counter, last values, GAE; update: see update_launches above
           "update_graph_steps": chunk, "ranks_in_sync": in_sync,
           "gradient_allreduce": ("none (one rank)" if world == 1 else
                                  "in-kernel over NVLink peer memory (last block of the gradient reduction)" if getattr(model, "_p2p", None)
                                  else "NCCL all_reduce between the gradient and Adam kernels"),
           "update_path": update_path,
           "gpu_launches": int(iters * (n_steps * 6 + 3 + run_epochs * update_launches))}
    if run_epochs < n_epochs:
        epoch_s = update_s / run_epochs
        full = rollout_s + n_epochs * epoch_s
        out.update({"full_iteration": False, "epochs_timed": run_epochs, "epoch_s": epoch_s,
                    "sps_timed_region": out.pop("sps"),
                    "sps": per_iter / full,
                    "sps_note": f"update timed for {run_epochs} of {n_epochs} epochs ({run_epochs * mb} optimiser steps); sps = env-steps "
                                f"of one rollout / (rollout_s + {n_epochs} x epoch_s), every epoch being {mb} identical optimiser "
                                "steps; `--ppo-a-full` runs all of them"})
    else:
        out["full_iteration"] = True
    env.close()
    del model
    torch.cuda.empty_cache()
    return out


def run_ours(args, rank: int, local_rank: int, world: int):
    import numpy as np
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the env step has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    import ctypes as C
    import pyflyt_drone_b200 as fw
    from pyflyt_drone_b200 import _lib
    from pyflyt_drone_b200.vec_env import FixedwingVecEnv

    cfg = fw.make_config(args.workload)
    N = args.envs
    state_bytes = N * (6 * 16 + 4 + (cfg.num_targets * 12) + (5 * 16 + 32 * 12 if cfg.task in (2, 4) else 0)
                       + (31 * 4 if cfg.task == 4 else 0))
    replicas = max(2, int(np.ceil(2 * L2_BYTES / state_bytes)))
    envs = [FixedwingVecEnv(N, config=cfg, device=local_rank, seed=1234, env_id0=(rank * replicas + r) * N)
            for r in range(replicas)]
    K, W = args.steps, max(3, args.warmup)
    graph = not args.no_graph
    spl = max(1, args.steps_per_launch)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def ev():
        return torch.cuda.Event(enable_timing=True)

    FixedwingVecEnv.rollout_random(envs, W, spl, use_graph=False)                 # W untimed warm-up steps
    FixedwingVecEnv.rollout_random(envs, K, spl, use_graph=graph)                 # builds + instantiates the graphs of K launches
    launches0 = sum(e.launch_count for e in envs)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    barrier()
    if sampler:
        sampler.start()
    e0, e1 = ev(), ev()
    FixedwingVecEnv.rollout_random(envs, replicas, spl, use_graph=graph)           # warm launch: the GPU is busy ...
    e0.record()                                                                    # ... so the region opens behind it, in enqueue order
    FixedwingVecEnv.rollout_random(envs, K, spl, use_graph=graph)
    e1.record()
    barrier()
    region_ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if sampler else None        # sampled during the timed region only
    launches = sum(e.launch_count for e in envs) - launches0
    step_ms = _max_over_ranks(region_ms / K, world)
    value = N * spl * world / (step_ms * 1e-3)
    kernel_ms = step_ms          # back-to-back launches of one kernel: the mean launch-to-launch duration
    env_outputs, outputs = {}, ({} if args.dump_outputs else None)
    if args.dump_outputs:        # every call of rollout_random starts at envs[0]: the last timed launch stepped this batch
        env_outputs = {f"step_{k}": v for k, v in envs[(K - 1) % replicas].get_state().items()}
    for e in envs:
        e.close()
    envs = []

    # ---- e2e: the VecEnv.step seam with host buffers (Waypoints-v3 task, obs/reward/flags come back) ----
    e2e_cfg = fw.make_config(E2E_WORKLOAD)
    venv = FixedwingVecEnv(N, config=e2e_cfg, device=local_rank, seed=99, env_id0=rank * N)
    venv.reset()
    rng = np.random.default_rng(rank)
    # the step's inputs wait in pinned host memory (bench contract); FixedwingVecEnv reads page-locked caller buffers in place
    pinned = [torch.empty((N, 4), dtype=torch.float32, pin_memory=True) for _ in range(4)]   # owns the memory
    acts = [b.numpy() for b in pinned]
    for a in acts:
        a[:] = rng.uniform(-1, 1, (N, 4)).astype(np.float32)
    for s in range(W):
        venv.step_arrays(acts[s % 4], want_terminal_obs=False)
    barrier()
    t0 = time.perf_counter()
    for s in range(K):
        obs, rew, flags, _ = venv.step_arrays(acts[s % 4], want_terminal_obs=False)
    torch.cuda.synchronize()
    e2e_step_s = _max_over_ranks((time.perf_counter() - t0) / K, world)
    e2e_value = N * world / e2e_step_s
    h2d = N * 4 * 4
    d2h = N * venv.obs_dim * 4 + N * 4 + N + N          # obs, reward, flag byte, targets-reached byte
    e2e_launches = K * (2 if N >= 16384 else 1)
    if args.dump_outputs:
        env_outputs.update(e2e_obs=obs.copy(), e2e_reward=rew.copy(), e2e_flags=flags.copy())
    venv.close()
    # what bounds e2e: the step's results cross PCIe (the kernel writes them into pinned host memory as it runs); the link's
    # device->host rate is measured here with plain pinned copies of 64 MiB (copy engine, nothing else on the link)
    pcie = None
    try:
        big_d = torch.empty(64 << 20, dtype=torch.uint8, device=f"cuda:{local_rank}")
        big_h = torch.empty(64 << 20, dtype=torch.uint8, pin_memory=True)
        for _ in range(3):
            big_h.copy_(big_d, non_blocking=True)
        p0, p1 = ev(), ev()
        p0.record()
        for _ in range(10):
            big_h.copy_(big_d, non_blocking=True)
        p1.record(); torch.cuda.synchronize()
        peak = 10 * (64 << 20) / (p0.elapsed_time(p1) * 1e-3) / 1e9
        ach = d2h / e2e_step_s / 1e9
        pcie = {"bound": "pcie_d2h", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "note": "achieved = d2h_bytes_per_step / step time of this rank's GPU; peak = 64 MiB pinned device->host copies "
                        "measured in this run; a step is synchronous (the next actions depend on its observations), so host "
                        "latency per step is inside"}
        del big_d, big_h
    except Exception as e:            # never lose the line over the side measurement
        pcie = {"error": f"{type(e).__name__}: {e}"}

    # ---- PPO SPS: every rank takes part (gradient all-reduce inside the timed region) ----
    ppo = None
    if not args.no_ppo and args.workload == "physics_only":
        ppo = {}
        try:
            ppo["waypoints_v3_B"] = ppo_measure("waypoints_v3", 4096, 128, 4096 * 128 // 4, 20, rank, local_rank, world, iters=3,
                                                outputs=outputs, name="waypoints_v3_B")
            ppo["waypoints_v3_A"] = ppo_measure("waypoints_v3", 4096, 2048, 128, 20, rank, local_rank, world, iters=1, warm=1,
                                                epochs_run=None if args.ppo_a_full else args.ppo_a_epochs,
                                                outputs=outputs, name="waypoints_v3_A")
            ppo["waypoint_objlock"] = ppo_measure("waypoint_objlock", 65536, 64, 65536 * 64 // 4, 20, rank, local_rank, world, iters=2,
                                                  outputs=outputs, name="waypoint_objlock")
        except Exception as e:
            ppo["error"] = f"{type(e).__name__}: {e}"
            if world > 1:
                raise

    if rank == 0:
        hbm_peak, peak_src = measured_peaks()
        tf, sms, khz = C.c_double(), C.c_int32(), C.c_int32()
        _lib.check(_lib.load().fw_measure_fp32_peak(local_rank, C.byref(tf), C.byref(sms), C.byref(khz)))
        per_gpu = N * spl / (kernel_ms * 1e-3)
        achieved_gbs = per_gpu * BYTES_PER_STEP[args.workload] / 1e9
        fp32_tf = per_gpu * FLOPS_PER_STEP[args.workload] / 1e12
        traffic, executed, tj = None, None, {}
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            try:
                tj = json.load(open(tpath))
                traffic = tj.get(f"{args.workload}_{N}")
                executed = tj.get(f"{args.workload}_executed_fp32_flop_per_env_step")
            except Exception:
                traffic = None
        roof = {"bound": "fp32", "achieved": fp32_tf, "peak": tf.value, "unit": "TFLOP/s", "frac": fp32_tf / tf.value,
                "traffic": traffic, "kernel": "fw_step_kernel", "kernel_ms": kernel_ms,
                "flops_per_env_step": FLOPS_PER_STEP[args.workload], "sm_count": sms.value,
                "peak_source": "FP32 FMA chain measured in this run (fw_measure_fp32_peak); MEASURED_PEAKS.json has no FP32 entry",
                "binding_pipe": "fp32 issue (arithmetic intensity 42 flop/B against a ridge of 11)",
                "hbm": {"achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": achieved_gbs / hbm_peak,
                        "algorithmic_bytes_per_env_step": BYTES_PER_STEP[args.workload], "peak_source": peak_src}}
        if executed:
            roof["executed_fp32_flop_per_env_step"] = executed
            roof["executed_frac"] = per_gpu * executed / 1e12 / tf.value
        winst = tj.get(f"{args.workload}_executed_warp_inst_per_env_step")
        if winst:
            # the ceiling that actually binds K1: one warp instruction per scheduler per clock (4 schedulers per SM); the mix is
            # 1 flop per instruction (FFMA 33 %, FMUL 23 %, FADD 12 %, the rest loads / compares / MUFU), so the FMA-chain
            # peak above is not reachable by this instruction stream
            mhz = (clocks or {}).get("sm_mhz") or khz.value / 1e3
            issue_peak = sms.value * 4 * mhz * 1e6
            issue_ach = per_gpu * winst / 32.0
            roof["issue"] = {"achieved": issue_ach, "peak": issue_peak, "unit": "warp-instructions/s", "frac": issue_ach / issue_peak,
                             "warp_inst_per_env_step": winst, "sm_mhz": mhz,
                             "note": "executed warp instructions per env-step from the ncu capture x env-steps/s / 32 lanes, "
                                     "against SMs x 4 schedulers x the SM clock sampled under load"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": bench_config(args),
            "timed": {"regions": 1, "timed_launches": K, "region_ms": region_ms, "statistic": "region / K, MAX over ranks",
                      "physics_substeps_per_sec": value * cfg.inner_per_step * cfg.substeps_per_inner,
                      "l2": f"rotating {replicas} env batches ({replicas * state_bytes / 2**20:.0f} MiB > 2x L2)",
                      "launch": "host loop" if args.no_graph else
                                f"CUDA graph of {replicas} launches chained by programmatic dependent launch edges (each launch steps "
                                f"another env batch; the next one places its blocks while this one drains; FWSIM_PDL=0 = plain edges)"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "us_per_step": e2e_step_s * 1e6, "steps_per_region": K, "regions": 1, "roofline": pcie},
            "gpu_launches": int(launches + e2e_launches),
            "clocks": clocks,
            "roofline": roof,
        }
        if ppo is not None:
            line["ppo"] = ppo
        if world == 1 and not args.no_cpu_baseline:
            v, sample = oracle_rate(args.workload, host_cores(), args.cpu_seconds)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": host_cores(), "kind": "port",
                                    "sample": sample + f"; {cpu_model()}"}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, env_outputs, outputs)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_ppo(args, rank: int, local_rank: int, world: int):
    """`--workload ppo`: one PPO workload as its own JSON line (a step = one rollout + one update)."""
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    N, T = args.ppo_envs, args.ppo_n_steps
    bs = args.ppo_batch_size if args.ppo_batch_size > 0 else N * T // args.ppo_minibatches
    K = args.steps
    outputs = {} if args.dump_outputs else None
    r = ppo_measure(args.ppo_preset, N, T, bs, args.ppo_epochs, rank, local_rank, world, iters=K, warm=1, outputs=outputs,
                    name=args.ppo_preset)
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {}, outputs)
        line = {"metric": "ppo_env_steps_per_sec", "value": r["sps"], "unit": "env-steps/s", "n_gpus": world,
                "steps": K, "warmup": 2, "ms_per_step": r["iter_ms"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": f"ppo: {args.ppo_preset} PPO rollout+update (BASELINE configs[2]/[3])", **r},
                "gpu_launches": r["gpu_launches"]}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.workload == "ppo":
        run_ppo(args, rank, local_rank, world)
        return
    run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
