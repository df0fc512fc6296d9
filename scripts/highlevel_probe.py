"""High-level waypoints (task 5): what the fused step costs, against task 1 and against composing it by hand, and whether the
hierarchy learns.

In one process, with the card's name and power limit read in the same run:
  * env-steps/s of a random-action batch (the action tensor refilled on the device between steps) at --envs, for
      task1  waypoints_v3, one fw_step per agent step;
      task5  highlevel with a tracker, one fw_step per agent step (the tracker runs inside the step kernel);
      comp   the hand composition a user would write without task 5: per agent step, 4 x (CUDA-core forward of the tracker
             (ppo_policy_forward_a, deterministic) + one task-3 fw_step) -- 8 launches;
    each timed with CUDA events over --steps steps after --warmup untimed steps, the three alternated --reps times (median);
  * the fp32 share of the fused step from the algorithmic count: 7,000 flop of physics per agent step plus
    4 decisions x 11,648 flop of tracker (2 x (21 x 64 + 64 x 64 + 64 x 6) multiply-adds + 64 + 64 tanh + normalisation),
    over the FP32 FMA-chain peak measured in the run (fw_measure_fp32_peak);
  * PPO SPS on task 5 at 4,096 envs x n_steps 128 (4 minibatches, 20 epochs: bench.py's configs[2] variant B);
  * a learning check: a tracker trained on ``lowlevel``, then a high-level policy trained on ``highlevel`` with dense reward
    through it; evaluate() before and after (mean return, targets reached per episode).

    python scripts/highlevel_probe.py --out-dir profiles
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PHYS_FLOP, TRK_FLOP, DECISIONS = 7000, 11648, 4


def card() -> dict:
    import torch
    out = {"device": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        out["nvidia_smi"] = r.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out["nvidia_smi"] = f"unavailable: {e}"
    return out


def timed(fn, steps: int, warmup: int) -> float:
    """env-steps of one batch per second: CUDA events around `steps` calls of fn after `warmup` untimed ones."""
    import torch
    for _ in range(warmup):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    e1.synchronize()
    return steps / (e0.elapsed_time(e1) * 1e-3)


def throughput(n: int, tracker, model_low, steps: int, warmup: int, reps: int) -> dict:
    import torch
    import pyflyt_drone_b200 as fw
    from pyflyt_drone_b200.ppo import _p, _stream
    from pyflyt_drone_b200 import _lib
    g = torch.Generator(device="cuda").manual_seed(0)
    act4 = torch.empty((n, 4), device="cuda")
    e1 = fw.FixedwingVecEnv(n, preset="waypoints_v3", seed=1)
    e5 = fw.FixedwingVecEnv(n, preset="highlevel", seed=1, tracker=tracker)
    e3 = fw.FixedwingVecEnv(n, preset="lowlevel", seed=1, max_steps=3600)
    for e in (e1, e5):
        e.reset_tensor()
    o3 = e3.reset_tensor()
    act6 = torch.zeros((n, 6), device="cuda")
    val = torch.zeros(n, device="cuda")
    lib, m = _lib.load(), model_low

    def step1():
        act4.uniform_(-1, 1, generator=g); e1.step_tensor(act4)

    def step5():
        act4.uniform_(-1, 1, generator=g); e5.step_tensor(act4)

    def comp():
        nonlocal o3
        act4.uniform_(-1, 1, generator=g)          # the same per-step host work as the other two
        for _ in range(DECISIONS):
            _lib.check(lib.ppo_policy_forward_a(_p(m.policy.theta), 21, 6, _p(o3), m._stats_ptr(), m.vecnorm.clip_obs, n, 0, 0, 0,
                                                None, 1, None, _p(act6), None, None, _p(val), _stream()))
            o3 = e3.step_tensor(act6)[0]
    res = {"task1": [], "task5": [], "comp": []}
    for _ in range(reps):
        res["task1"].append(timed(step1, steps, warmup))
        res["task5"].append(timed(step5, steps, warmup))
        res["comp"].append(timed(comp, steps, warmup))
    for e in (e1, e5, e3):
        e.close()
    med = {k: statistics.median(v) * n for k, v in res.items()}
    return {"envs": n, "env_steps_per_s": med, "fused_over_comp": med["task5"] / med["comp"],
            "task5_over_task1": med["task5"] / med["task1"], "reps": reps, "steps": steps}


def one_iteration(model) -> float:
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    model.collect_rollouts()
    model.vecnorm.sync_across_ranks()
    model.train()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def ppo_sps(tracker, n=4096, n_steps=128) -> dict:
    import pyflyt_drone_b200 as fw
    from pyflyt_drone_b200.ppo import PPO
    env = fw.FixedwingVecEnv(n, preset="highlevel", seed=2, tracker=tracker)
    model = PPO("MlpPolicy", env, n_steps=n_steps, batch_size=n * n_steps // 4, n_epochs=20, seed=2)
    model.learn(2 * n * n_steps)                   # eager warm-up and graph capture
    t = statistics.median(one_iteration(model) for _ in range(3))
    env.close()
    return {"envs": n, "n_steps": n_steps, "sps": n * n_steps / t, "iter_s": t}


def learning(tracker_steps: int, high_steps: int) -> tuple[dict, object]:
    import pyflyt_drone_b200 as fw
    from pyflyt_drone_b200.ppo import PPO
    from pyflyt_drone_b200.tracker import Tracker
    n = 4096
    low = fw.FixedwingVecEnv(n, preset="lowlevel", seed=3)
    lm = PPO("MlpPolicy", low, n_steps=128, batch_size=n * 128 // 4, n_epochs=10, seed=3)
    before_low = lm.evaluate(n_eval_episodes=256, max_steps=2100)
    t0 = time.perf_counter()
    lm.learn(tracker_steps)
    t_low = time.perf_counter() - t0
    after_low = lm.evaluate(n_eval_episodes=256, max_steps=2100)
    tracker = Tracker.from_ppo(lm)
    high = fw.FixedwingVecEnv(n, preset="highlevel", seed=4, tracker=tracker, sparse_reward=0)
    hm = PPO("MlpPolicy", high, n_steps=128, batch_size=n * 128 // 4, n_epochs=20, seed=4, ent_coef=0.001)
    ev = lambda: hm.evaluate(n_eval_episodes=512, max_steps=3700)  # noqa: E731
    b = ev()
    t0 = time.perf_counter()
    hm.learn(high_steps)
    t_high = time.perf_counter() - t0
    a = ev()
    out = {"tracker": {"timesteps": tracker_steps, "train_s": t_low, "return_before": before_low.mean_reward,
                       "return_after": after_low.mean_reward, "len_after": after_low.mean_length},
           "highlevel": {"timesteps": high_steps, "train_s": t_high, "return_before": b.mean_reward, "return_after": a.mean_reward,
                         "targets_before": b.mean_targets_reached, "targets_after": a.mean_targets_reached,
                         "len_before": b.mean_length, "len_after": a.mean_length}}
    low.close(); high.close()
    return out, lm


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--envs", type=int, nargs="+", default=[4096, 65536])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--tracker-steps", type=int, default=60_000_000)
    ap.add_argument("--high-steps", type=int, default=60_000_000)
    args = ap.parse_args()
    import torch
    from pyflyt_drone_b200 import _lib
    rows = [{"kind": "card", **card()}]
    learn, lm = learning(args.tracker_steps, args.high_steps)
    from pyflyt_drone_b200.tracker import Tracker
    tracker = Tracker.from_ppo(lm)
    for n in args.envs:
        rows.append({"kind": "throughput", **throughput(n, tracker, lm, args.steps, args.warmup, args.reps)})
    tf = C.c_double(0.0)
    _lib.check(_lib.load().fw_measure_fp32_peak(0, C.byref(tf), None, None))
    flop = PHYS_FLOP + DECISIONS * TRK_FLOP
    for r in rows:
        if r["kind"] == "throughput":
            r["fp32_frac_task5"] = r["env_steps_per_s"]["task5"] * flop / (tf.value * 1e12)
    rows.append({"kind": "fp32", "peak_tflops": tf.value, "flop_per_agent_step": flop, "tracker_over_physics": DECISIONS * TRK_FLOP / PHYS_FLOP})
    rows.append({"kind": "ppo", **ppo_sps(tracker)})
    rows.append({"kind": "learning", **learn})
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "r6_highlevel.jsonl"), "w") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")
    c = rows[0]
    md = ["# r6: high-level waypoints (task 5)", "",
          f"Measured by `scripts/highlevel_probe.py` on {c['device']} (`nvidia-smi`: {c['nvidia_smi']}, name, power limit, max SM "
          "clock), in one run; raw rows in `r6_highlevel.jsonl`.", "",
          "## Step throughput (random high-level actions, env-steps/s, median of alternated repetitions)", "",
          "| envs | task 1 | task 5 (fused) | hand composition (8 launches) | task 5 / composition | task 5 / task 1 | task-5 fp32 share |",
          "|---|---|---|---|---|---|---|"]
    for r in rows:
        if r["kind"] == "throughput":
            v = r["env_steps_per_s"]
            md.append(f"| {r['envs']:,} | {v['task1']:.3g} | {v['task5']:.3g} | {v['comp']:.3g} | {r['fused_over_comp']:.2f}x | "
                      f"{r['task5_over_task1']:.3f} | {r['fp32_frac_task5']:.1%} |")
    fp = [r for r in rows if r["kind"] == "fp32"][0]
    pp = [r for r in rows if r["kind"] == "ppo"][0]
    ln = learn
    md += ["", f"fp32 share = task-5 env-steps/s x {fp['flop_per_agent_step']:,} flop (7,000 physics + 4 x 11,648 tracker, the "
           f"tracker {fp['tracker_over_physics']:.1f}x the physics) over the FP32 FMA-chain peak measured in the run, "
           f"{fp['peak_tflops']:.1f} TFLOP/s.", "",
           "## PPO on task 5", "", f"{pp['envs']:,} envs x n_steps {pp['n_steps']}, 4 minibatches, 20 epochs: "
           f"{pp['sps']:.3g} SPS ({pp['iter_s'] * 1e3:.1f} ms per iteration, median of 3).", "",
           "## Learning check", "",
           f"Tracker: PPO on `lowlevel`, 4,096 envs, {ln['tracker']['timesteps']:,} steps ({ln['tracker']['train_s']:.0f} s): "
           f"evaluate() return {ln['tracker']['return_before']:.1f} -> {ln['tracker']['return_after']:.1f}.", "",
           f"High level: PPO on `highlevel` (dense reward) through that tracker, 4,096 envs, {ln['highlevel']['timesteps']:,} "
           f"steps ({ln['highlevel']['train_s']:.0f} s): return {ln['highlevel']['return_before']:.1f} -> "
           f"{ln['highlevel']['return_after']:.1f}, targets per episode {ln['highlevel']['targets_before']:.2f} -> "
           f"{ln['highlevel']['targets_after']:.2f}, episode length {ln['highlevel']['len_before']:.0f} -> "
           f"{ln['highlevel']['len_after']:.0f} (512 evaluation episodes each)."]
    with open(os.path.join(args.out_dir, "r6_highlevel.md"), "w") as f:
        f.write("\n".join(md) + "\n")
    print("\n".join(md))


if __name__ == "__main__":
    main()
