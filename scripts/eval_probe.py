"""PPO.evaluate (device ledger, chunked, graph-replayed) against PPO.evaluate_policy (host loop, one sync per step).

For Waypoints and Waypoint-ObjLock and n_eval_episodes in {20, 1,024, 16,384} (training batch of --n-envs envs, so the eval
batch is min(n_envs, n_eval_episodes) envs with SB3's quotas), both evaluate the same seeded, perturbed policy with a fixed
--max-steps on caller-supplied eval batches built from one seed.  The first pair of calls runs on two fresh batches and must
agree: evaluate()'s episode table equals a host-loop recording of evaluate_policy's loop, and the four means are bit-identical.
Then --reps timed calls of each are alternated (wall clock around a device synchronise); evaluate() keeps its batch and the
chunk graph captured on its first call, as EvalCallback does, and that first call (with the capture) is reported on its own.
Card name and power limit are read in the same run.

    python scripts/eval_probe.py --out profiles/r4_eval_probe.jsonl
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


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


def host_record(m, env, n_eval, max_steps):
    """evaluate_policy's loop step for step, recording each selected episode as (return, length, targets, env, step)."""
    import torch
    obs = env.reset_tensor()
    n = env.num_envs
    quota = torch.tensor(m.episode_quotas(n_eval, n), dtype=torch.int64, device=m.device)
    count = torch.zeros(n, dtype=torch.int64, device=m.device)
    ret = torch.zeros(n, dtype=torch.float64, device=m.device)
    length = torch.zeros(n, dtype=torch.int64, device=m.device)
    rec = []
    for s in range(max_steps):
        obs, rew, flags = env.step_tensor(m.predict(obs))
        ret += rew.double()
        length += 1
        fin = (flags & 3) != 0
        take = fin & (count < quota)
        if bool(take.any()):
            idx = take.nonzero().flatten()
            tr = env.targets_reached_tensor()[idx].tolist()
            rec += list(zip(ret[idx].tolist(), length[idx].tolist(), tr, idx.tolist(), [s] * len(idx)))
            count += take.to(torch.int64)
        ret[fin] = 0.0
        length[fin] = 0
        if bool((count >= quota).all()):
            break
    return rec


def measure(preset: str, n_envs: int, n_eval: int, max_steps: int, reps: int) -> dict:
    import torch
    from pyflyt_drone_b200.ppo import PPO
    from pyflyt_drone_b200.vec_env import FixedwingVecEnv
    train = FixedwingVecEnv(n_envs, preset=preset, seed=5)
    m = PPO("MlpPolicy", train, n_steps=16, batch_size=n_envs * 16, n_epochs=1, seed=5)
    with torch.no_grad():
        m.policy.theta.add_(0.05 * torch.randn(m.policy.count, device=m.device, generator=m._gen))
    n = min(n_envs, n_eval)
    mk = lambda: FixedwingVecEnv(n, preset=preset, seed=1234, env_id0=1 << 24)  # noqa: E731
    # agreement on fresh batches
    a, b, c = mk(), mk(), mk()
    rec = host_record(m, a, n_eval, max_steps)
    ref = m.evaluate_policy(env=b, n_eval_episodes=n_eval, max_steps=max_steps)
    keep = c
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = m.evaluate(env=keep, n_eval_episodes=n_eval, max_steps=max_steps)
    torch.cuda.synchronize()
    first_ms = 1e3 * (time.perf_counter() - t0)
    steps_first = int(m._eval_state["step"].item())
    table = list(zip(res.returns.tolist(), res.lengths.tolist(), res.targets_reached.tolist(), res.env_index.tolist(),
                     res.finish_step.tolist()))
    assert table == rec, "evaluate() episode table differs from the host loop"
    got = (res.mean_reward, res.std_reward, res.mean_length, res.mean_targets_reached)
    assert np.array_equal(np.array(got), np.array(ref), equal_nan=True), (got, ref)
    a.close()
    steps_ref = (max(r[4] for r in rec) + 1) if len(rec) == n_eval else max_steps
    t_ref, t_dev, steps_dev = [], [], []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        m.evaluate_policy(env=b, n_eval_episodes=n_eval, max_steps=max_steps)
        torch.cuda.synchronize()
        t_ref.append(1e3 * (time.perf_counter() - t0))
        t0 = time.perf_counter()
        m.evaluate(env=keep, n_eval_episodes=n_eval, max_steps=max_steps)
        torch.cuda.synchronize()
        t_dev.append(1e3 * (time.perf_counter() - t0))
        steps_dev.append(int(m._eval_state["step"].item()))
    out = dict(preset=preset, n_envs_train=n_envs, eval_envs=n, n_eval_episodes=n_eval, max_steps=max_steps,
               episodes=res.n_episodes, steps_first_call=dict(evaluate_policy=steps_ref, evaluate=steps_first),
               evaluate_policy_ms=dict(median=statistics.median(t_ref), min=min(t_ref), max=max(t_ref)),
               evaluate_ms=dict(median=statistics.median(t_dev), min=min(t_dev), max=max(t_dev)),
               evaluate_steps_run=steps_dev, evaluate_first_call_ms=first_ms,
               speedup_median=statistics.median(t_ref) / statistics.median(t_dev), tables_agree=True, means_bit_identical=True)
    m._eval_state = None
    for e in (b, keep, train):
        e.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-envs", type=int, default=4096)
    ap.add_argument("--max-steps", type=int, default=400)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--episodes", type=str, default="20,1024,16384")
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("eval_probe needs a CUDA device")
    lines = [dict(card=card())]
    print(json.dumps(lines[0]), flush=True)
    for preset in ("waypoints_v3", "waypoint_objlock"):
        for n_eval in (int(x) for x in args.episodes.split(",")):
            r = measure(preset, args.n_envs, n_eval, args.max_steps, args.reps)
            lines.append(r)
            print(json.dumps(r), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
