"""PPOPopulation against standalone PPO runs one after another: aggregate PPO throughput of P members trained together.

Two member shapes on Waypoints (waypoints_v3, the reference's hyper-parameters):
  ref  the reference's own run: 32 envs, n_steps 2048, batch 128, 20 epochs (multi-step kernel, P thread blocks)
  B    configs[2] variant B per member: 4,096 envs, n_steps 128, 4 minibatches per epoch, 20 epochs (window update per member)
and P in --members.  Per (shape, P), in one process:
  * a population of P members (seeds 42 + k) over P * n envs;
  * standalone PPO models for the first K = min(P, --standalone) members (PPO's defaults, fused observation moments on), each
    on its own n-env batch, run one after another;
  * member 0's exact twin (fused_obs_moments = False), untimed, whose parameters, Adam state, counters and buffers must equal
    member 0's at the end (asserted in the run).
Each side first runs two untimed iterations (the eager warm-up and the graph capture), then --reps timed iterations alternate:
one population iteration, then one iteration of each of the K standalone models.  A time is the wall clock around one
`learn` iteration ending in a device synchronise; rollout and update are split as PPO.learn splits them.  The time of P
standalone iterations is P x the median per-model iteration of the K models (K < P: scaled, and reported as such).
Aggregate SPS = P * n * n_steps / time.  Card name and power limit are read in the same run.

    python scripts/population_probe.py --out profiles/r5_population.jsonl
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HP = dict(learning_rate=3e-4, gamma=0.99, gae_lambda=0.95, clip_range=0.2, ent_coef=0.001, vf_coef=0.5, max_grad_norm=0.5)
SHAPES = {"ref": dict(n=32, n_steps=2048, batch_size=128, n_epochs=20),
          "B": dict(n=4096, n_steps=128, batch_size=4096 * 128 // 4, n_epochs=20)}


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


def one_iteration(model) -> tuple[float, float]:
    """One learn iteration (rollout + update), as PPO.learn runs it; returns (rollout_s, update_s)."""
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    model.collect_rollouts()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    if hasattr(model, "vecnorm"):
        model.vecnorm.sync_across_ranks()
    else:
        model.obs_accum.zero_(); model.ret_accum.zero_()
    model.train()
    torch.cuda.synchronize()
    return t1 - t0, time.perf_counter() - t1


def measure(shape: str, P: int, K: int, reps: int) -> dict:
    import torch
    from pyflyt_drone_b200 import FixedwingVecEnv
    from pyflyt_drone_b200.population import PPOPopulation
    from pyflyt_drone_b200.ppo import PPO
    s = SHAPES[shape]
    n, T = s["n"], s["n_steps"]
    shared = dict(n_steps=T, batch_size=s["batch_size"], n_epochs=s["n_epochs"])
    env = FixedwingVecEnv(P * n, preset="waypoints_v3", seed=7)
    pop = PPOPopulation("MlpPolicy", env, members=P, seed=42, **shared, **HP)
    K = min(K, P)
    solo = []
    for m in range(K):
        e = FixedwingVecEnv(n, config=env.cfg, seed=7, env_id0=env.env_id0 + m * n)
        solo.append(PPO("MlpPolicy", e, seed=42 + m, **shared, **HP))
    twin = PPO("MlpPolicy", FixedwingVecEnv(n, config=env.cfg, seed=7, env_id0=env.env_id0), seed=42, **shared, **HP)
    twin.fused_obs_moments = False
    for _ in range(2):                                    # eager warm-up, then the graph capture
        one_iteration(pop); one_iteration(twin)
        for mdl in solo:
            one_iteration(mdl)
    pop_t, solo_t = [], []
    for _ in range(reps):
        pop_t.append(one_iteration(pop))
        one_iteration(twin)
        for mdl in solo:
            solo_t.append(one_iteration(mdl))
    # member 0 against its exact twin, same number of iterations
    ok = (torch.equal(pop.theta[0], twin.policy.theta.data) and torch.equal(pop.adam_m[0], twin._adam_m)
          and torch.equal(pop.adam_v[0], twin._adam_v) and int(pop.adam_t[0]) == int(twin._adam_t.item())
          and pop.num_timesteps == twin.num_timesteps
          and all(torch.equal(pop.buf[k][:, :n], twin.buf[k]) for k in ("obs", "act", "logp", "val", "rew", "done", "adv", "ret")))
    assert ok, f"member 0 differs from its standalone twin ({shape}, P={P})"
    med = lambda xs: statistics.median(xs)  # noqa: E731
    pr, pu = med([r for r, _ in pop_t]), med([u for _, u in pop_t])
    pi = med([r + u for r, u in pop_t])
    si = med([r + u for r, u in solo_t])
    sr, su = med([r for r, _ in solo_t]), med([u for _, u in solo_t])
    steps = P * n * T
    out = {"shape": shape, "members": P, "envs_per_member": n, **shared, "reps": reps, "standalone_timed": K,
           "standalone_scaled": K < P, "pop_iter_s": pi, "pop_rollout_s": pr, "pop_update_s": pu,
           "standalone_iter_s_per_model": si, "standalone_rollout_s_per_model": sr, "standalone_update_s_per_model": su,
           "standalone_P_iters_s": si * P, "pop_sps": steps / pi, "standalone_sps": steps / (si * P),
           "speedup": si * P / pi, "member0_equals_twin": ok}
    for mdl in solo:
        mdl.env.close()
    twin.env.close()
    env.close()
    del pop, solo, twin
    torch.cuda.empty_cache()
    return out


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--members", default="1,4,16,64,148")
    ap.add_argument("--shapes", default="ref,B")
    ap.add_argument("--standalone", type=int, default=4, help="standalone models timed per size (K)")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("population_probe measures on the GPU; no CUDA device is visible")
    lines = [{"card": card()}]
    print(json.dumps(lines[0]), flush=True)
    for shape in args.shapes.split(","):
        for P in (int(x) for x in args.members.split(",")):
            r = measure(shape, P, args.standalone, args.reps)
            lines.append(r)
            print(json.dumps(r), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
