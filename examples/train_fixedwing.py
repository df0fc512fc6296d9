#!/usr/bin/env python
"""PPO training on the B200-native simulator with the reference's TRAIN_CONFIG keys.

Counterpart of /root/reference/train/train_Fixedwing_Waypoints_v3.py (--task waypoints) and
train_Fixedwing_Waypoints_ObjLock.py (--task objlock) / train_lowlevel_cmd.py (--task lowlevel) / train_objlock.py
(--task duck, the duck-only lock-and-strike env) / train_highlevel_cmd.py (--task highlevel --tracker PATH, waypoints flown
through a frozen --task lowlevel policy): same hyper-parameter dictionary, same flow
(vectorised env -> observation/reward normalisation -> PPO("MlpPolicy", ...).learn -> save model + vecnorm),
with SubprocVecEnv/VecNormalize/PPO replaced by their device-resident equivalents.

    python examples/train_fixedwing.py --task waypoints --num_envs 4096 --total_timesteps 20000000
    torchrun --nproc-per-node 8 --master-addr 127.0.0.1 examples/train_fixedwing.py --task objlock --num_envs 65536
"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

TRAIN_CONFIG = {
    "waypoints": {   # train_Fixedwing_Waypoints_v3.py:27-55
        "total_timesteps": 4_000_000, "num_envs": 32, "num_targets": 8, "goal_reach_distance": 4, "sparse_reward": True,
        "learning_rate": 3e-4, "n_steps": 2048, "batch_size": 128, "n_epochs": 20, "gamma": 0.99, "gae_lambda": 0.95,
        "clip_range": 0.2, "ent_coef": 0.001, "vf_coef": 0.5, "max_grad_norm": 0.5, "seed": 42,
        "model_dir": "models/waypoints_ppo_b200", "flight_dome_size": 100.0, "max_duration_seconds": 120.0,
        "context_length": 2, "preset": "waypoints_v3",
    },
    "objlock": {     # train_Fixedwing_Waypoints_ObjLock.py:35-92
        "total_timesteps": 20_000_000, "num_envs": 32, "num_targets": 8, "goal_reach_distance": 8, "sparse_reward": False,
        "learning_rate": 3e-4, "n_steps": 1024, "batch_size": 128, "n_epochs": 20, "gamma": 0.99, "gae_lambda": 0.95,
        "clip_range": 0.2, "ent_coef": 0.001, "vf_coef": 0.5, "max_grad_norm": 0.5, "seed": 42,
        "model_dir": "models/obj_strike_ppo_b200", "flight_dome_size": 100.0, "max_duration_seconds": 120.0,
        "context_length": 2, "preset": "waypoint_objlock",
    },
    "lowlevel": {    # train_lowlevel_cmd.py:27-49 (FixedwingLowLevelEnv: 6-channel actions, psi/h/V tracking)
        "total_timesteps": 2_000_000, "num_envs": 32, "learning_rate": 3e-4, "n_steps": 2048, "batch_size": 64, "n_epochs": 10,
        "gamma": 0.99, "gae_lambda": 0.95, "clip_range": 0.2, "ent_coef": 0.0, "vf_coef": 0.5, "max_grad_norm": 0.5, "seed": 42,
        "model_dir": "models/lowlevel_ppo_b200", "preset": "lowlevel",
    },
    "duck": {        # train_objlock.py:27-85 (FixedwingObjLockEnv + FlattenObjLockEnv: 56-float vision-history observation)
        "total_timesteps": 1_000_000, "num_envs": 16, "learning_rate": 3e-4, "n_steps": 2048, "batch_size": 64, "n_epochs": 10,
        "gamma": 0.99, "gae_lambda": 0.95, "clip_range": 0.2, "ent_coef": 0.001, "vf_coef": 0.5, "max_grad_norm": 0.5, "seed": 42,
        "model_dir": "models/obj_lock_only_ppo_b200", "preset": "objlock_duck",
    },
    "highlevel": {   # train_highlevel_cmd.py: the waypoints episode commanded through a frozen tracker (--tracker)
        "total_timesteps": 4_000_000, "num_envs": 32, "num_targets": 8, "goal_reach_distance": 4, "sparse_reward": True,
        "learning_rate": 3e-4, "n_steps": 2048, "batch_size": 128, "n_epochs": 20, "gamma": 0.99, "gae_lambda": 0.95,
        "clip_range": 0.2, "ent_coef": 0.001, "vf_coef": 0.5, "max_grad_norm": 0.5, "seed": 42,
        "model_dir": "models/highlevel_ppo_b200", "flight_dome_size": 100.0, "max_duration_seconds": 120.0,
        "context_length": 2, "preset": "highlevel",
    },
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--task", choices=list(TRAIN_CONFIG), default="waypoints")
    ap.add_argument("--num_envs", type=int, default=None, help="envs per GPU (the reference uses 32 processes)")
    ap.add_argument("--n_steps", type=int, default=None)
    ap.add_argument("--batch_size", type=int, default=None)
    ap.add_argument("--total_timesteps", type=int, default=None)
    ap.add_argument("--pretrained_model", type=str, default=None)
    ap.add_argument("--eval_freq", type=int, default=10_000, help="timesteps between evaluations (20 episodes each)")
    ap.add_argument("--save_freq", type=int, default=50_000, help="timesteps between checkpoints")
    ap.add_argument("--tracker", type=str, default=None,
                    help="--task highlevel: the low-level tracker (a PPO.save file of --task lowlevel, or an SB3 directory)")
    args = ap.parse_args()
    if (args.task == "highlevel") != (args.tracker is not None):
        ap.error("--tracker is required with --task highlevel, and only with it")
    cfg = dict(TRAIN_CONFIG[args.task])
    for k in ("num_envs", "n_steps", "batch_size", "total_timesteps"):
        if getattr(args, k) is not None:
            cfg[k] = getattr(args, k)

    import torch
    import torch.distributed as dist
    rank, local_rank, world = (int(os.environ.get(k, d)) for k, d in (("RANK", 0), ("LOCAL_RANK", 0), ("WORLD_SIZE", 1)))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from pyflyt_drone_b200.callbacks import CheckpointCallback, EvalCallback
    from pyflyt_drone_b200.ppo import PPO
    from pyflyt_drone_b200.tracker import Tracker
    from pyflyt_drone_b200.vec_env import FixedwingVecEnv

    if args.task in ("lowlevel", "duck"):       # the preset carries the whole env configuration of the script
        env = FixedwingVecEnv(cfg["num_envs"], preset=cfg["preset"], device=local_rank, seed=cfg["seed"],
                              env_id0=rank * cfg["num_envs"])
    else:
        env = FixedwingVecEnv(cfg["num_envs"], preset=cfg["preset"], device=local_rank, seed=cfg["seed"],
                              env_id0=rank * cfg["num_envs"], num_targets=cfg["num_targets"],
                              goal_reach=float(cfg["goal_reach_distance"]), sparse_reward=int(cfg["sparse_reward"]),
                              dome=cfg["flight_dome_size"], max_steps=int(30 * cfg["max_duration_seconds"]),
                              context_len=cfg["context_length"],
                              tracker=Tracker.load(args.tracker) if args.tracker else None)
    model = PPO("MlpPolicy", env, learning_rate=cfg["learning_rate"], n_steps=cfg["n_steps"], batch_size=cfg["batch_size"],
                n_epochs=cfg["n_epochs"], gamma=cfg["gamma"], gae_lambda=cfg["gae_lambda"], clip_range=cfg["clip_range"],
                ent_coef=cfg["ent_coef"], vf_coef=cfg["vf_coef"], max_grad_norm=cfg["max_grad_norm"], seed=cfg["seed"],
                verbose=1 if rank == 0 else 0)
    if args.pretrained_model:
        model.load(args.pretrained_model)
    # the reference's WaypointEvalCallback(eval_freq=10000 // num_envs, n_eval_episodes=20, best_model_save_path=model_dir)
    # and CheckpointCallback(save_freq=50000 // num_envs); here both frequencies count timesteps (rank 0 evaluates and writes)
    eval_cb = EvalCallback(eval_freq=args.eval_freq, n_eval_episodes=20, best_model_save_path=cfg["model_dir"],
                           log_path=os.path.join(cfg["model_dir"], "eval_logs"), verbose=1)
    ckpt_cb = CheckpointCallback(save_freq=args.save_freq, save_path=os.path.join(cfg["model_dir"], "checkpoints"),
                                 name_prefix="ppo_fixedwing")
    try:
        model.learn(total_timesteps=cfg["total_timesteps"], callback=lambda l, g: eval_cb(l, g) and ckpt_cb(l, g))
    except KeyboardInterrupt:
        print("Training interrupted by user.")
    finally:
        eval_cb.close()
        if rank == 0:
            os.makedirs(cfg["model_dir"], exist_ok=True)
            model.save(os.path.join(cfg["model_dir"], "final_model.pt"))
            print("saved", os.path.join(cfg["model_dir"], "final_model.pt"))
            paths = model.export_sb3(os.path.join(cfg["model_dir"], "sb3_export"))      # policy.pth + vecnorm.npz for SB3
            print("exported", paths)
            # the reference's eval flow (eval/eval_waypoints.py): frozen statistics, raw returns, deterministic actions
            res = model.evaluate(n_eval_episodes=100)
            print(f"evaluation over 100 episodes: reward {res.mean_reward:.2f} +/- {res.std_reward:.2f}, length "
                  f"{res.mean_length:.1f}, targets reached per episode {res.mean_targets_reached:.2f}, "
                  f"success rate {res.success_rate:.2f}")
        env.close()
        if world > 1:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
