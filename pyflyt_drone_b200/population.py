"""A population of independent PPO runs trained together: one env batch, one launch per kernel for every member.

``PPOPopulation`` trains P members over one ``FixedwingVecEnv`` of P * n envs.  Member m owns env rows
``[m * n, (m + 1) * n)`` (env ids from ``env.env_id0 + m * n``), its own parameters, Adam state and VecNormalize statistics,
and may have its own seed and loss / optimizer hyper-parameters.  Every rollout kernel (forward, running moments, reward
normalisation, time-limit bootstrap, GAE) runs once per agent step for all members, and the stable_baselines3-sized update
(``batch_size <= fused_steps_max_batch``) is one launch of P thread blocks per window of optimizer steps.

The contract is exact equivalence: member m computes, bit for bit, what a standalone ``PPO`` computes on that member's slice
of the envs (``PPO(..., seed=seed_m, **hp_m)`` over ``FixedwingVecEnv(n, config=env.cfg, seed=<env seed>,
env_id0=env.env_id0 + m * n)`` with ``fused_obs_moments = False``).  DESIGN.md section 5 "Populations" has the layout.
"""
from __future__ import annotations

import ctypes as C
import time

import numpy as np
import torch

from . import _lib
from .ppo import FlatMlpPolicy, PPO, RolloutStats, _p, _stream

# per-member keys: what may differ between members without changing buffer shapes or the launch structure
MEMBER_KEYS = ("seed", "learning_rate", "clip_range", "ent_coef", "vf_coef", "max_grad_norm", "gamma", "gae_lambda")
# column of each per-member hyper-parameter in the device record (PPO_POP_* of include/fwppo.h)
HP_COLUMNS = {"learning_rate": 0, "clip_range": 1, "ent_coef": 2, "vf_coef": 3, "max_grad_norm": 4, "gamma": 5, "gae_lambda": 6}
HP_WIDTH = 8
EPISODE_STAT_NAMES = ["episodes", "return_sum", "length_sum", "targets_reached_sum", "collisions", "out_of_bounds", "completed",
                      "strikes"]
# Adam's betas and eps are those of PPO's optimizer (torch defaults, stable_baselines3's eps), shared by every member
ADAM_BETAS, ADAM_EPS = (0.9, 0.999), 1e-5


def parse_members(members, num_envs: int, defaults: dict) -> tuple[list[dict], int]:
    """Per-member hyper-parameters and envs per member.

    ``members`` is a count P (member k gets ``seed = defaults["seed"] + k`` and the defaults otherwise) or a list of dicts,
    one per member, over the keys of ``MEMBER_KEYS``; a key a dict leaves out takes the default (the constructor's keyword
    argument).  Raises ``ValueError`` for an unknown key, an empty population or a P that does not divide ``num_envs``."""
    if isinstance(members, bool) or not isinstance(members, (int, list, tuple)):
        raise ValueError("members must be a positive int or a list of per-member dicts")
    if isinstance(members, int):
        if members < 1:
            raise ValueError("members must be at least 1")
        specs = [dict(defaults, seed=int(defaults["seed"]) + k) for k in range(members)]
    else:
        if len(members) == 0:
            raise ValueError("members must not be empty")
        specs = []
        for k, m in enumerate(members):
            if not isinstance(m, dict):
                raise ValueError(f"member {k}: expected a dict of hyper-parameters, got {type(m).__name__}")
            unknown = sorted(set(m) - set(MEMBER_KEYS))
            if unknown:
                raise ValueError(f"member {k}: unknown per-member key(s) {unknown}; per-member keys are {list(MEMBER_KEYS)}")
            specs.append(dict(defaults, **m))
    for s in specs:
        s["seed"] = int(s["seed"])
        for key in HP_COLUMNS:
            s[key] = float(s[key])
    P = len(specs)
    if num_envs % P != 0:
        raise ValueError(f"{P} members do not divide the env batch of {num_envs} envs")
    return specs, num_envs // P


class PPOPopulation:
    """P independent ``PPO`` runs over one ``FixedwingVecEnv`` of P * n envs (see the module docstring).

    Per member (``members`` entries, defaulting to the keyword arguments): ``seed``, ``learning_rate``, ``clip_range``,
    ``ent_coef``, ``vf_coef``, ``max_grad_norm``, ``gamma``, ``gae_lambda``.  Shared: ``n_steps``, ``batch_size``,
    ``n_epochs``, ``normalize``, ``norm_reward``, ``clip_obs``, ``use_cuda_graph``, ``tensor_core_forward`` and Adam's betas
    and eps.  Refused: ``update="torch"``, a ``torch.distributed`` world larger than 1, and action / observation widths the
    hand-written ``PPO`` update does not take (actions other than 4 or 6 wide, observations wider than 64 floats, or wider than
    32 with six actions)."""

    def __init__(self, policy: str, env, members=1, learning_rate: float = 3e-4, n_steps: int = 2048, batch_size: int = 64,
                 n_epochs: int = 10, gamma: float = 0.99, gae_lambda: float = 0.95, clip_range: float = 0.2, ent_coef: float = 0.0,
                 vf_coef: float = 0.5, max_grad_norm: float = 0.5, seed: int = 0, device=None, verbose: int = 0,
                 normalize: bool = True, norm_reward: bool = True, clip_obs: float = 10.0, use_cuda_graph: bool = True,
                 tensor_core_forward: bool = True, update: str = "kernel"):
        if policy != "MlpPolicy":
            raise ValueError("only 'MlpPolicy' (the policy the reference trains) is implemented")
        if update != "kernel":
            raise ValueError("a population trains through the hand-written kernels only (update='kernel'); "
                             "update='torch' is the standalone PPO's fp32 reference")
        defaults = dict(seed=seed, learning_rate=learning_rate, clip_range=clip_range, ent_coef=ent_coef, vf_coef=vf_coef,
                        max_grad_norm=max_grad_norm, gamma=gamma, gae_lambda=gae_lambda)
        self.members, self.n = parse_members(members, int(env.num_envs), defaults)
        self.P = len(self.members)
        self.d, self.a = int(env.obs_dim), int(getattr(env, "act_dim", 4))
        if self.a not in (4, 6):
            raise ValueError(f"PPO supports 4- or 6-channel actions; this env has {self.a}")
        if self.d < 1 or self.d > 64 or (self.d > 32 and self.a != 4):
            raise ValueError(f"observation width {self.d} with {self.a} actions has no hand-written PPO update "
                             "(1..32 floats, or up to 64 with four actions)")
        try:
            import torch.distributed as dist
            world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
        except Exception:
            world = 1
        if world > 1:
            raise ValueError("a population runs on one GPU; torch.distributed has a world of "
                             f"{world} (members on several GPUs are not supported)")
        if not torch.cuda.is_available():
            raise RuntimeError("PPO rollouts run on CUDA kernels of libfwsim.so; no CUDA device is visible")
        self.env = env
        self.device = torch.device("cuda", env.device_index)
        self.lib = _lib.load()
        self.n_envs = int(env.num_envs)
        self.n_steps, self.batch_size, self.n_epochs = int(n_steps), int(batch_size), int(n_epochs)
        self.normalize, self.norm_reward, self.clip_obs = bool(normalize), bool(normalize and norm_reward), float(clip_obs)
        self.clip_reward = 10.0
        self.use_graph, self.verbose = bool(use_cuda_graph), verbose
        self.tensor_core_forward = bool(tensor_core_forward) and (self.d <= 32 or self.a == 4)
        self.fused_steps_max_batch = 256          # PPO's default: minibatches up to this size take the multi-step kernel
        P, n, N, T, D = self.P, self.n, self.n_envs, self.n_steps, self.d
        dev = self.device
        f32, f64, i32 = (dict(dtype=t, device=dev) for t in (torch.float32, torch.float64, torch.int32))
        self.count = int(self.lib.ppo_param_count_a(D, self.a))
        self.theta = torch.stack([FlatMlpPolicy(D, dev, seed=m["seed"], act_dim=self.a).theta.data for m in self.members])
        self.seeds = torch.from_numpy(np.array([m["seed"] & (2 ** 64 - 1) for m in self.members], np.uint64).view(np.int64)).to(dev)
        hp = np.zeros((P, HP_WIDTH), np.float32)
        for k, m in enumerate(self.members):
            for key, col in HP_COLUMNS.items():
                hp[k, col] = m[key]
        self.hp = torch.from_numpy(hp).to(dev)
        self.adam_m, self.adam_v = torch.zeros((P, self.count), **f32), torch.zeros((P, self.count), **f32)
        self.adam_t = torch.zeros(P, **i32)
        self.grad, self.grad_norm, self.stats_mb = torch.zeros((P, self.count), **f32), torch.zeros(P, **f32), torch.zeros((P, 8), **f32)
        self._ws = torch.zeros(int(self.lib.ppo_update_workspace_floats_a(D, self.a)), **f32)
        # VecNormalize statistics per member (DeviceVecNormalize's layout, one row per member) and the per-env return
        self.obs_stats = torch.cat([torch.zeros((P, D), **f64), torch.ones((P, D), **f64), torch.full((P, 1), 1e-4, **f64)], 1)
        self.ret_stats = torch.tensor([0.0, 1.0, 1e-4], **f64).repeat(P, 1)
        self.obs_scratch, self.ret_scratch = torch.zeros((P, 2 * D + 2), **f64), torch.zeros((P, 4), **f64)
        self.obs_accum, self.ret_accum = torch.zeros((P, 2 * D + 1), **f64), torch.zeros((P, 3), **f64)
        self.ret = torch.zeros(N, **f32)
        self.buf = dict(obs=torch.zeros((T, N, D), **f32), act=torch.zeros((T, N, self.a), **f32),
                        rew=torch.zeros((T, N), **f32), done=torch.zeros((T, N), **f32), val=torch.zeros((T, N), **f32),
                        logp=torch.zeros((T, N), **f32), adv=torch.zeros((T, N), **f32), ret=torch.zeros((T, N), **f32))
        self.act_env = torch.zeros((N, self.a), **f32)
        self.last_values = torch.zeros(N, **f32)
        self._step_dev = torch.zeros(1, **i32)            # shared Philox step counter: every member is at the same step
        # training episode ledger: running return and length per env, finished-episode sums [8, N]
        self._ep_ret, self._ep_len, self._ep_acc = torch.zeros(N, **f64), torch.zeros(N, **i32), torch.zeros((8, N), **f64)
        self._perm = torch.empty((P, T * n), dtype=torch.int64, device=dev)
        self._perm_epoch = 0
        self.num_timesteps = 0
        self._obs = None
        self._graph, self._pending_capture = None, False
        self.stats = RolloutStats()

    # ------------------------------------------------------------------ rollout
    def _stats_ptr(self):
        return _p(self.obs_stats) if self.normalize else None

    def _update_obs_moments(self, obs_raw: torch.Tensor) -> None:
        if self.normalize:
            _lib.check(self.lib.ppo_pop_moments_update(self.P, self.n, _p(obs_raw), self.d, _p(self.obs_stats), _p(self.obs_scratch),
                                                       _p(self.obs_accum), _stream()))

    def collect_rollouts(self) -> None:
        """One rollout of n_steps agent steps for every member; captured once into a CUDA graph and replayed, as PPO does."""
        if self._obs is None:
            self._obs = self.env.reset_tensor()
            self.ret.zero_()
            self._update_obs_moments(self._obs)
        if not self.use_graph:
            self._rollout_body()
        elif self._graph is None:
            torch.cuda.synchronize()
            side = torch.cuda.Stream(device=self.device)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                self._rollout_body()                 # eager warm-up on a side stream (also a real rollout)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            self._graph = torch.cuda.CUDAGraph()
            self._pending_capture = True
        else:
            if self._pending_capture:
                with torch.cuda.graph(self._graph):
                    self._rollout_body()
                self._pending_capture = False
            self._graph.replay()
        self.num_timesteps += self.n_steps * self.n

    def _rollout_body(self) -> None:
        env, b, lib, P, n = self.env, self.buf, self.lib, self.P, self.n
        fwd = lib.ppo_pop_policy_forward_tc_a if self.tensor_core_forward else lib.ppo_pop_policy_forward_a
        has_targets = env.cfg.task in (1, 2, 5)
        for t in range(self.n_steps):
            _lib.check(fwd(P, n, _p(self.seeds), _p(self.theta), self.d, self.a, _p(self._obs), self._stats_ptr(), self.clip_obs,
                           env.env_id0, t, _p(self._step_dev), 0, _p(b["obs"][t]), _p(self.act_env), _p(b["act"][t]),
                           _p(b["logp"][t]), _p(b["val"][t]), _stream()))
            obs, rew, flags, term = env.step_tensor(self.act_env, want_terminal_obs=True)
            tidx = env.targets_reached_tensor() if has_targets else None
            _lib.check(lib.ppo_pop_episode_ledger(P, n, _p(rew), _p(flags), _p(tidx), _p(self._ep_ret), _p(self._ep_len),
                                                  _p(self._ep_acc), _stream()))
            self._update_obs_moments(obs)
            if self.norm_reward:
                _lib.check(lib.ppo_pop_reward_normalize(P, n, _p(self.hp), _p(rew), _p(flags), self.clip_reward, _p(self.ret),
                                                        _p(self.ret_stats), _p(self.ret_scratch), _p(self.ret_accum),
                                                        _p(b["rew"][t]), _p(b["done"][t]), _stream()))
            else:
                b["rew"][t].copy_(rew)
                b["done"][t].copy_((flags & 3) != 0)
            _lib.check(lib.ppo_pop_timeout_bootstrap_a(P, n, _p(self.hp), _p(self.theta), self.d, self.a, _p(term), self._stats_ptr(),
                                                       self.clip_obs, _p(flags), _p(b["rew"][t]), _stream()))
            self._obs = obs
        _lib.check(lib.ppo_counter_add(_p(self._step_dev), self.n_steps, _stream()))
        _lib.check(lib.ppo_pop_value_forward_a(P, n, _p(self.theta), self.d, self.a, _p(self._obs), self._stats_ptr(), self.clip_obs,
                                               _p(self.last_values), _stream()))
        _lib.check(lib.ppo_pop_gae(P, n, _p(self.hp), _p(b["rew"]), _p(b["val"]), _p(b["done"]), _p(self.last_values), self.n_steps,
                                   _p(b["adv"]), _p(b["ret"]), _stream()))

    # ------------------------------------------------------------------ update
    def _epoch_permutation(self) -> torch.Tensor:
        """Every member's standalone permutation of the next epoch (its seed, the shared epoch counter), as population rows."""
        self._perm_epoch += 1
        _lib.check(self.lib.ppo_pop_random_permutation(self.P, self.n, _p(self.seeds), _p(self._perm), self._perm.shape[1],
                                                       self._perm_epoch, _stream()))
        return self._perm

    def train(self) -> dict:
        """PPO.train for every member, on the path a standalone PPO takes at this batch size: one launch of P thread blocks per
        window of optimizer steps for batch_size <= fused_steps_max_batch, the existing per-model update kernels member by
        member otherwise.  Returns PPO.train's dict with one entry per member (numpy arrays of length P)."""
        lib, b, P = self.lib, self.buf, self.P
        total = self.n_steps * self.n
        bs = min(self.batch_size, total)
        b1, b2 = ADAM_BETAS
        eps = ADAM_EPS
        steps_per_epoch = total // bs
        bufs = (_p(b["obs"]), _p(b["act"]), _p(b["logp"]), _p(b["adv"]), _p(b["ret"]))
        if bs <= self.fused_steps_max_batch and total % bs == 0:
            chunk = max(c for c in range(1, min(steps_per_epoch, 256) + 1) if steps_per_epoch % c == 0)
            for _ in range(self.n_epochs):
                perm = self._epoch_permutation()
                for s in range(0, total, chunk * bs):
                    _lib.check(lib.ppo_pop_minibatch_steps_a(
                        P, _p(self.hp), _p(self.theta), self.d, self.a, *bufs, C.c_void_p(perm.data_ptr() + 8 * s), total, bs, chunk,
                        _p(self.adam_m), _p(self.adam_v), b1, b2, eps, _p(self.adam_t), _p(self.grad_norm), _p(self.grad),
                        _p(self.stats_mb), _stream()))
        elif total % bs == 0:
            chunk = max(c for c in range(1, min(steps_per_epoch, 16) + 1) if steps_per_epoch % c == 0)
            for _ in range(self.n_epochs):
                perm = self._epoch_permutation()
                for k, m in enumerate(self.members):
                    for s in range(0, total, chunk * bs):
                        _lib.check(lib.ppo_window_update_a(
                            _p(self.theta[k]), self.d, self.a, *bufs, _p(perm[k, s:s + chunk * bs]), bs, chunk, m["clip_range"],
                            m["ent_coef"], m["vf_coef"], _p(self.adam_m[k]), _p(self.adam_v[k]), m["learning_rate"], b1, b2, eps,
                            m["max_grad_norm"], _p(self.adam_t[k:k + 1]), _p(self.grad_norm[k:k + 1]), _p(self._ws), _p(self.grad[k]),
                            _p(self.stats_mb[k]), _stream()))
        else:                                   # ragged last minibatch: step by step, as PPO does
            for _ in range(self.n_epochs):
                perm = self._epoch_permutation()
                for k, m in enumerate(self.members):
                    for s in range(0, total, bs):
                        idx = perm[k, s:s + bs]
                        _lib.check(lib.ppo_minibatch_grad_a(
                            _p(self.theta[k]), self.d, self.a, *bufs, _p(idx), int(idx.numel()), m["clip_range"], m["ent_coef"],
                            m["vf_coef"], _p(self._ws), _p(self.grad[k]), _p(self.stats_mb[k]), _stream()))
                        _lib.check(lib.ppo_adam_step(_p(self.theta[k]), _p(self.grad[k]), _p(self.adam_m[k]), _p(self.adam_v[k]),
                                                     self.count, m["learning_rate"], b1, b2, eps, m["max_grad_norm"], 1.0,
                                                     _p(self.adam_t[k:k + 1]), _p(self.grad_norm[k:k + 1]), _stream()))
        st = self.stats_mb.cpu().numpy().astype(np.float64)
        n = np.maximum(st[:, 5], 1.0)
        vf = np.array([m["vf_coef"] for m in self.members])
        return dict(policy_loss=st[:, 0] / n, value_loss=st[:, 1] / n, approx_kl=st[:, 2] / n, clip_fraction=st[:, 3] / n,
                    loss=st[:, 0] / n + vf * (st[:, 1] / n), grad_norm=self.grad_norm.cpu().numpy().astype(np.float64))

    def learn(self, total_timesteps: int, log_interval: int = 1, callback=None, reset_num_timesteps: bool = True) -> "PPOPopulation":
        """Trains every member for ``total_timesteps`` timesteps PER MEMBER, counted as PPO.learn counts them (n_steps * n per
        iteration).  ``callback(locals(), globals())`` runs after every iteration; returning False stops.  With ``verbose``,
        one line per ``log_interval`` iterations: min / median / max over members of the training ``ep_rew_mean``."""
        if reset_num_timesteps:
            self.num_timesteps = 0
        it = 0
        while self.num_timesteps < total_timesteps:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            self.collect_rollouts()
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            self.obs_accum.zero_(); self.ret_accum.zero_()      # one process: no cross-rank reconciliation (PPO's world 1)
            info = self.train()
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            self.stats.env_steps += self.n_steps * self.n_envs
            self.stats.rollout_s += t1 - t0
            self.stats.update_s += t2 - t1
            it += 1
            if self.verbose and it % log_interval == 0:
                ep = self.episode_stats()
                rew = ep["return_sum"] / np.maximum(ep["episodes"], 1.0)
                print(f"[ppo-pop] iter {it} members {self.P} timesteps/member {self.num_timesteps} "
                      f"sps {self.n_steps * self.n_envs / (t2 - t0):.3e} rollout {t1 - t0:.3f}s update {t2 - t1:.3f}s "
                      f"ep_rew_mean min {rew.min():.2f} median {float(np.median(rew)):.2f} max {rew.max():.2f} "
                      f"loss median {float(np.median(info['loss'])):.4f}", flush=True)
            if callback is not None and callback(locals(), globals()) is False:
                break
        return self

    def episode_stats(self) -> dict[str, np.ndarray]:
        """Training episodes finished since the last call, per member: the eight sums of ``FixedwingVecEnv.episode_stats``
        (episodes, return_sum, length_sum, targets_reached_sum, collisions, out_of_bounds, completed, strikes) as float64
        arrays of length P.  Returns are summed per env in double in step order; each member's envs are added in env order."""
        acc = self._ep_acc.cpu().numpy().reshape(8, self.P, self.n)
        self._ep_acc.zero_()
        sums = np.cumsum(acc, axis=2)[:, :, -1]                 # sequential: env order
        return {name: sums[i].copy() for i, name in enumerate(EPISODE_STAT_NAMES)}

    # ------------------------------------------------------------------ members
    def member_env(self, k: int):
        """A fresh env batch equal to member k's slice: the same config, wind field and env seed, env ids from env_id0 + k * n."""
        from .vec_env import FixedwingVecEnv
        return FixedwingVecEnv(self.n, config=self.env.cfg, device=self.env.device_index, seed=self.env._seed,
                               env_id0=self.env.env_id0 + k * self.n, wind_field=getattr(self.env, "wind_field", None),
                               tracker=getattr(self.env, "tracker", None))

    def member(self, k: int, env=None) -> PPO:
        """A standalone ``PPO`` holding copies of member k's state: hyper-parameters, parameters, Adam moments and step,
        VecNormalize statistics, ``num_timesteps`` and the step counter.  Without ``env`` it gets ``member_env(k)``.
        ``evaluate``, ``export_sb3`` and ``save`` then behave as for a model trained alone; continuing training through it is
        not promised (env state and the permutation epoch are not carried over)."""
        k = int(k)
        if not 0 <= k < self.P:
            raise IndexError(f"member {k} out of range [0, {self.P})")
        m = self.members[k]
        model = PPO("MlpPolicy", env if env is not None else self.member_env(k), learning_rate=m["learning_rate"],
                    n_steps=self.n_steps, batch_size=self.batch_size, n_epochs=self.n_epochs, gamma=m["gamma"],
                    gae_lambda=m["gae_lambda"], clip_range=m["clip_range"], ent_coef=m["ent_coef"], vf_coef=m["vf_coef"],
                    max_grad_norm=m["max_grad_norm"], seed=m["seed"], normalize=self.normalize, norm_reward=self.norm_reward,
                    clip_obs=self.clip_obs, use_cuda_graph=self.use_graph, tensor_core_forward=self.tensor_core_forward)
        with torch.no_grad():
            model.policy.theta.copy_(self.theta[k])
            model._adam_m.copy_(self.adam_m[k]); model._adam_v.copy_(self.adam_v[k]); model._adam_t.copy_(self.adam_t[k:k + 1])
            vn = model.vecnorm
            vn.obs_stats.copy_(self.obs_stats[k]); vn.ret_stats.copy_(self.ret_stats[k])
            vn.obs_base.copy_(vn.obs_stats); vn.ret_base.copy_(vn.ret_stats)
            if vn.ret.numel() == self.n:
                vn.ret.copy_(self.ret[k * self.n:(k + 1) * self.n])
            model._step_dev.copy_(self._step_dev)
        model.num_timesteps = self.num_timesteps
        return model
