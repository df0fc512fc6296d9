"""PPO on device tensors around FixedwingVecEnv -- the training seam of the reference's scripts.

Mirrors the reference's use of stable_baselines3 (train/train_Fixedwing_Waypoints_v3.py:260,293-337):
``VecNormalize(env, norm_obs=True, norm_reward=True, clip_obs=10)`` then
``PPO("MlpPolicy", env, learning_rate, n_steps, batch_size, n_epochs, gamma, gae_lambda, clip_range, ent_coef,
vf_coef, max_grad_norm, seed, device).learn(total_timesteps)``.

Rollout path (every agent step, no host sync): hand-written kernels of libfwsim.so --
policy/value forward + Gaussian sampling (ppo_policy_forward[_tc]), env step (fw_step, whose epilogue also accumulates
the observation moments: fw_set_obs_accumulator + ppo_moments_finalize), reward normalisation (ppo_reward_normalize),
time-limit bootstrap (ppo_timeout_bootstrap), and GAE (ppo_gae) once per rollout; the whole rollout is one replayed
CUDA graph.  The minibatch update is hand-written too (update="kernel"): one fused tcgen05 forward+backward kernel
per minibatch on ONE flat parameter vector, whose gradient is a single contiguous 49 KB buffer, with clip + Adam in
the gradient reduction (ppo_window_update_a) or, for stable_baselines3-sized minibatches, whole windows of optimizer
steps in one single-block launch (ppo_minibatch_steps_a).  The one collective of the path, the gradient all-reduce
of a multi-GPU run, happens inside those kernels over NVLink peer memory (ppo_*_p2p_a; NCCL all_reduce between the
kernels when peer memory cannot be set up or FWPPO_P2P=0).  update="torch" keeps a plain autograd implementation as
the fp32 reference the tests compare against.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import time
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from .vec_env import FixedwingVecEnv

H, A = 64, 4


def _p(t: torch.Tensor | None):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream() -> C.c_void_p:
    return C.c_void_p(int(torch.cuda.current_stream().cuda_stream))


def export_vecnorm_npz(sd: dict, path: str) -> None:
    """VecNormalize statistics (DeviceVecNormalize.state_dict()) under SB3's attribute names, as a plain .npz."""
    np.savez(path, obs_rms_mean=np.asarray(sd["obs_rms.mean"], np.float64), obs_rms_var=np.asarray(sd["obs_rms.var"], np.float64),
             obs_rms_count=np.float64(sd["obs_rms.count"]), ret_rms_mean=np.float64(sd["ret_rms.mean"]),
             ret_rms_var=np.float64(sd["ret_rms.var"]), ret_rms_count=np.float64(sd["ret_rms.count"]),
             clip_obs=np.float64(sd["clip_obs"]), clip_reward=np.float64(sd["clip_reward"]), gamma=np.float64(sd["gamma"]),
             epsilon=np.float64(1e-8), norm_obs=np.bool_(sd.get("norm_obs", True)), norm_reward=np.bool_(sd.get("norm_reward", True)))


def import_vecnorm_npz(path: str) -> dict:
    z = np.load(path)
    return {"obs_rms.mean": z["obs_rms_mean"], "obs_rms.var": z["obs_rms_var"], "obs_rms.count": float(z["obs_rms_count"]),
            "ret_rms.mean": float(z["ret_rms_mean"]), "ret_rms.var": float(z["ret_rms_var"]),
            "ret_rms.count": float(z["ret_rms_count"]), "clip_obs": float(z["clip_obs"]),
            "clip_reward": float(z["clip_reward"]), "gamma": float(z["gamma"]),
            "norm_obs": bool(z["norm_obs"]), "norm_reward": bool(z["norm_reward"])}


class FlatMlpPolicy:
    """SB3 ``MlpPolicy`` (separate pi / vf towers [64, 64], tanh, state-independent log_std) stored as ONE flat
    fp32 parameter vector in the layout of include/fwppo.h."""

    def __init__(self, obs_dim: int, device: torch.device, seed: int = 0, act_dim: int = A):
        self.d = int(obs_dim)
        self.a = int(act_dim)
        self.device = device
        lib = _lib.load()
        self.count = int(lib.ppo_param_count_a(self.d, self.a))
        if self.count <= 0 or self.a not in (4, 6):
            raise ValueError(f"unsupported action width {self.a} (4 or 6)")
        shapes = [("pi.0.weight", (H, self.d)), ("pi.0.bias", (H,)), ("pi.2.weight", (H, H)), ("pi.2.bias", (H,)),
                  ("action_net.weight", (self.a, H)), ("action_net.bias", (self.a,)),
                  ("vf.0.weight", (H, self.d)), ("vf.0.bias", (H,)), ("vf.2.weight", (H, H)), ("vf.2.bias", (H,)),
                  ("value_net.weight", (1, H)), ("value_net.bias", (1,)), ("log_std", (self.a,))]
        self.slices, off = {}, 0
        for name, shp in shapes:
            n = int(np.prod(shp))
            self.slices[name] = (off, off + n, shp)
            off += n
        assert off == self.count, (off, self.count)
        g = torch.Generator(device="cpu").manual_seed(int(seed))
        flat = torch.zeros(self.count, dtype=torch.float32)
        gains = {"pi.0.weight": math.sqrt(2), "pi.2.weight": math.sqrt(2), "vf.0.weight": math.sqrt(2),
                 "vf.2.weight": math.sqrt(2), "action_net.weight": 0.01, "value_net.weight": 1.0}
        for name, (a, b, shp) in self.slices.items():
            if name in gains:       # SB3 ActorCriticPolicy: orthogonal init, biases zero, log_std_init = 0
                w = torch.empty(shp)
                torch.nn.init.orthogonal_(w, gain=gains[name], generator=g)
                flat[a:b] = w.reshape(-1)
        self.theta = torch.nn.Parameter(flat.to(device))

    def view(self, name: str, theta: torch.Tensor | None = None) -> torch.Tensor:
        a, b, shp = self.slices[name]
        return (self.theta if theta is None else theta)[a:b].view(shp)

    def state_dict(self) -> dict[str, torch.Tensor]:
        """Parameters under SB3's ActorCriticPolicy names (mlp_extractor.policy_net.{0,2}, action_net, ...)."""
        m = {"pi.0": "mlp_extractor.policy_net.0", "pi.2": "mlp_extractor.policy_net.2", "vf.0": "mlp_extractor.value_net.0",
             "vf.2": "mlp_extractor.value_net.2"}
        out = {}
        for name in self.slices:
            base, _, leaf = name.rpartition(".")
            key = f"{m[base]}.{leaf}" if base in m else name
            out[key] = self.view(name).detach().clone()
        return out

    def load_state_dict(self, sd: dict[str, torch.Tensor]) -> None:
        m = {"mlp_extractor.policy_net.0": "pi.0", "mlp_extractor.policy_net.2": "pi.2",
             "mlp_extractor.value_net.0": "vf.0", "mlp_extractor.value_net.2": "vf.2"}
        with torch.no_grad():
            for key, val in sd.items():
                base, _, leaf = key.rpartition(".")
                name = f"{m[base]}.{leaf}" if base in m else key
                if name in self.slices:
                    self.view(name).copy_(val.to(self.device))

    # ---- torch reference of the two towers (used by the update and by the tests as the fp32 reference)
    def towers(self, obs_norm: torch.Tensor, theta: torch.Tensor | None = None):
        v = lambda n: self.view(n, theta)  # noqa: E731
        h = torch.tanh(torch.addmm(v("pi.0.bias"), obs_norm, v("pi.0.weight").t()))
        h = torch.tanh(torch.addmm(v("pi.2.bias"), h, v("pi.2.weight").t()))
        mean = torch.addmm(v("action_net.bias"), h, v("action_net.weight").t())
        g = torch.tanh(torch.addmm(v("vf.0.bias"), obs_norm, v("vf.0.weight").t()))
        g = torch.tanh(torch.addmm(v("vf.2.bias"), g, v("vf.2.weight").t()))
        value = torch.addmm(v("value_net.bias"), g, v("value_net.weight").t()).squeeze(-1)
        return mean, value

    def evaluate_actions(self, obs_norm: torch.Tensor, actions: torch.Tensor):
        mean, value = self.towers(obs_norm)
        log_std = self.view("log_std")
        z = (actions - mean) * torch.exp(-log_std)
        logp = (-0.5 * z * z - log_std - 0.5 * math.log(2 * math.pi)).sum(-1)
        entropy = (0.5 + 0.5 * math.log(2 * math.pi) + log_std).sum().expand_as(logp)
        return value, logp, entropy


class DeviceVecNormalize:
    """stable_baselines3 ``VecNormalize`` statistics kept on the device in float64 (RunningMeanStd(eps=1e-4))."""

    def __init__(self, obs_dim: int, num_envs: int, device: torch.device, norm_obs: bool = True, norm_reward: bool = True,
                 clip_obs: float = 10.0, clip_reward: float = 10.0, gamma: float = 0.99, training: bool = True):
        self.d, self.n = obs_dim, num_envs
        self.norm_obs, self.norm_reward, self.training = norm_obs, norm_reward, training
        self.clip_obs, self.clip_reward, self.gamma = float(clip_obs), float(clip_reward), float(gamma)
        f64 = dict(dtype=torch.float64, device=device)
        self.obs_stats = torch.cat([torch.zeros(obs_dim, **f64), torch.ones(obs_dim, **f64), torch.full((1,), 1e-4, **f64)])
        self.ret_stats = torch.tensor([0.0, 1.0, 1e-4], **f64)
        self.ret = torch.zeros(num_envs, dtype=torch.float32, device=device)
        self.obs_scratch = torch.zeros(2 * obs_dim + 2, **f64)
        self.ret_scratch = torch.zeros(4, **f64)
        # raw batch sums since the last cross-rank sync (multi-GPU reconciliation), and the stats at that sync
        self.obs_accum = torch.zeros(2 * obs_dim + 1, **f64)
        self.ret_accum = torch.zeros(3, **f64)
        self.obs_base = self.obs_stats.clone()
        self.ret_base = self.ret_stats.clone()

    def state_dict(self) -> dict:
        d = self.d
        return {"obs_rms.mean": self.obs_stats[:d].cpu().numpy(), "obs_rms.var": self.obs_stats[d:2 * d].cpu().numpy(),
                "obs_rms.count": float(self.obs_stats[2 * d]), "ret_rms.mean": float(self.ret_stats[0]),
                "ret_rms.var": float(self.ret_stats[1]), "ret_rms.count": float(self.ret_stats[2]),
                "clip_obs": self.clip_obs, "clip_reward": self.clip_reward, "gamma": self.gamma,
                "norm_obs": self.norm_obs, "norm_reward": self.norm_reward}

    def load_state_dict(self, sd: dict) -> None:
        d = self.d
        dev = self.obs_stats.device
        self.obs_stats[:d] = torch.as_tensor(sd["obs_rms.mean"], dtype=torch.float64, device=dev)
        self.obs_stats[d:2 * d] = torch.as_tensor(sd["obs_rms.var"], dtype=torch.float64, device=dev)
        self.obs_stats[2 * d] = float(sd["obs_rms.count"])
        self.ret_stats[:] = torch.tensor([sd["ret_rms.mean"], sd["ret_rms.var"], sd["ret_rms.count"]], dtype=torch.float64)
        self.obs_base.copy_(self.obs_stats); self.ret_base.copy_(self.ret_stats)
        self.obs_accum.zero_(); self.ret_accum.zero_()

    @staticmethod
    def _merge(base: torch.Tensor, accum: torch.Tensor, d: int) -> torch.Tensor:
        """base (mean, var, count) merged with raw sums (sum, sumsq, n) -- Chan et al., in float64."""
        n = accum[2 * d]
        if float(n) <= 0:
            return base.clone()
        bmean = accum[:d] / n
        bvar = (accum[d:2 * d] / n - bmean * bmean).clamp_min(0.0)
        mean, var, count = base[:d], base[d:2 * d], base[2 * d]
        tot = count + n
        delta = bmean - mean
        out = base.clone()
        out[:d] = mean + delta * n / tot
        out[d:2 * d] = (var * count + bvar * n + delta * delta * count * n / tot) / tot
        out[2 * d] = tot
        return out

    def sync_across_ranks(self) -> None:
        """Exact reconciliation of the per-rank running statistics: all-reduce the raw batch sums accumulated
        since the last sync and re-apply them to the common base (a 0.5 KB collective once per rollout)."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1):
            self.obs_base.copy_(self.obs_stats); self.ret_base.copy_(self.ret_stats)
            self.obs_accum.zero_(); self.ret_accum.zero_()
            return
        buf = torch.cat([self.obs_accum, self.ret_accum])
        dist.all_reduce(buf)
        self.obs_stats.copy_(self._merge(self.obs_base, buf[: 2 * self.d + 1], self.d))
        self.ret_stats.copy_(self._merge(self.ret_base, buf[2 * self.d + 1:], 1))
        self.obs_base.copy_(self.obs_stats); self.ret_base.copy_(self.ret_stats)
        self.obs_accum.zero_(); self.ret_accum.zero_()


@dataclass
class RolloutStats:
    env_steps: int = 0
    rollout_s: float = 0.0
    update_s: float = 0.0


@dataclass
class EvalResult:
    """The episodes ``PPO.evaluate`` selected and the reference's evaluation metrics over them.

    Per-episode arrays, in the order stable_baselines3's ``evaluate_policy`` appends episodes (finish step, then env index):
    ``returns`` (float64, raw rewards summed in step order), ``lengths``, ``targets_reached`` (``info["num_targets_reached"]``
    before the auto-reset; 0 on tasks without targets), ``flags`` (the flag byte of the episode's last step),
    ``env_index`` and ``finish_step`` (evaluation step index of the last step).

    The means are those of ``PPO.evaluate_policy``, computed the same way on the same device, so they agree bit for bit:
    ``mean_reward``, ``std_reward`` (population), ``mean_length``, ``mean_targets_reached`` (0.0 without targets).  With no
    finished episode every mean and rate is NaN.

    The rates are the reference's ``eval/*`` metrics (SURVEY §5 "metrics / logging": what ``WaypointEvalCallback`` and the
    ObjLock script's callback read from the info dict of each finished episode), as fractions of the episodes:
      ``wp_reach_rate[i - 1]``  ``eval/wp{i}_reach_rate``: ``num_targets_reached >= i``, i = 1..num_targets (empty without
                                targets)
      ``success_rate``          ``eval/success_rate``: ``duck_strike`` on the ObjLock tasks (the duck-only env's
                                ``is_success``), ``env_complete`` (every waypoint reached) on the others
      ``duck_strike_rate``      ``eval/duck_strike_rate``: ``duck_strike``
      ``collision_rate``, ``out_of_bounds_rate``  ``collision`` / ``out_of_bounds`` of the last step
      ``truncation_rate``       ``TimeLimit.truncated``: time limit reached without termination
    """
    returns: np.ndarray
    lengths: np.ndarray
    targets_reached: np.ndarray
    flags: np.ndarray
    env_index: np.ndarray
    finish_step: np.ndarray
    task: int
    num_targets: int
    mean_reward: float
    std_reward: float
    mean_length: float
    mean_targets_reached: float
    wp_reach_rate: np.ndarray
    success_rate: float
    duck_strike_rate: float
    collision_rate: float
    out_of_bounds_rate: float
    truncation_rate: float

    @property
    def has_targets(self) -> bool:
        return self.task in (1, 2)

    @property
    def n_episodes(self) -> int:
        return int(self.returns.shape[0])

    @property
    def successes(self) -> np.ndarray:
        """Per-episode success (the definition of ``success_rate``)."""
        from .config import FLAG_COMPLETE, FLAG_STRIKE
        bit = FLAG_STRIKE if self.task in (2, 4) else FLAG_COMPLETE
        return (self.flags & bit) != 0

    @classmethod
    def from_episodes(cls, returns, lengths, targets_reached, flags, env_index, finish_step, task: int, num_targets: int,
                      device: str | torch.device = "cpu") -> "EvalResult":
        """Orders the episodes by (finish step, env index) and computes the metrics; the means are reduced by torch on
        ``device`` (the device ``evaluate_policy`` reduces on, for bitwise agreement with it)."""
        from .config import FLAG_COLLISION, FLAG_OOB, FLAG_STRIKE, FLAG_TERM, FLAG_TRUNC
        finish_step, env_index = np.asarray(finish_step, np.int32), np.asarray(env_index, np.int32)
        order = np.lexsort((env_index, finish_step))
        returns = np.asarray(returns, np.float64)[order]
        lengths = np.asarray(lengths, np.int32)[order]
        targets_reached = np.asarray(targets_reached, np.uint8)[order]
        flags = np.asarray(flags, np.uint8)[order]
        has_targets = task in (1, 2)
        if not has_targets:
            targets_reached = np.zeros_like(targets_reached)
        nt = int(num_targets) if has_targets else 0
        out = dict(returns=returns, lengths=lengths, targets_reached=targets_reached, flags=flags, env_index=env_index[order],
                   finish_step=finish_step[order], task=int(task), num_targets=nt)
        if returns.shape[0] == 0:
            nan = float("nan")
            return cls(**out, mean_reward=nan, std_reward=nan, mean_length=nan, mean_targets_reached=nan,
                       wp_reach_rate=np.full(nt, nan), success_rate=nan, duck_strike_rate=nan, collision_rate=nan,
                       out_of_bounds_rate=nan, truncation_rate=nan)
        r = torch.from_numpy(returns).to(device)
        rate = lambda m: float(np.count_nonzero(m)) / returns.shape[0]  # noqa: E731
        res = cls(**out, mean_reward=float(r.mean()), std_reward=float(r.std(unbiased=False)),
                  mean_length=float(torch.from_numpy(lengths).to(device).double().mean()),
                  mean_targets_reached=float(torch.from_numpy(targets_reached).to(device).double().mean()) if has_targets else 0.0,
                  wp_reach_rate=np.array([rate(targets_reached >= i) for i in range(1, nt + 1)], np.float64),
                  success_rate=0.0, duck_strike_rate=rate(flags & FLAG_STRIKE), collision_rate=rate(flags & FLAG_COLLISION),
                  out_of_bounds_rate=rate(flags & FLAG_OOB),
                  truncation_rate=rate(((flags & FLAG_TRUNC) != 0) & ((flags & FLAG_TERM) == 0)))
        res.success_rate = rate(res.successes)
        return res

    def metrics(self) -> dict[str, float]:
        """The metrics under the names the reference's training scripts log (SURVEY §5 "metrics / logging")."""
        m = {"eval/mean_reward": self.mean_reward, "eval/mean_ep_length": self.mean_length,
             "eval/success_rate": self.success_rate}
        for i, v in enumerate(self.wp_reach_rate, 1):
            m[f"eval/wp{i}_reach_rate"] = float(v)
        if self.task in (2, 4):
            m["eval/duck_strike_rate"] = self.duck_strike_rate
        return m


class PPO:
    """Keyword-compatible with the reference's ``PPO("MlpPolicy", env, ...)`` call
    (train/train_Fixedwing_Waypoints_v3.py:293-310); ``env`` is a FixedwingVecEnv."""

    def __init__(self, policy: str, env: FixedwingVecEnv, learning_rate: float = 3e-4, n_steps: int = 2048,
                 batch_size: int = 64, n_epochs: int = 10, gamma: float = 0.99, gae_lambda: float = 0.95,
                 clip_range: float = 0.2, ent_coef: float = 0.0, vf_coef: float = 0.5, max_grad_norm: float = 0.5,
                 seed: int = 0, device: str | torch.device | None = None, verbose: int = 0, tensorboard_log=None,
                 normalize: bool = True, norm_reward: bool = True, clip_obs: float = 10.0, use_cuda_graph: bool = True,
                 tensor_core_forward: bool = True, update: str = "kernel"):
        if policy != "MlpPolicy":
            raise ValueError("only 'MlpPolicy' (the policy the reference trains) is implemented")
        if not torch.cuda.is_available():
            raise RuntimeError("PPO rollouts run on CUDA kernels of libfwsim.so; no CUDA device is visible")
        self.env = env
        self.device = torch.device("cuda", env.device_index)
        self.lib = _lib.load()
        self.n_envs, self.d = env.num_envs, env.obs_dim
        self.a = int(getattr(env, "act_dim", A))
        if self.a not in (4, 6):
            raise ValueError(f"PPO supports 4- or 6-channel actions; this env has {self.a}")
        self.n_steps, self.batch_size, self.n_epochs = int(n_steps), int(batch_size), int(n_epochs)
        self.gamma, self.gae_lambda, self.clip_range = float(gamma), float(gae_lambda), float(clip_range)
        self.ent_coef, self.vf_coef, self.max_grad_norm = float(ent_coef), float(vf_coef), float(max_grad_norm)
        self.seed, self.verbose = int(seed), verbose
        self.policy = FlatMlpPolicy(self.d, self.device, seed=seed, act_dim=self.a)
        self.optimizer = torch.optim.Adam([self.policy.theta], lr=learning_rate, eps=1e-5)   # SB3 default eps
        self.vecnorm = DeviceVecNormalize(self.d, self.n_envs, self.device, norm_obs=normalize,
                                          norm_reward=normalize and norm_reward, clip_obs=clip_obs, gamma=gamma)
        T, N, D = self.n_steps, self.n_envs, self.d
        f32 = dict(dtype=torch.float32, device=self.device)
        self.buf = dict(obs=torch.zeros((T, N, D), **f32), act=torch.zeros((T, N, self.a), **f32),
                        rew=torch.zeros((T, N), **f32), done=torch.zeros((T, N), **f32), val=torch.zeros((T, N), **f32),
                        logp=torch.zeros((T, N), **f32), adv=torch.zeros((T, N), **f32), ret=torch.zeros((T, N), **f32))
        self.act_env = torch.zeros((N, self.a), **f32)
        self.last_values = torch.zeros(N, **f32)
        self._vterm = torch.zeros(N, **f32)
        self.num_timesteps = 0
        self._step_dev = torch.zeros(1, dtype=torch.int32, device=self.device)    # Philox step counter (uint32 bits)
        if update not in ("kernel", "torch"):
            raise ValueError("update must be 'kernel' (hand-written tcgen05 kernels) or 'torch' (autograd reference)")
        self.update = update
        if self.d > 32 and self.a != 4:
            # The fused update (K6) is built for (action width, observation slab) = (4, 32), (6, 32) and (4, 64): the
            # Waypoints / Waypoint-ObjLock / low-level / duck-only ObjLock policies (28, 29, 21 and 56 floats).  A six-channel
            # policy over more than 32 floats has no reference script; it would update through the torch autograd path.
            self.update = "torch"
        P = self.policy.count
        self._ws = torch.zeros(int(self.lib.ppo_update_workspace_floats_a(self.d, self.a)), **f32)
        self._grad = torch.zeros(P, **f32)
        self._adam_m, self._adam_v = torch.zeros(P, **f32), torch.zeros(P, **f32)
        self._adam_t = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._grad_norm = torch.zeros(1, **f32)
        self._stats, self._stats_mb = torch.zeros(8, **f32), torch.zeros(8, **f32)
        self.use_graph = bool(use_cuda_graph)
        # the tcgen05 forward is built for (action width, observation slab) = (4, 32), (6, 32), (4, 64); anything else uses
        # the CUDA-core forward
        self.tensor_core_forward = bool(tensor_core_forward) and (self.d <= 32 or self.a == 4)
        self._graph = None
        self._pending_capture = False
        # the update's optimizer steps as a replayed graph of up to update_graph_steps consecutive minibatches (see _train_kernel)
        # obs running moments accumulated by the env-step kernels' epilogue (SURVEY 8 f1) instead of a pass over the batch
        self.fused_obs_moments = os.environ.get("FWPPO_FUSED_MOMENTS", "1") != "0"
        self._obs_acc = torch.zeros(64 * 2 * self.d, dtype=torch.float64, device=self.device)
        self._side = torch.cuda.Stream(device=self.device)
        self.update_graph = os.environ.get("FWPPO_UPDATE_GRAPH", "1") != "0"
        self.update_graph_steps = 256
        # minibatches up to this size take the single-CTA multi-step kernel when there is no gradient all-reduce (world 1)
        self.fused_steps_max_batch = int(os.environ.get("FWPPO_FUSED_MAX_BATCH", "256"))
        self._ugraph, self._ugraph_key, self._perm_win = None, None, None
        self._perm_ctr = torch.zeros(2, dtype=torch.int32, device=self.device)
        self._perm_epoch = 0
        self._obs = None               # raw observation tensor (view of the env's persistent buffer)
        self._eval_state = None        # PPO.evaluate's buffers and captured chunk for its last eval env
        self._gen = torch.Generator(device=self.device).manual_seed(seed)
        self.stats = RolloutStats()
        self.world = 1
        try:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized():
                self.world = dist.get_world_size()
                dist.broadcast(self.policy.theta.data, src=0)          # one ncclBroadcast of the initial weights
        except Exception:
            self.world = 1
        # gradient all-reduce inside the gradient reduction kernel over NVLink peer memory (one NVLink node, world <= 8);
        # FWPPO_P2P=0 keeps the NCCL all-reduce between the kernels
        self._p2p = None
        if self.world > 1 and self.update == "kernel" and os.environ.get("FWPPO_P2P", "1") != "0":
            self._setup_p2p()

    def _setup_p2p(self) -> None:
        """One exchange buffer per rank (cudaMalloc), shared with every other rank through CUDA IPC handles; all ranks agree
        (an all-reduce of a success flag) whether the peer path is on."""
        import torch.distributed as dist
        rank, world, ok = dist.get_rank(), self.world, 1.0
        own, peers, opened = C.c_void_p(), (C.c_void_p * world)(), []
        try:
            if world > 8:
                raise RuntimeError("more than 8 ranks")
            _lib.check(self.lib.ppo_peer_alloc(C.byref(own)))
            handle = (C.c_uint8 * 64)()
            _lib.check(self.lib.ppo_peer_export(own, handle))
            mine = torch.tensor(list(bytes(handle)), dtype=torch.uint8, device=self.device)
            gathered = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(gathered, mine)
            for j in range(world):
                if j == rank:
                    peers[j] = own.value
                else:
                    h = (C.c_uint8 * 64)(*gathered[j].cpu().tolist())
                    pj = C.c_void_p()
                    _lib.check(self.lib.ppo_peer_import(h, C.byref(pj)))
                    peers[j] = pj.value
                    opened.append(pj)
        except Exception as e:          # no peer access / IPC refused: every rank falls back to NCCL together
            ok = 0.0
            self._p2p_error = f"{type(e).__name__}: {e}"
        flag = torch.tensor([ok], device=self.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if float(flag) < 0.5:
            for pj in opened:
                self.lib.ppo_peer_close(pj)
            if own.value:
                self.lib.ppo_peer_free(own)
            return
        self._p2p = dict(own=own, peers=peers, opened=opened, rank=rank,
                         seq=torch.zeros(1, dtype=torch.int32, device=self.device))
        torch.cuda.synchronize()
        dist.barrier()

    def close_p2p(self) -> None:
        """Unmap the peers' exchange buffers and free this rank's (idempotent; every rank should call it, or none)."""
        pp, self._p2p = getattr(self, "_p2p", None), None
        if not pp:
            return
        try:
            torch.cuda.synchronize()
            for pj in pp["opened"]:
                self.lib.ppo_peer_close(pj)
            self.lib.ppo_peer_free(pp["own"])
        except Exception:
            pass

    # ------------------------------------------------------------------ kernels
    def _stats_ptr(self):
        return _p(self.vecnorm.obs_stats) if self.vecnorm.norm_obs else None

    def _update_obs_moments(self, obs_raw: torch.Tensor) -> None:
        vn = self.vecnorm
        if vn.norm_obs and vn.training:
            _lib.check(self.lib.ppo_moments_update(_p(obs_raw), self.n_envs, self.d, _p(vn.obs_stats), _p(vn.obs_scratch),
                                                   _p(vn.obs_accum), _stream()))

    def _forward(self, obs_raw, t, deterministic=False):
        b = self.buf
        fwd = self.lib.ppo_policy_forward_tc_a if self.tensor_core_forward else self.lib.ppo_policy_forward_a
        _lib.check(fwd(
            _p(self.policy.theta), self.d, self.a, _p(obs_raw), self._stats_ptr(), self.vecnorm.clip_obs, self.n_envs,
            self.seed, self.env.env_id0, t, _p(self._step_dev), int(deterministic), _p(b["obs"][t]), _p(self.act_env),
            _p(b["act"][t]), _p(b["logp"][t]), _p(b["val"][t]), _stream()))

    def collect_rollouts(self) -> None:
        """One rollout of n_steps agent steps.  The kernel sequence is identical every time (persistent buffers,
        step counter on the device), so it is captured once into a CUDA graph and replayed: ~7 launches per agent
        step are then issued back to back by the GPU front end instead of by Python."""
        env, vn = self.env, self.vecnorm
        if self._obs is None:
            self._obs = env.reset_tensor()
            vn.ret.zero_()
            self._update_obs_moments(self._obs)
        if not self.use_graph:
            self._rollout_body()
        elif self._graph is None:
            torch.cuda.synchronize()
            side = torch.cuda.Stream(device=self.device)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                self._rollout_body()                 # eager warm-up on the side stream (also a real rollout)
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
        self.num_timesteps += self.n_steps * self.n_envs * self.world

    def _rollout_body(self) -> None:
        env, vn, b = self.env, self.vecnorm, self.buf
        fused = self.fused_obs_moments and vn.norm_obs and vn.training
        env.set_obs_accumulator(self._obs_acc if fused else None)
        try:
            self._rollout_steps(fused)
        finally:
            env.set_obs_accumulator(None)        # other callers of env.step (evaluation, user code) must not feed the sums

    def _rollout_steps(self, fused: bool) -> None:
        env, vn, b = self.env, self.vecnorm, self.buf
        for t in range(self.n_steps):
            self._forward(self._obs, t)
            obs, rew, flags, term = env.step_tensor(self.act_env, want_terminal_obs=True)
            if fused:
                # the finalize of the observation moments only feeds the NEXT forward: it runs on a side stream beside the
                # reward normalisation and the bootstrap (a fork / join inside the captured graph)
                cur = torch.cuda.current_stream()
                self._side.wait_stream(cur)
                with torch.cuda.stream(self._side):
                    _lib.check(self.lib.ppo_moments_finalize(_p(self._obs_acc), 64, self.n_envs, self.d, _p(vn.obs_stats),
                                                             _p(vn.obs_accum), _stream()))
            else:
                self._update_obs_moments(obs)
            if vn.norm_reward:
                _lib.check(self.lib.ppo_reward_normalize(_p(rew), _p(flags), self.n_envs, vn.gamma, vn.clip_reward, _p(vn.ret),
                                                         _p(vn.ret_stats), _p(vn.ret_scratch), _p(vn.ret_accum),
                                                         _p(b["rew"][t]), _p(b["done"][t]), _stream()))
            else:
                b["rew"][t].copy_(rew)
                b["done"][t].copy_((flags & 3) != 0)
            _lib.check(self.lib.ppo_timeout_bootstrap_a(_p(self.policy.theta), self.d, self.a, _p(term), self._stats_ptr(),
                                                        vn.clip_obs, _p(flags), self.n_envs, self.gamma, _p(b["rew"][t]),
                                                        _stream()))
            if fused:
                torch.cuda.current_stream().wait_stream(self._side)
            self._obs = obs
        _lib.check(self.lib.ppo_counter_add(_p(self._step_dev), self.n_steps, _stream()))
        _lib.check(self.lib.ppo_value_forward_a(_p(self.policy.theta), self.d, self.a, _p(self._obs), self._stats_ptr(),
                                                vn.clip_obs, self.n_envs, _p(self.last_values), _stream()))
        _lib.check(self.lib.ppo_gae(_p(b["rew"]), _p(b["val"]), _p(b["done"]), _p(self.last_values), self.n_steps,
                                    self.n_envs, self.gamma, self.gae_lambda, _p(b["adv"]), _p(b["ret"]), _stream()))

    # ------------------------------------------------------------------ update
    def _minibatch_grad_kernel(self, idx: torch.Tensor, grad: torch.Tensor, stats: torch.Tensor | None = None) -> None:
        """Fused tcgen05 forward+backward of one minibatch (csrc/ppo_update_tc.cu) into `grad`."""
        b = self.buf
        _lib.check(self.lib.ppo_minibatch_grad_a(
            _p(self.policy.theta), self.d, self.a, _p(b["obs"]), _p(b["act"]), _p(b["logp"]), _p(b["adv"]), _p(b["ret"]), _p(idx),
            int(idx.numel()), self.clip_range, self.ent_coef, self.vf_coef, _p(self._ws), _p(grad), _p(stats), _stream()))

    def train(self) -> dict:
        return self._train_kernel() if self.update == "kernel" else self._train_torch()

    def _train_kernel(self) -> dict:
        """SB3 PPO.train with hand-written kernels: per minibatch one fused gradient kernel (tensor cores), the
        NCCL all-reduce of the 49 KB gradient when world > 1, and one clip+Adam kernel.  No host sync inside."""
        total = self.n_steps * self.n_envs
        bs = min(self.batch_size, total)
        lr, (b1, b2), eps = (self.optimizer.param_groups[0][k] for k in ("lr", "betas", "eps"))
        self._stats.zero_()
        self._train_calls = getattr(self, "_train_calls", 0) + 1
        steps_per_epoch = total // bs
        # Optimizer steps are launch-latency sized at small minibatches (batch 128: four ~5 us kernels): from the second call
        # on, a window of consecutive steps is one CUDA graph, replayed for every window of every epoch (the permutation
        # position lives on the device).  The first call runs eagerly -- it is the warm-up a capture needs.
        if (self.world == 1 or self._p2p is not None) and bs <= self.fused_steps_max_batch and total % bs == 0:
            # stable_baselines3-sized minibatches (batch_size 128 = one 128-row tile): a window of consecutive optimizer steps
            # is ONE single-CTA launch (ppo_minibatch_steps_a) -- advantage statistics, gradient, clip and Adam per step, no
            # launch in between
            b = self.buf
            chunk = max(c for c in range(1, min(steps_per_epoch, self.update_graph_steps) + 1) if steps_per_epoch % c == 0)
            for _ in range(self.n_epochs):
                perm = self._epoch_permutation(total)
                for s in range(0, total, chunk * bs):
                    args = (_p(self.policy.theta.data), self.d, self.a, _p(b["obs"]), _p(b["act"]), _p(b["logp"]), _p(b["adv"]),
                            _p(b["ret"]), _p(perm[s:s + chunk * bs]), bs, chunk, self.clip_range, self.ent_coef, self.vf_coef,
                            _p(self._adam_m), _p(self._adam_v), lr, b1, b2, eps, self.max_grad_norm, _p(self._adam_t),
                            _p(self._grad_norm), _p(self._grad), _p(self._stats_mb))
                    if self.world > 1:       # every rank's block exchanges the step's gradient over NVLink peer memory
                        pp = self._p2p
                        _lib.check(self.lib.ppo_minibatch_steps_p2p_a(*args, self.world, pp["rank"], pp["peers"], _p(pp["seq"]),
                                                                      _stream()))
                    else:
                        _lib.check(self.lib.ppo_minibatch_steps_a(*args, _stream()))
        elif total % bs == 0:
            # windows of consecutive minibatches: a single process runs each window through ppo_window_update_a (one launch
            # for the window's advantage statistics, clip + Adam inside the gradient reduction: 2 n + 1 launches for n
            # steps); with an all-reduce between gradient and optimizer the steps stay four launches + NCCL each
            cap = 16 if (self.world == 1 or self._p2p is not None) else self.update_graph_steps
            chunk = max(c for c in range(1, min(steps_per_epoch, cap) + 1) if steps_per_epoch % c == 0)
            if self.use_graph and self.update_graph and self._train_calls > 1:
                key = (total, bs, chunk, lr, b1, b2, eps, self.clip_range, self.ent_coef, self.vf_coef, self.max_grad_norm)
                if self._ugraph is None or self._ugraph_key != key:
                    self._capture_update_graph(total, bs, chunk, lr, b1, b2, eps)
                    self._ugraph_key = key
                self._perm_ctr.copy_(torch.tensor([self._perm_epoch + 1, 0], dtype=torch.int32), non_blocking=False)
                for _ in range(self.n_epochs * (steps_per_epoch // chunk)):
                    self._ugraph.replay()
                self._perm_epoch += self.n_epochs
            else:
                for _ in range(self.n_epochs):
                    perm = self._epoch_permutation(total)
                    for s in range(0, total, chunk * bs):
                        self._window_steps(perm[s:s + chunk * bs], bs, chunk, lr, b1, b2, eps)
        else:                                          # ragged last minibatch (stable_baselines3 allows it): step by step
            for _ in range(self.n_epochs):
                perm = self._epoch_permutation(total)
                for s in range(0, total, bs):
                    self._optimizer_step(perm[s:s + bs], lr, b1, b2, eps)
        st = self._stats_mb
        n = max(float(st[5]), 1.0)
        return dict(policy_loss=float(st[0]) / n, value_loss=float(st[1]) / n, approx_kl=float(st[2]) / n,
                    clip_fraction=float(st[3]) / n, loss=float(st[0]) / n + self.vf_coef * float(st[1]) / n,
                    grad_norm=float(self._grad_norm))

    def _optimizer_step(self, idx: torch.Tensor, lr: float, b1: float, b2: float, eps: float) -> None:
        self._minibatch_grad_kernel(idx, self._grad, self._stats_mb)
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(self._grad)                               # the path's one collective: 49 KB over NVLink
        _lib.check(self.lib.ppo_adam_step(_p(self.policy.theta.data), _p(self._grad), _p(self._adam_m), _p(self._adam_v),
                                          self.policy.count, lr, b1, b2, eps, self.max_grad_norm, 1.0 / self.world,
                                          _p(self._adam_t), _p(self._grad_norm), _stream()))

    def _window_steps(self, idx: torch.Tensor, bs: int, nmb: int, lr: float, b1: float, b2: float, eps: float) -> None:
        """`nmb` consecutive optimizer steps over the index window `idx` (nmb * bs entries)."""
        if self.world > 1 and self._p2p is not None:
            b, pp = self.buf, self._p2p
            _lib.check(self.lib.ppo_window_update_p2p_a(
                _p(self.policy.theta.data), self.d, self.a, _p(b["obs"]), _p(b["act"]), _p(b["logp"]), _p(b["adv"]), _p(b["ret"]),
                _p(idx), bs, nmb, self.clip_range, self.ent_coef, self.vf_coef, _p(self._adam_m), _p(self._adam_v), lr, b1, b2, eps,
                self.max_grad_norm, _p(self._adam_t), _p(self._grad_norm), _p(self._ws), _p(self._grad), _p(self._stats_mb),
                self.world, pp["rank"], pp["peers"], _p(pp["seq"]), _stream()))
        elif self.world == 1:
            b = self.buf
            _lib.check(self.lib.ppo_window_update_a(
                _p(self.policy.theta.data), self.d, self.a, _p(b["obs"]), _p(b["act"]), _p(b["logp"]), _p(b["adv"]), _p(b["ret"]),
                _p(idx), bs, nmb, self.clip_range, self.ent_coef, self.vf_coef, _p(self._adam_m), _p(self._adam_v), lr, b1, b2, eps,
                self.max_grad_norm, _p(self._adam_t), _p(self._grad_norm), _p(self._ws), _p(self._grad), _p(self._stats_mb),
                _stream()))
        else:
            for k in range(nmb):
                self._optimizer_step(idx[k * bs:(k + 1) * bs], lr, b1, b2, eps)

    def _capture_update_graph(self, total: int, bs: int, chunk: int, lr: float, b1: float, b2: float, eps: float) -> None:
        """Graph of one window: indices of the next `chunk` minibatches (ppo_random_permutation_window advances the device
        counters), then per minibatch the gradient kernels, the NCCL all-reduce when world > 1, and clip + Adam."""
        if self._perm_win is None or self._perm_win.numel() != chunk * bs:
            self._perm_win = torch.empty(chunk * bs, dtype=torch.int64, device=self.device)
        torch.cuda.synchronize()
        self._ugraph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._ugraph):
            _lib.check(self.lib.ppo_random_permutation_window(_p(self._perm_win), total, self.seed & (2 ** 64 - 1),
                                                              _p(self._perm_ctr), chunk * bs, _stream()))
            self._window_steps(self._perm_win, bs, chunk, lr, b1, b2, eps)

    def _epoch_permutation(self, total: int) -> torch.Tensor:
        """Minibatch order of the next epoch (RolloutBuffer.get's np.random.permutation): a keyed Feistel bijection
        from one small kernel -- torch.randperm is a multi-pass radix sort of ``total`` keys, ~0.4 ms at 4 M samples."""
        if getattr(self, "_perm", None) is None or self._perm.numel() != total:
            self._perm = torch.empty(total, dtype=torch.int64, device=self.device)
        self._perm_epoch += 1
        _lib.check(self.lib.ppo_random_permutation(_p(self._perm), total, self.seed & (2 ** 64 - 1), self._perm_epoch,
                                                   _stream()))
        return self._perm

    def _train_torch(self) -> dict:
        b = self.buf
        T, N, D = self.n_steps, self.n_envs, self.d
        total = T * N
        obs, act = b["obs"].view(total, D), b["act"].view(total, self.a)
        val, logp_old = b["val"].view(total), b["logp"].view(total)
        adv, ret = b["adv"].view(total), b["ret"].view(total)
        bs = min(self.batch_size, total)
        theta = self.policy.theta
        info = {}
        for _ in range(self.n_epochs):
            perm = self._epoch_permutation(total)
            for s in range(0, total, bs):
                idx = perm[s:s + bs]
                a = adv[idx]
                if len(idx) > 1:
                    a = (a - a.mean()) / (a.std() + 1e-8)
                values, logp, entropy = self.policy.evaluate_actions(obs[idx], act[idx])
                ratio = torch.exp(logp - logp_old[idx])
                pl = -torch.min(a * ratio, a * torch.clamp(ratio, 1 - self.clip_range, 1 + self.clip_range)).mean()
                vl = torch.nn.functional.mse_loss(ret[idx], values)
                el = -entropy.mean()
                loss = pl + self.ent_coef * el + self.vf_coef * vl
                self.optimizer.zero_grad(set_to_none=False)
                loss.backward()
                if self.world > 1:
                    import torch.distributed as dist
                    dist.all_reduce(theta.grad)                       # the path's one collective: 49 KB over NVLink
                    theta.grad.div_(self.world)
                torch.nn.utils.clip_grad_norm_([theta], self.max_grad_norm)
                self.optimizer.step()
        info.update(policy_loss=float(pl.detach()), value_loss=float(vl.detach()), loss=float(loss.detach()))
        return info

    def learn(self, total_timesteps: int, log_interval: int = 1, callback=None, progress_bar: bool = False,
              reset_num_timesteps: bool = True) -> "PPO":
        if reset_num_timesteps:
            self.num_timesteps = 0
        it = 0
        while self.num_timesteps < total_timesteps:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            self.collect_rollouts()
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            self.vecnorm.sync_across_ranks()
            info = self.train()
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            self.stats.env_steps += self.n_steps * self.n_envs * self.world
            self.stats.rollout_s += t1 - t0
            self.stats.update_s += t2 - t1
            it += 1
            if self.verbose and it % log_interval == 0:
                ep = self.env.episode_stats()
                n = max(ep["episodes"], 1.0)
                print(f"[ppo] iter {it} timesteps {self.num_timesteps} sps {self.n_steps * self.n_envs * self.world / (t2 - t0):.3e} "
                      f"rollout {t1 - t0:.3f}s update {t2 - t1:.3f}s ep_rew_mean {ep['return_sum'] / n:.2f} "
                      f"ep_len_mean {ep['length_sum'] / n:.1f} targets/ep {ep['targets_reached_sum'] / n:.2f} "
                      f"loss {info['loss']:.4f}", flush=True)
            if callback is not None and callback(locals(), globals()) is False:
                break
        return self

    # ------------------------------------------------------------------ inference / checkpoint
    def predict(self, obs_raw: torch.Tensor, deterministic: bool = True) -> torch.Tensor:
        """Actions for raw (un-normalised) observations.  Stochastic predictions draw fresh Philox noise on every call
        (a call counter is the step index of the draw; the key is offset from the training stream's)."""
        obs_raw = obs_raw.to(self.device, torch.float32).contiguous()
        n = obs_raw.shape[0]
        act = torch.zeros((n, self.a), dtype=torch.float32, device=self.device)
        val = torch.zeros(n, dtype=torch.float32, device=self.device)
        self._predict_calls = getattr(self, "_predict_calls", 0) + 1
        _lib.check(self.lib.ppo_policy_forward_a(_p(self.policy.theta), self.d, self.a, _p(obs_raw), self._stats_ptr(),
                                                 self.vecnorm.clip_obs, n, (self.seed ^ 0x5BD1E995) & (2 ** 63 - 1), 0,
                                                 self._predict_calls & 0x3FFFFFFF, _p(self._step_dev),
                                                 int(deterministic), None, _p(act), None, None, _p(val), _stream()))
        return act

    @staticmethod
    def episode_quotas(n_eval_episodes: int, n_envs: int) -> list[int]:
        """How many episodes each env contributes, as stable_baselines3.common.evaluation.evaluate_policy divides them:
        ``(n_eval_episodes + i) // n_envs`` for env ``i``.  Counting only up to the quota keeps fast-failing envs (a crash
        takes ~100 steps, a full flight 3,600) from filling the sample with short, bad episodes."""
        return [(int(n_eval_episodes) + i) // int(n_envs) for i in range(int(n_envs))]

    def evaluate_policy(self, env=None, n_eval_episodes: int = 100, deterministic: bool = True, max_steps: int | None = None):
        """stable_baselines3.common.evaluation.evaluate_policy as the reference uses it (eval/eval_waypoints.py:96-160,
        WaypointEvalCallback in train_Fixedwing_Waypoints_v3.py:163-172): frozen VecNormalize statistics, raw (un-normalised)
        rewards, deterministic actions by default, and SB3's per-env episode quotas (``episode_quotas``).  Runs on the device
        until every env of ``env`` (default: the training env's configuration on a fresh batch of at most
        ``n_eval_episodes`` envs) has delivered its quota; returns ``(mean_reward, std_reward, mean_length,
        mean_targets_reached)`` -- all four over the same selected episodes."""
        from .vec_env import FixedwingVecEnv
        own = env is None
        if own:
            n = max(1, min(self.n_envs, int(n_eval_episodes)))
            env = FixedwingVecEnv(n, config=self.env.cfg, device=self.env.device_index, seed=self.seed + 7919,
                                  env_id0=self.env.env_id0 + (1 << 24), wind_field=getattr(self.env, "wind_field", None))
        obs = env.reset_tensor()
        n = env.num_envs
        quota = torch.tensor(self.episode_quotas(n_eval_episodes, n), dtype=torch.int64, device=self.device)
        count = torch.zeros(n, dtype=torch.int64, device=self.device)
        ret = torch.zeros(n, dtype=torch.float64, device=self.device)
        length = torch.zeros(n, dtype=torch.int64, device=self.device)
        has_targets = env.cfg.task in (1, 2)
        done_ret, done_len, done_tr = [], [], []
        # every env needs at most quota episodes of at most max_steps + 2 steps
        limit = max_steps if max_steps is not None else (int(quota.max()) * (int(env.cfg.max_steps) + 2) + 8)
        for _ in range(limit):
            act = self.predict(obs, deterministic=deterministic)
            obs, rew, flags = env.step_tensor(act)
            ret += rew.double()
            length += 1
            fin = (flags & 3) != 0
            take = fin & (count < quota)
            if bool(take.any()):
                done_ret.append(ret[take].clone()); done_len.append(length[take].clone())
                if has_targets:
                    done_tr.append(env.targets_reached_tensor()[take].double())
                count += take.to(torch.int64)
            ret[fin] = 0.0; length[fin] = 0
            if bool((count >= quota).all()):
                break
        if own:
            env.close()
        if not done_ret:
            return float("nan"), float("nan"), float("nan"), float("nan")
        r = torch.cat(done_ret)
        ln = torch.cat(done_len).double()
        targets = float(torch.cat(done_tr).mean()) if done_tr else 0.0
        return float(r.mean()), float(r.std(unbiased=False)), float(ln.mean()), targets

    # agent steps per evaluation chunk: the host reads the count of unfinished envs once per chunk.  Even, because the camera
    # tasks alternate a refill parity on every step and a replayed chunk must end on the parity it was captured with.
    EVAL_CHUNK = 32

    def make_eval_env(self, n_eval_episodes: int) -> FixedwingVecEnv:
        """The batch ``evaluate`` builds when given no env: the training env's configuration (and wind field) on a fresh batch
        of at most ``n_eval_episodes`` envs, seed ``seed + 7919``, env ids from ``env_id0 + 2**24`` -- ``evaluate_policy``'s."""
        n = max(1, min(self.n_envs, int(n_eval_episodes)))
        return FixedwingVecEnv(n, config=self.env.cfg, device=self.env.device_index, seed=self.seed + 7919,
                               env_id0=self.env.env_id0 + (1 << 24), wind_field=getattr(self.env, "wind_field", None))

    def evaluate(self, env=None, n_eval_episodes: int = 100, deterministic: bool = True,
                 max_steps: int | None = None) -> EvalResult:
        """``evaluate_policy`` with the bookkeeping on the device and the per-episode table it does not return.

        Same arguments, defaults, own-env rule (``make_eval_env``), per-env quotas and episodes: every step runs the CUDA-core
        forward of ``predict`` (frozen VecNormalize statistics, no moment accumulation), ``fw_step``, the copy of the pre-reset
        targets-reached plane and ``ppo_eval_ledger``, which records each env's first ``quota`` finished episodes into a table
        slot fixed by env and episode number.  Steps run in chunks of ``EVAL_CHUNK``; with ``use_cuda_graph`` a chunk is
        captured once per eval env and replayed, and the host reads the count of envs below quota between chunks -- one sync
        per chunk instead of one per step.  ``max_steps`` is exact: steps at or after it record nothing.

        The episodes, and the four means (``EvalResult.mean_*``), are bit-identical to ``evaluate_policy``'s.  The env's state
        afterwards is not: ``evaluate`` may step a caller-supplied env up to ``EVAL_CHUNK - 1`` steps past the step on which
        the last needed episode ended, where ``evaluate_policy`` stops on that step.

        ``deterministic=False`` samples the Gaussian policy with Philox noise keyed by the model seed and counted by the
        evaluation's own step index (restarting at 0 on every call): the training counter and ``predict``'s call counter are
        neither read nor advanced, so evaluating never changes what training draws."""
        own = env is None
        if own:
            env = self.make_eval_env(n_eval_episodes)
        try:
            return self._evaluate(env, int(n_eval_episodes), bool(deterministic), max_steps)
        finally:
            if own:
                self._eval_state = None            # the captured chunk names the env's buffers: it goes first
                env.close()

    def _evaluate(self, env, n_eval_episodes: int, deterministic: bool, max_steps: int | None) -> EvalResult:
        n, K = env.num_envs, self.EVAL_CHUNK
        quotas = np.asarray(self.episode_quotas(n_eval_episodes, n), np.int64)
        limit = max_steps if max_steps is not None else int(quotas.max()) * (int(env.cfg.max_steps) + 2) + 8
        limit = min(max(int(limit), 0), 2 ** 31 - 1)
        key = (n_eval_episodes, deterministic, limit)
        s = self._eval_state
        if s is None or s["env"] is not env or s["key"] != key:
            self._eval_state = None
            dev = self.device
            i32, f64 = dict(dtype=torch.int32, device=dev), dict(dtype=torch.float64, device=dev)
            E = max(int(quotas.sum()), 1)
            s = dict(env=env, key=key, graph=None, quota=torch.tensor(quotas, **i32),
                     offset=torch.tensor(np.cumsum(quotas) - quotas, **i32), ret=torch.zeros(n, **f64),
                     len=torch.zeros(n, **i32), count=torch.zeros(n, **i32), step=torch.zeros(1, **i32),
                     remaining=torch.zeros(1, **i32), act=torch.zeros((n, self.a), dtype=torch.float32, device=dev),
                     val=torch.zeros(n, dtype=torch.float32, device=dev), ep_ret=torch.zeros(E, **f64),
                     ep_len=torch.zeros(E, **i32), ep_tr=torch.zeros(E, dtype=torch.uint8, device=dev),
                     ep_flags=torch.zeros(E, dtype=torch.uint8, device=dev), ep_step=torch.zeros(E, **i32))
            self._eval_state = s
        s["obs"] = env.reset_tensor()
        for k in ("ret", "len", "count", "step"):
            s[k].zero_()
        active = int((quotas > 0).sum())
        s["remaining"].fill_(active)
        done = 0
        while done < limit and active > 0:
            if self.use_graph and s["graph"] is not None:
                s["graph"].replay()
            else:
                self._eval_chunk(s, env, deterministic, limit)
            done += K
            if int(s["remaining"].item()) == 0:
                break
            if self.use_graph and s["graph"] is None:
                # the chunk that just ran eagerly was the warm-up; capture does not execute the launches it records
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._eval_chunk(s, env, deterministic, limit)
                s["graph"] = g
        count = s["count"].cpu().numpy().astype(np.int64)
        slot = np.repeat(np.cumsum(quotas) - quotas, count) + (np.arange(int(count.sum())) - np.repeat(np.cumsum(count) - count, count))
        take = lambda name: s[name].cpu().numpy()[slot]  # noqa: E731
        return EvalResult.from_episodes(take("ep_ret"), take("ep_len"), take("ep_tr"), take("ep_flags"),
                                        np.repeat(np.arange(n), count), take("ep_step"), env.cfg.task, env.cfg.num_targets,
                                        device=self.device)

    def _eval_chunk(self, s: dict, env, deterministic: bool, limit: int) -> None:
        """EVAL_CHUNK agent steps of an evaluation: forward, env step, targets-reached copy, ledger; then the step index
        advances by the chunk.  Every pointer is persistent, so the same launches serve as a replayed graph."""
        n, lib = env.num_envs, self.lib
        tidx = None
        seed = (self.seed ^ 0x1B873593) & (2 ** 63 - 1)        # a key of its own: neither the training's nor predict's
        for k in range(self.EVAL_CHUNK):
            _lib.check(lib.ppo_policy_forward_a(_p(self.policy.theta), self.d, self.a, _p(s["obs"]), self._stats_ptr(),
                                                self.vecnorm.clip_obs, n, seed, env.env_id0 & 0xFFFFFFFF, k, _p(s["step"]),
                                                int(deterministic), None, _p(s["act"]), None, None, _p(s["val"]), _stream()))
            _, rew, flags = env.step_tensor(s["act"])
            if env.cfg.task in (1, 2):
                tidx = env.targets_reached_tensor()
            _lib.check(lib.ppo_eval_ledger(_p(rew), _p(flags), _p(tidx), n, _p(s["ret"]), _p(s["len"]), _p(s["count"]),
                                           _p(s["quota"]), _p(s["offset"]), k, _p(s["step"]), limit, _p(s["remaining"]),
                                           _p(s["ep_ret"]), _p(s["ep_len"]), _p(s["ep_tr"]), _p(s["ep_flags"]), _p(s["ep_step"]),
                                           _stream()))
        _lib.check(lib.ppo_counter_add(_p(s["step"]), self.EVAL_CHUNK, _stream()))

    def save(self, path: str) -> None:
        torch.save({"policy": self.policy.state_dict(), "optimizer": self.optimizer.state_dict(),
                    "adam": {"m": self._adam_m.clone(), "v": self._adam_v.clone(), "t": int(self._adam_t.item())},
                    "vecnorm": self.vecnorm.state_dict(), "num_timesteps": self.num_timesteps,
                    "global_step": int(self._step_dev.item()), "seed": self.seed, "obs_dim": self.d}, path)

    def load(self, path: str) -> "PPO":
        ck = torch.load(path, map_location=self.device, weights_only=False)
        self.policy.load_state_dict(ck["policy"])
        self.optimizer.load_state_dict(ck["optimizer"])
        if "adam" in ck:
            self._adam_m.copy_(ck["adam"]["m"]); self._adam_v.copy_(ck["adam"]["v"]); self._adam_t.fill_(int(ck["adam"]["t"]))
        self.vecnorm.load_state_dict(ck["vecnorm"])
        self.num_timesteps = ck["num_timesteps"]
        self._step_dev.fill_(int(ck["global_step"]))
        return self

    def export_sb3(self, directory: str, space_dtype=np.float64) -> dict:
        """Write what stable_baselines3 needs to replay this policy in the reference's eval scripts
        (eval/eval_waypoints.py:96-107: ``VecNormalize.load(vecnorm_path, env)`` then ``PPO.load(model_path, env=env)``):
          final_model.zip -- SB3's own archive layout (sb3_io.write_model_zip): ``data`` JSON, ``policy.pth``,
                             ``policy.optimizer.pth``, ``pytorch_variables.pth``, version and system info
          vecnorm.pkl     -- a pickled ``VecNormalize`` without its venv (sb3_io.write_vecnorm_pkl)
          policy.pth      -- ``ActorCriticPolicy.state_dict()`` on its own (MlpPolicy, net_arch pi = vf = [64, 64], Tanh)
          vecnorm.npz     -- the running moments as plain arrays under VecNormalize's attribute names
        The two SB3 containers are written without SB3 (it is not installable here) from its on-disk format; INTEGRATION.md
        section 5 has the one-line load check for a machine that has it.  Returns the four paths."""
        import os
        from . import sb3_io
        os.makedirs(directory, exist_ok=True)
        pol_path, vn_path = os.path.join(directory, "policy.pth"), os.path.join(directory, "vecnorm.npz")
        torch.save({k: v.detach().cpu() for k, v in self.policy.state_dict().items()}, pol_path)
        export_vecnorm_npz(self.vecnorm.state_dict(), vn_path)
        zip_path = sb3_io.write_model_zip(os.path.join(directory, "final_model.zip"), self, space_dtype)
        pkl_path = sb3_io.write_vecnorm_pkl(os.path.join(directory, "vecnorm.pkl"), self.vecnorm.state_dict(), self.d, self.a,
                                            self.n_envs, space_dtype)
        return {"policy": pol_path, "vecnorm": vn_path, "model_zip": zip_path, "vecnorm_pkl": pkl_path}

    def import_sb3(self, directory: str) -> "PPO":
        """Inverse of export_sb3.  Also takes what SB3 itself wrote: ``final_model.zip`` / ``best_model.zip`` (``model.save``)
        and ``vecnorm.pkl`` (``VecNormalize.save``) of the reference's training runs, or a bare ``policy.pth``."""
        import os
        from . import sb3_io
        zips = [f for f in ("final_model.zip", "best_model.zip", "model.zip") if os.path.exists(os.path.join(directory, f))]
        if zips:
            ck = sb3_io.read_model_zip(os.path.join(directory, zips[0]))
            self.policy.load_state_dict(ck["policy"])
            for i, st in ck.get("optimizer", {}).get("state", {}).items():          # Adam moments, SB3 parameter order
                key = sb3_io.SB3_PARAM_ORDER[int(i)]
                base, _, leaf = key.rpartition(".")
                m = {"mlp_extractor.policy_net.0": "pi.0", "mlp_extractor.policy_net.2": "pi.2",
                     "mlp_extractor.value_net.0": "vf.0", "mlp_extractor.value_net.2": "vf.2"}
                a, b, _ = self.policy.slices[f"{m[base]}.{leaf}" if base in m else key]
                self._adam_m[a:b] = st["exp_avg"].reshape(-1).to(self.device)
                self._adam_v[a:b] = st["exp_avg_sq"].reshape(-1).to(self.device)
                self._adam_t.fill_(int(float(st["step"])))
        else:
            sd = torch.load(os.path.join(directory, "policy.pth"), map_location="cpu", weights_only=True)
            self.policy.load_state_dict(sd)
        pkl, npz = os.path.join(directory, "vecnorm.pkl"), os.path.join(directory, "vecnorm.npz")
        if os.path.exists(pkl):
            self.vecnorm.load_state_dict(sb3_io.read_vecnorm_pkl(pkl))
        elif os.path.exists(npz):
            self.vecnorm.load_state_dict(import_vecnorm_npz(npz))
        return self

    def get_parameters(self) -> dict:
        return {"policy": self.policy.state_dict()}

    def set_parameters(self, params: dict) -> None:
        self.policy.load_state_dict(params["policy"])


def smoke() -> None:
    """Tiny rollout + update on cuda:0 (called from __graft_entry__.smoke)."""
    env = FixedwingVecEnv(256, preset="waypoints_v3", seed=3)
    model = PPO("MlpPolicy", env, n_steps=8, batch_size=512, n_epochs=2, seed=3)
    model.learn(256 * 8 * 2)
    assert torch.isfinite(model.policy.theta).all()
    env.close()
