"""The frozen low-level tracker of the high-level waypoint task (task 5, ``highlevel`` preset).

The reference trains a low-level tracker (train/train_lowlevel_cmd.py: FixedwingLowLevelEnv, mode -1, six surface / thrust
channels tracking ``[psi_ref, h_ref, V_ref]``) so that a high-level policy can command it (train/train_highlevel_cmd.py,
examples/lowlevel.py).  Here that tracker runs inside the step kernel: the high-level action ``a`` is a command
``psi = atan2(a1, a0)``, ``h = h_lo + (clip(a2) + 1) / 2 (h_hi - h_lo)``, ``V = v_lo + (clip(a3) + 1) / 2 (v_hi - v_lo)``,
and every 120 Hz inner iteration evaluates the tracker's policy mean on the task-3 observation built with that command,
bit-identical to ``PPO.predict(obs, deterministic=True)`` of the tracker model (include/fwsim.h ``FwTracker``).

    tracker = Tracker.load("runs/lowlevel/final_model.pt")         # PPO.save file, or an export_sb3 / SB3 directory
    env = FixedwingVecEnv(4096, preset="highlevel", tracker=tracker)
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Sequence

import numpy as np

OBS_DIM, ACT_DIM, HIDDEN = 21, 6, 64
# the flat parameter vector of include/fwppo.h for (obs 21, action 6): pi tower, vf tower, log_std
POLICY_TOWER = HIDDEN * OBS_DIM + HIDDEN + HIDDEN * HIDDEN + HIDDEN + ACT_DIM * HIDDEN + ACT_DIM
PARAM_COUNT = POLICY_TOWER + HIDDEN * OBS_DIM + HIDDEN + HIDDEN * HIDDEN + HIDDEN + HIDDEN + 1 + ACT_DIM
# the low-level env's reference distribution (fw_sample_targets, task 3): h ~ U(5, 20) m, V ~ U(10, 20) m/s
H_RANGE, V_RANGE = (5.0, 20.0), (10.0, 20.0)


def _range(r, name: str) -> tuple[float, float]:
    a = np.asarray(r, dtype=np.float64).reshape(-1)
    if a.shape != (2,) or not np.all(np.isfinite(a)) or not a[0] < a[1]:
        raise ValueError(f"{name} must be a finite (lo, hi) pair with lo < hi, got {r!r}")
    return float(a[0]), float(a[1])


class Tracker:
    """A frozen (21 -> 6) MlpPolicy: the flat parameter vector (``PARAM_COUNT`` float32, include/fwppo.h layout; only the
    policy tower is used), its frozen VecNormalize statistics (``obs_mean`` / ``obs_var``, both None for an un-normalised
    policy) and ``clip_obs``, and the altitude / airspeed ranges the high-level command is mapped onto."""

    def __init__(self, params, obs_mean=None, obs_var=None, clip_obs: float = 10.0,
                 h_range: Sequence[float] = H_RANGE, v_range: Sequence[float] = V_RANGE):
        p = np.ascontiguousarray(np.asarray(params, dtype=np.float32).reshape(-1))
        if p.shape != (PARAM_COUNT,):
            raise ValueError(f"params must hold {PARAM_COUNT} floats (the (21, 6) policy of include/fwppo.h), got {p.size}")
        if not np.all(np.isfinite(p[:POLICY_TOWER])):
            raise ValueError("tracker policy parameters must be finite")
        self.params = p
        if (obs_mean is None) != (obs_var is None):
            raise ValueError("obs_mean and obs_var are both given (normalised tracker) or both None")
        self.obs_mean = self.obs_var = None
        if obs_mean is not None:
            m = np.ascontiguousarray(np.asarray(obs_mean, dtype=np.float64).reshape(-1))
            v = np.ascontiguousarray(np.asarray(obs_var, dtype=np.float64).reshape(-1))
            if m.shape != (OBS_DIM,) or v.shape != (OBS_DIM,):
                raise ValueError(f"obs_mean and obs_var must have {OBS_DIM} entries, got {m.size} and {v.size}")
            if not (np.all(np.isfinite(m)) and np.all(np.isfinite(v)) and np.all(v >= 0)):
                raise ValueError("obs_mean must be finite and obs_var finite and >= 0")
            self.obs_mean, self.obs_var = m, v
        self.clip_obs = float(clip_obs)
        if not (np.isfinite(self.clip_obs) and self.clip_obs > 0):
            raise ValueError(f"clip_obs must be finite and > 0, got {clip_obs!r}")
        self.h_range = _range(h_range, "h_range")
        self.v_range = _range(v_range, "v_range")

    @staticmethod
    def _check_widths(obs_dim: int, act_dim: int) -> None:
        if (obs_dim, act_dim) != (OBS_DIM, ACT_DIM):
            raise ValueError(f"a tracker is a low-level policy with a {OBS_DIM}-float observation and {ACT_DIM} actions "
                             f"(the lowlevel preset); this one has {obs_dim} and {act_dim}")

    @classmethod
    def _from_state(cls, policy_sd: dict, vecnorm: dict | None, **kw) -> "Tracker":
        """From an SB3-named policy state dict and a ``DeviceVecNormalize.state_dict``-layout statistics dict (or None)."""
        import torch
        from .ppo import FlatMlpPolicy
        w1, wa = policy_sd["mlp_extractor.policy_net.0.weight"], policy_sd["action_net.weight"]
        cls._check_widths(int(w1.shape[1]), int(wa.shape[0]))
        pol = FlatMlpPolicy(OBS_DIM, torch.device("cpu"), act_dim=ACT_DIM)
        pol.load_state_dict({k: torch.as_tensor(v) for k, v in policy_sd.items()})
        norm = vecnorm is not None and bool(vecnorm.get("norm_obs", True))
        return cls(pol.theta.detach().numpy(), vecnorm["obs_rms.mean"] if norm else None,
                   vecnorm["obs_rms.var"] if norm else None, vecnorm["clip_obs"] if vecnorm is not None else 10.0, **kw)

    @classmethod
    def from_ppo(cls, model, **kw) -> "Tracker":
        """The policy a ``PPO`` (trained on the ``lowlevel`` preset) holds now, with its frozen observation statistics."""
        cls._check_widths(int(model.d), int(model.a))
        vn = model.vecnorm
        stats = vn.obs_stats.detach().cpu().numpy() if vn.norm_obs else None
        return cls(model.policy.theta.detach().cpu().numpy(), stats[:OBS_DIM] if stats is not None else None,
                   stats[OBS_DIM:2 * OBS_DIM] if stats is not None else None, vn.clip_obs, **kw)

    @classmethod
    def load(cls, path: str, **kw) -> "Tracker":
        """A ``PPO.save`` file, or a directory in the ``PPO.export_sb3`` / stable-baselines3 layout (``final_model.zip`` /
        ``best_model.zip`` / ``model.zip`` or ``policy.pth``, with ``vecnorm.pkl`` or ``vecnorm.npz``)."""
        if os.path.isdir(path):
            from . import sb3_io
            ck = sb3_io.read_directory(path)
            return cls._from_state(ck["policy"], ck.get("vecnorm"), **kw)
        import torch
        ck = torch.load(path, map_location="cpu", weights_only=False)
        if not isinstance(ck, dict) or "policy" not in ck:
            raise ValueError(f"{path} is not a PPO.save checkpoint")
        return cls._from_state(ck["policy"], ck.get("vecnorm"), **kw)

    def to_c(self):
        """The ``FwTracker`` descriptor (its pointers refer to this object's arrays: keep the object alive)."""
        from ._lib import FwTrackerC
        c = FwTrackerC()
        c.params = self.params.ctypes.data_as(C.c_void_p).value
        c.obs_mean = self.obs_mean.ctypes.data_as(C.c_void_p).value if self.obs_mean is not None else None
        c.obs_var = self.obs_var.ctypes.data_as(C.c_void_p).value if self.obs_var is not None else None
        c.clip_obs = self.clip_obs
        c.h_range[0], c.h_range[1] = self.h_range
        c.v_range[0], c.v_range[1] = self.v_range
        return c

    def command(self, actions: np.ndarray) -> np.ndarray:
        """``[psi_ref, h_ref, V_ref]`` of high-level actions ``[..., 4]`` (float64; the kernel computes it in float32)."""
        a = np.asarray(actions, dtype=np.float64)
        c = np.clip(a[..., 2:4], -1.0, 1.0)
        h = self.h_range[0] + (c[..., 0] + 1.0) / 2.0 * (self.h_range[1] - self.h_range[0])
        v = self.v_range[0] + (c[..., 1] + 1.0) / 2.0 * (self.v_range[1] - self.v_range[0])
        return np.stack([np.arctan2(a[..., 1], a[..., 0]), h, v], axis=-1)

    def __repr__(self) -> str:
        return (f"Tracker(normalised={self.obs_mean is not None}, clip_obs={self.clip_obs}, h_range={self.h_range}, "
                f"v_range={self.v_range})")
