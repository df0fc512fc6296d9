"""FixedwingVecEnv -- the batched seam (SURVEY section 8 b, B1/B1').

Drop-in for the one line of the reference that builds its training env
(train/train_Fixedwing_Waypoints_v3.py:251, train/train_Fixedwing_Waypoints_ObjLock.py:306)::

    env = SubprocVecEnv([make_env(i, seed) for i in range(num_envs)])        # reference
    env = FixedwingVecEnv(num_envs, preset="waypoints_v3", seed=seed)        # this package

It honours the stable-baselines3 ``VecEnv`` contract (attrs ``num_envs``/``observation_space``/``action_space``;
``reset``/``step_async``/``step_wait``/``step``/``close``/``seed``/``get_attr``/``set_attr``/``env_method``/
``env_is_wrapped``; auto-reset inside ``step`` with ``infos[i]["terminal_observation"]`` and
``infos[i]["TimeLimit.truncated"]``) with host NumPy arrays, and adds a device-tensor lane (``step_tensor``)
that never leaves HBM.  All arithmetic happens in libfwsim.so (sm_100a CUDA); there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from typing import Any, Sequence

import numpy as np

from . import _lib
from .compat import spaces
from .compat.vec_env import VecEnv
from .config import (EnvConfig, FLAG_COLLISION, FLAG_COMPLETE, FLAG_FAULT, FLAG_OOB, FLAG_STRIKE, FLAG_TERM, FLAG_TRUNC,
                     make_config)
from .wind import WindField

_STATE_FIELDS = {
    "pos": (np.float32, 3), "quat": (np.float32, 4), "vel": (np.float32, 3), "omega": (np.float32, 3),
    "act": (np.float32, 6), "targets": (np.float32, None), "target_idx": (np.int32, 0),
    "step_count": (np.int32, 0), "physics_steps": (np.int32, 0), "episode": (np.uint32, 0),
    "new_dist": (np.float32, 0), "wind": (np.float32, 7),
    # ObjLock task only
    "duck": (np.float32, 3), "obst": (np.float32, (32, 3)), "ol_f": (np.float32, 12), "ol_i": (np.int32, 9),
    # duck-only task: MAX_HIST history rows of 9 (newest first) + 4 deltas
    "vis_hist": (np.float32, 4 * 9 + 4),
}
_OBJLOCK_FIELDS = ("duck", "obst", "ol_f", "ol_i")
_DUCK_FIELDS = ("vis_hist",)


class FixedwingVecEnv(VecEnv):
    """``num_envs`` fixed-wing environments stepped by one CUDA kernel launch per agent step.

    Derives from ``stable_baselines3.common.vec_env.VecEnv`` when SB3 is importable (compat.vec_env keeps a stand-in of
    the same shape otherwise), so ``VecNormalize(env)``, ``PPO("MlpPolicy", env)`` and ``evaluate_policy(model, env,
    callback=...)`` of the reference's scripts take it as they take a ``SubprocVecEnv``."""

    metadata = {"render_modes": []}

    def __init__(self, num_envs: int, preset: str = "waypoints_v3", config: EnvConfig | None = None,
                 device: int = 0, seed: int = 0, env_id0: int = 0, info_mode: str = "auto", wind_field: WindField | None = None,
                 **overrides):
        self.cfg = config if config is not None else make_config(preset, **overrides)
        if config is not None and overrides:
            self.cfg = self.cfg.replace(**overrides)
        # gridded wind (wind_mode 3): the config keeps its wind_start_substep / wind_randomize; the field is installed by _open()
        if wind_field is not None:
            if not isinstance(wind_field, WindField):
                raise TypeError("wind_field must be a pyflyt_drone_b200.wind.WindField")
            self.cfg = self.cfg.replace(wind_mode=3)
        elif self.cfg.wind_mode == 3:
            raise ValueError("wind_mode 3 (gridded field) needs wind_field=WindField(...)")
        self.wind_field = wind_field
        self.num_envs = int(num_envs)
        self.device_index = int(device)
        self._seed = int(seed)
        self.env_id0 = int(env_id0)
        self.lib = _lib.load()
        self._c_cfg = self.cfg.to_c()
        if info_mode == "auto":
            info_mode = "full" if self.num_envs <= 4096 else "lazy"
        if info_mode not in ("full", "lazy"):
            raise ValueError("info_mode must be 'auto', 'full' or 'lazy'")
        self.info_mode = info_mode
        self._open()
        VecEnv.__init__(self, self.num_envs, self.observation_space, self.action_space)
        self._user_attrs: dict[str, list] = {}     # set_attr() storage (per-env Python-side attributes)
        self._pending: np.ndarray | None = None
        self._t = None  # lazily created torch buffers for the tensor lane
        self._closed = False

    def _open(self) -> None:
        """Create the device batch and map the library's pinned staging buffers as NumPy views."""
        self._h = C.c_void_p()
        _lib.check(self.lib.fw_create(C.byref(self._c_cfg), self.num_envs, self.device_index, self._seed,
                                      self.env_id0, C.byref(self._h)))
        if self.wind_field is not None:
            desc = self.wind_field.to_c()
            rc = self.lib.fw_set_wind_field(self._h, C.byref(desc))
            if rc != 0:
                msg = self.lib.fw_last_error()
                self.lib.fw_destroy(self._h)
                self._h = C.c_void_p()
                raise _lib.FwError(f"libfwsim error {rc}: {msg.decode() if msg else '?'}")
        self.obs_dim = int(self.lib.fw_obs_dim(self._h))
        self.act_dim = int(self.lib.fw_act_dim(self._h))     # 4, or 6 for the low-level task
        D = max(self.obs_dim, 1)
        self.observation_space = spaces.Box(low=-np.inf, high=np.inf, shape=(self.obs_dim,), dtype=np.float32)
        self.action_space = spaces.Box(low=-1.0, high=1.0, shape=(self.act_dim,), dtype=np.float32)
        # host arrays = NumPy views of the library's pinned staging buffers: the DMA engines read actions from
        # and write observations to the very memory the caller sees (no extra host memcpy on either side)
        ptrs = [C.c_void_p() for _ in range(5)]
        _lib.check(self.lib.fw_host_buffers(self._h, *[C.byref(p) for p in ptrs]))

        def view(ptr, shape, ctype, dtype):
            n = int(np.prod(shape))
            return np.frombuffer((ctype * n).from_address(ptr.value), dtype=dtype).reshape(shape)

        self._h_act = view(ptrs[0], (self.num_envs, self.act_dim), C.c_float, np.float32)
        self._h_obs = view(ptrs[1], (self.num_envs, D), C.c_float, np.float32)
        self._h_rew = view(ptrs[2], (self.num_envs,), C.c_float, np.float32)
        self._h_flags = view(ptrs[3], (self.num_envs,), C.c_uint8, np.uint8)
        self._h_term = view(ptrs[4], (self.num_envs, D), C.c_float, np.float32)
        tp = C.c_void_p()
        _lib.check(self.lib.fw_host_info_buffer(self._h, C.byref(tp)))
        self._h_tidx = view(tp, (self.num_envs,), C.c_uint8, np.uint8)      # info["num_targets_reached"], pre-reset

    # ------------------------------------------------------------------ SB3 VecEnv (host NumPy lane)
    def reset(self) -> np.ndarray:
        _lib.check(self.lib.fw_reset_host(self._h, self._h_obs.ctypes.data_as(C.c_void_p)))
        self.reset_infos = [{} for _ in range(self.num_envs)]
        return self._h_obs[:, : self.obs_dim].copy()

    def observe(self) -> np.ndarray:
        """Observation of the current state of every env, nothing reset (see fw_observe_host)."""
        _lib.check(self.lib.fw_observe_host(self._h, self._h_obs.ctypes.data_as(C.c_void_p)))
        return self._h_obs[:, : self.obs_dim].copy()

    def step_async(self, actions: np.ndarray) -> None:
        if self._pending is not None:
            raise RuntimeError("step_async called twice without step_wait")
        a = np.ascontiguousarray(actions, dtype=np.float32)
        if a.shape != (self.num_envs, self.act_dim):
            raise ValueError(f"actions must have shape ({self.num_envs}, {self.act_dim}), got {a.shape}")
        self._pending = a

    def step_arrays(self, actions: np.ndarray, want_terminal_obs: bool = True):
        """Host-buffer step without the per-env info dicts: (obs, rewards, flags, terminal_obs).
        The returned arrays are views of pinned memory owned by the env, valid until the next step."""
        if np.shape(actions) != (self.num_envs, self.act_dim):
            raise ValueError(f"actions must have shape ({self.num_envs}, {self.act_dim}), got {np.shape(actions)}")
        # the library stages caller-owned actions into its pinned buffer chunk by chunk, overlapped with the GPU work;
        # actions written straight into ``action_buffer`` skip that copy
        a = actions if (isinstance(actions, np.ndarray) and actions.dtype == np.float32 and actions.flags.c_contiguous) \
            else np.ascontiguousarray(actions, dtype=np.float32)
        p = lambda x: x.ctypes.data_as(C.c_void_p)  # noqa: E731
        _lib.check(self.lib.fw_step_host(self._h, p(a), p(self._h_obs), p(self._h_rew), p(self._h_flags),
                                         p(self._h_term) if want_terminal_obs else None))
        return self._h_obs[:, : self.obs_dim], self._h_rew, self._h_flags, self._h_term[:, : self.obs_dim]

    @property
    def action_buffer(self) -> np.ndarray:
        """The env's pinned [num_envs, 4] float32 action staging buffer: a policy that writes its actions here and
        passes this very array to ``step_arrays`` avoids the host-side staging copy."""
        return self._h_act

    def step_wait(self):
        if self._pending is None:
            raise RuntimeError("step_wait called without step_async")
        a, self._pending = self._pending, None
        obs, rew, flags, term = self.step_arrays(a)
        dones = (flags & (FLAG_TERM | FLAG_TRUNC)) != 0
        infos = self._make_infos(flags, dones, term)
        return obs.copy(), rew.copy(), dones, infos

    def step(self, actions: np.ndarray):
        self.step_async(actions)
        return self.step_wait()

    def _info_of(self, f: int, tidx: int | None) -> dict:
        d = {"out_of_bounds": bool(f & FLAG_OOB), "collision": bool(f & FLAG_COLLISION),
             "env_complete": bool(f & FLAG_COMPLETE)}
        if tidx is not None:
            d["num_targets_reached"] = tidx
        if self.cfg.task in (2, 4):
            d["duck_strike"] = bool(f & FLAG_STRIKE)
        if self.cfg.task == 4:
            d["is_success"] = bool(f & FLAG_STRIKE)          # fixedwing_objlock_env.py:235,372
        if f & FLAG_FAULT:
            d["state_fault"] = True                          # non-finite state: force-reset by the kernel (no reference key)
        return d

    def _make_infos(self, flags: np.ndarray, dones: np.ndarray, term: np.ndarray) -> list[dict]:
        """The info dicts of the reference env (fixedwing_base_env.py:212-215; fixedwing_waypoint_objlock_env.py:296,
        336-337).  ``num_targets_reached`` is the value the env held BEFORE the auto-reset of a finished episode -- the
        one WaypointEvalCallback._log_success_callback reads on every done (train_Fixedwing_Waypoints_v3.py:136-138).
        ``info_mode="lazy"`` (default above 4,096 envs) builds full dicts for finished envs only; the others share one
        blank dict, and the per-env values stay available as arrays (``last_flags``, ``last_targets_reached``)."""
        has_t = self.cfg.task in (1, 2)
        tr = self._h_tidx
        idx = np.nonzero(dones)[0]
        if self.info_mode == "lazy":
            blank = self._info_of(0, None)                       # no per-env value in the shared dict: the key is absent
            infos: list[dict] = [blank] * self.num_envs
        else:
            infos = [self._info_of(int(f), int(t) if has_t else None) for f, t in zip(flags, tr)]
        for i in idx:
            f = int(flags[i])
            d = self._info_of(f, int(tr[i]) if has_t else None)
            d["terminal_observation"] = term[i].copy()
            d["TimeLimit.truncated"] = bool(f & FLAG_TRUNC) and not bool(f & FLAG_TERM)
            infos[i] = d
        return infos

    @property
    def last_flags(self) -> np.ndarray:
        """Flag bytes of the last host-lane step (view of pinned memory, valid until the next step)."""
        return self._h_flags

    @property
    def last_targets_reached(self) -> np.ndarray:
        """``info["num_targets_reached"]`` of the last host-lane step for every env, taken before any auto-reset."""
        return self._h_tidx

    def close(self) -> None:
        if not self._closed and self._h:
            self._h_act = self._h_obs = self._h_rew = self._h_flags = self._h_term = self._h_tidx = None   # views die with the handle
            self.lib.fw_destroy(self._h)
            self._h = C.c_void_p()
            self._t = None
            self._closed = True

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def seed(self, seed: int | None = None) -> list[int | None]:
        """SB3 ``VecEnv.seed``: env ``i`` gets ``seed + i``.  The Philox key is fixed per batch, so passing a seed
        ALWAYS rebuilds the batch -- also when it equals the current one, which makes ``seed(s); reset()`` reproduce
        the same first episode every time (the gymnasium ``reset(seed=s)`` contract the reference's eval scripts use)."""
        if seed is not None:
            self._seed = int(seed)
            self._h_act = self._h_obs = self._h_rew = self._h_flags = self._h_term = self._h_tidx = None
            self._t = None
            self.lib.fw_destroy(self._h)
            self._open()
        return [self._seed + self.env_id0 + i for i in range(self.num_envs)]

    def _indices(self, indices) -> Sequence[int]:
        if indices is None:
            return range(self.num_envs)
        if isinstance(indices, int):
            return [indices]
        return indices

    # Python-level per-env attributes / methods (SB3 reaches the sub-envs of a SubprocVecEnv with these).  The batch has
    # no sub-env objects: attributes are the VecEnv's own, then the shared EnvConfig, then whatever set_attr stored;
    # env_method calls the VecEnv's batched method of that name once and hands every selected env the same result.
    def get_attr(self, attr_name: str, indices=None) -> list[Any]:
        idx = self._indices(indices)
        if attr_name in self._user_attrs:
            return [self._user_attrs[attr_name][i] for i in idx]
        if attr_name == "render_mode":
            return [None for _ in idx]
        if hasattr(self, attr_name):
            val = getattr(self, attr_name)
        elif hasattr(self.cfg, attr_name):
            val = getattr(self.cfg, attr_name)
        else:
            raise AttributeError(f"FixedwingVecEnv envs have no attribute {attr_name!r}")
        return [val for _ in idx]

    def set_attr(self, attr_name: str, value: Any, indices=None) -> None:
        """Stores a Python-side attribute per env (returned by ``get_attr``).  Fields of the compiled batch
        configuration cannot change under a live batch: build a new ``FixedwingVecEnv`` for that."""
        if hasattr(self.cfg, attr_name):
            raise AttributeError(f"{attr_name!r} is part of the compiled batch configuration (EnvConfig); "
                                 "build a new FixedwingVecEnv with that override instead of set_attr")
        slot = self._user_attrs.setdefault(attr_name, [None] * self.num_envs)
        for i in self._indices(indices):
            slot[i] = value

    def env_method(self, method_name: str, *args, indices=None, **kwargs) -> list[Any]:
        fn = getattr(self, method_name, None)
        if method_name.startswith("_") or not callable(fn) or method_name in ("reset", "step", "step_async", "step_wait",
                                                                              "close", "seed", "env_method"):
            raise AttributeError(f"FixedwingVecEnv envs have no per-env method {method_name!r} (a batch is stepped and "
                                 "reset as a whole; use reset()/step() or the *_tensor lane)")
        out = fn(*args, **kwargs)
        return [out for _ in self._indices(indices)]

    def env_is_wrapped(self, wrapper_class, indices=None) -> list[bool]:
        return [False for _ in self._indices(indices)]

    def get_images(self):
        raise NotImplementedError("rendered frames are out of scope (DESIGN.md section 9)")

    # ------------------------------------------------------------------ device-tensor lane (B1')
    def _tensors(self):
        if self._t is None:
            import torch
            dev = torch.device("cuda", self.device_index)
            D = max(self.obs_dim, 1)
            self._t = dict(
                obs=torch.zeros((self.num_envs, D), dtype=torch.float32, device=dev),
                rew=torch.zeros(self.num_envs, dtype=torch.float32, device=dev),
                flags=torch.zeros(self.num_envs, dtype=torch.uint8, device=dev),
                term=torch.zeros((self.num_envs, D), dtype=torch.float32, device=dev),
                tidx=torch.zeros(self.num_envs, dtype=torch.uint8, device=dev),
            )
        return self._t

    @staticmethod
    def _stream() -> int:
        import torch
        return int(torch.cuda.current_stream().cuda_stream)

    def reset_tensor(self, mask=None):
        t = self._tensors()
        mp = None if mask is None else C.c_void_p(mask.data_ptr())
        _lib.check(self.lib.fw_reset(self._h, mp, C.c_void_p(t["obs"].data_ptr()), C.c_void_p(self._stream())))
        return t["obs"][:, : self.obs_dim]

    def step_tensor(self, actions, want_terminal_obs: bool = False):
        """actions: CUDA float32 [N,4] contiguous.  Returns views of persistent CUDA tensors
        (obs, reward, flags[, terminal_obs]); valid until the next call.  No host sync."""
        t = self._tensors()
        if actions.dtype is not t["obs"].dtype or not actions.is_contiguous() or tuple(actions.shape) != (self.num_envs, self.act_dim):
            raise ValueError(f"actions must be a contiguous CUDA float32 tensor of shape (num_envs, {self.act_dim})")
        _lib.check(self.lib.fw_step(
            self._h, C.c_void_p(actions.data_ptr()), C.c_void_p(t["obs"].data_ptr()) if self.obs_dim else None,
            C.c_void_p(t["rew"].data_ptr()), C.c_void_p(t["flags"].data_ptr()),
            C.c_void_p(t["term"].data_ptr()) if (want_terminal_obs and self.obs_dim) else None,
            C.c_void_p(self._stream())))
        if want_terminal_obs:
            return t["obs"][:, : self.obs_dim], t["rew"], t["flags"], t["term"][:, : self.obs_dim]
        return t["obs"][:, : self.obs_dim], t["rew"], t["flags"]

    def targets_reached_tensor(self):
        """Device lane: ``info["num_targets_reached"]`` of the last ``step_tensor`` for every env (uint8 CUDA tensor,
        pre-reset values; an asynchronous copy on the current stream)."""
        t = self._tensors()
        _lib.check(self.lib.fw_targets_reached(self._h, C.c_void_p(t["tidx"].data_ptr()), C.c_void_p(self._stream())))
        return t["tidx"]

    def set_obs_accumulator(self, acc) -> None:
        """Device float64 tensor of FW_OBS_ACC_SLOTS x 2 x obs_dim zeros (or None): the step kernels add the column sums and
        sums of squares of the observations they return to it (``fw_set_obs_accumulator``); ``ppo_moments_finalize`` folds
        them into the running statistics.  Applies to steps enqueued from now on."""
        if acc is not None and (acc.numel() != 64 * 2 * self.obs_dim or str(acc.dtype) != "torch.float64" or not acc.is_cuda):
            raise ValueError("accumulator must be a CUDA float64 tensor of 64 * 2 * obs_dim elements")
        _lib.check(self.lib.fw_set_obs_accumulator(self._h, C.c_void_p(acc.data_ptr()) if acc is not None else None))

    def render_layers(self, env_index: int = 0, width: int | None = None, height: int | None = None) -> dict:
        """Debug / evaluation frame of one env (``fw_render``): ``rgba`` uint8 [H,W,4], ``seg`` int32 [H,W] (-1 sky, 0 ground,
        1 duck, 2+k obstacle k, 64+t waypoint t) and ``depth`` float32 [H,W] (OpenGL depth-buffer values, what pybullet's
        ``getCameraImage`` returns) as NumPy arrays; default size = the task camera's resolution.  The scene is the analytic
        one the vision features are computed from, seen through the task's own camera (DESIGN.md section 4.8)."""
        import torch
        W = int(width or self.cfg.cam_res); H = int(height or self.cfg.cam_res)
        dev = torch.device("cuda", self.device_index)
        rgba = torch.empty((H, W, 4), dtype=torch.uint8, device=dev)
        seg = torch.empty((H, W), dtype=torch.int32, device=dev)
        depth = torch.empty((H, W), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            st = torch.cuda.current_stream().cuda_stream
            _lib.check(self.lib.fw_render(self._h, int(env_index), W, H, C.c_void_p(rgba.data_ptr()), C.c_void_p(seg.data_ptr()),
                                          C.c_void_p(depth.data_ptr()), C.c_void_p(st)))
        return dict(rgba=rgba.cpu().numpy(), seg=seg.cpu().numpy(), depth=depth.cpu().numpy())

    def render(self, mode: str = "rgb_array", env_index: int = 0, width: int | None = None, height: int | None = None):
        """``FixedwingBaseEnv.render`` [REF fixedwing_base_env.py:350-369]: the RGBA frame (uint8 [H,W,4]) of one env."""
        if mode != "rgb_array":
            raise ValueError("only mode='rgb_array' is available (there is no window to draw into)")
        return self.render_layers(env_index, width, height)["rgba"]

    def get_images(self):
        """stable_baselines3 ``VecEnv.get_images``: one frame per env -- meant for a handful of envs."""
        return [self.render(env_index=i) for i in range(self.num_envs)]

    def fault_count(self) -> int:
        """Envs force-reset so far because their state went non-finite (FLAG_FAULT)."""
        out = C.c_int64(0)
        _lib.check(self.lib.fw_fault_count(self._h, C.byref(out)))
        return int(out.value)

    def spare_stats(self) -> dict[str, int]:
        """Camera tasks: in-step auto-resets served from a pre-warmed spare episode / inline (fw_spare_stats)."""
        out = (C.c_int64 * 2)()
        _lib.check(self.lib.fw_spare_stats(self._h, out))
        return {"from_spare": int(out[0]), "inline": int(out[1])}

    def step_random(self, n_steps: int = 1, with_outputs: bool = False):
        """Random-action workload (BASELINE config 2): actions drawn in-kernel, one launch per env-step."""
        t = self._tensors() if with_outputs else None
        _lib.check(self.lib.fw_step_random(
            self._h, int(n_steps),
            C.c_void_p(t["rew"].data_ptr()) if t else None, C.c_void_p(t["flags"].data_ptr()) if t else None,
            C.c_void_p(self._stream())))
        return (t["rew"], t["flags"]) if t else None

    @staticmethod
    def rollout_random(envs: "Sequence[FixedwingVecEnv]", n_launches: int, steps_per_launch: int = 1,
                       use_graph: bool = True) -> None:
        """Round-robin random-action sweep over several env batches of one device (see fw_rollout_random)."""
        arr = (C.c_void_p * len(envs))(*[e._h for e in envs])
        _lib.check(envs[0].lib.fw_rollout_random(arr, len(envs), int(n_launches), int(steps_per_launch),
                                                 1 if use_graph else 0, C.c_void_p(envs[0]._stream())))

    # ------------------------------------------------------------------ parity injection / inspection
    def get_state(self) -> dict[str, np.ndarray]:
        n, T = self.num_envs, max(self.cfg.num_targets, 1)
        out = {}
        s = _lib.FwStateHostC()
        for k, (dt, w) in _STATE_FIELDS.items():
            if (k in _OBJLOCK_FIELDS and self.cfg.task not in (2, 4)) or (k in _DUCK_FIELDS and self.cfg.task != 4):
                continue
            shape = self._state_shape(k, w, n, T)
            out[k] = np.zeros(shape, dtype=dt)
            setattr(s, k, out[k].ctypes.data_as(C.c_void_p).value)
        _lib.check(self.lib.fw_get_state(self._h, C.byref(s)))
        return out

    @staticmethod
    def _state_shape(k, w, n, T):
        if k == "targets":
            return (n, T, 3)
        if isinstance(w, tuple):
            return (n, *w)
        return (n,) if w == 0 else (n, w)

    def set_state(self, state: dict[str, np.ndarray]) -> None:
        n, T = self.num_envs, max(self.cfg.num_targets, 1)
        s = _lib.FwStateHostC()
        keep = []
        for k, v in state.items():
            if k not in _STATE_FIELDS:
                raise KeyError(f"unknown state field {k!r}")
            dt, w = _STATE_FIELDS[k]
            if (k in _OBJLOCK_FIELDS and self.cfg.task not in (2, 4)) or (k in _DUCK_FIELDS and self.cfg.task != 4):
                continue
            shape = self._state_shape(k, w, n, T)
            a = np.ascontiguousarray(np.asarray(v).astype(dt)).reshape(shape)
            keep.append(a)
            setattr(s, k, a.ctypes.data_as(C.c_void_p).value)
        _lib.check(self.lib.fw_set_state(self._h, C.byref(s)))

    def episode_stats(self) -> dict[str, float]:
        out = (C.c_double * 8)()
        _lib.check(self.lib.fw_episode_stats(self._h, out))
        names = ["episodes", "return_sum", "length_sum", "targets_reached_sum", "collisions", "out_of_bounds",
                 "completed", "strikes"]
        return dict(zip(names, list(out)))

    @property
    def launch_count(self) -> int:
        return int(self.lib.fw_launch_count(self._h))
