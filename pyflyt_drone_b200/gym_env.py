"""Single-environment gymnasium-style view (SURVEY section 8 b, seam B2).

Mirrors what the reference's scripts obtain from ``gym.make("PyFlyt/Fixedwing-Waypoints-v3", ...)``
(train/train_Fixedwing_Waypoints_v3.py:100-110, eval/eval_waypoints.py:47-55) or from
``FixedwingWaypointObjLockEnv(...)`` (train/train_Fixedwing_Waypoints_ObjLock.py:119-165):
``reset(seed=, options=) -> (obs_dict, info)``, ``step(a) -> (obs_dict, reward, terminated, truncated, info)``,
``observation_space`` Dict{attitude, target_deltas[, duck_vision]}, ``.unwrapped.waypoints.targets`` (probed by
FlattenWaypointEnv, envs/flatten_waypoint_env.py:33-38), ``.env`` exposing the wind hook
(envs/utils.py:133-138), ``.np_random``, ``.state``, ``close()``.

It is a thin view over a one-env device batch: all arithmetic still happens in libfwsim.so.  Use it for
evaluation / debugging; training goes through FixedwingVecEnv.
"""
from __future__ import annotations

from typing import Any

import numpy as np

from .compat import spaces
from .config import (EnvConfig, FLAG_COLLISION, FLAG_COMPLETE, FLAG_OOB, FLAG_STRIKE, FLAG_TERM, FLAG_TRUNC, make_config,
                     _wind_fields)
from .vec_env import FixedwingVecEnv


def _field_of(wind_config: dict | None):
    """The WindField of a wind_config dict in mode "field" (None otherwise); _wind_fields validates the dict."""
    if wind_config and wind_config.get("enabled", False) and str(wind_config.get("mode", "")).lower() == "field":
        return wind_config["field"]
    return None


def _quat_to_mat(q: np.ndarray) -> np.ndarray:
    x, y, z, w = (float(v) for v in q)
    s = 2.0 / (x * x + y * y + z * z + w * w)
    return np.array([[1 - s * (y * y + z * z), s * (x * y - w * z), s * (x * z + w * y)],
                     [s * (x * y + w * z), 1 - s * (x * x + z * z), s * (y * z - w * x)],
                     [s * (x * z - w * y), s * (y * z + w * x), 1 - s * (x * x + y * y)]])


class _Waypoints:
    """The slice of PyFlyt's WaypointHandler the reference touches."""

    def __init__(self, owner: "FixedwingWaypointsEnv"):
        self._o = owner

    @property
    def targets(self) -> np.ndarray:
        st = self._o._state()
        idx = int(st["target_idx"][0])
        return st["targets"][0, idx:self._o.cfg.num_targets].astype(np.float64)

    @property
    def num_targets_reached(self) -> int:
        return int(self._o._state()["target_idx"][0])

    @property
    def all_targets_reached(self) -> bool:
        return self.num_targets_reached >= self._o.cfg.num_targets

    @property
    def distance_to_next_target(self) -> float:
        return float(self._o._state()["new_dist"][0])


class _AviaryView:
    """Stand-in for the PyFlyt Aviary handle (``env.env``): only the wind hook survives the move to the GPU."""

    def __init__(self, owner: "FixedwingWaypointsEnv"):
        self._o = owner

    def register_wind_field_function(self, wind_field, *, origin=None, spacing=None, shape=None, n_slices: int = 1,
                                     t_step: float | None = None) -> None:
        """PyFlyt's hook for a custom wind ``f(time_s, positions[n, 3]) -> [n, 3]``.  A Python closure cannot run inside
        the CUDA step: with the lattice keywords the function is sampled once (``WindField.from_function``) and the
        gridded field is flown from the next ``reset()`` on, interpolated at every lifting surface."""
        if origin is None or spacing is None or shape is None:
            raise NotImplementedError(
                "Python wind closures cannot run inside the CUDA step: pass the sampling lattice, "
                "register_wind_field_function(f, origin=(x, y, z), spacing=metres, shape=(nx, ny, nz)[, n_slices=, "
                "t_step=]), and f is sampled once into a gridded field (pyflyt_drone_b200.wind.WindField); or pass the "
                "wind_config dict the reference feeds to _register_wind_field (envs/utils.py:141-205) to the env or to "
                "env.set_wind_config(dict).")
        from .wind import WindField
        field = WindField.from_function(wind_field, origin=origin, spacing=spacing, shape=shape, n_slices=n_slices,
                                        t_step=t_step)
        self._o.set_wind_config({"enabled": True, "mode": "field", "field": field})

    def state(self, index: int = 0) -> np.ndarray:
        return self._o._raw_state()

    def aux_state(self, index: int = 0) -> np.ndarray:
        return self._o._state()["act"][0].astype(np.float64)

    def disconnect(self) -> None:
        pass


class FixedwingWaypointsEnv:
    """``PyFlyt/Fixedwing-Waypoints-v3`` (task="waypoints") or ``FixedwingWaypointObjLockEnv`` (task="objlock")."""

    metadata = {"render_modes": ["rgb_array"], "render_fps": 30}

    def __init__(self, sparse_reward: bool = False, num_targets: int = 4, goal_reach_distance: float = 2.0,
                 flight_mode: int = 0, flight_dome_size: float = 100.0, max_duration_seconds: float = 120.0,
                 angle_representation: str = "quaternion", agent_hz: int = 30, render_mode=None,
                 wind_config: dict | None = None, task: str = "waypoints", device: int = 0, seed: int = 0, **objlock_kwargs):
        if 120 % agent_hz != 0:
            lowest = int(120 / (int(120 / agent_hz) + 1))
            highest = int(120 / int(120 / agent_hz))
            raise ValueError(f"`agent_hz` must be round denominator of 120, try {lowest} or {highest}.")
        if angle_representation not in ("euler", "quaternion"):
            raise ValueError(f"angle_representation must be either `euler` or `quaternion`, not {angle_representation}")
        if flight_mode != 0:
            raise ValueError("only flight_mode 0 (roll, pitch, yaw, thrust) is implemented")
        if render_mode not in (None, "rgb_array"):
            raise ValueError("only render_mode None or 'rgb_array' is available (no window to draw into)")
        self.render_mode = render_mode
        self.render_resolution = (480, 480)                          # fixedwing_base_env.py:96 default
        preset = {"waypoints": "waypoints_v3", "objlock": "waypoint_objlock"}[task]
        over = dict(sparse_reward=int(bool(sparse_reward)), num_targets=int(num_targets), goal_reach=float(goal_reach_distance),
                    dome=float(flight_dome_size), spawn_size=float(flight_dome_size),
                    max_steps=int(agent_hz * max_duration_seconds), inner_per_step=int(120 / agent_hz),
                    angle_repr=0 if angle_representation == "euler" else 1, context_len=min(int(num_targets) + 1, 4))
        names = {"num_obstacles": "num_obstacles", "obstacle_radius": "obst_radius", "obstacle_safe_distance_m": "obst_safe",
                 "obstacle_avoid_reward_scale": "obst_scale", "obstacle_avoid_max_penalty": "obst_max_pen",
                 "duck_lock_hold_steps": "lock_hold_steps", "duck_strike_distance_m": "strike_dist",
                 "duck_strike_reward": "strike_reward", "duck_lock_step_reward": "lock_step_reward",
                 "duck_approach_reward_scale": "approach_scale", "duck_switch_min_consecutive_seen": "switch_min_seen",
                 "duck_switch_min_area": "switch_min_area"}
        for k, v in objlock_kwargs.items():
            if k == "obstacle_height_range":
                over["obst_h_lo"], over["obst_h_hi"] = float(min(v)), float(max(v))
            elif k == "duck_camera_capture_interval_steps":
                over["cam_interval_substeps"] = 2 * int(v)
            elif k in names:
                over[names[k]] = v
            else:
                raise TypeError(f"unexpected keyword {k!r}")
        self.cfg: EnvConfig = make_config(preset, wind=wind_config, **over) if wind_config is not None or task == "waypoints" \
            else make_config(preset, **over)
        if task == "waypoints" and wind_config is not None:
            self.cfg = self.cfg.replace(**_wind_fields(wind_config, "env"))
        self._device, self._seed0 = device, int(seed)
        self._wind_field = _field_of(wind_config)
        self._vec = FixedwingVecEnv(1, config=self.cfg, device=device, seed=self._seed0, wind_field=self._wind_field)
        att = (12 if self.cfg.angle_repr == 0 else 13) + 4 + 6
        self._att = att
        self.attitude_space = spaces.Box(low=-np.inf, high=np.inf, shape=(att - 10,), dtype=np.float64)
        self.auxiliary_space = spaces.Box(low=-np.inf, high=np.inf, shape=(6,), dtype=np.float64)
        self.action_space = spaces.Box(low=-np.ones(4), high=np.ones(4), dtype=np.float64)
        self.combined_space = spaces.Box(low=-np.inf, high=np.inf, shape=(att,), dtype=np.float64)
        sp = {"attitude": self.combined_space,
              "target_deltas": spaces.Sequence(spaces.Box(low=-2 * flight_dome_size, high=2 * flight_dome_size, shape=(3,),
                                                          dtype=np.float64), stack=True)}
        if task == "objlock":
            sp["duck_vision"] = spaces.Box(low=-np.inf, high=np.inf, shape=(9,), dtype=np.float32)
        self.observation_space = spaces.Dict(sp)
        self.task = task
        self.waypoints = _Waypoints(self)
        self.env = _AviaryView(self)
        self.np_random = np.random.default_rng(self._seed0)
        self.state: dict | None = None
        self.info: dict = {}
        self.termination = self.truncation = False
        self.step_count = 0
        self.action = np.zeros(4)
        self._needs_reset = True
        self._cache = None

    # gymnasium.Env conveniences
    @property
    def unwrapped(self):
        return self

    def _state(self) -> dict:
        if self._cache is None:
            self._cache = self._vec.get_state()
        return self._cache

    def _raw_state(self) -> np.ndarray:
        st = self._state()
        R = _quat_to_mat(st["quat"][0])
        from math import asin, atan2
        x, y, z, w = (float(v) for v in st["quat"][0])
        sarg = -2.0 * (x * z - w * y)
        if sarg <= -0.99999:
            rpy = (0.0, -np.pi / 2, 2 * atan2(x, -y))
        elif sarg >= 0.99999:
            rpy = (0.0, np.pi / 2, 2 * atan2(-x, y))
        else:
            rpy = (atan2(2 * (y * z + w * x), w * w - x * x - y * y + z * z), asin(sarg),
                   atan2(2 * (x * y + w * z), w * w + x * x - y * y - z * z))
        return np.stack([R.T @ st["omega"][0], np.array(rpy), R.T @ st["vel"][0], st["pos"][0].astype(np.float64)])

    def _obs_dict(self, flat: np.ndarray, terminal: bool) -> dict:
        """Dict observation.  The flattened row carries the attitude; every remaining target delta (not only the
        first context rows) is recomputed on the host from the state when it is still the live state."""
        att = flat[: self._att].astype(np.float64)
        rows = flat[self._att:].reshape(-1, 3).astype(np.float64)
        if not terminal:
            st = self._state()
            R = _quat_to_mat(st["quat"][0])
            idx = int(st["target_idx"][0])
            tg = st["targets"][0, idx:self.cfg.num_targets].astype(np.float64)
            rows = (tg - st["pos"][0]) @ R if len(tg) else np.zeros((0, 3))
            if self.task == "objlock":
                rows = np.vstack([rows, ((st["duck"][0] - st["pos"][0]) @ R).reshape(1, 3)])
        out = {"attitude": att, "target_deltas": rows}
        if self.task == "objlock":
            st = self._state()
            f, i = st["ol_f"][0], st["ol_i"][0]
            vis = 1.0 if (i[3] and i[4]) else 0.0
            out["duck_vision"] = np.array([vis, f[0], f[1], f[2], f[3], i[7] / 60.0, f[8], f[9], f[10]], dtype=np.float32)
        return out

    def set_wind_config(self, wind_config: dict | None) -> None:
        """What WindOnResetWrapper does for the reference: takes effect from the next reset()."""
        self.cfg = self.cfg.replace(**_wind_fields(wind_config, "wrapper"))
        self._wind_field = _field_of(wind_config)
        self._vec.close()
        self._vec = FixedwingVecEnv(1, config=self.cfg, device=self._device, seed=self._seed0, wind_field=self._wind_field)
        self._needs_reset = True
        self._auto_reset_done = False

    def reset(self, *, seed: int | None = None, options: dict | None = None) -> tuple[dict, dict]:
        if seed is not None:
            self._seed0 = int(seed)
            self.np_random = np.random.default_rng(self._seed0)
            self._vec.seed(self._seed0)                  # always rebuilds: reset(seed=s) is reproducible
            self._auto_reset_done = False
        # after a finished episode the device batch has already opened the next one (SubprocVecEnv semantics): hand out
        # its first observation instead of discarding a whole episode (and, for ObjLock, its warm-up and camera frame)
        flat = self._vec.observe()[0] if getattr(self, "_auto_reset_done", False) else self._vec.reset()[0]
        self._auto_reset_done = False
        self._cache = None
        self.step_count, self.termination, self.truncation = 0, False, False
        self.action = np.zeros(4)
        self.info = {"out_of_bounds": False, "collision": False, "env_complete": False, "num_targets_reached": 0}
        if self.task == "objlock":
            self.info["duck_strike"] = False
        self.state = self._obs_dict(flat, terminal=False)
        self._needs_reset = False
        return self.state, self.info

    def step(self, action) -> tuple[dict, float, bool, bool, dict]:
        if self._needs_reset:
            raise RuntimeError("call reset() before step() (the previous episode has ended)")
        a = np.asarray(action, dtype=np.float32).reshape(1, 4)
        self.action = a[0].astype(np.float64)
        pre_idx = self.waypoints.num_targets_reached
        obs, rew, flags, term = self._vec.step_arrays(a, want_terminal_obs=True)
        self._cache = None
        f = int(flags[0])
        self.termination, self.truncation = bool(f & FLAG_TERM), bool(f & FLAG_TRUNC)
        done = self.termination or self.truncation
        self.step_count += 1
        self.info["collision"] = self.info["collision"] or bool(f & FLAG_COLLISION)
        self.info["out_of_bounds"] = self.info["out_of_bounds"] or bool(f & FLAG_OOB)
        self.info["env_complete"] = bool(f & FLAG_COMPLETE)
        if self.task == "objlock":
            self.info["duck_strike"] = bool(f & FLAG_STRIKE)
        if done:
            # the device batch has already auto-reset (SubprocVecEnv semantics); hand back the terminal observation
            self.state = self._obs_dict(term[0].copy(), terminal=True)
            self.info["num_targets_reached"] = int(self._vec.last_targets_reached[0])
            self._needs_reset = True
            self._auto_reset_done = True
        else:
            self.info["num_targets_reached"] = max(pre_idx, self.waypoints.num_targets_reached)
            self.state = self._obs_dict(obs[0].copy(), terminal=False)
        return self.state, float(rew[0]), self.termination, self.truncation, self.info

    def close(self) -> None:
        self._vec.close()

    def render(self) -> np.ndarray:
        """FixedwingBaseEnv.render (fixedwing_base_env.py:350-369): RGBA uint8 [H,W,4] at render_resolution, through the
        aircraft's camera; the analytic scene (vec_env.render_layers), not pybullet's meshes."""
        if self.render_mode is None:
            raise ValueError("Please set `render_mode='human'` or `render_mode='rgb_array'` in init to use this function.")
        return self._vec.render(env_index=0, width=self.render_resolution[1], height=self.render_resolution[0])


class FixedwingLowLevelEnv:
    """Single-env gymnasium view of the low-level tracking task, the interface of
    envs/fixedwing_envs/fixedwing_lowlevel_env.py:10-163: 6-channel action [left_ail, right_ail, hstab, vstab, flap,
    thrust] in [-1, 1], 21-float observation, ``info["target"] = [psi_ref, h_ref, V_ref]``."""

    metadata = {"render_modes": [], "name": "fixedwing_lowlevel_env"}

    def __init__(self, render_mode=None, wind_config: dict | None = None, device: int = 0, seed: int = 0):
        if render_mode is not None:
            raise ValueError("rendering is out of scope for the batched simulator")
        self.cfg: EnvConfig = make_config("lowlevel", wind=wind_config)
        self._vec = FixedwingVecEnv(1, config=self.cfg, device=device, seed=int(seed), wind_field=_field_of(wind_config))
        self.observation_space = spaces.Box(low=-np.inf, high=np.inf, shape=(21,), dtype=np.float64)
        self.action_space = spaces.Box(low=-1.0, high=1.0, shape=(6,), dtype=np.float64)
        self.prev_action = np.zeros(6)
        self.target = np.zeros(3)
        self._needs_reset = True
        self.unwrapped = self

    def reset(self, *, seed: int | None = None, options: dict | None = None):
        if seed is not None:
            self._vec.seed(int(seed))
        obs = self._vec.reset()[0].astype(np.float64)
        self.prev_action = np.zeros(6)
        self.target = obs[18:21].copy()
        self._needs_reset = False
        return obs, {"target": self.target.copy()}

    def step(self, action):
        if self._needs_reset:
            raise RuntimeError("call reset() before step() (the previous episode has ended)")
        a = np.asarray(action, dtype=np.float32).reshape(1, 6)
        self.prev_action = a[0].astype(np.float64)
        obs, rew, flags, term = self._vec.step_arrays(a, want_terminal_obs=True)
        f = int(flags[0])
        terminated, truncated = bool(f & FLAG_TERM), bool(f & FLAG_TRUNC)
        if terminated or truncated:          # the device batch has already auto-reset: hand back the terminal observation
            self._needs_reset = True
            out = term[0].astype(np.float64)
        else:
            out = obs[0].astype(np.float64)
        return out, float(rew[0]), terminated, truncated, {"target": self.target.copy()}

    def close(self) -> None:
        self._vec.close()


class FixedwingObjLockEnv:
    """Single-env gymnasium view of the duck-only lock/strike task, the interface of
    envs/fixedwing_objlock_env.py:17-175: same keyword names and defaults as the reference's constructor, Dict
    observation {attitude, target_vector(3), duck_vision(9*history [+4])}, ``info`` keys ``duck_strike`` /
    ``env_complete`` / ``is_success`` / ``collision`` / ``out_of_bounds``.  The camera is the analytic stand-in
    (DESIGN.md): ``camera_FOV_degrees`` must be 90, ``duck_urdf_path`` / ``use_egl`` are accepted and ignored,
    ``render_mode="rgb_array"`` selects the capture resolution the way the reference does (:213-218) and enables
    ``render()`` (frames of the analytic scene, see FixedwingVecEnv.render_layers)."""

    metadata = {"render_modes": ["rgb_array"], "render_fps": 30}

    def __init__(self, sparse_reward: bool = False, flight_mode: int = 0, flight_dome_size: float = 100.0,
                 max_duration_seconds: float = 120.0, angle_representation: str = "quaternion", agent_hz: int = 30,
                 render_mode=None, render_resolution=(480, 480), duck_urdf_path=None, use_egl: bool = False,
                 camera_profile: str = "cockpit_fpv", camera_position_offset=None, camera_angle_degrees=None,
                 camera_FOV_degrees=None, camera_resolution=None,
                 num_obstacles: int = 5, obstacle_radius: float = 2.0, obstacle_height_range=(10.0, 30.0),
                 obstacle_safe_distance_m: float = 20.0, obstacle_avoid_reward_scale: float = 1.0,
                 obstacle_avoid_max_penalty: float = 2.0,
                 duck_camera_capture_interval_steps: int = 12, duck_lock_hold_steps: int = 10,
                 duck_strike_distance_m: float = 2.0, duck_strike_reward: float = 200.0,
                 duck_lock_step_reward: float = 0.1, duck_approach_reward_scale: float = 0.05,
                 duck_global_scaling: float = 20.0, duck_vision_history_len: int = 3, duck_vision_use_deltas: bool = True,
                 duck_distance_reward_scale: float = 1.0, duck_lock_center_radius: float = 0.55,
                 duck_centering_reward_scale: float = 3, duck_visible_step_reward: float = 2,
                 duck_area_reward_scale: float = 5.0, duck_lock_decay_steps: int = 1, duck_lock_lost_penalty: float = 0.5,
                 duck_approach_reward_clip_m: float = 2.0, wind_config: dict | None = None,
                 device: int = 0, seed: int = 0):
        if 120 % agent_hz != 0:
            lowest = int(120 / (int(120 / agent_hz) + 1))
            highest = int(120 / int(120 / agent_hz))
            raise ValueError(f"`agent_hz` must be round denominator of 120, try {lowest} or {highest}.")
        if angle_representation not in ("euler", "quaternion"):
            raise ValueError(f"angle_representation must be either `euler` or `quaternion`, not {angle_representation}")
        if flight_mode != 0:
            raise ValueError("only flight_mode 0 (roll, pitch, yaw, thrust) is implemented")
        if render_mode not in (None, "rgb_array"):
            raise ValueError("only render_mode None or 'rgb_array' is available (no window to draw into)")
        self.render_mode = render_mode
        if camera_FOV_degrees is not None and int(camera_FOV_degrees) != 90:
            raise ValueError("the analytic camera is built for the reference's 90 degree field of view")
        if camera_profile == "cockpit_fpv":                          # fixedwing_objlock_env.py:184-192,226-229
            offset, angle, mode = [0.8, 0.0, 0.12], -5, 1
        else:                                                        # "chase", and PyFlyt's own default camera
            offset, angle, mode = [-3.0, 0.0, 1.0], 0, 0
        if camera_position_offset is not None:
            offset = [float(x) for x in camera_position_offset]
        if camera_angle_degrees is not None:
            angle = int(camera_angle_degrees)
        res = camera_resolution if camera_resolution is not None else (render_resolution if render_mode is not None else (128, 128))
        hlo, hhi = float(min(obstacle_height_range)), float(max(obstacle_height_range))
        over = dict(
            sparse_reward=int(bool(sparse_reward)), dome=float(flight_dome_size), spawn_size=float(flight_dome_size),
            max_steps=int(agent_hz * max_duration_seconds), inner_per_step=int(120 / agent_hz),
            angle_repr=0 if angle_representation == "euler" else 1,
            cam_mode=mode, cam_offset=offset, cam_tilt_deg=float(angle), cam_res=int(res[1]),
            num_obstacles=int(num_obstacles), obst_radius=float(obstacle_radius), obst_h_lo=hlo, obst_h_hi=hhi,
            obst_safe=float(obstacle_safe_distance_m), obst_scale=float(obstacle_avoid_reward_scale),
            obst_max_pen=float(obstacle_avoid_max_penalty),
            cam_interval_substeps=2 * int(duck_camera_capture_interval_steps), lock_hold_steps=int(duck_lock_hold_steps),
            strike_dist=float(duck_strike_distance_m), strike_reward=float(duck_strike_reward),
            lock_step_reward=float(duck_lock_step_reward), approach_scale=float(duck_approach_reward_scale),
            duck_radius=0.05 * float(duck_global_scaling), vision_hist_len=int(max(1, duck_vision_history_len)),
            vision_use_deltas=int(bool(duck_vision_use_deltas)), duck_dist_scale=float(duck_distance_reward_scale),
            lock_center_radius=float(duck_lock_center_radius), centering_scale=float(duck_centering_reward_scale),
            visible_step_reward=float(duck_visible_step_reward), area_reward_scale=float(duck_area_reward_scale),
            lock_decay_steps=int(max(1, duck_lock_decay_steps)), lock_lost_penalty=float(duck_lock_lost_penalty),
            approach_clip=float(max(0.0, duck_approach_reward_clip_m)))
        self.cfg: EnvConfig = make_config("objlock_duck", wind=wind_config if wind_config is not None else {"enabled": False},
                                          **over)
        self._device, self._seed0 = device, int(seed)
        self._vec = FixedwingVecEnv(1, config=self.cfg, device=device, seed=self._seed0, wind_field=_field_of(wind_config))
        att = (12 if self.cfg.angle_repr == 0 else 13) + 4 + 6
        self._att = att
        self.combined_space = spaces.Box(low=-np.inf, high=np.inf, shape=(att,), dtype=np.float64)
        self.action_space = spaces.Box(low=-np.ones(4), high=np.ones(4), dtype=np.float64)
        nv = 9 * self.cfg.vision_hist_len + (4 if self.cfg.vision_use_deltas else 0)
        self.observation_space = spaces.Dict({
            "attitude": self.combined_space,
            "target_vector": spaces.Box(low=-np.inf, high=np.inf, shape=(3,), dtype=np.float64),
            "duck_vision": spaces.Box(low=-np.inf, high=np.inf, shape=(nv,), dtype=np.float32)})
        self.sparse_reward = bool(sparse_reward)
        self.np_random = np.random.default_rng(self._seed0)
        self.state: dict | None = None
        self.info: dict = {}
        self.termination = self.truncation = False
        self.step_count = 0
        self.action = np.zeros(4)
        self._needs_reset = True

    @property
    def unwrapped(self):
        return self

    @property
    def duck_pos(self) -> np.ndarray:
        return self._vec.get_state()["duck"][0].astype(np.float64)

    def _obs_dict(self, flat: np.ndarray) -> dict:
        a = self._att
        return {"attitude": flat[:a].astype(np.float64), "target_vector": flat[a:a + 3].astype(np.float64),
                "duck_vision": flat[a + 3:].astype(np.float32)}

    def reset(self, *, seed: int | None = None, options: dict | None = None) -> tuple[dict, dict]:
        if seed is not None:
            self._seed0 = int(seed)
            self.np_random = np.random.default_rng(self._seed0)
            self._vec.seed(self._seed0)
        flat = self._vec.reset()[0]
        self.step_count, self.termination, self.truncation = 0, False, False
        self.action = np.zeros(4)
        self.info = {"out_of_bounds": False, "collision": False, "env_complete": False, "duck_strike": False,
                     "is_success": False}
        self.state = self._obs_dict(flat)
        self._needs_reset = False
        return self.state, self.info

    def step(self, action) -> tuple[dict, float, bool, bool, dict]:
        if self._needs_reset:
            raise RuntimeError("call reset() before step() (the previous episode has ended)")
        a = np.asarray(action, dtype=np.float32).reshape(1, 4)
        self.action = a[0].astype(np.float64)
        obs, rew, flags, term = self._vec.step_arrays(a, want_terminal_obs=True)
        f = int(flags[0])
        self.termination, self.truncation = bool(f & FLAG_TERM), bool(f & FLAG_TRUNC)
        self.step_count += 1
        self.info["collision"] = self.info["collision"] or bool(f & FLAG_COLLISION)
        self.info["out_of_bounds"] = self.info["out_of_bounds"] or bool(f & FLAG_OOB)
        self.info["env_complete"] = bool(f & FLAG_COMPLETE)
        self.info["duck_strike"] = self.info["is_success"] = bool(f & FLAG_STRIKE)
        if self.termination or self.truncation:      # the device batch has already auto-reset: hand back the terminal observation
            self.state = self._obs_dict(term[0].copy())
            self._needs_reset = True
        else:
            self.state = self._obs_dict(obs[0].copy())
        return self.state, float(rew[0]), self.termination, self.truncation, self.info

    def close(self) -> None:
        self._vec.close()

    def render(self) -> np.ndarray:
        """RGBA uint8 [H,W,4] through the task camera at the capture resolution (see FixedwingWaypointsEnv.render)."""
        if self.render_mode is None:
            raise ValueError("Please set `render_mode='human'` or `render_mode='rgb_array'` in init to use this function.")
        return self._vec.render(env_index=0)


class FlattenObjLockEnv:
    """Dict -> Box flattening of FixedwingObjLockEnv, as envs/flatten_objlock_env.py:8-46:
    ``concatenate([attitude, target_vector, duck_vision]).astype(float32)``."""

    def __init__(self, env: FixedwingObjLockEnv):
        self.env = env
        sp = env.observation_space
        self.attitude_shape = sp["attitude"].shape[0]
        self.target_shape = sp["target_vector"].shape[0]
        self.vision_shape = sp["duck_vision"].shape[0]
        self.observation_space = spaces.Box(low=-np.inf, high=np.inf,
                                            shape=(self.attitude_shape + self.target_shape + self.vision_shape,),
                                            dtype=np.float32)
        self.action_space = env.action_space

    @property
    def unwrapped(self):
        return self.env.unwrapped

    def _flatten_obs(self, obs: dict) -> np.ndarray:
        return np.concatenate([obs["attitude"], obs["target_vector"], obs["duck_vision"]], axis=0).astype(np.float32)

    def reset(self, **kwargs):
        obs, info = self.env.reset(**kwargs)
        return self._flatten_obs(obs), info

    def step(self, action):
        obs, reward, term, trunc, info = self.env.step(action)
        return self._flatten_obs(obs), reward, term, trunc, info

    def close(self):
        self.env.close()


class FlattenWaypointEnv:
    """Dict -> Box flattening of a waypoints env, as envs/flatten_waypoint_env.py:14-72 (zero padded)."""

    def __init__(self, env, context_length: int = 2):
        if not hasattr(env.unwrapped, "waypoints") and not hasattr(env, "waypoints"):
            raise AttributeError("Only a waypoints environment can be used with the `FlattenWaypointEnv` wrapper.")
        self.env = env
        self.context_length = int(context_length)
        self.attitude_shape = env.observation_space["attitude"].shape[0]
        self.target_shape = env.observation_space["target_deltas"].feature_space.shape[0]
        self.observation_space = spaces.Box(low=-np.inf, high=np.inf,
                                            shape=(self.attitude_shape + self.target_shape * self.context_length,),
                                            dtype=np.float64)
        self.action_space = env.action_space

    @property
    def unwrapped(self):
        return self.env.unwrapped

    def observation(self, observation: dict) -> np.ndarray:
        targets = np.zeros((self.context_length, self.target_shape), dtype=np.float64)
        src = observation["target_deltas"]
        if src.shape[0] > 0:
            n = min(self.context_length, src.shape[0])
            targets[:n] = src[:n]
        return np.concatenate([observation["attitude"], targets.flatten()])

    def reset(self, **kwargs):
        obs, info = self.env.reset(**kwargs)
        return self.observation(obs), info

    def step(self, action):
        obs, r, term, trunc, info = self.env.step(action)
        return self.observation(obs), r, term, trunc, info

    def close(self):
        self.env.close()


def make(env_id: str, **kwargs) -> Any:
    """``gym.make`` for the ids the reference uses (train_Fixedwing_Waypoints_v3.py:101)."""
    if env_id == "PyFlyt/Fixedwing-Waypoints-v3":
        return FixedwingWaypointsEnv(task="waypoints", **kwargs)
    raise KeyError(f"unknown env id {env_id!r}")
