"""Env/aircraft configuration: one Python dataclass <-> the C struct ``FwConfig`` of include/fwsim.h.

Presets carry the exact numbers of the reference's training scripts:
  * ``waypoints_v3``     train/train_Fixedwing_Waypoints_v3.py:27-55,100-110
  * ``waypoint_objlock`` train/train_Fixedwing_Waypoints_ObjLock.py:35-92
  * ``physics_only``     BASELINE.json configs[1] (dynamics + ground/dome termination, random actions)
"""
from __future__ import annotations

import ctypes as C
import dataclasses
from dataclasses import dataclass, field
from typing import Any

import numpy as np

from . import aircraft

NSURF, MAX_TARGETS, MAX_COL, MAX_OBST = 5, 16, 16, 32

TASK_PHYSICS, TASK_WAYPOINTS, TASK_OBJLOCK, TASK_LOWLEVEL, TASK_DUCK = 0, 1, 2, 3, 4
MAX_HIST = 4

FLAG_TERM, FLAG_TRUNC, FLAG_COLLISION, FLAG_OOB, FLAG_COMPLETE, FLAG_STRIKE, FLAG_FAULT = 1, 2, 4, 8, 16, 32, 64

_D = C.c_double
_I = C.c_int32


class FwConfigC(C.Structure):
    """ctypes mirror of ``struct FwConfig`` (include/fwsim.h) -- field order must match exactly."""
    _fields_ = [
        ("cl_alpha_2d", _D * NSURF), ("chord", _D * NSURF), ("span", _D * NSURF), ("flap_to_chord", _D * NSURF),
        ("eta", _D * NSURF), ("alpha0_base_deg", _D * NSURF), ("stall_p_base_deg", _D * NSURF),
        ("stall_n_base_deg", _D * NSURF), ("cd0", _D * NSURF), ("defl_limit_deg", _D * NSURF), ("surf_tau", _D * NSURF),
        ("lift_unit", (_D * 3) * NSURF), ("fwd_unit", (_D * 3) * NSURF), ("r_surf", (_D * 3) * NSURF),
        ("total_thrust", _D), ("thrust_coef", _D), ("torque_coef", _D), ("noise_ratio", _D), ("motor_tau", _D),
        ("r_motor", _D * 3), ("thrust_unit", _D * 3),
        ("mass", _D), ("com", _D * 3), ("inertia_o", _D * 9),
        ("col_pts", (_D * 3) * MAX_COL),
        ("contact_margin", _D),
        ("dt", _D), ("gravity", _D), ("rho", _D), ("max_coord_vel", _D),
        ("ail_left_sign", _D), ("ail_right_sign", _D), ("pitch_sign", _D), ("yaw_sign", _D),
        ("goal_reach", _D), ("dome", _D), ("spawn_size", _D), ("min_height", _D),
        ("start_pos", _D * 3), ("start_vel", _D * 3),
        ("wind_base", _D * 3), ("wind_base_lo", _D * 3), ("wind_base_hi", _D * 3),
        ("gust_amp", _D * 3), ("gust_amp_lo", _D * 3), ("gust_amp_hi", _D * 3),
        ("gust_freq", _D), ("gust_phase", _D),
        ("obst_radius", _D), ("obst_h_lo", _D), ("obst_h_hi", _D), ("obst_safe", _D), ("obst_scale", _D),
        ("obst_max_pen", _D),
        ("strike_dist", _D), ("strike_reward", _D), ("lock_step_reward", _D), ("approach_scale", _D),
        ("switch_min_area", _D),
        ("duck_radius", _D), ("cam_offset", _D * 3), ("cam_near", _D), ("cam_far", _D),
        ("cam_tilt_deg", _D), ("duck_dist_scale", _D), ("lock_center_radius", _D), ("centering_scale", _D),
        ("visible_step_reward", _D), ("area_reward_scale", _D), ("lock_lost_penalty", _D), ("approach_clip", _D),
        ("n_col", _I),
        ("physics_per_control", _I), ("substeps_per_inner", _I), ("inner_per_step", _I), ("warmup_inner", _I),
        ("freestream_3d", _I), ("cd90_degrees", _I),
        ("task", _I), ("num_targets", _I), ("sparse_reward", _I), ("angle_repr", _I), ("max_steps", _I),
        ("context_len", _I),
        ("early_return_on_crash", _I), ("complete_truncates", _I),
        ("wind_mode", _I), ("wind_randomize", _I), ("wind_rand_phase", _I), ("wind_start_substep", _I),
        ("num_obstacles", _I), ("cam_interval_substeps", _I), ("lock_hold_steps", _I), ("switch_min_seen", _I),
        ("cam_res", _I),
        ("force_generic_kernel", _I),
        ("cam_mode", _I), ("vision_hist_len", _I), ("vision_use_deltas", _I), ("lock_decay_steps", _I),
        ("packed_pairs", _I),
    ]


def _z3():
    return [0.0, 0.0, 0.0]


@dataclass
class EnvConfig:
    # ---- aircraft (filled by with_aircraft) ----
    cl_alpha_2d: list = field(default_factory=lambda: [0.0] * NSURF)
    chord: list = field(default_factory=lambda: [0.0] * NSURF)
    span: list = field(default_factory=lambda: [0.0] * NSURF)
    flap_to_chord: list = field(default_factory=lambda: [0.0] * NSURF)
    eta: list = field(default_factory=lambda: [0.0] * NSURF)
    alpha0_base_deg: list = field(default_factory=lambda: [0.0] * NSURF)
    stall_p_base_deg: list = field(default_factory=lambda: [0.0] * NSURF)
    stall_n_base_deg: list = field(default_factory=lambda: [0.0] * NSURF)
    cd0: list = field(default_factory=lambda: [0.0] * NSURF)
    defl_limit_deg: list = field(default_factory=lambda: [0.0] * NSURF)
    surf_tau: list = field(default_factory=lambda: [0.0] * NSURF)
    lift_unit: list = field(default_factory=lambda: [_z3() for _ in range(NSURF)])
    fwd_unit: list = field(default_factory=lambda: [_z3() for _ in range(NSURF)])
    r_surf: list = field(default_factory=lambda: [_z3() for _ in range(NSURF)])
    total_thrust: float = 0.0
    thrust_coef: float = 0.0
    torque_coef: float = 0.0
    noise_ratio: float = 0.0
    motor_tau: float = 0.0
    r_motor: list = field(default_factory=_z3)
    thrust_unit: list = field(default_factory=lambda: [1.0, 0.0, 0.0])
    mass: float = 0.0
    com: list = field(default_factory=_z3)
    inertia_o: list = field(default_factory=lambda: [0.0] * 9)
    col_pts: list = field(default_factory=list)          # list of [x,y,z]
    contact_margin: float = 0.02                         # [UP-RECALL] Bullet contact breaking threshold
    # ---- simulator: PyFlyt Aviary physics 240 Hz / control 120 Hz; env agent_hz 30 ----
    dt: float = 1.0 / 240.0
    gravity: float = 9.81
    rho: float = 1.225
    max_coord_vel: float = 100.0
    physics_per_control: int = 2
    substeps_per_inner: int = 2
    inner_per_step: int = 4                              # env_step_ratio, fixedwing_base_env.py:102
    warmup_inner: int = 10                               # end_reset, fixedwing_base_env.py:254-255
    # ---- upstream conventions not verifiable offline (SURVEY appendix B rank 2) ----
    ail_left_sign: float = 1.0
    ail_right_sign: float = -1.0
    pitch_sign: float = 1.0
    yaw_sign: float = 1.0
    freestream_3d: int = 1
    cd90_degrees: int = 1
    # ---- env ----
    task: int = TASK_WAYPOINTS
    num_targets: int = 4
    goal_reach: float = 2.0
    sparse_reward: int = 0
    angle_repr: int = 1                                  # 0 euler, 1 quaternion (upstream default)
    dome: float = 100.0
    max_steps: int = 3600                                # int(agent_hz * max_duration_seconds)
    context_len: int = 2
    start_pos: list = field(default_factory=lambda: [0.0, 0.0, 10.0])
    start_vel: list = field(default_factory=lambda: [20.0, 0.0, 0.0])
    spawn_size: float = 100.0
    min_height: float = 0.5
    early_return_on_crash: int = 0
    complete_truncates: int = 1
    # ---- wind ----
    wind_mode: int = 0
    wind_randomize: int = 0
    wind_rand_phase: int = 1
    wind_start_substep: int = 0
    wind_base: list = field(default_factory=_z3)
    wind_base_lo: list = field(default_factory=_z3)
    wind_base_hi: list = field(default_factory=_z3)
    gust_amp: list = field(default_factory=_z3)
    gust_amp_lo: list = field(default_factory=_z3)
    gust_amp_hi: list = field(default_factory=_z3)
    gust_freq: float = 0.0
    gust_phase: float = 0.0
    # ---- objlock (defaults of FixedwingWaypointObjLockEnv.__init__, objlock_env.py:42-76) ----
    num_obstacles: int = 5
    cam_interval_substeps: int = 12
    obst_radius: float = 2.0
    obst_h_lo: float = 10.0
    obst_h_hi: float = 30.0
    obst_safe: float = 20.0
    obst_scale: float = 1.0
    obst_max_pen: float = 2.0
    lock_hold_steps: int = 10
    switch_min_seen: int = 2
    strike_dist: float = 2.0
    strike_reward: float = 200.0
    lock_step_reward: float = 0.1
    approach_scale: float = 0.05
    switch_min_area: float = 0.0005
    duck_radius: float = 1.5
    cam_offset: list = field(default_factory=lambda: [-3.0, 0.0, 1.0])
    cam_near: float = 0.1
    cam_far: float = 255.0
    cam_res: int = 128
    cam_mode: int = 0                                    # 0 tracking chase camera, 1 fixed (cockpit) camera tilted by cam_tilt_deg
    # ---- duck-only task (defaults of FixedwingObjLockEnv.__init__, envs/fixedwing_objlock_env.py:37-81) ----
    cam_tilt_deg: float = 0.0                            # camera_angle_degrees; [UP-RECALL] about body +y, positive = nose-down
    duck_dist_scale: float = 1.0
    lock_center_radius: float = 0.55
    centering_scale: float = 3.0
    visible_step_reward: float = 2.0
    area_reward_scale: float = 5.0
    lock_lost_penalty: float = 0.5
    approach_clip: float = 2.0
    vision_hist_len: int = 3
    vision_use_deltas: int = 1
    lock_decay_steps: int = 1
    force_generic_kernel: int = 0                       # testing: run the generic kernels even for the standard layout
    packed_pairs: int = 0                               # 1: two envs per thread on the packed fp32x2 path (csrc/fw_pack.cuh; opt-in)

    # ------------------------------------------------------------------
    @property
    def obs_dim(self) -> int:
        if self.task == TASK_PHYSICS:
            return 0
        if self.task == TASK_LOWLEVEL:
            return 21
        att = (12 if self.angle_repr == 0 else 13) + 4 + 6
        if self.task == TASK_DUCK:                        # flatten_objlock_env.py:20-31
            return att + 3 + 9 * self.vision_hist_len + (4 if self.vision_use_deltas else 0)
        return att + 3 * self.context_len

    @property
    def n_col(self) -> int:
        return len(self.col_pts)

    def replace(self, **kw) -> "EnvConfig":
        return dataclasses.replace(self, **kw)

    def as_dict(self) -> dict[str, Any]:
        d = dataclasses.asdict(self)
        d["n_col"] = self.n_col
        return d

    def with_aircraft(self, urdf_path: str | None = None, aero_path: str | None = None,
                      body: "aircraft.RigidBody | None" = None) -> "EnvConfig":
        """Fill the aircraft fields from a URDF (or an already reduced ``RigidBody``, e.g. aircraft.body_from_bullet of a
        PyFlyt recording) and the aero table."""
        if body is None:
            body = aircraft.load_urdf(urdf_path or aircraft.DEFAULT_URDF)
        aero = aircraft.load_aero(aero_path or aircraft.DEFAULT_AERO)
        cols = aero.cols
        out = self.replace(
            cl_alpha_2d=cols["Cl_alpha_2D"].tolist(), chord=cols["chord"].tolist(), span=cols["span"].tolist(),
            flap_to_chord=cols["flap_to_chord"].tolist(), eta=cols["eta"].tolist(),
            alpha0_base_deg=cols["alpha_0_base"].tolist(), stall_p_base_deg=cols["alpha_stall_P_base"].tolist(),
            stall_n_base_deg=cols["alpha_stall_N_base"].tolist(), cd0=cols["Cd_0"].tolist(),
            defl_limit_deg=cols["deflection_limit"].tolist(), surf_tau=cols["tau"].tolist(),
            lift_unit=aero.lift_unit.tolist(), fwd_unit=aero.fwd_unit.tolist(),
            r_surf=[body.link_offsets[l].tolist() for l in aero.links],
            total_thrust=float(aero.motor["total_thrust"]), thrust_coef=float(aero.motor["thrust_coef"]),
            torque_coef=float(aero.motor["torque_coef"]), noise_ratio=float(aero.motor["noise_ratio"]),
            motor_tau=float(aero.motor["tau"]), r_motor=body.link_offsets[aero.motor["link"]].tolist(),
            thrust_unit=[float(x) for x in aero.motor["thrust_unit"]],
            mass=body.mass, com=body.com.tolist(), inertia_o=body.inertia_o.reshape(-1).tolist(),
            col_pts=body.collision_points[:MAX_COL].tolist(),
        )
        return out

    def to_c(self) -> FwConfigC:
        c = FwConfigC()
        names = {f[0] for f in FwConfigC._fields_}
        d = self.as_dict()
        for name, ctype in FwConfigC._fields_:
            v = d[name]
            if name == "col_pts":
                for i, p in enumerate(v):
                    for k in range(3):
                        c.col_pts[i][k] = float(p[k])
            elif isinstance(v, list):
                arr = getattr(c, name)
                if v and isinstance(v[0], list):
                    for i, row in enumerate(v):
                        for k, x in enumerate(row):
                            arr[i][k] = float(x)
                else:
                    for i, x in enumerate(v):
                        arr[i] = float(x)
            else:
                setattr(c, name, v)
        missing = [k for k in d if k not in names]
        if missing:
            raise RuntimeError(f"EnvConfig fields without a C counterpart: {missing}")
        return c


def _wind_fields(wind: dict | None, hook: str) -> dict:
    """Translate the reference's wind_config dict (fixedwing_base_env.py:108-173) into flat fields.

    hook: "env" -> applied in begin_reset (FixedwingBaseEnv(wind_config=...)); "wrapper" -> applied by
    WindOnResetWrapper after reset's warm-up (envs/utils.py:208-218).
    """
    if not wind or not bool(wind.get("enabled", False)):
        return dict(wind_mode=0)
    mode = str(wind.get("mode", "constant")).lower()
    if mode not in ("constant", "gust_sine", "field"):
        raise ValueError(f"Unsupported wind mode: {mode}")
    rnd = bool(wind.get("randomize_on_reset", False))
    if mode == "field":
        # gridded field (pyflyt_drone_b200/wind.py): the WindField itself travels beside the config, to FixedwingVecEnv
        from .wind import WindField
        if not isinstance(wind.get("field"), WindField):
            raise ValueError("wind mode 'field' needs wind_config['field'] = a pyflyt_drone_b200.wind.WindField")
        return dict(wind_mode=3, wind_randomize=int(rnd), wind_start_substep=0 if hook == "env" else 20)

    def vec(key):
        return [float(x) for x in np.asarray(wind.get(key, (0.0, 0.0, 0.0)), dtype=np.float64).reshape(3)]

    def rng(key, base):
        r = wind.get(key, None)
        if r is None:
            return base, base
        if not isinstance(r, (list, tuple)) or len(r) != 3 or not all(isinstance(x, (list, tuple)) and len(x) == 2 for x in r):
            raise ValueError(f"Invalid {key}: {r}")
        return [float(x[0]) for x in r], [float(x[1]) for x in r]

    base = vec("wind_enu_mps")
    amp = vec("gust_amp_enu_mps")
    blo, bhi = rng("wind_enu_mps_range", base)
    alo, ahi = rng("gust_amp_enu_mps_range", amp)
    return dict(
        wind_mode=1 if mode == "constant" else 2, wind_randomize=int(rnd),
        wind_rand_phase=int(bool(wind.get("randomize_gust_phase", True))),
        wind_start_substep=0 if hook == "env" else 20,
        wind_base=base, wind_base_lo=blo, wind_base_hi=bhi, gust_amp=amp, gust_amp_lo=alo, gust_amp_hi=ahi,
        gust_freq=float(wind.get("gust_freq_hz", 0.0)), gust_phase=float(wind.get("gust_phase_rad", 0.0)),
    )


def waypoints_v3(wind: dict | None = None, **overrides) -> EnvConfig:
    """PyFlyt/Fixedwing-Waypoints-v3 as built by train_Fixedwing_Waypoints_v3.py:97-118."""
    cfg = EnvConfig(
        task=TASK_WAYPOINTS, num_targets=8, goal_reach=4.0, sparse_reward=1, angle_repr=0, dome=100.0,
        max_steps=int(30 * 120.0), context_len=2, spawn_size=100.0, early_return_on_crash=0, complete_truncates=1,
        **_wind_fields(wind, "wrapper"),
    ).with_aircraft()
    return cfg.replace(**overrides) if overrides else cfg


def waypoint_objlock(wind: dict | None = None, **overrides) -> EnvConfig:
    """FixedwingWaypointObjLockEnv as built by train_Fixedwing_Waypoints_ObjLock.py:119-165."""
    if wind is None:
        wind = {
            "enabled": True, "mode": "gust_sine", "wind_enu_mps": [0.0, 0.0, 0.0],
            "wind_enu_mps_range": [[-5.0, 5.0], [-5.0, 5.0], [-0.5, 0.5]],
            "gust_amp_enu_mps": [0.0, 0.0, 0.0], "gust_amp_enu_mps_range": [[0.0, 3.0], [0.0, 3.0], [0.0, 0.3]],
            "gust_freq_hz": 0.2, "gust_phase_rad": 0.0, "randomize_on_reset": True, "randomize_gust_phase": True,
        }
    cfg = EnvConfig(
        task=TASK_OBJLOCK, num_targets=8, goal_reach=8.0, sparse_reward=0, angle_repr=0, dome=100.0,
        max_steps=int(30 * 120.0), context_len=2, spawn_size=100.0, early_return_on_crash=1, complete_truncates=0,
        num_obstacles=20, obst_radius=2.0, obst_h_lo=10.0, obst_h_hi=30.0, obst_safe=5.0, obst_scale=1.0,
        obst_max_pen=2.0, cam_interval_substeps=12, lock_hold_steps=10, strike_dist=8.0, strike_reward=200.0,
        lock_step_reward=0.1, approach_scale=0.05, switch_min_seen=2, switch_min_area=0.0005, duck_radius=1.5,
        **_wind_fields(wind, "env"),
    ).with_aircraft()
    return cfg.replace(**overrides) if overrides else cfg


def physics_only(**overrides) -> EnvConfig:
    """BASELINE.json configs[1]: batched physics step only, random actions, reset on ground/dome."""
    cfg = EnvConfig(task=TASK_PHYSICS, num_targets=0, dome=100.0, max_steps=2 ** 30, context_len=0,
                    angle_repr=0).with_aircraft()
    return cfg.replace(**overrides) if overrides else cfg


def lowlevel(wind: dict | None = None, **overrides) -> EnvConfig:
    """FixedwingLowLevelEnv (envs/fixedwing_envs/fixedwing_lowlevel_env.py:22-72): mode -1 six-channel control, start
    (0,0,10) at 15 m/s, one Aviary.step per env step, no warm-up, 2,000-step episodes, psi/h/V tracking."""
    cfg = EnvConfig(task=TASK_LOWLEVEL, num_targets=1, angle_repr=0, max_steps=2000, context_len=0, inner_per_step=1,
                    warmup_inner=0, start_pos=[0.0, 0.0, 10.0], start_vel=[15.0, 0.0, 0.0],
                    **_wind_fields(wind, "env")).with_aircraft()
    return cfg.replace(**overrides) if overrides else cfg


def objlock_duck(wind: dict | None = None, **overrides) -> EnvConfig:
    """FixedwingObjLockEnv + FlattenObjLockEnv as built by train/train_objlock.py:27-146 (duck-only lock and strike):
    start (0,0,100), 200 m dome, 60 s episodes, cockpit camera (offset (0.8,0,0.12), -5 deg, not tracking) captured every
    2*12 physics steps at render_resolution 480 (render_mode="rgb_array"), no obstacles, 3-frame vision history + deltas,
    56-float observation.  duck_radius is the analytic stand-in for the duck mesh at globalScaling 60 (0.05 m per unit
    of scaling, the ratio the waypoint_objlock preset uses at scaling 30)."""
    if wind is None:
        wind = {
            "enabled": True, "mode": "gust_sine", "wind_enu_mps": [0.0, 0.0, 0.0],
            "wind_enu_mps_range": [[-10.0, 10.0], [-10.0, 10.0], [-0.10, 0.10]],
            "gust_amp_enu_mps": [0.0, 0.0, 0.0], "gust_amp_enu_mps_range": [[0.0, 3.0], [0.0, 3.0], [0.0, 0.3]],
            "gust_freq_hz": 0.2, "gust_phase_rad": 0.0, "randomize_on_reset": True, "randomize_gust_phase": True,
        }
    cfg = EnvConfig(
        task=TASK_DUCK, num_targets=0, sparse_reward=0, angle_repr=0, dome=200.0, spawn_size=200.0,
        max_steps=int(30 * 60.0), context_len=0, start_pos=[0.0, 0.0, 100.0], early_return_on_crash=1, complete_truncates=0,
        num_obstacles=0, obst_radius=2.0, obst_h_lo=10.0, obst_h_hi=30.0, obst_safe=10.0, obst_scale=1.0, obst_max_pen=5.0,
        cam_interval_substeps=2 * 12, lock_hold_steps=5, strike_dist=10.0, strike_reward=400.0, lock_step_reward=0.2,
        approach_scale=0.1, duck_radius=3.0, cam_mode=1, cam_offset=[0.8, 0.0, 0.12], cam_tilt_deg=-5.0, cam_res=480,
        vision_hist_len=3, vision_use_deltas=1,
        **_wind_fields(wind, "env"),
    ).with_aircraft()
    return cfg.replace(**overrides) if overrides else cfg


PRESETS = {"waypoints_v3": waypoints_v3, "waypoint_objlock": waypoint_objlock, "physics_only": physics_only,
           "lowlevel": lowlevel, "objlock_duck": objlock_duck}


def from_gym_kwargs(preset: str = "waypoints_v3", *, sparse_reward=None, num_targets=None, goal_reach_distance=None,
                    flight_dome_size=None, max_duration_seconds=None, agent_hz=None, angle_representation=None,
                    context_length=None, wind=None, **overrides) -> EnvConfig:
    """Preset + the keyword names the reference passes to ``gym.make`` / ``FlattenWaypointEnv``
    (train/train_Fixedwing_Waypoints_v3.py:100-117), translated to EnvConfig fields.  ``None`` keeps the preset."""
    over = dict(overrides)
    if sparse_reward is not None:
        over["sparse_reward"] = int(bool(sparse_reward))
    if num_targets is not None:
        over["num_targets"] = int(num_targets)
    if goal_reach_distance is not None:
        over["goal_reach"] = float(goal_reach_distance)
    if flight_dome_size is not None:
        over["dome"] = over["spawn_size"] = float(flight_dome_size)
    if agent_hz is not None:
        if 120 % int(agent_hz) != 0:
            raise ValueError("agent_hz must divide 120")           # fixedwing_base_env.py:97-100
        over["inner_per_step"] = 120 // int(agent_hz)
    if max_duration_seconds is not None:
        over["max_steps"] = int((agent_hz or 30) * max_duration_seconds)
    if angle_representation is not None:
        if angle_representation not in ("euler", "quaternion"):
            raise ValueError(f"angle_representation must be either `euler` or `quaternion`, not {angle_representation}")
        over["angle_repr"] = 0 if angle_representation == "euler" else 1
    if context_length is not None:
        over["context_len"] = int(context_length)
    return PRESETS[preset](wind=wind, **over) if preset != "physics_only" else PRESETS[preset](**over)


def make_config(preset: str = "waypoints_v3", **overrides) -> EnvConfig:
    if preset not in PRESETS:
        raise KeyError(f"unknown preset {preset!r}; choose from {sorted(PRESETS)}")
    return PRESETS[preset](**overrides)
