"""CPU tests of the host side: URDF reduction, aero table, presets mirroring the reference's TRAIN_CONFIGs."""
import json
import math
import os

import numpy as np
import pytest

import pyflyt_drone_b200 as fw
from pyflyt_drone_b200 import aircraft
from pyflyt_drone_b200.config import _wind_fields


def test_placeholder_urdf_is_flagged_and_totals_2p5kg():
    body = aircraft.load_urdf()
    assert body.placeholder
    assert body.mass == pytest.approx(2.5)
    assert set(body.link_offsets) >= {"motor_link", "main_wing_link", "left_wing_flapped_link"}
    assert body.collision_points.shape == (8, 3)


def test_parallel_axis_and_composite_inertia(tmp_path):
    urdf = tmp_path / "two.urdf"
    urdf.write_text("""<robot name="t"><link name="base"><inertial><origin xyz="0 0 0"/><mass value="2"/>
      <inertia ixx="1" ixy="0" ixz="0" iyy="1" iyz="0" izz="1"/></inertial></link>
      <link name="tip"><inertial><origin xyz="0 0 0"/><mass value="1"/>
      <inertia ixx="0.1" ixy="0" ixz="0" iyy="0.2" iyz="0" izz="0.3"/></inertial></link>
      <joint name="j" type="fixed"><parent link="base"/><child link="tip"/><origin xyz="2 0 0" rpy="0 0 0"/></joint>
      </robot>""")
    b = aircraft.load_urdf(str(urdf))
    assert b.mass == 3 and b.com == pytest.approx([2 / 3, 0, 0])
    # about the base CoM: tip adds m*d^2 = 4 on yy and zz
    assert np.diag(b.inertia_o) == pytest.approx([1.1, 1.2 + 4, 1.3 + 4])
    S = b.spatial_inertia()
    assert S.shape == (6, 6) and np.allclose(S @ b.spatial_inertia_inv(), np.eye(6))
    # pure force through the composite CoM produces no angular acceleration
    f = np.array([0.0, 3.0, 0.0])
    wrench = np.concatenate([np.cross(b.com, f), f])
    acc = b.spatial_inertia_inv() @ wrench
    assert acc[:3] == pytest.approx([0, 0, 0], abs=1e-12) and acc[3:] == pytest.approx(f / 3)


def test_rotated_joint_and_inertial_frames(tmp_path):
    urdf = tmp_path / "rot.urdf"
    urdf.write_text(f"""<robot name="t"><link name="base"><inertial><mass value="1"/>
      <inertia ixx="1" ixy="0" ixz="0" iyy="1" iyz="0" izz="1"/></inertial></link>
      <link name="tip"><inertial><origin xyz="1 0 0" rpy="0 0 0"/><mass value="1"/>
      <inertia ixx="1" ixy="0" ixz="0" iyy="2" iyz="0" izz="3"/></inertial></link>
      <joint name="j" type="fixed"><parent link="base"/><child link="tip"/><origin xyz="0 0 0" rpy="0 0 {math.pi/2}"/></joint>
      </robot>""")
    b = aircraft.load_urdf(str(urdf))
    assert b.link_offsets["tip"] == pytest.approx([0, 1, 0], abs=1e-12)
    tip = next(l for l in b.links if l.name == "tip")
    assert np.diag(tip.inertia) == pytest.approx([2, 1, 3], abs=1e-12)


def test_non_fixed_joint_rejected(tmp_path):
    urdf = tmp_path / "bad.urdf"
    urdf.write_text("""<robot name="t"><link name="a"><inertial><mass value="1"/><inertia ixx="1" iyy="1" izz="1"/></inertial></link>
      <link name="b"><inertial><mass value="1"/><inertia ixx="1" iyy="1" izz="1"/></inertial></link>
      <joint name="j" type="revolute"><parent link="a"/><child link="b"/></joint></robot>""")
    with pytest.raises(ValueError):
        aircraft.load_urdf(str(urdf))


def test_aero_table_carries_reference_numbers():
    t = aircraft.load_aero()
    assert t.names == list(aircraft.SURFACE_ORDER)
    assert t.cols["span"].tolist() == [0.3, 0.3, 0.625, 0.312, 1.6]
    assert t.cols["deflection_limit"].tolist() == [30, 30, 20, 20, 0]
    assert t.cols["alpha_stall_P_base"].tolist() == [14, 14, 9, 9, 14]
    assert t.lift_unit[3].tolist() == [0, 1, 0]
    assert t.motor["total_thrust"] == 18 and t.motor["thrust_coef"] == 3.16e-10
    areas = t.cols["chord"] * t.cols["span"]
    assert areas == pytest.approx([0.09, 0.09, 0.125, 0.0624, 0.48])


def test_reference_yaml_numbers_match_if_reference_is_mounted():
    """Every number of the original project's fixed-wing parameter file, stored under tests/golden, is in the aero table."""
    with open(os.path.join(os.path.dirname(__file__), "golden", "reference_fixedwing_params.json")) as f:
        doc = json.load(f)
    t = aircraft.load_aero()
    keymap = {"left_wing_flapped": "left_wing_flapped_params", "right_wing_flapped": "right_wing_flapped_params",
              "horizontal_tail": "horizontal_tail_params", "vertical_tail": "vertical_tail_params",
              "main_wing": "main_wing_params"}
    for i, n in enumerate(t.names):
        for k, v in doc[keymap[n]].items():
            assert t.cols[k][i] == pytest.approx(float(v)), (n, k)
    for k, v in doc["motor_params"].items():
        assert float(t.motor[k]) == pytest.approx(float(v))


def test_presets_mirror_train_configs():
    w = fw.waypoints_v3()
    assert (w.num_targets, w.goal_reach, w.sparse_reward, w.angle_repr, w.context_len) == (8, 4.0, 1, 0, 2)
    assert w.max_steps == 3600 and w.inner_per_step == 4 and w.obs_dim == 28 and w.wind_mode == 0
    assert w.complete_truncates == 1 and w.early_return_on_crash == 0
    o = fw.waypoint_objlock()
    assert (o.num_targets, o.goal_reach, o.sparse_reward, o.num_obstacles, o.obst_safe) == (8, 8.0, 0, 20, 5.0)
    assert o.wind_mode == 2 and o.wind_randomize == 1 and o.gust_freq == 0.2 and o.wind_start_substep == 0
    assert o.wind_base_lo == [-5.0, -5.0, -0.5] and o.gust_amp_hi == [3.0, 3.0, 0.3]
    assert o.strike_dist == 8.0 and o.cam_interval_substeps == 12 and o.early_return_on_crash == 1
    ph = fw.physics_only()
    assert ph.task == 0 and ph.obs_dim == 0
    q = fw.waypoints_v3(angle_repr=1)
    assert q.obs_dim == 29


def test_wind_config_translation_and_validation():
    assert _wind_fields(None, "env") == dict(wind_mode=0)
    assert _wind_fields({"enabled": False}, "env") == dict(wind_mode=0)
    f = _wind_fields({"enabled": True, "mode": "constant", "wind_enu_mps": [1, 2, 3]}, "wrapper")
    assert f["wind_mode"] == 1 and f["wind_start_substep"] == 20 and f["wind_base"] == [1.0, 2.0, 3.0]
    with pytest.raises(ValueError):
        _wind_fields({"enabled": True, "mode": "tornado"}, "env")
    with pytest.raises(ValueError):
        _wind_fields({"enabled": True, "wind_enu_mps_range": [[0, 1]]}, "env")


def test_config_round_trips_into_c_struct():
    c = fw.waypoint_objlock().to_c()
    assert c.num_targets == 8 and c.n_col == 8 and c.wind_mode == 2
    assert c.r_surf[4][2] == pytest.approx(0.05) and c.col_pts[0][0] == pytest.approx(0.6)
    assert c.lift_unit[3][1] == 1.0 and c.gust_amp_hi[2] == pytest.approx(0.3)


def test_from_gym_kwargs_reproduces_the_training_script_preset():
    """The keyword names of the reference's gym.make call (train_Fixedwing_Waypoints_v3.py:100-110) map onto the preset."""
    import pytest
    from pyflyt_drone_b200 import from_gym_kwargs, waypoints_v3
    cfg = from_gym_kwargs("waypoints_v3", sparse_reward=True, num_targets=8, goal_reach_distance=4.0,
                          angle_representation="euler", flight_dome_size=100.0, max_duration_seconds=120.0, agent_hz=30,
                          context_length=2, wind=None)
    assert cfg == waypoints_v3()
    other = from_gym_kwargs("waypoints_v3", num_targets=4, goal_reach_distance=2.0, agent_hz=60, max_duration_seconds=10.0,
                            angle_representation="quaternion")
    assert (other.num_targets, other.goal_reach, other.inner_per_step, other.max_steps, other.angle_repr) == (4, 2.0, 2, 600, 1)
    with pytest.raises(ValueError):
        from_gym_kwargs("waypoints_v3", agent_hz=50)           # fixedwing_base_env.py:97-100: agent_hz must divide 120
    with pytest.raises(ValueError):
        from_gym_kwargs("waypoints_v3", angle_representation="dcm")


def test_duck_only_config_round_trips_and_rejects_bad_arguments():
    """objlock_duck preset -> C struct (the task-4 fields added in ABI 9), and the argument checks of the single-env view
    that fire before any device is touched (envs/fixedwing_objlock_env.py:37-118 keyword names)."""
    c = fw.make_config("objlock_duck").to_c()
    assert c.task == 4 and c.num_targets == 0 and c.context_len == 0 and c.cam_mode == 1 and c.cam_res == 480
    assert c.cam_tilt_deg == -5.0 and c.cam_offset[0] == pytest.approx(0.8) and c.cam_offset[2] == pytest.approx(0.12)
    assert (c.vision_hist_len, c.vision_use_deltas, c.lock_decay_steps) == (3, 1, 1)
    assert (c.duck_dist_scale, c.lock_center_radius, c.centering_scale, c.visible_step_reward, c.area_reward_scale,
            c.lock_lost_penalty, c.approach_clip) == (1.0, 0.55, 3.0, 2.0, 5.0, 0.5, 2.0)
    assert c.strike_reward == 400.0 and c.lock_hold_steps == 5 and c.wind_base_hi[0] == 10.0
    from pyflyt_drone_b200.gym_env import FixedwingObjLockEnv
    with pytest.raises(ValueError, match="agent_hz"):
        FixedwingObjLockEnv(agent_hz=50)
    with pytest.raises(ValueError, match="angle_representation"):
        FixedwingObjLockEnv(angle_representation="axis_angle")
    with pytest.raises(ValueError, match="flight_mode"):
        FixedwingObjLockEnv(flight_mode=-1)
    with pytest.raises(ValueError, match="render_mode"):
        FixedwingObjLockEnv(render_mode="human")
    with pytest.raises(ValueError, match="90 degree"):
        FixedwingObjLockEnv(camera_FOV_degrees=60)
