"""High-level waypoints (task 5) without a GPU: preset and dimensions, the action -> command mapping, Tracker validation and
loading from PPO.save / export_sb3 files, and the C entry points' argument checks, which return before touching a device."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import pyflyt_drone_b200 as fw
from pyflyt_drone_b200 import _lib, tracker as trk
from pyflyt_drone_b200.config import TASK_HIGHLEVEL, make_config
from pyflyt_drone_b200.tracker import Tracker


def random_tracker(seed=0, **kw) -> Tracker:
    rng = np.random.default_rng(seed)
    p = rng.normal(0.0, 0.2, trk.PARAM_COUNT).astype(np.float32)
    return Tracker(p, rng.normal(0, 1, 21), rng.uniform(0.5, 2.0, 21), **kw)


def test_preset_and_dimensions():
    cfg = make_config("highlevel")
    wp = make_config("waypoints_v3")
    assert TASK_HIGHLEVEL == 5 and cfg.task == 5
    assert cfg.replace(task=1) == wp                       # the waypoints_v3 numbers with task 5
    assert cfg.obs_dim == wp.obs_dim == 28
    assert make_config("highlevel", angle_repr=1).obs_dim == 29
    assert cfg.inner_per_step == 4 and cfg.substeps_per_inner == 2
    assert trk.PARAM_COUNT == 11597 and trk.POLICY_TOWER == 5958


def test_param_count_matches_the_library():
    lib = _lib.load()
    assert lib.ppo_param_count_a(21, 6) == trk.PARAM_COUNT


def test_action_to_command_mapping():
    t = random_tracker(h_range=(5.0, 20.0), v_range=(10.0, 20.0))
    a = np.array([[1.0, 0.0, -1.0, -1.0], [0.0, 1.0, 1.0, 1.0], [-1.0, 0.0, 0.0, 0.0], [0.0, -2.0, 3.0, -7.0],
                  [0.0, 0.0, 0.5, -0.5]])
    c = t.command(a)
    np.testing.assert_allclose(c[:, 0], [0.0, np.pi / 2, np.pi, -np.pi / 2, 0.0])      # atan2(0, 0) = 0
    np.testing.assert_allclose(c[:, 1], [5.0, 20.0, 12.5, 20.0, 16.25])                 # clamped to [-1, 1]
    np.testing.assert_allclose(c[:, 2], [10.0, 20.0, 15.0, 10.0, 12.5])
    # a direction vector: scaling it does not change the heading, so a Gaussian policy sees no wrap at +-pi
    np.testing.assert_allclose(t.command(a[:2] * [[3.0, 3.0, 1.0, 1.0]])[:, 0], c[:2, 0])


def test_tracker_validation():
    p = np.zeros(trk.PARAM_COUNT, np.float32)
    Tracker(p)
    with pytest.raises(ValueError, match="floats"):
        Tracker(p[:-1])
    bad = p.copy(); bad[17] = np.nan
    with pytest.raises(ValueError, match="finite"):
        Tracker(bad)
    bad = p.copy(); bad[-1] = np.nan                        # log_std is not read by the tracker
    Tracker(bad)
    with pytest.raises(ValueError, match="both"):
        Tracker(p, obs_mean=np.zeros(21))
    with pytest.raises(ValueError, match="21"):
        Tracker(p, np.zeros(20), np.ones(20))
    with pytest.raises(ValueError, match=">= 0"):
        Tracker(p, np.zeros(21), -np.ones(21))
    with pytest.raises(ValueError, match="clip_obs"):
        Tracker(p, clip_obs=0.0)
    with pytest.raises(ValueError, match="h_range"):
        Tracker(p, h_range=(20.0, 5.0))
    with pytest.raises(ValueError, match="v_range"):
        Tracker(p, v_range=(10.0, np.inf))


def _sb3_state(d, a, seed=0):
    g = torch.Generator().manual_seed(seed)
    sd = {"mlp_extractor.policy_net.0.weight": (64, d), "mlp_extractor.policy_net.0.bias": (64,),
          "mlp_extractor.policy_net.2.weight": (64, 64), "mlp_extractor.policy_net.2.bias": (64,),
          "action_net.weight": (a, 64), "action_net.bias": (a,),
          "mlp_extractor.value_net.0.weight": (64, d), "mlp_extractor.value_net.0.bias": (64,),
          "mlp_extractor.value_net.2.weight": (64, 64), "mlp_extractor.value_net.2.bias": (64,),
          "value_net.weight": (1, 64), "value_net.bias": (1,), "log_std": (a,)}
    return {k: torch.randn(s, generator=g) for k, s in sd.items()}


def _vecnorm(d, norm_obs=True):
    return {"obs_rms.mean": np.linspace(-1, 1, d), "obs_rms.var": np.linspace(0.5, 2, d), "obs_rms.count": 10.0,
            "ret_rms.mean": 0.0, "ret_rms.var": 1.0, "ret_rms.count": 1.0, "clip_obs": 7.0, "clip_reward": 10.0,
            "gamma": 0.99, "norm_obs": norm_obs, "norm_reward": True}


def test_tracker_load_from_ppo_save_file(tmp_path):
    sd = _sb3_state(21, 6)
    path = os.path.join(tmp_path, "tracker.pt")
    torch.save({"policy": sd, "vecnorm": _vecnorm(21), "obs_dim": 21}, path)
    t = Tracker.load(path)
    assert t.params[:64 * 21].tolist() == sd["mlp_extractor.policy_net.0.weight"].reshape(-1).tolist()
    np.testing.assert_array_equal(t.params[-6:], sd["log_std"].numpy())
    np.testing.assert_array_equal(t.obs_mean, np.linspace(-1, 1, 21))
    assert t.clip_obs == 7.0 and t.h_range == (5.0, 20.0) and t.v_range == (10.0, 20.0)
    torch.save({"policy": sd, "vecnorm": _vecnorm(21, norm_obs=False)}, path)
    assert Tracker.load(path, h_range=(2.0, 30.0)).obs_mean is None and Tracker.load(path, h_range=(2.0, 30.0)).h_range == (2.0, 30.0)


@pytest.mark.parametrize("d,a", [(28, 4), (21, 4), (28, 6)])
def test_tracker_refuses_other_widths(tmp_path, d, a):
    path = os.path.join(tmp_path, "m.pt")
    torch.save({"policy": _sb3_state(d, a), "vecnorm": _vecnorm(d)}, path)
    with pytest.raises(ValueError, match="21-float observation and 6 actions"):
        Tracker.load(path)


def test_tracker_load_from_sb3_directory(tmp_path):
    from pyflyt_drone_b200 import sb3_io
    from pyflyt_drone_b200.ppo import export_vecnorm_npz
    sd = _sb3_state(21, 6, seed=3)
    d = str(tmp_path)
    torch.save(sd, os.path.join(d, "policy.pth"))                    # a bare policy.pth + vecnorm.npz
    export_vecnorm_npz(_vecnorm(21), os.path.join(d, "vecnorm.npz"))
    t = Tracker.load(d)
    np.testing.assert_array_equal(t.params[64 * 21:64 * 22], sd["mlp_extractor.policy_net.0.bias"].numpy())
    np.testing.assert_array_equal(t.obs_var, np.linspace(0.5, 2, 21))
    # vecnorm.pkl (VecNormalize.save's pickle) takes precedence over the npz
    sb3_io.write_vecnorm_pkl(os.path.join(d, "vecnorm.pkl"), {**_vecnorm(21), "clip_obs": 5.0}, 21, 6, 8)
    assert Tracker.load(d).clip_obs == 5.0


def test_vec_env_requires_a_tracker_for_task_5_only():
    with pytest.raises(ValueError, match="tracker"):
        fw.FixedwingVecEnv(4, preset="highlevel")
    with pytest.raises(ValueError, match="tracker"):
        fw.FixedwingVecEnv(4, preset="waypoints_v3", tracker=random_tracker())
    with pytest.raises(TypeError):
        fw.FixedwingVecEnv(4, preset="highlevel", tracker=object())


def test_entry_points_validate_before_touching_a_device():
    lib = _lib.load()
    t = random_tracker()
    desc = t.to_c()
    assert lib.fw_set_tracker(None, None) == -1
    assert lib.fw_set_tracker(None, C.byref(desc)) == -1 and b"null handle" in lib.fw_last_error()
    bad = Tracker(t.params.copy(), t.obs_mean, t.obs_var)
    for field, value, msg in [("clip_obs", 0.0, b"clip_obs"), ("clip_obs", float("nan"), b"clip_obs")]:
        d = bad.to_c(); setattr(d, field, value)
        assert lib.fw_set_tracker(None, C.byref(d)) == -1 and msg in lib.fw_last_error()
    d = bad.to_c(); d.h_range[0], d.h_range[1] = 20.0, 5.0
    assert lib.fw_set_tracker(None, C.byref(d)) == -1 and b"h_range" in lib.fw_last_error()
    d = bad.to_c(); d.v_range[1] = float("inf")
    assert lib.fw_set_tracker(None, C.byref(d)) == -1 and b"v_range" in lib.fw_last_error()
    d = bad.to_c(); d.obs_var = None
    assert lib.fw_set_tracker(None, C.byref(d)) == -1 and b"both" in lib.fw_last_error()
    d = bad.to_c(); d.params = None
    assert lib.fw_set_tracker(None, C.byref(d)) == -1 and b"params" in lib.fw_last_error()
    p = t.params.copy(); p[100] = np.inf
    d = bad.to_c(); d.params = p.ctypes.data_as(C.c_void_p).value
    assert lib.fw_set_tracker(None, C.byref(d)) == -1 and b"not finite" in lib.fw_last_error()
    v = t.obs_var.copy(); v[3] = -1.0
    d = bad.to_c(); d.obs_var = v.ctypes.data_as(C.c_void_p).value
    assert lib.fw_set_tracker(None, C.byref(d)) == -1 and b"obs_var" in lib.fw_last_error()
    buf = np.zeros((4, 6), np.float32)
    assert lib.fw_get_tracker_state(None, buf.ctypes.data_as(C.c_void_p)) == -1
    assert lib.fw_get_tracker_state(None, None) == -1
    assert lib.fw_set_tracker_state(None, buf.ctypes.data_as(C.c_void_p)) == -1
    assert lib.fw_set_tracker_obs_buffer(None, None) == -1
