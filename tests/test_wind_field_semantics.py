"""Gridded wind fields (wind_mode 3) without a device: the fp64 field reference (tests/field_oracle.py) -- interpolation and
per-surface sampling --, the
WindField host class, the wind_config translation and the argument checks of fw_set_wind_field."""
import ctypes as C

import numpy as np
import pytest

import pyflyt_drone_b200 as fw
from oracle import fw_oracle as fo
from pyflyt_drone_b200 import _lib
from tests import field_oracle as fwf
from pyflyt_drone_b200.config import _wind_fields
from pyflyt_drone_b200.wind import WindField

# an affine field w = A x + b t + c whose lattice values are dyadic (exact in float32): interpolation reproduces it exactly
A = np.array([[0.5, -0.25, 0.125], [0.25, 0.5, -0.5], [-0.125, 0.25, 0.75]])
B = np.array([1.0, -2.0, 0.5])
CC = np.array([3.0, -1.0, 0.25])
ORIGIN, SPACING, SHAPE, NT, TSTEP = np.array([-4.0, -2.0, 0.0]), np.array([0.5, 1.0, 2.0]), (9, 5, 6), 4, 0.25


def _affine(t, x):
    return x @ A.T + B * t + CC


def _affine_field(**kw):
    return WindField.from_function(_affine, ORIGIN, SPACING, SHAPE, n_slices=NT, t_step=TSTEP, **kw)


def _oracle_field(wf: WindField):
    return fwf.make_field(wf)


def _box_hi():
    return ORIGIN + SPACING * (np.array(SHAPE) - 1)


def test_trilinear_linear_in_time_reproduces_an_affine_field():
    wf = _affine_field()
    assert np.array_equal(wf.values[2, 3, 1, 4], _affine(2 * TSTEP, ORIGIN + SPACING * [4, 1, 3]).astype(np.float32))
    of = _oracle_field(wf)
    rng = np.random.default_rng(0)
    for _ in range(200):
        x = rng.uniform(ORIGIN, _box_hi())
        t = rng.uniform(0.0, (NT - 1) * TSTEP)             # inside the slices: no wrap
        np.testing.assert_allclose(fwf.wind_at(of, t, x), _affine(t, x), rtol=0, atol=1e-12)


def test_outside_the_box_clamps_to_the_edge_and_time_is_periodic():
    of = _oracle_field(_affine_field())
    rng = np.random.default_rng(1)
    lo, hi = ORIGIN, _box_hi()
    for _ in range(100):
        x = rng.uniform(lo - 20.0, hi + 20.0)
        t = rng.uniform(0.0, (NT - 1) * TSTEP)
        np.testing.assert_allclose(fwf.wind_at(of, t, x), _affine(t, np.clip(x, lo, hi)), rtol=0, atol=1e-12)
    period = NT * TSTEP
    x = (lo + hi) / 2
    for t in (0.1, 0.3, 0.6):
        w = fwf.wind_at(of, t, x)
        np.testing.assert_allclose(fwf.wind_at(of, t + period, x), w, atol=1e-12)
        np.testing.assert_allclose(fwf.wind_at(of, t - 3 * period, x), w, atol=1e-12)
    # between the last slice and the first: the slice after the last is slice 0
    last, first = _affine((NT - 1) * TSTEP, x), _affine(0.0, x)
    np.testing.assert_allclose(fwf.wind_at(of, (NT - 0.5) * TSTEP, x), 0.5 * (last + first), atol=1e-12)


def test_one_point_axes_are_constant():
    wf = WindField.from_function(lambda t, x: _affine(t, x), origin=(1.0, 2.0, 3.0), spacing=1.0, shape=(4, 1, 1))
    of = _oracle_field(wf)
    for y, z in ((-50.0, 0.0), (2.0, 3.0), (80.0, 99.0)):
        np.testing.assert_allclose(fwf.wind_at(of, 5.0, (2.5, y, z)), _affine(0.0, np.array([2.5, 2.0, 3.0])),
                                   atol=1e-12)


def _cfg(**kw):
    base = dict(noise_ratio=0.0, wind_start_substep=0)
    base.update(kw)
    return fw.make_config("waypoints_v3", **base).as_dict()


def _quat(roll, pitch, yaw):
    q = np.zeros(4)
    fo.lib().fwo_euler_to_quat((C.c_double * 3)(roll, pitch, yaw), q.ctypes.data_as(C.POINTER(C.c_double)))
    return q


def test_each_surface_sees_the_field_at_its_own_link_com():
    wf = _affine_field()
    cfg = _cfg()
    orc = fwf.FieldOracleVecEnv(cfg, 1, seed=3, wind_field=wf)
    orc.reset()
    q = _quat(0.7, -0.3, 1.1)                              # rolled, pitched, yawed
    pos, vel, omg = np.array([-1.0, 0.5, 4.0]), np.array([12.0, -1.0, 0.5]), np.array([1.5, -0.4, 0.8])
    ps = 37
    orc.set_state(dict(pos=pos[None], quat=q[None], vel=vel[None], omega=omg[None], physics_steps=np.array([ps]),
                       wind=np.array([[0.25, -0.5, 0.125, 0, 0, 0, 0.05]])))
    R = np.zeros(9)
    fo.lib().fwo_quat_to_mat(q.ctypes.data_as(C.POINTER(C.c_double)), R.ctypes.data_as(C.POINTER(C.c_double)))
    R = R.reshape(3, 3)
    shift, t = np.array([0.25, -0.5, 0.125]), (ps - 1) * cfg["dt"] + 0.05
    e = orc.envs[0]
    for s in range(5):
        rw = R @ np.array(cfg["r_surf"][s])
        x = np.clip(pos + rw - shift, ORIGIN, _box_hi())
        u = (t / TSTEP) % NT
        assert u < NT - 1
        w = _affine(t, x)
        want = R.T @ (vel + np.cross(omg, rw) - w)
        np.testing.assert_allclose(np.array(e.surf_vel[s][:]), want, rtol=0, atol=1e-9)
    # the surfaces do not all see the same wind: the field differs across the airframe
    assert np.ptp([e.surf_vel[s][2] for s in range(5)]) > 1e-3


def test_one_point_field_equals_constant_wind_over_240_substeps():
    v = np.array([2.5, -1.25, 0.5])
    const = fo.OracleVecEnv(_cfg(wind_mode=1, wind_base=list(v)), 4, seed=5)
    wf = WindField(np.broadcast_to(v.astype(np.float32), (1, 1, 1, 1, 3)), origin=0.0, spacing=1.0)
    field = fwf.FieldOracleVecEnv(_cfg(), 4, seed=5, wind_field=wf)
    np.testing.assert_allclose(field.reset(), const.reset(), rtol=1e-12, atol=1e-12)
    rng = np.random.default_rng(2)
    for _ in range(30):                                    # 30 agent steps x 8 substeps
        a = rng.uniform(-1, 1, (4, 4))
        oc, rc, fc, _ = const.step(a)
        of, rf, ff, _ = field.step(a)
        np.testing.assert_allclose(of, oc, rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(rf, rc, rtol=1e-12, atol=1e-12)
        np.testing.assert_array_equal(ff, fc)


def test_spanwise_updraft_gradient_rolls_the_aircraft():
    """An updraft that grows along the span gives a rolling moment whose sign follows the gradient's: a uniform wind
    cannot do that."""
    def roll_rate_change(g):
        wf = WindField.from_function(lambda t, x: np.stack([0 * x[:, 0], 0 * x[:, 0], g * x[:, 1]], axis=1),
                                     origin=(-50.0, -50.0, 0.0), spacing=(100.0, 1.0, 100.0), shape=(2, 101, 2))
        orc = fwf.FieldOracleVecEnv(_cfg(), 1, seed=1, wind_field=wf)
        orc.reset()
        orc.set_state(dict(pos=np.array([[0.0, 0.0, 20.0]]), quat=np.array([[0.0, 0.0, 0.0, 1.0]]),
                           vel=np.array([[15.0, 0.0, 0.0]]), omega=np.zeros((1, 3)), act=np.zeros((1, 6)),
                           physics_steps=np.array([40])))
        orc.step(np.zeros((1, 4)))
        return orc.get_state()["omega"][0, 0]

    calm, up, down = roll_rate_change(0.0), roll_rate_change(0.5), roll_rate_change(-0.5)
    assert abs(up - calm) > 1e-3 and abs(down - calm) > 1e-3
    assert np.sign(up - calm) == -np.sign(down - calm)


def test_from_function_samples_at_the_lattice_points_and_times():
    calls = []

    def f(t, pos):
        calls.append((t, pos.copy()))
        return np.stack([pos[:, 0], pos[:, 1] * 10, pos[:, 2] * 100 + t], axis=1)

    wf = WindField.from_function(f, origin=(1.0, 2.0, 3.0), spacing=(0.5, 1.0, 2.0), shape=(3, 2, 4), n_slices=3, t_step=0.5)
    assert [c[0] for c in calls] == [0.0, 0.5, 1.0]
    assert wf.values.shape == (3, 4, 2, 3, 3) and wf.shape == (3, 2, 4) and wf.n_slices == 3
    k, j, i = 3, 1, 2
    assert np.allclose(wf.values[2, k, j, i], [1.0 + 0.5 * i, (2.0 + j) * 10, (3.0 + 2 * k) * 100 + 1.0])
    assert wf.device_bytes == 3 * 4 * 2 * 3 * 16


@pytest.mark.parametrize("kw, msg", [
    (dict(values=np.full((1, 2, 2, 2, 3), np.nan)), "finite"),
    (dict(spacing=(1.0, 0.0, 1.0)), "spacing"),
    (dict(spacing=-1.0), "spacing"),
    (dict(values=np.zeros((2, 2, 2, 3))[..., :2]), "shape"),
    (dict(values=np.zeros((2, 2, 2, 2, 3)), t_step=None), "t_step"),
    (dict(shift_range=[(1.0, 0.0)] * 3), "shift_range"),
])
def test_wind_field_validation(kw, msg):
    args = dict(values=np.zeros((1, 2, 2, 2, 3)), origin=0.0, spacing=1.0, t_step=1.0)
    args.update(kw)
    with pytest.raises(ValueError, match=msg):
        WindField(**args)
    with pytest.raises(ValueError, match="t_step"):
        WindField.from_function(lambda t, x: 0 * x, 0.0, 1.0, (2, 2, 2), n_slices=2)


def test_wind_config_field_mode_translates():
    wf = _affine_field()
    d = _wind_fields({"enabled": True, "mode": "field", "field": wf, "randomize_on_reset": True}, "wrapper")
    assert d == dict(wind_mode=3, wind_randomize=1, wind_start_substep=20)
    d = _wind_fields({"enabled": True, "mode": "field", "field": wf}, "env")
    assert d == dict(wind_mode=3, wind_randomize=0, wind_start_substep=0)
    with pytest.raises(ValueError, match="WindField"):
        _wind_fields({"enabled": True, "mode": "field"}, "env")
    with pytest.raises(ValueError, match="Unsupported wind mode"):
        _wind_fields({"enabled": True, "mode": "tornado"}, "env")


def test_set_wind_field_argument_checks_need_no_device():
    lib = _lib.load()
    assert "fw_set_wind_field" in {s[0] for s in _lib.SYMBOLS}
    assert lib.fw_set_wind_field(None, None) == -1
    wf = _affine_field()

    def bad(**kw):
        d = wf.to_c()
        for k, v in kw.items():
            if k in ("spacing", "origin"):
                getattr(d, k)[0] = v
            else:
                setattr(d, k, v)
        return lib.fw_set_wind_field(None, C.byref(d)), lib.fw_last_error().decode()

    assert bad(nx=0) == (-1, "wind field: every dimension must be >= 1")
    assert bad(spacing=0.0)[1].startswith("wind field: spacing")
    assert bad(origin=float("inf"))[1].startswith("wind field: origin")
    assert bad(t_step=-1.0)[1].startswith("wind field: t_step")
    assert bad(values=None)[1] == "wind field: values is null"
    assert bad(nx=1 << 16, ny=1 << 16)[1].startswith("wind field: nx * ny * nz * nt")
    nan = wf.values.copy()
    nan[1, 2, 3, 4, 1] = np.nan
    d = wf.to_c()
    d.values = nan.ctypes.data_as(C.c_void_p).value
    assert lib.fw_set_wind_field(None, C.byref(d)) == -1 and "not finite" in lib.fw_last_error().decode()
    # a well-formed descriptor without a handle
    assert lib.fw_set_wind_field(None, C.byref(wf.to_c())) == -1 and lib.fw_last_error().decode() == "null handle"
