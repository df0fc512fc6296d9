"""Gridded wind fields (wind_mode 3) on the GPU: the FIELD step kernels against the fp64 reference (tests/field_oracle.py:
the oracle with the field), against the uniform wind, across shardings and spare-episode resets, the fw_set_wind_field
lifecycle, PPO and the gym views.  Tolerances as in test_parity_gpu.py (1e-4 norm-wise with a floor of 1 per state group,
flags and sparse rewards exact)."""
import ctypes as C

import numpy as np
import pytest

import pyflyt_drone_b200 as fw
from pyflyt_drone_b200 import _lib
from pyflyt_drone_b200.config import FLAG_TERM, FLAG_TRUNC
from pyflyt_drone_b200.vec_env import FixedwingVecEnv
from pyflyt_drone_b200.wind import WindField
from tests import field_oracle as fwf

pytestmark = pytest.mark.gpu

RTOL = 1e-4
PRESETS = {1: "waypoints_v3", 2: "waypoint_objlock", 3: "lowlevel", 4: "objlock_duck"}


def shear_thermal(t, x):
    """Boundary-layer shear along +x, a drifting, pulsing thermal and a weak crosswind: varies in x, y, z and t."""
    z = np.maximum(x[:, 2], 0.0)
    u = 6.0 * (1.0 - np.exp(-z / 15.0))
    cx, cy = 20.0 + 2.0 * t, -10.0
    r2 = (x[:, 0] - cx) ** 2 + (x[:, 1] - cy) ** 2
    up = (2.5 + 0.8 * np.sin(0.7 * t)) * np.exp(-r2 / 300.0) * np.minimum(z / 10.0, 1.0)
    return np.stack([u, 0.5 + 0.02 * x[:, 0], up], axis=1)


def make_field(randomize_time=True):
    return WindField.from_function(shear_thermal, origin=(-100.0, -100.0, 0.0), spacing=(10.0, 10.0, 5.0),
                                   shape=(21, 21, 21), n_slices=8, t_step=0.5,
                                   shift_range=[(-10.0, 10.0), (-10.0, 10.0), (-2.0, 2.0)], randomize_time=randomize_time)


def field_cfg(task, field, **kw):
    wind = {"enabled": True, "mode": "field", "field": field, "randomize_on_reset": True}
    cfg = fw.make_config(PRESETS[task], wind=wind, noise_ratio=0.0, **kw)
    return cfg.replace(wind_start_substep=0)      # env-hook flavour: the field acts during the warm-up too


STATE_GROUPS = ("pos", "quat", "vel", "omega", "act")


def state_err(sg, sc, ok):
    out = {}
    for k in STATE_GROUPS:
        d = np.abs(sg[k][ok] - sc[k][ok]).max(axis=1)
        scale = np.maximum(np.abs(sc[k][ok]).max(axis=1), 1.0)
        out[k] = float((d / scale).max()) if len(d) else 0.0
    return out


@pytest.mark.parametrize("generic", [False, True], ids=["std", "generic"])
@pytest.mark.parametrize("task", [1, 2, 3, 4])
def test_field_single_step_parity_from_injected_state(task, generic):
    field = make_field()
    cfg = field_cfg(task, field, force_generic_kernel=int(generic))
    N = 256
    env = FixedwingVecEnv(N, config=cfg, seed=7, wind_field=field)
    orc = fwf.FieldOracleVecEnv(cfg.as_dict(), N, seed=7, wind_field=field)
    env.reset(); orc.reset()
    sg, sc = env.get_state(), orc.get_state()
    np.testing.assert_allclose(sg["wind"], sc["wind"], rtol=0, atol=1e-5 * 10)       # the per-episode draws
    assert np.ptp(sc["wind"][:, 0]) > 1.0 and np.all(sc["wind"][:, 3:6] == 0)
    rng = np.random.default_rng(task)
    A = env.act_dim
    worst, mism, n_done, rew_bad, rew_n = {}, 0, 0, 0, 0
    for k in range(25):
        env.set_state(orc.get_state())
        a = rng.uniform(-1, 1, (N, A)).astype(np.float32)
        if task in (2, 4):
            a[:, :3] *= 0.3
        _, rg, fg, _ = env.step_arrays(a)
        rg, fg = rg.copy(), fg.copy().astype(np.int32)
        _, rc, fc, _ = orc.step(a.astype(np.float64))
        ok = fg == fc
        mism += int((~ok).sum())
        done = (fc & (FLAG_TERM | FLAG_TRUNC)) != 0
        n_done += int(done.sum())
        sg, sc = env.get_state(), orc.get_state()
        for g, v in state_err(sg, sc, ok & ~done).items():
            worst[g] = max(worst.get(g, 0.0), v)
        scale = max(1.0, np.abs(rc).max())
        if task in (2, 4):        # the obstacle penalty / visual rewards follow a flipped pixel (test_objlock_gpu.py)
            rew_bad += int((np.abs(rg - rc)[ok] > 2e-4 * scale).sum()); rew_n += int(ok.sum())
        else:
            assert np.abs(rg - rc)[ok].max() <= 1e-4 * scale, k
        sparse_like = ok & np.isin(np.round(rc, 6), (-0.1, 100.0, -100.0))
        if task == 1:
            assert np.abs(rg - rc)[sparse_like].max(initial=0.0) < 1e-6
    print(f"\n[field task {task} {'generic' if generic else 'std'}] worst state rel err "
          + ", ".join(f"{g}={v:.1e}" for g, v in worst.items()) + f"; flag mismatches {mism}; episodes ended {n_done}")
    # camera tasks: a pixel-column ray grazing a silhouette can flip a visibility counter (test_objlock_gpu.py)
    assert mism <= (2 if task in (2, 4) else 0)
    assert rew_bad <= 0.002 * max(rew_n, 1)
    assert max(worst.values()) < RTOL


def test_field_one_second_free_run_divergence():
    field = make_field()
    cfg = field_cfg(1, field)
    N = 1024
    env = FixedwingVecEnv(N, config=cfg, seed=2, wind_field=field)
    orc = fwf.FieldOracleVecEnv(cfg.as_dict(), N, seed=2, wind_field=field)
    env.reset(); orc.reset()
    rng = np.random.default_rng(2)
    alive = np.ones(N, bool)
    div = []
    for _ in range(30):
        a = rng.uniform(-1, 1, (N, 4)).astype(np.float32)
        og, _, fg, _ = env.step_arrays(a)
        oc, _, fc, _ = orc.step(a.astype(np.float64))
        alive &= (fg.astype(np.int32) == fc) & ((fc & 3) == 0)
        div.append(float(np.abs(og[alive][:, 9:12] - oc[alive][:, 9:12]).max()) if alive.any() else 0.0)
    print(f"\n[field] 1 s free-run (240 substeps, {int(alive.sum())}/{N} envs alive in both): max position divergence "
          f"{div[-1]:.3e} m; trace {['%.1e' % d for d in div[::5]]}")
    assert alive.mean() > 0.9
    assert div[-1] < 5e-3


def test_one_point_field_equals_constant_wind_on_the_gpu():
    v = np.array([3.0, -2.0, 0.5], np.float32)
    field = WindField(np.broadcast_to(v, (1, 1, 1, 1, 3)), origin=0.0, spacing=1.0)
    base = dict(noise_ratio=0.0, wind_start_substep=0)
    env_f = FixedwingVecEnv(512, config=fw.waypoints_v3(**base), seed=4, wind_field=field)
    env_c = FixedwingVecEnv(512, config=fw.waypoints_v3(**base).replace(wind_mode=1, wind_base=[float(x) for x in v]), seed=4)
    env_f.reset(); env_c.reset()
    rng = np.random.default_rng(0)
    worst = 0.0
    for _ in range(20):
        env_f.set_state(env_c.get_state() | {"wind": np.zeros((512, 7), np.float32)})
        a = rng.uniform(-1, 1, (512, 4)).astype(np.float32)
        of, rf, ff, _ = (x.copy() for x in env_f.step_arrays(a))
        oc, rc, fc, _ = (x.copy() for x in env_c.step_arrays(a))
        assert np.array_equal(ff, fc)
        worst = max(worst, float((np.abs(of - oc) / np.maximum(np.abs(oc), 1.0)).max()))
    print(f"\n[1x1x1x1 field vs constant wind] worst rel obs difference {worst:.1e}")
    assert worst < 1e-5


def test_field_sharding_is_split_invariant():
    field = make_field()
    cfg = field_cfg(1, field, max_steps=20)      # short episodes: new shift / time offset draws inside the window
    full = FixedwingVecEnv(256, config=cfg, seed=3, wind_field=field)
    lo = FixedwingVecEnv(128, config=cfg, seed=3, env_id0=0, wind_field=field)
    hi = FixedwingVecEnv(128, config=cfg, seed=3, env_id0=128, wind_field=field)
    assert np.array_equal(full.reset(), np.concatenate([lo.reset(), hi.reset()]))
    full.step_random(60); lo.step_random(60); hi.step_random(60)
    sf, sl, sh = full.get_state(), lo.get_state(), hi.get_state()
    for k in ("pos", "quat", "vel", "episode", "targets", "wind", "act"):
        assert np.array_equal(sf[k], np.concatenate([sl[k], sh[k]])), k
    assert int(sf["episode"].min()) >= 2
    for e in (full, lo, hi):
        e.close()


@pytest.mark.parametrize("task", [2, 4])
def test_field_spare_episodes_equal_inline_resets(task, monkeypatch):
    field = make_field()
    cfg = field_cfg(task, field, num_obstacles=4, max_steps=12)      # short episodes: many resets in the window
    spare = FixedwingVecEnv(128, config=cfg, seed=5, wind_field=field)
    monkeypatch.setenv("FWSIM_SPARE", "0")
    inline = FixedwingVecEnv(128, config=cfg, seed=5, wind_field=field)
    assert np.array_equal(spare.reset(), inline.reset())
    rng = np.random.default_rng(1)
    for _ in range(80):
        a = rng.uniform(-1, 1, (128, 4)).astype(np.float32)
        os_, rs, fs, ts = (x.copy() for x in spare.step_arrays(a))
        oi, ri, fi, ti = (x.copy() for x in inline.step_arrays(a))
        assert np.array_equal(fs, fi) and np.array_equal(os_, oi) and np.array_equal(rs, ri)
    st = spare.spare_stats()
    assert st["from_spare"] > 0, st
    assert inline.spare_stats()["from_spare"] == 0
    spare.close(); inline.close()


def test_set_wind_field_lifecycle_and_state_round_trip():
    lib = _lib.load()
    field = make_field()
    cfg = field_cfg(1, field)
    c = cfg.to_c()
    h = C.c_void_p()
    _lib.check(lib.fw_create(C.byref(c), 64, 0, 1, 0, C.byref(h)))
    try:
        assert lib.fw_step_random(h, 1, None, None, None) == -4          # FW_ESTATE before the field is set
        assert lib.fw_reset_host(h, None) == -4
        desc = field.to_c()
        assert lib.fw_set_wind_field(h, C.byref(desc)) == 0
        assert lib.fw_set_wind_field(h, C.byref(desc)) == -4             # one field per handle
        assert lib.fw_step_random(h, 2, None, None, None) == 0
    finally:
        lib.fw_destroy(h)
    c2 = fw.waypoints_v3(wind={"enabled": True, "mode": "gust_sine"}).to_c()
    h2 = C.c_void_p()
    _lib.check(lib.fw_create(C.byref(c2), 8, 0, 1, 0, C.byref(h2)))
    try:
        assert lib.fw_set_wind_field(h2, C.byref(field.to_c())) == -1    # not a wind_mode 3 handle
    finally:
        lib.fw_destroy(h2)
    with pytest.raises(ValueError, match="wind_field"):
        FixedwingVecEnv(8, config=cfg)
    env = FixedwingVecEnv(64, config=cfg, seed=1, wind_field=field)
    w = env.get_state()["wind"]
    assert np.all(w[:, 0:2] >= -10) and np.all(w[:, 0:2] <= 10) and np.all(np.abs(w[:, 2]) <= 2)
    assert np.all(w[:, 3:6] == 0) and np.all((w[:, 6] >= 0) & (w[:, 6] < 8 * 0.5)) and np.ptp(w[:, 6]) > 0.5
    w2 = w.copy()
    w2[:, 0] = np.linspace(-3, 3, 64); w2[:, 6] = np.linspace(0, 3.5, 64)
    env.set_state({"wind": w2})
    assert np.array_equal(env.get_state()["wind"], w2)
    env.seed(9)                                   # a rebuild keeps the field
    assert env.wind_field is field
    env.step_random(3)
    env.close()


def test_ppo_learns_on_a_field_env_and_evaluates_in_the_same_field():
    import torch
    from pyflyt_drone_b200.ppo import PPO
    field = make_field()
    env = FixedwingVecEnv(1024, config=field_cfg(1, field), seed=3, wind_field=field)
    m = PPO("MlpPolicy", env, n_steps=16, batch_size=4096, n_epochs=2, seed=5)
    before = m.policy.theta.clone()
    m.learn(3 * 16 * 1024)
    assert torch.isfinite(m.policy.theta).all() and not torch.equal(before, m.policy.theta)
    seen = {}
    orig = FixedwingVecEnv.__init__

    def spy(self, *a, **kw):
        orig(self, *a, **kw)
        seen["field"] = self.wind_field
        seen["mode"] = self.cfg.wind_mode

    FixedwingVecEnv.__init__ = spy
    try:
        r = m.evaluate_policy(n_eval_episodes=32)
    finally:
        FixedwingVecEnv.__init__ = orig
    assert seen["field"] is field and seen["mode"] == 3
    assert all(np.isfinite(x) for x in r)
    env.close()


def test_gym_views_fly_the_field():
    from pyflyt_drone_b200.gym_env import FixedwingLowLevelEnv, FixedwingWaypointsEnv
    field = make_field(randomize_time=False)
    g1 = FixedwingWaypointsEnv(wind_config={"enabled": True, "mode": "field", "field": field}, seed=11)
    assert g1.cfg.wind_mode == 3 and g1.cfg.wind_start_substep == 0 and g1.cfg.wind_randomize == 0
    ref = FixedwingVecEnv(1, config=g1.cfg, seed=11, wind_field=field)
    g2 = FixedwingWaypointsEnv(seed=11)
    with pytest.raises(NotImplementedError, match="origin="):
        g2.env.register_wind_field_function(shear_thermal)
    g2.env.register_wind_field_function(shear_thermal, origin=(-100.0, -100.0, 0.0), spacing=(10.0, 10.0, 5.0),
                                        shape=(21, 21, 21), n_slices=8, t_step=0.5)
    assert g2.cfg.wind_mode == 3 and g2.cfg.wind_start_substep == 20
    g1.reset(); g2.reset()
    calm = FixedwingWaypointsEnv(seed=11)
    calm.reset()
    o_ref = ref.reset()
    a = np.array([0.1, 0.2, 0.0, 0.6])
    for _ in range(20):
        s1, *_ = g1.step(a)
        s2, *_ = g2.step(a)
        sc, *_ = calm.step(a)
        o_ref, *_ = ref.step_arrays(a[None].astype(np.float32))
    p_ref = ref.get_state()["pos"][0]
    p1, p2, pc = g1._state()["pos"][0], g2._state()["pos"][0], calm._state()["pos"][0]
    np.testing.assert_allclose(p1, p_ref, rtol=0, atol=1e-4)    # the env-hook gym view and the vec env fly the same field
    assert np.linalg.norm(p2 - pc) > 1e-2         # register_wind_field_function changes the flight
    assert np.linalg.norm(p1 - pc) > 1e-2
    ll = FixedwingLowLevelEnv(wind_config={"enabled": True, "mode": "field", "field": field}, seed=3)
    ll.reset()
    for _ in range(5):
        ll.step(np.zeros(6))
    for e in (g1, g2, calm, ll):
        e.close()
    ref.close()
