"""High-level waypoints (task 5) on the device: single steps against the fp64 reference of tests/highlevel_oracle.py, the
bitwise contract with PPO.predict of the tracker model, lane / graph / sharding equivalences, the lifecycle of the tracker,
and PPO / PPOPopulation on the task."""
import ctypes as C

import numpy as np
import pytest
import torch

import pyflyt_drone_b200 as fw
from pyflyt_drone_b200 import _lib
from pyflyt_drone_b200.tracker import Tracker

pytestmark = pytest.mark.gpu
RTOL = 1e-4
OBS_GROUPS = {"ang_vel": slice(0, 3), "euler": slice(3, 6), "lin_vel": slice(6, 9), "pos": slice(9, 12),
              "action": slice(12, 16), "aux": slice(16, 22), "targets": slice(22, 28)}
TRK_GROUPS = {"ang_vel": slice(0, 3), "euler": slice(3, 6), "lin_vel": slice(6, 9), "pos": slice(9, 12),
              "prev_action": slice(12, 18), "command": slice(18, 21)}


def make_tracker(seed=0, gain=60.0) -> Tracker:
    """A non-trivial tracker: SB3's init with the action head scaled up from its 0.01 gain, random frozen statistics."""
    from pyflyt_drone_b200.ppo import FlatMlpPolicy
    pol = FlatMlpPolicy(21, torch.device("cpu"), seed=seed, act_dim=6)
    with torch.no_grad():
        pol.view("action_net.weight").mul_(gain)
        pol.view("action_net.bias").uniform_(-0.3, 0.3)
    rng = np.random.default_rng(seed)
    scale = np.r_[np.full(3, 1.0), np.full(3, 1.0), np.full(3, 10.0), np.full(3, 20.0), np.full(6, 0.5), [1.5, 10.0, 15.0]]
    mean = rng.normal(0, 0.3, 21) * scale
    var = (scale * rng.uniform(0.5, 1.5, 21)) ** 2
    return Tracker(pol.theta.detach().numpy(), mean, var, clip_obs=10.0)


def group_err(got, ref, groups, angles=slice(3, 6)):
    d = got - ref
    d[:, angles] = (d[:, angles] + np.pi) % (2 * np.pi) - np.pi
    out = {}
    for k, sl in groups.items():
        if sl.start >= ref.shape[1]:
            continue
        scale = np.maximum(np.abs(ref[:, sl]).max(axis=1), 1.0)
        out[k] = float((np.abs(d[:, sl]).max(axis=1) / scale).max()) if len(d) else 0.0
    return out


def _field():
    from pyflyt_drone_b200.wind import WindField

    def f(t, x):
        z = np.maximum(x[:, 2], 0.0)
        return np.stack([6.0 * (1.0 - np.exp(-z / 15.0)), 0.5 + 0.02 * x[:, 0], 1.5 * np.exp(-(x[:, 0] ** 2 + x[:, 1] ** 2) / 300.0)], 1)
    return WindField.from_function(f, origin=(-100.0, -100.0, 0.0), spacing=(10.0, 10.0, 5.0), shape=(21, 21, 21), n_slices=4,
                                   t_step=0.5, shift_range=[(-10.0, 10.0), (-10.0, 10.0), (-2.0, 2.0)], randomize_time=True)


def _pair(oracle_mod, wind, generic, n, tracker, **kw):
    from tests.field_oracle import FieldOracleVecEnv
    from tests.highlevel_oracle import HighLevelOracle
    field = None
    if wind == "constant":
        kw["wind"] = dict(enabled=True, mode="constant", wind_enu_mps_range=[[-5, 5], [-5, 5], [-0.5, 0.5]], randomize_on_reset=True)
    if wind == "field":
        field = _field()
        kw["wind"] = {"enabled": True, "mode": "field", "field": field, "randomize_on_reset": True}
    cfg = fw.make_config("highlevel", force_generic_kernel=int(generic), **kw)
    env = fw.FixedwingVecEnv(n, config=cfg, seed=7, tracker=tracker, wind_field=field)
    d1 = cfg.replace(task=1).as_dict()
    base = FieldOracleVecEnv(d1, n, seed=7, wind_field=field) if field is not None else oracle_mod.OracleVecEnv(d1, n, seed=7)
    return env, HighLevelOracle(base, tracker), cfg


@pytest.mark.parametrize("generic", [False, True], ids=["std", "generic"])
@pytest.mark.parametrize("wind", ["off", "constant", "field"])
def test_single_steps_against_the_fp64_reference(oracle_mod, wind, generic):
    N = 1024
    tracker = make_tracker(1)
    env, orc, cfg = _pair(oracle_mod, wind, generic, N, tracker, sparse_reward=1)
    tob = torch.zeros((N, 21), dtype=torch.float32, device="cuda")
    env.set_tracker_obs_buffer(tob)
    e = group_err(env.reset().astype(np.float64), orc.reset(), OBS_GROUPS)
    assert max(e.values()) < RTOL, e
    rng = np.random.default_rng(3)
    worst, worst_trk, worst_act, n_done, n_reach = {}, {}, 0.0, 0, 0
    for k in range(8):
        st = orc.get_state()
        if k % 4 == 1:                                # step limit, dome edge, and a waypoint within reach
            st["step_count"][:16] = cfg.max_steps + 1
            st["pos"][16:32] = st["pos"][16:32] / np.linalg.norm(st["pos"][16:32], axis=1, keepdims=True) * 99.9
            tix = np.minimum(st["target_idx"][32:64], cfg.num_targets - 1)
            st["targets"][np.arange(32, 64), tix] = st["pos"][32:64] + [1.0, 0.5, 0.0]
            orc.set_state(st)
            st = orc.get_state()
        env.set_state(st)
        orc.prev[:] = orc.prev.astype(np.float32)
        env.set_tracker_state(orc.prev)
        a = rng.uniform(-1.2, 1.2, (N, 4)).astype(np.float32)
        og, rg, fg, tg = (x.astype(np.float64) for x in env.step_arrays(a))
        oc, rc, fc, tc = orc.step(a.astype(np.float64))
        assert np.array_equal(fg.astype(np.int32), fc), (k, np.nonzero(fg.astype(np.int32) != fc))
        done = (fc & 3) != 0
        n_done += int(done.sum())
        n_reach += int((rc == 100.0).sum())
        # sparse rewards are exact (-0.1, -100, 100)
        assert np.array_equal(rg, rc.astype(np.float32).astype(np.float64)), k
        ge = group_err(og, oc, OBS_GROUPS)
        if done.any():
            et = group_err(tg[done], tc[done], OBS_GROUPS)
            ge = {g: max(ge[g], et.get(g, 0.0)) for g in ge}
        for g, v in ge.items():
            worst[g] = max(worst.get(g, 0.0), v)
        live = ~done
        # the tracker's last decision of the step: its observation and its action (zeroed by the reset of a done env)
        te = group_err(tob.cpu().numpy().astype(np.float64), orc.last_tracker_obs, TRK_GROUPS)
        for g, v in te.items():
            worst_trk[g] = max(worst_trk.get(g, 0.0), v)
        prev = env.get_tracker_state().astype(np.float64)
        worst_act = max(worst_act, float(np.abs(prev[live] - orc.last_tracker_act[live]).max()))
        assert not prev[done].any()
    print(f"\n[highlevel/{wind}/{'generic' if generic else 'std'}] obs {worst}; tracker obs {worst_trk}; "
          f"tracker action {worst_act:.2e}; done {n_done}, waypoints reached {n_reach}")
    assert n_done > 0 and n_reach > 0
    assert max(worst.values()) < RTOL, worst
    assert max(worst_trk.values()) < RTOL, worst_trk
    assert worst_act < 1e-5
    env.close()


@pytest.mark.parametrize("agent_hz", [120, 30])
def test_tracker_action_is_ppo_predict_bit_for_bit(agent_hz):
    from pyflyt_drone_b200.ppo import PPO
    low = fw.FixedwingVecEnv(64, preset="lowlevel", seed=1)
    model = PPO("MlpPolicy", low, seed=4, n_steps=8, batch_size=256)
    with torch.no_grad():
        model.policy.view("action_net.weight").mul_(60.0)
    rng = np.random.default_rng(0)
    vn = model.vecnorm.obs_stats
    vn[:21] = torch.as_tensor(rng.normal(0, 1, 21)); vn[21:42] = torch.as_tensor(rng.uniform(0.2, 30.0, 21))
    tracker = Tracker.from_ppo(model)
    N = 2048
    env = fw.FixedwingVecEnv(N, preset="highlevel", seed=2, tracker=tracker, inner_per_step=120 // agent_hz)
    tob = torch.zeros((N, 21), dtype=torch.float32, device="cuda")
    env.set_tracker_obs_buffer(tob)
    env.reset_tensor()
    g = torch.Generator(device="cuda").manual_seed(0)
    checked = 0
    for _ in range(20):
        act = torch.rand((N, 4), device="cuda", generator=g) * 2.4 - 1.2
        _, _, flags = env.step_tensor(act.contiguous())
        live = (flags & 3) == 0
        pred = model.predict(tob, deterministic=True)
        got = torch.as_tensor(env.get_tracker_state(), device="cuda")
        assert torch.equal(got[live], pred[live])
        checked += int(live.sum())
    assert checked > 10 * N
    env.close(); low.close()


def _run(env, acts, lane):
    out = []
    for a in acts:
        if lane == "host":
            o, r, f, _ = env.step_arrays(a.cpu().numpy())
            out.append((torch.as_tensor(o.copy()), torch.as_tensor(r.copy()), torch.as_tensor(f.copy())))
        else:
            o, r, f = env.step_tensor(a)
            out.append((o.cpu(), r.cpu(), f.cpu()))
    return out


def test_device_lane_host_lane_graph_and_split_agree():
    tracker = make_tracker(2)
    N = 4096
    g = torch.Generator(device="cuda").manual_seed(1)
    acts = [(torch.rand((N, 4), device="cuda", generator=g) * 2 - 1).contiguous() for _ in range(40)]
    mk = lambda n=N, env_id0=0: fw.FixedwingVecEnv(n, preset="highlevel", seed=9, env_id0=env_id0, tracker=tracker)  # noqa: E731
    dev, host = mk(), mk()
    dev.reset_tensor(); host.reset()
    a_dev, a_host = _run(dev, acts, "device"), _run(host, acts, "host")
    for x, y in zip(a_dev, a_host):
        for u, v in zip(x, y):
            assert torch.equal(u, v)
    # eager against a captured, replayed CUDA graph of the step
    eager, graphed = mk(), mk()
    eager.reset_tensor(); graphed.reset_tensor()
    buf = acts[0].clone()
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        graphed.step_tensor(buf)                          # warm-up launch (module load, smem opt-in)
    torch.cuda.current_stream().wait_stream(st)
    eager.step_tensor(acts[0])
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        go, grw, gf = graphed.step_tensor(buf)
    for a in acts[1:]:
        buf.copy_(a)
        gr.replay()
        eo, er, ef = eager.step_tensor(a)
        assert torch.equal(go, eo) and torch.equal(grw, er) and torch.equal(gf, ef)
    # one handle against the same envs split over two (global-env-id Philox: random actions and resets agree)
    one, lo, hi = mk(), mk(N // 2, 0), mk(N // 2, N // 2)
    for e in (one, lo, hi):
        e.step_random(30)
    s1, sl, sh = one.get_state(), lo.get_state(), hi.get_state()
    for k in ("pos", "quat", "vel", "step_count", "episode", "target_idx"):
        assert np.array_equal(s1[k], np.concatenate([sl[k], sh[k]])), k
    assert np.array_equal(one.get_tracker_state(), np.concatenate([lo.get_tracker_state(), hi.get_tracker_state()]))
    assert one.get_tracker_state().any()
    for e in (dev, host, eager, graphed, one, lo, hi):
        e.close()


def test_lifecycle():
    lib = _lib.load()
    tracker = make_tracker(3)
    cfg = fw.make_config("highlevel").to_c()
    h = C.c_void_p()
    _lib.check(lib.fw_create(C.byref(cfg), 64, 0, 1, 0, C.byref(h)))
    assert lib.fw_obs_dim(h) == 28 and lib.fw_act_dim(h) == 4
    obs = torch.zeros((64, 28), device="cuda")
    act = torch.zeros((64, 4), device="cuda")
    prev = np.zeros((64, 6), np.float32)
    assert lib.fw_reset(h, None, C.c_void_p(obs.data_ptr()), None) == -4
    assert lib.fw_step(h, C.c_void_p(act.data_ptr()), C.c_void_p(obs.data_ptr()), None, None, None, None) == -4
    assert lib.fw_step_random(h, 1, None, None, None) == -4
    assert lib.fw_reset_host(h, None) == -4 and lib.fw_observe_host(h, None) == -4
    assert lib.fw_get_tracker_state(h, prev.ctypes.data_as(C.c_void_p)) == -4
    desc = tracker.to_c()
    _lib.check(lib.fw_set_tracker(h, C.byref(desc)))
    assert lib.fw_set_tracker(h, C.byref(desc)) == -4                     # one-shot
    _lib.check(lib.fw_reset(h, None, C.c_void_p(obs.data_ptr()), None))
    _lib.check(lib.fw_step(h, C.c_void_p(act.data_ptr()), C.c_void_p(obs.data_ptr()), None, None, None, None))
    arr = (C.c_void_p * 1)(h.value)
    assert lib.fw_rollout_random(arr, 1, 1, 1, 0, None) == -1
    rgba = torch.zeros((8, 8, 4), dtype=torch.uint8, device="cuda")
    assert lib.fw_render(h, 0, 8, 8, C.c_void_p(rgba.data_ptr()), None, None, None) == -1
    lib.fw_destroy(h)
    cfg1 = fw.make_config("waypoints_v3").to_c()
    _lib.check(lib.fw_create(C.byref(cfg1), 64, 0, 1, 0, C.byref(h)))
    assert lib.fw_set_tracker(h, C.byref(desc)) == -1 and lib.fw_set_tracker_obs_buffer(h, None) == -1
    lib.fw_destroy(h)
    # seed() rebuilds the batch and keeps the tracker (and the tracker observation buffer)
    env = fw.FixedwingVecEnv(256, preset="highlevel", seed=1, tracker=tracker)
    tob = torch.zeros((256, 21), device="cuda")
    env.set_tracker_obs_buffer(tob)
    env.seed(5)
    ref = fw.FixedwingVecEnv(256, preset="highlevel", seed=5, tracker=tracker)
    a = np.random.default_rng(0).uniform(-1, 1, (256, 4)).astype(np.float32)
    env.reset(); ref.reset()
    for _ in range(5):
        o1 = env.step_arrays(a)[0].copy()
        o2 = ref.step_arrays(a)[0].copy()
        assert np.array_equal(o1, o2)
    assert np.array_equal(env.get_tracker_state(), ref.get_tracker_state()) and tob.abs().sum() > 0
    # a masked device-lane reset zeroes the tracker's previous action of the reset envs only
    mask = torch.zeros(256, dtype=torch.uint8, device="cuda"); mask[:10] = 1
    before = env.get_tracker_state()
    env.reset_tensor(mask)
    after = env.get_tracker_state()
    assert not after[:10].any() and np.array_equal(after[10:], before[10:]) and before[10:].any()
    env.close(); ref.close()


def test_ppo_learn_evaluate_and_population_twin():
    from pyflyt_drone_b200.population import PPOPopulation
    from pyflyt_drone_b200.ppo import PPO
    tracker = make_tracker(4)
    env = fw.FixedwingVecEnv(512, preset="highlevel", seed=3, tracker=tracker, sparse_reward=0)
    model = PPO("MlpPolicy", env, n_steps=16, batch_size=512, n_epochs=2, seed=3)
    model.learn(512 * 16 * 2)
    assert torch.isfinite(model.policy.theta).all()
    res = model.evaluate(n_eval_episodes=20, max_steps=400)
    assert res.has_targets and res.n_episodes > 0 and np.isfinite(res.mean_reward)
    assert model.make_eval_env(4).tracker is tracker
    env.close()
    # a two-member population equals its standalone twins
    n, shared = 128, dict(n_steps=8, batch_size=256, n_epochs=2)
    penv = fw.FixedwingVecEnv(2 * n, preset="highlevel", seed=5, env_id0=1000, tracker=tracker, sparse_reward=0)
    pop = PPOPopulation("MlpPolicy", penv, members=2, seed=11, **shared)
    pop.learn(2 * 8 * n)
    assert pop.member_env(1).tracker is tracker
    for m in range(2):
        tenv = fw.FixedwingVecEnv(n, config=penv.cfg, seed=5, env_id0=1000 + m * n, tracker=tracker)
        twin = PPO("MlpPolicy", tenv, **pop.members[m], **shared)
        twin.fused_obs_moments = False
        twin.learn(2 * 8 * n)
        assert torch.equal(pop.theta[m], twin.policy.theta.data)
        for k in ("obs", "act", "rew", "done"):
            assert torch.equal(pop.buf[k][:, m * n:(m + 1) * n], twin.buf[k]), k
        tenv.close()
    penv.close()
