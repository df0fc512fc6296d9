"""PPO.evaluate (device-resident evaluation, ppo_eval_ledger) against the host loop of PPO.evaluate_policy, and the
EvalCallback / CheckpointCallback around PPO.learn."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

CONFIGS = {
    "waypoints_sparse_euler": ("waypoints_v3", {}),
    "waypoints_dense_quaternion": ("waypoints_v3", {"sparse_reward": 0, "angle_repr": 1}),
    "waypoint_objlock": ("waypoint_objlock", {}),
    "lowlevel": ("lowlevel", {}),
    "objlock_duck": ("objlock_duck", {}),
    "wind_field": ("waypoints_v3", {"wind_field": True}),
}


def _field():
    from pyflyt_drone_b200.wind import WindField

    def f(t, x):
        z = np.maximum(x[:, 2], 0.0)
        return np.stack([5.0 * (1.0 - np.exp(-z / 15.0)), 0.5 + 0.02 * x[:, 0], 1.5 * np.sin(0.05 * x[:, 1] + 0.3 * t)], axis=1)
    return WindField.from_function(f, origin=(-100.0, -100.0, 0.0), spacing=(10.0, 10.0, 5.0), shape=(21, 21, 21), n_slices=4,
                                   t_step=1.0)


def _model(name, n_envs=16, seed=5, **ppo_kw):
    from pyflyt_drone_b200.ppo import PPO
    from pyflyt_drone_b200.vec_env import FixedwingVecEnv
    preset, over = CONFIGS[name]
    over = dict(over)
    field = _field() if over.pop("wind_field", False) else None
    env = FixedwingVecEnv(n_envs, preset=preset, seed=seed, wind_field=field, **over)
    m = PPO("MlpPolicy", env, n_steps=16, batch_size=n_envs * 16, n_epochs=2, seed=seed, **ppo_kw)
    with torch.no_grad():           # actions away from the near-zero initial head, so episodes differ between envs
        m.policy.theta.add_(0.05 * torch.randn(m.policy.count, device=m.device, generator=m._gen))
    return m


def _host_record(m, env, n_eval_episodes, max_steps=None):
    """evaluate_policy's loop, step for step, recording each selected episode (return, length, targets, flags, env, step)."""
    obs = env.reset_tensor()
    n = env.num_envs
    quota = torch.tensor(m.episode_quotas(n_eval_episodes, n), dtype=torch.int64, device=m.device)
    count = torch.zeros(n, dtype=torch.int64, device=m.device)
    ret = torch.zeros(n, dtype=torch.float64, device=m.device)
    length = torch.zeros(n, dtype=torch.int64, device=m.device)
    has_targets = env.cfg.task in (1, 2)
    limit = max_steps if max_steps is not None else int(quota.max()) * (int(env.cfg.max_steps) + 2) + 8
    rec = []
    for s in range(limit):
        act = m.predict(obs, deterministic=True)
        obs, rew, flags = env.step_tensor(act)
        ret += rew.double()
        length += 1
        fin = (flags & 3) != 0
        take = fin & (count < quota)
        if bool(take.any()):
            idx = take.nonzero().flatten()
            tr = env.targets_reached_tensor()[idx].tolist() if has_targets else [0] * len(idx)
            rec += list(zip(ret[idx].tolist(), length[idx].tolist(), tr, flags[idx].tolist(), idx.tolist(), [s] * len(idx)))
            count += take.to(torch.int64)
        ret[fin] = 0.0
        length[fin] = 0
        if bool((count >= quota).all()):
            break
    return rec


def _table(res):
    return list(zip(res.returns.tolist(), res.lengths.tolist(), res.targets_reached.tolist(), res.flags.tolist(),
                    res.env_index.tolist(), res.finish_step.tolist()))


def _same(a, b):
    for k in ("returns", "lengths", "targets_reached", "flags", "env_index", "finish_step"):
        assert np.array_equal(getattr(a, k), getattr(b, k)), k
    for k in ("mean_reward", "std_reward", "mean_length", "mean_targets_reached"):
        assert np.array_equal(getattr(a, k), getattr(b, k), equal_nan=True), k


def _check_parity(m, n_eval, max_steps=None):
    env = m.make_eval_env(n_eval)
    host = _host_record(m, env, n_eval, max_steps)
    env.close()
    res = m.evaluate(n_eval_episodes=n_eval, max_steps=max_steps)
    ref = m.evaluate_policy(n_eval_episodes=n_eval, max_steps=max_steps)
    assert _table(res) == host                                          # every episode, bit for bit, in SB3's order
    got = (res.mean_reward, res.std_reward, res.mean_length, res.mean_targets_reached)
    assert np.array_equal(np.array(got), np.array(ref), equal_nan=True), (got, ref)
    return res


@pytest.mark.parametrize("name", list(CONFIGS))
def test_episodes_and_means_equal_the_host_loop(name):
    m = _model(name)
    res = _check_parity(m, 37)                          # 16 envs, quotas of 2 and 3
    assert res.n_episodes == 37 and np.array_equal(np.bincount(res.env_index, minlength=16), m.episode_quotas(37, 16))
    assert np.isfinite(res.returns).all() and (res.flags & 3).all()
    m.env.close()


def test_briefly_trained_policy_reaches_waypoints_and_stays_bit_identical():
    from pyflyt_drone_b200.ppo import PPO
    from pyflyt_drone_b200.vec_env import FixedwingVecEnv
    env = FixedwingVecEnv(2048, preset="waypoints_v3", seed=21)
    m = PPO("MlpPolicy", env, n_steps=64, batch_size=2048 * 16, n_epochs=10, seed=21)
    m.learn(40 * 64 * 2048)
    res = _check_parity(m, 256)
    assert (res.targets_reached > 0).any() and res.wp_reach_rate[0] > 0
    print(f"\n[evaluate] trained 5.2 M steps: {res.metrics()}")
    env.close()


def test_quotas_with_a_caller_supplied_env():
    from pyflyt_drone_b200.vec_env import FixedwingVecEnv
    m = _model("waypoints_sparse_euler")
    for n_envs, n_eval in ((7, 20), (7, 5)):            # fewer envs than episodes; more envs than episodes (zero quotas)
        a = FixedwingVecEnv(n_envs, preset="waypoints_v3", seed=77)
        b = FixedwingVecEnv(n_envs, preset="waypoints_v3", seed=77)
        host = _host_record(m, a, n_eval)
        res = m.evaluate(env=b, n_eval_episodes=n_eval)
        assert _table(res) == host
        assert np.array_equal(np.bincount(res.env_index, minlength=n_envs), m.episode_quotas(n_eval, n_envs))
        a.close(); b.close()
    m.env.close()


def test_max_steps_cuts_inside_a_chunk():
    m = _model("waypoints_sparse_euler")
    for max_steps in (150, 3):                          # neither a multiple of the chunk; the second ends before any episode
        res = _check_parity(m, 200, max_steps=max_steps)
        assert res.n_episodes < 200 and (res.finish_step < max_steps).all()
    m.env.close()


@pytest.mark.parametrize("name", ["waypoints_sparse_euler", "objlock_duck"])
def test_graph_replay_equals_the_eager_path(name):
    from pyflyt_drone_b200.vec_env import FixedwingVecEnv
    m = _model(name)

    def run(use_graph):
        env = FixedwingVecEnv(12, preset=CONFIGS[name][0], seed=9)
        m.use_graph, m._eval_state = use_graph, None
        out = [m.evaluate(env=env, n_eval_episodes=40) for _ in range(2)]    # the second call replays the graph kept for env
        assert (m._eval_state["graph"] is not None) == use_graph
        m._eval_state = None
        env.close()
        return out

    eager, graph = run(False), run(True)
    for e, g in zip(eager, graph):
        assert e.n_episodes == 40
        _same(e, g)
    m.env.close()


def test_stochastic_evaluation_is_reproducible_and_leaves_the_training_counters_alone():
    m = _model("waypoints_sparse_euler")
    step0 = m._step_dev.clone()
    calls0 = getattr(m, "_predict_calls", 0)
    a = m.evaluate(n_eval_episodes=30, deterministic=False)
    b = m.evaluate(n_eval_episodes=30, deterministic=False)
    _same(a, b)
    d = m.evaluate(n_eval_episodes=30, deterministic=True)
    assert not np.array_equal(a.returns, d.returns)
    assert torch.equal(m._step_dev, step0) and getattr(m, "_predict_calls", 0) == calls0
    other = _model("waypoints_sparse_euler", seed=6)
    with torch.no_grad():
        other.policy.theta.copy_(m.policy.theta)
    c = other.evaluate(n_eval_episodes=30, deterministic=False)
    assert not np.array_equal(a.returns, c.returns)
    m.env.close(); other.env.close()


def _train(with_callback, tmp_path=None):
    from pyflyt_drone_b200.callbacks import EvalCallback
    from pyflyt_drone_b200.ppo import PPO
    from pyflyt_drone_b200.vec_env import FixedwingVecEnv
    env = FixedwingVecEnv(512, preset="waypoints_v3", seed=13)
    m = PPO("MlpPolicy", env, n_steps=32, batch_size=512 * 8, n_epochs=2, seed=13, ent_coef=0.001)
    cb = EvalCallback(eval_freq=32 * 512, n_eval_episodes=24) if with_callback else None
    m.learn(4 * 32 * 512, callback=cb)
    return m, env, cb


def test_evaluation_does_not_disturb_training():
    m0, env0, _ = _train(False)
    m1, env1, cb = _train(True)
    assert len(cb.evaluations_timesteps) == 4 and cb.last_result.n_episodes == 24
    for a, b in ((m0.policy.theta, m1.policy.theta), (m0._adam_m, m1._adam_m), (m0._adam_v, m1._adam_v),
                 (m0._adam_t, m1._adam_t), (m0._step_dev, m1._step_dev), (m0.vecnorm.obs_stats, m1.vecnorm.obs_stats),
                 (m0.vecnorm.ret_stats, m1.vecnorm.ret_stats), (m0.vecnorm.ret, m1.vecnorm.ret)):
        assert torch.equal(a, b)
    s0, s1 = env0.get_state(), env1.get_state()
    assert s0.keys() == s1.keys() and all(np.array_equal(s0[k], s1[k]) for k in s0)
    cb.close(); env0.close(); env1.close()


def test_callback_files(tmp_path):
    from pyflyt_drone_b200.callbacks import CheckpointCallback, EvalCallback
    from pyflyt_drone_b200.ppo import PPO
    from pyflyt_drone_b200.vec_env import FixedwingVecEnv
    env = FixedwingVecEnv(256, preset="waypoint_objlock", seed=4)
    m = PPO("MlpPolicy", env, n_steps=16, batch_size=256 * 8, n_epochs=2, seed=4)
    ev = EvalCallback(eval_freq=10_000, n_eval_episodes=10, best_model_save_path=str(tmp_path / "best"),
                      log_path=str(tmp_path / "logs"))
    ck = CheckpointCallback(save_freq=8_192, save_path=str(tmp_path / "ckpt"), name_prefix="objlock")
    m.learn(6 * 16 * 256, callback=lambda l, g: ev(l, g) and ck(l, g))     # 4,096 timesteps per iteration
    z = np.load(tmp_path / "logs" / "evaluations.npz")
    assert sorted(z.files) == ["ep_lengths", "results", "successes", "timesteps"]
    assert z["timesteps"].tolist() == [12_288, 20_480]
    assert z["results"].shape == z["ep_lengths"].shape == z["successes"].shape == (2, 10)
    assert z["results"].dtype == np.float64 and z["successes"].dtype == np.bool_
    assert "eval/duck_strike_rate" in ev.last_metrics and "eval/wp8_reach_rate" in ev.last_metrics
    names = sorted(os.listdir(tmp_path / "ckpt"))
    assert names == sorted(f"objlock_{s}{t}_steps.{x}" for t in (8_192, 16_384, 24_576)
                           for s, x in (("", "zip"), ("vecnormalize_", "pkl")))
    # the best model round-trips through import_sb3: force a save of the current parameters and statistics
    ev.best_mean_reward = -np.inf
    ev.evaluate(m)
    m2 = PPO("MlpPolicy", FixedwingVecEnv(8, preset="waypoint_objlock", seed=1), n_steps=16, batch_size=128, seed=99)
    m2.import_sb3(str(tmp_path / "best"))
    assert torch.equal(m2.policy.theta, m.policy.theta)
    assert torch.equal(m2._adam_m, m._adam_m) and torch.equal(m2._adam_v, m._adam_v)
    assert torch.equal(m2.vecnorm.obs_stats, m.vecnorm.obs_stats) and torch.equal(m2.vecnorm.ret_stats, m.vecnorm.ret_stats)
    ev.close(); m2.env.close(); env.close()
