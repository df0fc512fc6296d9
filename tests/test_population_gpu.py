"""PPOPopulation on the device: every member is bit-identical to a standalone PPO trained on that member's slice of the envs.

The standalone twin of member m is ``PPO("MlpPolicy", FixedwingVecEnv(n, config=env.cfg, seed=<env seed>,
env_id0=env.env_id0 + m * n), seed=s_m, **hp_m, **shared)`` with ``fused_obs_moments = False`` (a population folds the
observation moments with the batched moments kernel).  Float tensors must agree bit for bit; the fp64 running statistics to a
relative 1e-12, because both sides' moment and return kernels add block partials with double atomicAdd, whose order varies
from run to run."""
import numpy as np
import pytest
import torch

from pyflyt_drone_b200.population import PPOPopulation

pytestmark = pytest.mark.gpu

ENV_SEED = 5
HPS = [dict(seed=11, learning_rate=3e-4, clip_range=0.2, ent_coef=0.0, vf_coef=0.5, max_grad_norm=0.5, gamma=0.99, gae_lambda=0.95),
       dict(seed=12, learning_rate=1e-3, clip_range=0.1, ent_coef=0.01, vf_coef=0.25, max_grad_norm=1.0, gamma=0.95, gae_lambda=0.9),
       dict(seed=913, learning_rate=5e-5, clip_range=0.3, ent_coef=0.001, vf_coef=1.0, max_grad_norm=0.3, gamma=0.999,
            gae_lambda=0.8)]
BUFFERS = ("obs", "act", "logp", "val", "rew", "done", "adv", "ret")


def _env(P, n, preset, **kw):
    from pyflyt_drone_b200 import FixedwingVecEnv
    return FixedwingVecEnv(P * n, preset=preset, seed=ENV_SEED, env_id0=1000, **kw)


def _twin(pop, m, shared):
    from pyflyt_drone_b200 import FixedwingVecEnv
    from pyflyt_drone_b200.ppo import PPO
    env = FixedwingVecEnv(pop.n, config=pop.env.cfg, seed=ENV_SEED, env_id0=pop.env.env_id0 + m * pop.n)
    model = PPO("MlpPolicy", env, **pop.members[m], **shared)
    model.fused_obs_moments = False
    return model


def _rel(a, b):
    return float(((a - b).abs() / b.abs().clamp_min(1e-300)).max())


def _assert_member_equals(pop, m, model):
    assert torch.equal(pop.theta[m], model.policy.theta.data), "parameters"
    assert torch.equal(pop.adam_m[m], model._adam_m) and torch.equal(pop.adam_v[m], model._adam_v), "Adam moments"
    assert int(pop.adam_t[m]) == int(model._adam_t.item()), "Adam step"
    assert pop.num_timesteps == model.num_timesteps
    cols = slice(m * pop.n, (m + 1) * pop.n)
    for k in BUFFERS:
        assert torch.equal(pop.buf[k][:, cols], model.buf[k]), k
    vn = model.vecnorm
    if vn.norm_obs:
        assert _rel(pop.obs_stats[m], vn.obs_stats) <= 1e-12
    if vn.norm_reward:
        assert _rel(pop.ret_stats[m], vn.ret_stats) <= 1e-12


CASES = [  # preset, envs per member, n_steps, batch_size
    ("waypoints_v3", 200, 16, 128),      # a = 4, d = 28; 200 rows: a masked tail tile per member; multi-step kernel, P blocks
    ("lowlevel", 64, 8, 128),            # a = 6
    ("objlock_duck", 64, 8, 128),        # d = 56: the 64-wide builds
    ("waypoint_objlock", 64, 8, 128),
    ("waypoints_v3", 128, 16, 1024),     # window update per member
    ("waypoints_v3", 64, 8, 200),        # ragged last minibatch
]


@pytest.mark.parametrize("preset,n,n_steps,batch", CASES, ids=[f"{c[0]}-n{c[1]}-b{c[3]}" for c in CASES])
def test_members_are_bit_identical_to_standalone_runs(preset, n, n_steps, batch):
    shared = dict(n_steps=n_steps, batch_size=batch, n_epochs=2)
    env = _env(3, n, preset)
    pop = PPOPopulation("MlpPolicy", env, members=HPS, **shared)
    pop.learn(2 * n_steps * n)             # iteration 1 eager, iteration 2 a captured, replayed rollout graph
    assert pop.num_timesteps == 2 * n_steps * n
    for m in range(3):
        model = _twin(pop, m, shared)
        model.learn(2 * n_steps * n)
        _assert_member_equals(pop, m, model)
        model.env.close()
    env.close()


def test_population_of_one_equals_standalone():
    shared = dict(n_steps=16, batch_size=128, n_epochs=3)
    env = _env(1, 256, "waypoints_v3")
    pop = PPOPopulation("MlpPolicy", env, members=[HPS[1]], **shared)
    pop.learn(2 * 16 * 256)
    model = _twin(pop, 0, shared)
    model.learn(2 * 16 * 256)
    _assert_member_equals(pop, 0, model)


def _state(pop):
    return [pop.theta.clone(), pop.adam_m.clone(), pop.adam_v.clone(), pop.adam_t.clone()] + [pop.buf[k].clone() for k in BUFFERS]


def test_cuda_graph_and_eager_give_the_same_bits():
    shared = dict(n_steps=16, batch_size=128, n_epochs=2)
    out = []
    for graph in (False, True):
        env = _env(3, 96, "waypoints_v3")
        pop = PPOPopulation("MlpPolicy", env, members=HPS, use_cuda_graph=graph, **shared)
        pop.learn(3 * 16 * 96)
        out.append(_state(pop))
        env.close()
    for a, b in zip(*out):
        assert torch.equal(a, b)


def test_changing_one_member_leaves_the_others_bit_identical():
    shared = dict(n_steps=16, batch_size=128, n_epochs=2)
    states = []
    for hp1 in (HPS[1], dict(HPS[1], learning_rate=2e-3, ent_coef=0.05, gamma=0.9, seed=99)):
        env = _env(3, 64, "waypoints_v3")
        pop = PPOPopulation("MlpPolicy", env, members=[HPS[0], hp1, HPS[2]], **shared)
        pop.learn(2 * 16 * 64)
        states.append(pop)
    a, b = states
    assert not torch.equal(a.theta[1], b.theta[1])
    for m in (0, 2):
        cols = slice(m * 64, (m + 1) * 64)
        assert torch.equal(a.theta[m], b.theta[m]) and torch.equal(a.adam_v[m], b.adam_v[m])
        for k in BUFFERS:
            assert torch.equal(a.buf[k][:, cols], b.buf[k][:, cols]), k


@pytest.mark.parametrize("preset", ["waypoints_v3", "objlock_duck"])
def test_episode_stats_equal_host_sums_of_the_raw_steps(preset):
    P, n, T = 3, 64, 64
    env = _env(P, n, preset, max_steps=40)        # short episodes: time-limit truncations and crashes inside the rollout
    pop = PPOPopulation("MlpPolicy", env, members=HPS, n_steps=T, batch_size=128, n_epochs=1, use_cuda_graph=False)
    rec = []
    step, targets = env.step_tensor, env.targets_reached_tensor

    def rec_step(act, want_terminal_obs=False):
        out = step(act, want_terminal_obs=want_terminal_obs)
        rec.append([out[1].double().cpu().numpy(), out[2].cpu().numpy().astype(np.int64), None])
        return out

    def rec_targets():
        t = targets()
        rec[-1][2] = t.cpu().numpy().astype(np.float64)
        return t

    env.step_tensor, env.targets_reached_tensor = rec_step, rec_targets
    pop.learn(2 * T * n)
    got = pop.episode_stats()
    N = P * n
    ret, length, acc = np.zeros(N), np.zeros(N), np.zeros((8, N))
    for rew, flags, tidx in rec:
        ret += rew
        length += 1
        done = (flags & 3) != 0
        acc[0] += done
        acc[1] += np.where(done, ret, 0.0)
        acc[2] += np.where(done, length, 0.0)
        if tidx is not None:
            acc[3] += np.where(done, tidx, 0.0)
        for i, bit in zip(range(4, 8), (4, 8, 16, 32)):
            acc[i] += done & ((flags & bit) != 0)
        ret[done] = 0.0
        length[done] = 0.0
    want = np.cumsum(acc.reshape(8, P, n), axis=2)[:, :, -1]
    assert want[0].sum() > 0, "no episode finished"
    for i, name in enumerate(["episodes", "return_sum", "length_sum", "targets_reached_sum", "collisions", "out_of_bounds",
                              "completed", "strikes"]):
        np.testing.assert_array_equal(got[name], want[i], err_msg=name)
    assert all(v.sum() == 0 for v in pop.episode_stats().values())      # read-and-reset, like FixedwingVecEnv.episode_stats


def test_member_evaluates_like_its_standalone_twin(tmp_path):
    shared = dict(n_steps=16, batch_size=128, n_epochs=2)
    env = _env(3, 64, "waypoints_v3")
    pop = PPOPopulation("MlpPolicy", env, members=HPS, **shared)
    pop.learn(2 * 16 * 64)
    model = _twin(pop, 1, shared)
    model.learn(2 * 16 * 64)
    mem = pop.member(1)
    assert mem.num_timesteps == model.num_timesteps and int(mem._step_dev.item()) == int(model._step_dev.item())
    a = mem.evaluate(n_eval_episodes=12, max_steps=300)
    b = model.evaluate(n_eval_episodes=12, max_steps=300)
    for k in ("returns", "lengths", "targets_reached", "flags", "env_index", "finish_step"):
        np.testing.assert_array_equal(getattr(a, k), getattr(b, k), err_msg=k)
    assert a.mean_reward == b.mean_reward or (np.isnan(a.mean_reward) and np.isnan(b.mean_reward))
    paths = mem.export_sb3(str(tmp_path / "m1"))
    assert all(p for p in paths.values())
