"""PPOPopulation host logic without a device: member-spec parsing, refused modes, and the argument checks of the ppo_pop_*
entry points (every one returns FW_EINVAL before anything is launched)."""
import ctypes as C
import types

import pytest

from pyflyt_drone_b200 import _lib
from pyflyt_drone_b200.population import HP_COLUMNS, MEMBER_KEYS, PPOPopulation, parse_members

DEFAULTS = dict(seed=42, learning_rate=3e-4, clip_range=0.2, ent_coef=0.001, vf_coef=0.5, max_grad_norm=0.5, gamma=0.99,
                gae_lambda=0.95)


def test_int_members_get_consecutive_seeds_and_the_defaults():
    specs, n = parse_members(4, 128, DEFAULTS)
    assert n == 32 and [s["seed"] for s in specs] == [42, 43, 44, 45]
    for s in specs:
        assert {k: s[k] for k in HP_COLUMNS} == {k: DEFAULTS[k] for k in HP_COLUMNS}


def test_list_members_override_only_what_they_name():
    specs, n = parse_members([{"seed": 0, "learning_rate": 1e-4}, {"seed": 1, "ent_coef": 0.01}, {}], 30, DEFAULTS)
    assert n == 10
    assert specs[0]["seed"] == 0 and specs[0]["learning_rate"] == 1e-4 and specs[0]["ent_coef"] == 0.001
    assert specs[1]["seed"] == 1 and specs[1]["ent_coef"] == 0.01 and specs[1]["learning_rate"] == 3e-4
    assert specs[2] == dict(DEFAULTS)                          # an empty dict is the keyword arguments, seed included
    assert set(MEMBER_KEYS) == set(HP_COLUMNS) | {"seed"}


@pytest.mark.parametrize("members, match", [
    ([{"seed": 0, "n_steps": 64}], "unknown per-member key"),
    ([{"batch_size": 64}], "unknown per-member key"),
    (0, "at least 1"),
    ([], "must not be empty"),
    (True, "positive int or a list"),
    ([3], "expected a dict"),
    (3, "do not divide"),
])
def test_bad_member_specs_raise(members, match):
    with pytest.raises(ValueError, match=match):
        parse_members(members, 64, DEFAULTS)


def _stub_env(num_envs=64, obs_dim=28, act_dim=4):
    return types.SimpleNamespace(num_envs=num_envs, obs_dim=obs_dim, act_dim=act_dim, env_id0=0, device_index=0)


@pytest.mark.parametrize("kwargs, env, match", [
    (dict(update="torch"), _stub_env(), "update='kernel'"),
    (dict(), _stub_env(act_dim=3), "4- or 6-channel"),
    (dict(), _stub_env(obs_dim=56, act_dim=6), "no hand-written PPO update"),
    (dict(), _stub_env(obs_dim=65), "no hand-written PPO update"),
    (dict(members=3), _stub_env(num_envs=64), "do not divide"),
    (dict(members=[{"lr": 1e-3}]), _stub_env(), "unknown per-member key"),
])
def test_refused_modes(kwargs, env, match):
    with pytest.raises(ValueError, match=match):
        PPOPopulation("MlpPolicy", env, **kwargs)


def test_refuses_a_distributed_world(monkeypatch):
    import torch.distributed as dist
    monkeypatch.setattr(dist, "is_available", lambda: True)
    monkeypatch.setattr(dist, "is_initialized", lambda: True)
    monkeypatch.setattr(dist, "get_world_size", lambda: 2)
    with pytest.raises(ValueError, match="one GPU"):
        PPOPopulation("MlpPolicy", _stub_env(), members=2)


# ---- C ABI: (name, valid argument list, indices of required pointers, index of `members`, index of `rows_per_member` or None)
ONE = C.c_void_p(16)                  # any non-null address: never dereferenced on these paths
ENTRY_POINTS = [
    ("ppo_pop_policy_forward_a", [2, 8, ONE, ONE, 28, 4, ONE, None, 10.0, 0, 0, None, 0, None, ONE, None, None, ONE, None],
     (2, 3, 6, 14, 17), 0, 1),
    ("ppo_pop_policy_forward_tc_a", [2, 8, ONE, ONE, 28, 4, ONE, None, 10.0, 0, 0, None, 0, None, ONE, None, None, ONE, None],
     (2, 3, 6, 14, 17), 0, 1),
    ("ppo_pop_value_forward_a", [2, 8, ONE, 28, 4, ONE, None, 10.0, ONE, None], (2, 5, 8), 0, 1),
    ("ppo_pop_timeout_bootstrap_a", [2, 8, ONE, ONE, 28, 4, ONE, None, 10.0, ONE, ONE, None], (2, 3, 6, 9, 10), 0, 1),
    ("ppo_pop_moments_update", [2, 8, ONE, 28, ONE, ONE, None, None], (2, 4, 5), 0, 1),
    ("ppo_pop_reward_normalize", [2, 8, ONE, ONE, ONE, 10.0, ONE, ONE, ONE, None, ONE, None, None], (2, 3, 4, 6, 7, 8, 10), 0, 1),
    ("ppo_pop_gae", [2, 8, ONE, ONE, ONE, ONE, ONE, 16, ONE, ONE, None], (2, 3, 4, 5, 6, 8, 9), 0, 1),
    ("ppo_pop_random_permutation", [2, 8, ONE, ONE, 64, 1, None], (2, 3), 0, 1),
    ("ppo_pop_minibatch_steps_a", [2, ONE, ONE, 28, 4, ONE, ONE, ONE, ONE, ONE, ONE, 1024, 128, 4, ONE, ONE, 0.9, 0.999, 1e-5, ONE,
                                   None, ONE, ONE, None], (1, 2, 5, 6, 7, 8, 9, 10, 14, 15, 19, 21, 22), 0, None),
    ("ppo_pop_episode_ledger", [2, 8, ONE, ONE, None, ONE, ONE, ONE, None], (2, 3, 5, 6, 7), 0, 1),
]


@pytest.mark.parametrize("name, ok, required, i_members, i_rows", ENTRY_POINTS, ids=[e[0] for e in ENTRY_POINTS])
def test_pop_entry_points_validate_arguments_without_a_device(name, ok, required, i_members, i_rows):
    lib = _lib.load()
    fn = getattr(lib, name)
    for i in required:
        bad = list(ok); bad[i] = None
        assert fn(*bad) == -1 and b"null" in lib.fw_last_error(), (name, i)
    for members in (0, -1, 65536):
        bad = list(ok); bad[i_members] = members
        assert fn(*bad) == -1 and b"members" in lib.fw_last_error(), (name, members)
    if i_rows is not None:
        bad = list(ok); bad[i_rows] = 0
        assert fn(*bad) == -1 and b"rows_per_member" in lib.fw_last_error(), name
        bad = list(ok); bad[i_members], bad[i_rows] = 65535, 1 << 16
        assert fn(*bad) == -1 and b"2^31" in lib.fw_last_error(), name


def test_pop_entry_points_check_widths_and_ranges():
    lib = _lib.load()
    fwd = [2, 8, ONE, ONE, 28, 4, ONE, None, 10.0, 0, 0, None, 0, None, ONE, None, None, ONE, None]
    for i, v in ((4, 0), (4, 65), (5, 5)):
        bad = list(fwd); bad[i] = v
        assert lib.ppo_pop_policy_forward_a(*bad) == -1
    bad = list(fwd); bad[4], bad[5] = 56, 6                   # the tensor-core forward has no 64-wide six-action build
    assert lib.ppo_pop_policy_forward_tc_a(*bad) == -1
    bad = list(fwd); bad[14] = C.c_void_p(20)                 # misaligned action buffer
    assert lib.ppo_pop_policy_forward_a(*bad) == -1 and b"aligned" in lib.fw_last_error()
    perm = [2, 8, ONE, ONE, 60, 1, None]                      # n must be a whole number of time steps of the member's rows
    assert lib.ppo_pop_random_permutation(*perm) == -1 and b"multiple" in lib.fw_last_error()
    gae = [2, 8, ONE, ONE, ONE, ONE, ONE, 0, ONE, ONE, None]
    assert lib.ppo_pop_gae(*gae) == -1 and b"T must" in lib.fw_last_error()
    steps = [2, ONE, ONE, 28, 4, ONE, ONE, ONE, ONE, ONE, ONE, 1024, 128, 4, ONE, ONE, 0.9, 0.999, 1e-5, ONE, None, ONE, ONE, None]
    for i, v in ((12, 0), (12, 4097), (13, 0), (11, -1), (4, 5)):
        bad = list(steps); bad[i] = v
        assert lib.ppo_pop_minibatch_steps_a(*bad) == -1, (i, v)
