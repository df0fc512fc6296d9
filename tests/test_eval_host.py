"""CPU checks of the evaluation layer: EvalResult's ordering and metrics on synthetic episode tables, the scheduling and
file layout of EvalCallback / CheckpointCallback against a stub model, and the argument checks of ppo_eval_ledger."""
import ctypes as C
import math
import os

import numpy as np
import pytest

from pyflyt_drone_b200 import _lib, callbacks
from pyflyt_drone_b200.config import FLAG_COLLISION, FLAG_COMPLETE, FLAG_OOB, FLAG_STRIKE, FLAG_TERM, FLAG_TRUNC
from pyflyt_drone_b200.ppo import EvalResult

T, R = FLAG_TERM, FLAG_TRUNC


def _table():
    # five episodes, given out of order: (return, length, targets, flags, env, finish step)
    rows = [(-10.0, 40, 2, T | FLAG_COLLISION, 3, 39),
            (-5.5, 12, 0, T | FLAG_OOB, 1, 11),
            (80.0, 300, 8, T | FLAG_COMPLETE, 0, 299),
            (-1.0, 40, 1, R, 0, 39),
            (7.25, 500, 3, T | R | FLAG_STRIKE, 2, 520)]
    return [np.array(c) for c in zip(*rows)]


def test_episodes_are_ordered_by_finish_step_then_env():
    ret, ln, tr, fl, env, step = _table()
    r = EvalResult.from_episodes(ret, ln, tr, fl, env, step, task=1, num_targets=8)
    assert r.finish_step.tolist() == [11, 39, 39, 299, 520]
    assert r.env_index.tolist() == [1, 0, 3, 0, 2]
    assert r.returns.tolist() == [-5.5, -1.0, -10.0, 80.0, 7.25]
    assert r.lengths.dtype == np.int32 and r.targets_reached.dtype == np.uint8 and r.flags.dtype == np.uint8
    assert r.n_episodes == 5


def test_waypoint_metrics():
    ret, ln, tr, fl, env, step = _table()
    r = EvalResult.from_episodes(ret, ln, tr, fl, env, step, task=1, num_targets=8)
    assert r.mean_reward == pytest.approx(np.mean(ret)) and r.std_reward == pytest.approx(np.std(ret))
    assert r.mean_length == pytest.approx(np.mean(ln)) and r.mean_targets_reached == pytest.approx(np.mean(tr))
    assert r.wp_reach_rate.tolist() == [0.8, 0.6, 0.4, 0.2, 0.2, 0.2, 0.2, 0.2]
    assert r.success_rate == 0.2                                   # env_complete on Waypoints
    assert r.duck_strike_rate == 0.2 and r.collision_rate == 0.2 and r.out_of_bounds_rate == 0.2
    assert r.truncation_rate == 0.2                                # the truncated-and-terminated episode is not a truncation
    m = r.metrics()
    assert m["eval/mean_reward"] == r.mean_reward and m["eval/mean_ep_length"] == r.mean_length
    assert [m[f"eval/wp{i}_reach_rate"] for i in range(1, 9)] == r.wp_reach_rate.tolist()
    assert m["eval/success_rate"] == 0.2 and "eval/duck_strike_rate" not in m


@pytest.mark.parametrize("task", [2, 4])
def test_objlock_success_is_the_duck_strike(task):
    ret, ln, tr, fl, env, step = _table()
    r = EvalResult.from_episodes(ret, ln, tr, fl, env, step, task=task, num_targets=8)
    assert r.successes.tolist() == [False, False, False, False, True]
    assert r.success_rate == r.duck_strike_rate == 0.2
    assert r.metrics()["eval/duck_strike_rate"] == 0.2


@pytest.mark.parametrize("task", [3, 4])
def test_tasks_without_targets(task):
    ret, ln, tr, fl, env, step = _table()
    r = EvalResult.from_episodes(ret, ln, tr, fl, env, step, task=task, num_targets=1)
    assert r.num_targets == 0 and r.wp_reach_rate.shape == (0,)
    assert r.mean_targets_reached == 0.0 and not r.targets_reached.any()
    assert not any(k.startswith("eval/wp") for k in r.metrics())


def test_no_finished_episode_gives_nan():
    e = np.zeros(0)
    r = EvalResult.from_episodes(e, e, e, e, e, e, task=1, num_targets=4)
    assert r.n_episodes == 0
    for v in (r.mean_reward, r.std_reward, r.mean_length, r.mean_targets_reached, r.success_rate, r.duck_strike_rate,
              r.collision_rate, r.out_of_bounds_rate, r.truncation_rate):
        assert math.isnan(v)
    assert r.wp_reach_rate.shape == (4,) and np.isnan(r.wp_reach_rate).all()


# ---------------------------------------------------------------- callbacks against a stub model
class _StubModel:
    d, a, n_envs = 28, 4, 8

    def __init__(self):
        self.num_timesteps = 0
        self.evals = []
        self.built = 0

    def make_eval_env(self, n):
        self.built += 1
        return ("env", n)

    def evaluate(self, env, n_eval_episodes, deterministic):
        self.evals.append((env, n_eval_episodes, deterministic, self.num_timesteps))
        k = len(self.evals)
        ret = np.array([float(k) * (1 if k != 3 else -1)] * n_eval_episodes)   # improves, improves, worse, improves
        if k == 4:
            ret += 10
        fl = np.full(n_eval_episodes, T | FLAG_COMPLETE)
        return EvalResult.from_episodes(ret, np.arange(n_eval_episodes) + 1, np.zeros(n_eval_episodes), fl,
                                        np.arange(n_eval_episodes), np.arange(n_eval_episodes), task=1, num_targets=2)


def _run(cb, model, per_iter, iters):
    fired = []
    for _ in range(iters):
        model.num_timesteps += per_iter
        assert cb({"self": model}, {}) is True
        fired.append(model.num_timesteps)
    return fired


def test_frequency_counts_timesteps_and_fires_once_per_crossing():
    e = callbacks._Every(10_000)
    seq = [3_000, 6_000, 9_000, 12_000, 15_000, 35_000, 39_000, 40_000]
    assert [e.due(t) for t in seq] == [False, False, False, True, False, True, False, True]
    e = callbacks._Every(100)
    assert [e.due(t) for t in (100, 0, 50, 100)] == [True, False, False, True]      # a new learn() restarts the count
    with pytest.raises(ValueError):
        callbacks._Every(0)


def test_eval_callback_schedule_files_and_best_model(tmp_path, monkeypatch):
    saved = []
    monkeypatch.setattr(callbacks, "_save_model", lambda m, zp, vp: saved.append((m.num_timesteps, zp, vp)))
    model = _StubModel()
    cb = callbacks.EvalCallback(eval_freq=5_000, n_eval_episodes=6, best_model_save_path=str(tmp_path / "best"),
                                log_path=str(tmp_path / "logs"))
    _run(cb, model, 2_048, 12)                      # 24,576 timesteps: crossings at 6,144 / 10,240 / 16,384 / 20,480
    assert [e[3] for e in model.evals] == [6_144, 10_240, 16_384, 20_480]
    assert model.built == 1 and all(e[0] == ("env", 6) and e[1] == 6 and e[2] is True for e in model.evals)
    z = np.load(tmp_path / "logs" / "evaluations.npz")
    assert sorted(z.files) == ["ep_lengths", "results", "successes", "timesteps"]
    assert z["timesteps"].tolist() == [6_144, 10_240, 16_384, 20_480]
    assert z["results"].shape == z["ep_lengths"].shape == z["successes"].shape == (4, 6)
    assert z["results"][:, 0].tolist() == [1.0, 2.0, -3.0, 14.0] and z["successes"].all()
    best = str(tmp_path / "best")
    assert saved == [(t, os.path.join(best, "best_model.zip"), os.path.join(best, "vecnorm.pkl")) for t in (6_144, 10_240, 20_480)]
    assert cb.best_mean_reward == 14.0
    assert cb.last_metrics["eval/mean_reward"] == 14.0 and cb.last_metrics["eval/success_rate"] == 1.0
    assert set(cb.last_metrics) >= {"eval/mean_ep_length", "eval/wp1_reach_rate", "eval/wp2_reach_rate"}


def test_eval_callback_uses_a_given_env_and_runs_on_rank_0_only(monkeypatch):
    model = _StubModel()
    cb = callbacks.EvalCallback(eval_freq=1_000, n_eval_episodes=3, deterministic=False, eval_env="mine")
    monkeypatch.setattr(callbacks, "_is_rank0", lambda: False)
    _run(cb, model, 1_000, 2)
    assert model.evals == []
    monkeypatch.setattr(callbacks, "_is_rank0", lambda: True)
    _run(cb, model, 1_000, 1)
    assert model.evals == [("mine", 3, False, 3_000)] and model.built == 0


def test_checkpoint_callback_names_and_timesteps(tmp_path, monkeypatch):
    saved = []
    monkeypatch.setattr(callbacks, "_save_model", lambda m, zp, vp: saved.append((zp, vp)))
    model = _StubModel()
    cb = callbacks.CheckpointCallback(save_freq=50_000, save_path=str(tmp_path), name_prefix="ppo_fixedwing")
    _run(cb, model, 32_768, 5)                      # crossings at 65,536 / 131,072 / 163,840
    p = str(tmp_path)
    assert saved == [(os.path.join(p, f"ppo_fixedwing_{t}_steps.zip"), os.path.join(p, f"ppo_fixedwing_vecnormalize_{t}_steps.pkl"))
                     for t in (65_536, 131_072, 163_840)]
    assert cb.last_paths == list(saved[-1])
    saved.clear()
    cb = callbacks.CheckpointCallback(save_freq=10, save_path=str(tmp_path), save_vecnormalize=False)
    model.num_timesteps = 0
    _run(cb, model, 10, 1)
    assert saved == [(os.path.join(p, "rl_model_10_steps.zip"), None)]


def test_eval_ledger_validates_arguments_without_a_device():
    lib = _lib.load()
    one = C.c_void_p(16)                         # any non-null address: never dereferenced on these paths
    ok = [one, one, None, 4, one, one, one, one, one, 0, one, 10, one, one, one, one, one, one, None]
    for i in (0, 1, 4, 5, 6, 7, 8, 10, 12, 13, 14, 15, 16, 17):          # every required pointer
        bad = list(ok); bad[i] = None
        assert lib.ppo_eval_ledger(*bad) == -1, i
    bad = list(ok); bad[3] = 0
    assert lib.ppo_eval_ledger(*bad) == -1 and b"positive" in lib.fw_last_error()
    bad = list(ok); bad[11] = -1
    assert lib.ppo_eval_ledger(*bad) == -1 and b"step_limit" in lib.fw_last_error()
