"""stable_baselines3's ``EvalCallback`` and ``CheckpointCallback`` for ``PPO.learn``.

The reference trains under ``callback=[WaypointEvalCallback, CheckpointCallback]`` (train/train_Fixedwing_Waypoints_v3.py:
163-172,284-288,332-337; SURVEY §3.1 and §5 "checkpoint / resume", "metrics / logging").  Both classes here are plain callables
with ``PPO.learn``'s ``callback(locals, globals)`` signature, called once per PPO iteration; pass one, or a lambda that calls
several.  Frequencies count environment timesteps (``model.num_timesteps``), not callback calls: the reference's
``eval_freq = 10000 // num_envs`` step calls become ``eval_freq=10000``.  A callback fires on the first call at or after each
multiple of its frequency (once, if one iteration crosses several).

Multi-GPU: the ranks hold bit-identical parameters and statistics, so only rank 0 evaluates and writes files.  The other ranks
go straight on to their next rollout and wait for rank 0 in the statistics all-reduce that follows it.
"""
from __future__ import annotations

import os

import numpy as np


def _is_rank0() -> bool:
    try:
        import torch.distributed as dist
        return not (dist.is_available() and dist.is_initialized()) or dist.get_rank() == 0
    except ImportError:
        return True


class _Every:
    """Fires when ``num_timesteps`` has crossed a multiple of ``freq`` since the last call (a new ``learn`` that restarts the
    count fires at its first crossing)."""

    def __init__(self, freq: int):
        if int(freq) <= 0:
            raise ValueError("frequency must be a positive number of timesteps")
        self.freq = int(freq)
        self._bucket = 0

    def due(self, num_timesteps: int) -> bool:
        b = int(num_timesteps) // self.freq
        fire = b > 0 and b != self._bucket
        self._bucket = b
        return fire


def _save_model(model, model_path: str, vecnorm_path: str | None) -> None:
    from . import sb3_io
    sb3_io.write_model_zip(model_path, model)
    if vecnorm_path is not None:
        sb3_io.write_vecnorm_pkl(vecnorm_path, model.vecnorm.state_dict(), model.d, model.a, model.n_envs)


class EvalCallback:
    """``stable_baselines3.common.callbacks.EvalCallback`` over ``PPO.evaluate``.

    Every ``eval_freq`` timesteps: ``n_eval_episodes`` episodes on ``eval_env`` (default: one batch built by
    ``model.make_eval_env`` on first use and kept, with its captured evaluation graph, for every later evaluation).
    ``last_result`` is the ``EvalResult``; ``last_metrics`` its metrics under the reference's names (``eval/mean_reward``,
    ``eval/mean_ep_length``, ``eval/wp{i}_reach_rate``, ``eval/success_rate``, ``eval/duck_strike_rate``).
    ``log_path``: ``evaluations.npz`` rewritten after each evaluation with SB3's keys -- ``timesteps`` [n_evals],
    ``results`` and ``ep_lengths`` [n_evals, n_eval_episodes], ``successes`` [n_evals, n_eval_episodes].
    ``best_model_save_path``: ``best_model.zip`` and ``vecnorm.pkl`` (SB3's containers, ``sb3_io``) whenever the mean reward
    improves; ``PPO.import_sb3`` reads that directory back.  ``close()`` frees a batch the callback built."""

    def __init__(self, eval_freq: int, n_eval_episodes: int = 20, deterministic: bool = True, eval_env=None,
                 best_model_save_path: str | None = None, log_path: str | None = None, verbose: int = 0):
        self._every = _Every(eval_freq)
        self.eval_freq = self._every.freq
        self.n_eval_episodes, self.deterministic = int(n_eval_episodes), bool(deterministic)
        self.eval_env, self._own_env = eval_env, eval_env is None
        self.best_model_save_path, self.log_path, self.verbose = best_model_save_path, log_path, verbose
        self.best_mean_reward = -np.inf
        self.last_result, self.last_metrics = None, {}
        self.evaluations_timesteps, self.evaluations_results, self.evaluations_length, self.evaluations_successes = [], [], [], []

    def __call__(self, locals_: dict, globals_: dict) -> bool:
        model = locals_["self"]
        if self._every.due(model.num_timesteps) and _is_rank0():
            self.evaluate(model)
        return True

    def evaluate(self, model) -> None:
        """One evaluation now, with its logging and best-model bookkeeping."""
        if self.eval_env is None:
            self.eval_env = model.make_eval_env(self.n_eval_episodes)
        res = model.evaluate(env=self.eval_env, n_eval_episodes=self.n_eval_episodes, deterministic=self.deterministic)
        self.last_result, self.last_metrics = res, res.metrics()
        self.evaluations_timesteps.append(int(model.num_timesteps))
        self.evaluations_results.append(res.returns)
        self.evaluations_length.append(res.lengths)
        self.evaluations_successes.append(res.successes)
        if self.log_path is not None:
            os.makedirs(self.log_path, exist_ok=True)
            np.savez(os.path.join(self.log_path, "evaluations"), timesteps=np.asarray(self.evaluations_timesteps),
                     results=np.asarray(self.evaluations_results), ep_lengths=np.asarray(self.evaluations_length),
                     successes=np.asarray(self.evaluations_successes))
        if self.verbose:
            print(f"Eval num_timesteps={model.num_timesteps}, episode_reward={res.mean_reward:.2f} +/- {res.std_reward:.2f}, "
                  f"episode_length={res.mean_length:.2f}, success_rate={res.success_rate:.3f}", flush=True)
        if res.mean_reward > self.best_mean_reward:
            self.best_mean_reward = res.mean_reward
            if self.best_model_save_path is not None:
                os.makedirs(self.best_model_save_path, exist_ok=True)
                _save_model(model, os.path.join(self.best_model_save_path, "best_model.zip"),
                            os.path.join(self.best_model_save_path, "vecnorm.pkl"))
                if self.verbose:
                    print("New best mean reward!", flush=True)

    def close(self) -> None:
        if self._own_env and self.eval_env is not None:
            self.eval_env.close()
            self.eval_env = None


class CheckpointCallback:
    """``stable_baselines3.common.callbacks.CheckpointCallback``: every ``save_freq`` timesteps, SB3's
    ``{name_prefix}_{num_timesteps}_steps.zip`` and (``save_vecnormalize``) ``{name_prefix}_vecnormalize_{num_timesteps}_steps.pkl``
    in ``save_path``.  ``last_paths`` lists the files of the latest checkpoint."""

    def __init__(self, save_freq: int, save_path: str, name_prefix: str = "rl_model", save_vecnormalize: bool = True):
        self._every = _Every(save_freq)
        self.save_freq = self._every.freq
        self.save_path, self.name_prefix, self.save_vecnormalize = save_path, name_prefix, bool(save_vecnormalize)
        self.last_paths: list[str] = []

    def __call__(self, locals_: dict, globals_: dict) -> bool:
        model = locals_["self"]
        if self._every.due(model.num_timesteps) and _is_rank0():
            os.makedirs(self.save_path, exist_ok=True)
            t = int(model.num_timesteps)
            paths = [os.path.join(self.save_path, f"{self.name_prefix}_{t}_steps.zip")]
            if self.save_vecnormalize:
                paths.append(os.path.join(self.save_path, f"{self.name_prefix}_vecnormalize_{t}_steps.pkl"))
            _save_model(model, paths[0], paths[1] if self.save_vecnormalize else None)
            self.last_paths = paths
        return True
