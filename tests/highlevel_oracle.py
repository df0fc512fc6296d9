"""fp64 reference of the high-level waypoint task (task 5), composed on the test side from the unmodified oracle.

Each agent step of an env is the Waypoints step of the oracle (oracle/fw_oracle.c ``fwo_step``, task 1) with the tracker
between the action and the physics, restated here:
  * the command ``[psi, h, V]`` of the high-level action (``Tracker.command``);
  * per inner iteration: the tracker's 21-float observation (task 3's ``lowlevel_obs`` with the command as the target and
    the tracker's previous action), its VecNormalize normalisation and policy tower in float64, the clipped mean as the
    mode -1 setpoint, ``substeps_per_inner`` oracle substeps under a task-3 configuration (whose only difference in the
    substep is that mode -1 control), then ``fwo_compute_obs`` and ``term_trunc_reward``'s Waypoints branch (restated:
    the oracle keeps it static);
  * the SubprocVecEnv reset-on-done through ``fwo_reset`` of the task-1 configuration, the tracker's previous action zeroed.
The wind of every mode, motor noise and resets are the oracle's own code; a gridded field goes through
tests/field_oracle.py's library.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

H = 64


def tower(params: np.ndarray, x: np.ndarray) -> np.ndarray:
    """The policy mean of the (21, 6) flat vector, float64, rows of x already normalised."""
    p = np.asarray(params, np.float64)
    d, a, o = 21, 6, 0
    def take(n, shape):
        nonlocal o
        v = p[o:o + n].reshape(shape)
        o += n
        return v
    w1, b1 = take(H * d, (H, d)), take(H, (H,))
    w2, b2 = take(H * H, (H, H)), take(H, (H,))
    w3, b3 = take(a * H, (a, H)), take(a, (a,))
    h = np.tanh(x @ w1.T + b1)
    h = np.tanh(h @ w2.T + b2)
    return h @ w3.T + b3


def tracker_act(tracker, obs_raw: np.ndarray) -> np.ndarray:
    """The tracker's action for raw observations: VecNormalize (frozen, eps 1e-8, clip), policy mean, clip to [-1, 1]."""
    x = np.asarray(obs_raw, np.float64)
    if tracker.obs_mean is not None:
        x = np.clip((x - tracker.obs_mean) / np.sqrt(tracker.obs_var + 1e-8), -tracker.clip_obs, tracker.clip_obs)
    return np.clip(tower(tracker.params, x), -1.0, 1.0)


class HighLevelOracle:
    """N fp64 task-5 envs: ``base`` is an oracle VecEnv (fw_oracle.OracleVecEnv or field_oracle.FieldOracleVecEnv) built with
    the task-1 form of the configuration; ``prev`` [N, 6] is the tracker's previous action."""

    def __init__(self, base, tracker):
        self.base, self.tracker = base, tracker
        self.L, self.n = base.L, base.n
        from oracle import fw_oracle as fo
        D, cfg, env = C.c_double, C.POINTER(fo.OConfig), C.POINTER(fo.OEnv)
        self.L.fwo_substep.argtypes = [cfg, env, C.c_uint64]
        self.L.fwo_reset.argtypes = [cfg, env, C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p]
        self.L.fwo_compute_obs.argtypes = [cfg, env, C.c_void_p, C.c_int]
        self.L.fwo_quat_to_mat.argtypes = [C.POINTER(D), C.POINTER(D)]
        self.L.fwo_quat_to_euler.argtypes = [C.POINTER(D), C.POINTER(D)]
        self.c1 = base.cfg
        self.c3 = type(base.cfg).from_buffer_copy(base.cfg)
        self.c3.task = 3
        self.prev = np.zeros((self.n, 6))
        self.last_tracker_obs = np.zeros((self.n, 21))
        self.last_tracker_act = np.zeros((self.n, 6))

    def _install(self):
        if hasattr(self.base, "_install"):
            self.base._install()

    def reset(self):
        self.prev[:] = 0.0
        return self.base.reset()

    def get_state(self):
        return self.base.get_state()

    def set_state(self, s):
        self.base.set_state(s)

    def _tracker_obs(self, e, ref) -> np.ndarray:
        D = C.c_double
        q = (D * 4)(*e.quat[:])
        R, rpy = (D * 9)(), (D * 3)()
        self.L.fwo_quat_to_mat(q, R)
        self.L.fwo_quat_to_euler(q, rpy)
        R = np.array(R[:]).reshape(3, 3)
        return np.concatenate([R.T @ np.array(e.omega[:]), np.array(rpy[:]), R.T @ np.array(e.vel[:]), np.array(e.pos[:]),
                               np.zeros(6), ref])

    def step(self, actions: np.ndarray):
        self._install()
        a = np.asarray(actions, np.float64)
        n, c1, c3, L, seed = self.n, self.c1, self.c3, self.L, self.base.seed
        D = int(L.fwo_obs_dim(C.byref(c1)))
        obs, term = np.zeros((n, D)), np.zeros((n, D))
        rew, flags = np.zeros(n), np.zeros(n, np.int32)
        tr = np.zeros(n, np.int32)
        refs = self.tracker.command(a)
        envs = self.base.envs
        for i in range(n):
            envs[i].reward = -0.1                 # the info bits stay as fwo_step leaves them (env_complete is sticky)
        obs_buf = (C.c_double * 64)()
        for it in range(int(c1.inner_per_step)):
            idx = [i for i in range(n) if not (envs[i].termination or envs[i].truncation)]
            if not idx:
                break
            tob = np.stack([self._tracker_obs(envs[i], refs[i]) for i in idx])
            tob[:, 12:18] = self.prev[idx]
            act = tracker_act(self.tracker, tob)
            self.prev[idx] = act
            self.last_tracker_obs[idx] = tob
            self.last_tracker_act[idx] = act
            for j, i in enumerate(idx):
                e = envs[i]
                for k in range(6):
                    e.setpoint[k] = float(act[j, k])
                e.contact = 0
                for _ in range(int(c1.substeps_per_inner)):
                    L.fwo_substep(C.byref(c3), C.byref(e), seed)
                for k in range(4):
                    e.last_action[k] = float(a[i, k])
                L.fwo_compute_obs(C.byref(c1), C.byref(e), C.cast(obs_buf, C.c_void_p), 1)
                obs[i] = obs_buf[:D]
                self._head(e)
        for i in range(n):
            e = envs[i]
            e.step_count += 1
            rew[i] = e.reward
            flags[i] = (1 if e.termination else 0) | (2 if e.truncation else 0) | (4 if e.info_collision else 0) | \
                       (8 if e.info_oob else 0) | (16 if e.info_complete else 0)
            tr[i] = c1.num_targets - e.n_remaining
            if flags[i] & 3:
                term[i] = obs[i]
                L.fwo_reset(C.byref(c1), C.byref(e), seed, e.env_id, e.episode + 1, C.cast(obs_buf, C.c_void_p))
                obs[i] = obs_buf[:D]
                self.prev[i] = 0.0
        self.last_targets_reached = tr
        return obs, rew, flags, term

    def _head(self, e):
        """term_trunc_reward of the oracle, Waypoints branch (oracle/fw_oracle.c)."""
        c = self.c1
        if e.step_count > c.max_steps:
            e.truncation = 1
        if e.contact:
            e.reward = -100.0; e.info_collision = 1; e.termination = 1
        p = np.array(e.pos[:])
        if np.sqrt(p @ p) > c.dome:
            e.reward = -100.0; e.info_oob = 1; e.termination = 1
        if c.early_return_on_crash and (e.info_collision or e.info_oob):
            return
        if e.n_remaining == 0:
            return
        if not c.sparse_reward:
            prog = 0.0 if (np.isinf(e.old_dist) or np.isinf(e.new_dist)) else e.old_dist - e.new_dist
            e.reward += max(3.0 * prog, 0.0)
            e.reward += 1.0 / e.new_dist
        if e.new_dist < c.goal_reach:
            e.reward = 100.0
            for t in range(1, e.n_remaining):
                e.targets[t - 1][:] = e.targets[t][:]
            e.n_remaining -= 1
            e.target_idx += 1
            done = e.n_remaining == 0
            if c.complete_truncates and done:
                e.truncation = 1
            e.info_complete = int(done)
            e.num_targets_reached = c.num_targets - e.n_remaining
