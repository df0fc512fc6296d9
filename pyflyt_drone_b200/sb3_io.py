"""stable-baselines3 checkpoint containers written and read WITHOUT stable-baselines3 (SURVEY.md section 8 f2).

The reference saves ``final_model.zip`` + ``vecnorm.pkl`` (train/train_Fixedwing_Waypoints_v3.py:343-344) and its eval scripts load
exactly those two files (eval/eval_waypoints.py:96-107, eval/eval_waypoint_objlock.py:200-207: ``VecNormalize.load(path, env)``,
``PPO.load(path, env=env)``).  SB3 and gymnasium are not installable in this image, so the containers are produced from their
documented on-disk format [UP-RECALL u10]:

``model.zip``   zip of ``data`` (JSON of the algorithm's attributes; entries that are not JSON-native are
                ``{":type:", ":serialized:" = base64(cloudpickle)}``), ``policy.pth`` (``ActorCriticPolicy.state_dict()``),
                ``policy.optimizer.pth`` (Adam state dict over the 13 parameter tensors in module order),
                ``pytorch_variables.pth``, ``_stable_baselines3_version``, ``system_info.txt``.
``vecnorm.pkl`` pickle of a ``VecNormalize`` without its ``venv``: ``obs_rms`` / ``ret_rms`` (``RunningMeanStd``: mean, var,
                count), ``clip_obs``, ``clip_reward``, ``gamma``, ``epsilon``, ``norm_obs``, ``norm_reward``, ``training``, spaces.

Objects of foreign classes (``Box``, ``ActorCriticPolicy``, ``VecNormalize``, ``RunningMeanStd``) are pickled BY REFERENCE -- a
pickle only names ``module.qualname`` -- through stand-in classes registered under those names while the real packages are
absent (the real classes are used when importable).  What cannot be checked here is the load on a machine that has SB3; the
structure is tested against stubs (tests/test_sb3_io.py) and a one-line check for that machine is in INTEGRATION.md section 5.
"""
from __future__ import annotations

import base64
import contextlib
import importlib
import io
import json
import pickle
import sys
import types
import zipfile

import numpy as np
import torch

SB3_VERSION = "2.3.2"          # format generation the layout below follows
# ActorCriticPolicy.named_parameters() order: own parameters first (log_std), then children in registration order
SB3_PARAM_ORDER = ("log_std",
                   "mlp_extractor.policy_net.0.weight", "mlp_extractor.policy_net.0.bias",
                   "mlp_extractor.policy_net.2.weight", "mlp_extractor.policy_net.2.bias",
                   "mlp_extractor.value_net.0.weight", "mlp_extractor.value_net.0.bias",
                   "mlp_extractor.value_net.2.weight", "mlp_extractor.value_net.2.bias",
                   "action_net.weight", "action_net.bias", "value_net.weight", "value_net.bias")
_FOREIGN = {
    "Box": ("gymnasium.spaces.box", "Box"),
    "ActorCriticPolicy": ("stable_baselines3.common.policies", "ActorCriticPolicy"),
    "VecNormalize": ("stable_baselines3.common.vec_env.vec_normalize", "VecNormalize"),
    "RunningMeanStd": ("stable_baselines3.common.running_mean_std", "RunningMeanStd"),
}


class _StubBox:
    """Stand-in for gymnasium.spaces.Box: reduces to ``Box(low, high, shape, dtype)`` -- the real constructor on load."""

    def __init__(self, low, high, shape, dtype):
        self.low, self.high, self.shape, self.dtype = low, high, tuple(shape), np.dtype(dtype)

    def __reduce__(self):
        return (type(self), (self.low, self.high, self.shape, self.dtype.type))


class _StubState:
    """Stand-in whose pickle is ``cls.__new__(cls)`` + ``__setstate__(state)`` / ``__dict__.update(state)`` on load."""

    def __init__(self, **state):
        self.__dict__.update(state)


@contextlib.contextmanager
def foreign_classes():
    """The four foreign classes under their real import paths: the real ones when importable, stand-ins otherwise (installed
    into ``sys.modules`` for the duration of the block, so that pickle can name them, and removed again)."""
    installed, out = [], {}
    try:
        for key, (mod, name) in _FOREIGN.items():
            try:
                out[key] = getattr(importlib.import_module(mod), name)
                continue
            except Exception:
                pass
            parts = mod.split(".")
            for k in range(1, len(parts) + 1):
                m = ".".join(parts[:k])
                if m not in sys.modules:
                    sys.modules[m] = types.ModuleType(m)
                    installed.append(m)
                    if k > 1:
                        setattr(sys.modules[".".join(parts[:k - 1])], parts[k - 1], sys.modules[m])
            base = _StubBox if key == "Box" else (_StubState if key != "ActorCriticPolicy" else object)
            cls = type(name, (base,), {"__module__": mod, "__qualname__": name})
            setattr(sys.modules[mod], name, cls)
            out[key] = cls
        yield out
    finally:
        for m in reversed(installed):
            sys.modules.pop(m, None)


def _serialized(obj) -> dict:
    return {":type:": str(type(obj)), ":serialized:": base64.b64encode(pickle.dumps(obj, protocol=4)).decode()}


def sb3_state_dict(policy_state: dict) -> "dict[str, torch.Tensor]":
    return {k: policy_state[k].detach().cpu().contiguous() for k in SB3_PARAM_ORDER}


def adam_state_dict(policy, adam_m: torch.Tensor, adam_v: torch.Tensor, step: int, lr: float, eps: float) -> dict:
    """torch.optim.Adam.state_dict() over the 13 tensors in SB3's parameter order, from the flat moment vectors."""
    names = {"mlp_extractor.policy_net.0": "pi.0", "mlp_extractor.policy_net.2": "pi.2", "mlp_extractor.value_net.0": "vf.0",
             "mlp_extractor.value_net.2": "vf.2"}
    state = {}
    for i, key in enumerate(SB3_PARAM_ORDER):
        base, _, leaf = key.rpartition(".")
        flat = f"{names[base]}.{leaf}" if base in names else key
        a, b, shp = policy.slices[flat]
        if step > 0:
            state[i] = {"step": torch.tensor(float(step)), "exp_avg": adam_m[a:b].view(shp).detach().cpu().clone(),
                        "exp_avg_sq": adam_v[a:b].view(shp).detach().cpu().clone()}
    group = {"lr": lr, "betas": (0.9, 0.999), "eps": eps, "weight_decay": 0, "amsgrad": False, "maximize": False, "foreach": None,
             "capturable": False, "differentiable": False, "fused": None, "params": list(range(len(SB3_PARAM_ORDER)))}
    return {"state": state, "param_groups": [group]}


def write_model_zip(path: str, model, space_dtype=np.float64) -> str:
    """``PPO.save`` as SB3 writes it.  ``space_dtype``: dtype of the Box spaces recorded in the archive -- float64 is what the
    reference's envs declare (fixedwing_base_env.py:60-75, flatten_waypoint_env.py:40-47) and what ``PPO.load(path, env=env)``
    compares the eval env's spaces with."""
    if not path.endswith(".zip"):
        path += ".zip"
    d, a = model.d, model.a
    lr = float(model.optimizer.param_groups[0]["lr"])
    with foreign_classes() as fc:
        obs_space = fc["Box"](np.full((d,), -np.inf, space_dtype), np.full((d,), np.inf, space_dtype), (d,), space_dtype)
        act_space = fc["Box"](np.full((a,), -1.0, space_dtype), np.full((a,), 1.0, space_dtype), (a,), space_dtype)
        data = {
            "policy_class": _serialized(fc["ActorCriticPolicy"]),
            "verbose": 0, "policy_kwargs": {}, "num_timesteps": int(model.num_timesteps), "_total_timesteps": int(model.num_timesteps),
            "_num_timesteps_at_start": 0, "seed": int(model.seed), "action_noise": None, "learning_rate": lr,
            "tensorboard_log": None, "_last_obs": None, "_last_episode_starts": None, "_last_original_obs": None, "_episode_num": 0,
            "use_sde": False, "sde_sample_freq": -1, "_current_progress_remaining": 0.0, "_stats_window_size": 100,
            "ep_info_buffer": None, "ep_success_buffer": None, "_n_updates": int(model._adam_t.item()),
            "observation_space": _serialized(obs_space), "action_space": _serialized(act_space),
            "n_envs": int(model.n_envs), "n_steps": int(model.n_steps), "gamma": model.gamma, "gae_lambda": model.gae_lambda,
            "ent_coef": model.ent_coef, "vf_coef": model.vf_coef, "max_grad_norm": model.max_grad_norm,
            "batch_size": int(model.batch_size), "n_epochs": int(model.n_epochs),
            # plain floats: PPO._setup_model wraps them with get_schedule_fn, like a freshly constructed model
            "clip_range": model.clip_range, "clip_range_vf": None, "normalize_advantage": True, "target_kl": None,
        }
    sd = sb3_state_dict(model.policy.state_dict())
    opt = adam_state_dict(model.policy, model._adam_m, model._adam_v, int(model._adam_t.item()), lr,
                          float(model.optimizer.param_groups[0]["eps"]))

    def blob(obj) -> bytes:
        b = io.BytesIO()
        torch.save(obj, b)
        return b.getvalue()

    with zipfile.ZipFile(path, "w") as z:
        z.writestr("data", json.dumps(data, indent=4))
        z.writestr("pytorch_variables.pth", blob(None))
        z.writestr("policy.pth", blob(sd))
        z.writestr("policy.optimizer.pth", blob(opt))
        z.writestr("_stable_baselines3_version", SB3_VERSION)
        z.writestr("system_info.txt", f"- written by pyflyt_drone_b200 (device PPO on libfwsim.so), torch {torch.__version__}, "
                                      f"numpy {np.__version__}; layout of stable-baselines3 {SB3_VERSION}\n")
    return path


def write_vecnorm_pkl(path: str, vn_state: dict, d: int, a: int, num_envs: int, space_dtype=np.float64) -> str:
    """``VecNormalize.save``: the wrapper without its venv (``__getstate__`` drops ``venv``, ``class_attributes``, ``returns``)."""
    with foreign_classes() as fc:
        rms = lambda mean, var, count: fc["RunningMeanStd"](mean=np.asarray(mean, np.float64), var=np.asarray(var, np.float64),  # noqa: E731
                                                              count=float(count))
        obs_space = fc["Box"](np.full((d,), -np.inf, space_dtype), np.full((d,), np.inf, space_dtype), (d,), space_dtype)
        act_space = fc["Box"](np.full((a,), -1.0, space_dtype), np.full((a,), 1.0, space_dtype), (a,), space_dtype)
        obj = fc["VecNormalize"](
            num_envs=int(num_envs), observation_space=obs_space, action_space=act_space, reset_infos=[{} for _ in range(int(num_envs))],
            _seeds=[None] * int(num_envs), _options=[{} for _ in range(int(num_envs))], render_mode=None,
            norm_obs_keys=None, obs_rms=rms(vn_state["obs_rms.mean"], vn_state["obs_rms.var"], vn_state["obs_rms.count"]),
            ret_rms=rms(vn_state["ret_rms.mean"], vn_state["ret_rms.var"], vn_state["ret_rms.count"]),
            clip_obs=float(vn_state["clip_obs"]), clip_reward=float(vn_state["clip_reward"]), gamma=float(vn_state["gamma"]),
            epsilon=1e-8, training=True, norm_obs=bool(vn_state.get("norm_obs", True)), norm_reward=bool(vn_state.get("norm_reward", True)),
            old_obs=np.zeros((int(num_envs), d), np.float32), old_reward=np.zeros(int(num_envs), np.float32))
        with open(path, "wb") as f:
            pickle.dump(obj, f, protocol=4)
    return path


class _StubUnpickler(pickle.Unpickler):
    """Resolves the foreign classes to the stand-ins (and nothing else outside numpy / builtins): reads SB3-written files here."""

    def find_class(self, module, name):
        for key, (mod, nm) in _FOREIGN.items():
            if name == nm and (module == mod or module.startswith(mod.split(".")[0])):
                return self._fc[key]
        if module.split(".")[0] in ("numpy", "builtins", "collections", "copyreg", "_codecs"):
            return super().find_class(module, name)
        raise pickle.UnpicklingError(f"refusing to load {module}.{name}")


def _loads(blob: bytes, fc: dict):
    u = _StubUnpickler(io.BytesIO(blob))
    u._fc = fc
    return u.load()


def read_model_zip(path: str) -> dict:
    """``policy`` state dict, ``optimizer`` state dict and the ``data`` attributes of an SB3 ``model.zip`` (ours or SB3's own).
    Serialized ``data`` entries that name anything but the four known classes are left as their JSON stubs."""
    out = {}
    with zipfile.ZipFile(path) as z, foreign_classes() as fc:
        data = json.loads(z.read("data").decode())
        for k, v in list(data.items()):
            if isinstance(v, dict) and ":serialized:" in v:
                try:
                    data[k] = _loads(base64.b64decode(v[":serialized:"].encode()), fc)
                except Exception:
                    pass
        out["data"] = data
        out["policy"] = torch.load(io.BytesIO(z.read("policy.pth")), map_location="cpu", weights_only=True)
        if "policy.optimizer.pth" in z.namelist():
            out["optimizer"] = torch.load(io.BytesIO(z.read("policy.optimizer.pth")), map_location="cpu", weights_only=False)
    return out


def read_vecnorm_pkl(path: str) -> dict:
    """The running statistics of a ``vecnorm.pkl`` in the key layout of ``DeviceVecNormalize.load_state_dict``."""
    with foreign_classes() as fc, open(path, "rb") as f:
        vn = _loads(f.read(), fc)
    g = vn.__dict__
    return {"obs_rms.mean": np.asarray(g["obs_rms"].mean, np.float64), "obs_rms.var": np.asarray(g["obs_rms"].var, np.float64),
            "obs_rms.count": float(g["obs_rms"].count), "ret_rms.mean": float(np.asarray(g["ret_rms"].mean)),
            "ret_rms.var": float(np.asarray(g["ret_rms"].var)), "ret_rms.count": float(g["ret_rms"].count),
            "clip_obs": float(g["clip_obs"]), "clip_reward": float(g["clip_reward"]), "gamma": float(g["gamma"]),
            "norm_obs": bool(g.get("norm_obs", True)), "norm_reward": bool(g.get("norm_reward", True))}


def read_directory(directory: str) -> dict:
    """What ``PPO.export_sb3`` writes, or what SB3 itself wrote: ``policy`` (state dict) and ``optimizer`` from the first of
    ``final_model.zip`` / ``best_model.zip`` / ``model.zip`` (else ``policy`` from a bare ``policy.pth``), and ``vecnorm``
    (``DeviceVecNormalize.load_state_dict`` layout) from ``vecnorm.pkl`` or ``vecnorm.npz`` when one exists."""
    import os
    out = {}
    zips = [f for f in ("final_model.zip", "best_model.zip", "model.zip") if os.path.exists(os.path.join(directory, f))]
    if zips:
        ck = read_model_zip(os.path.join(directory, zips[0]))
        out["policy"] = ck["policy"]
        if "optimizer" in ck:
            out["optimizer"] = ck["optimizer"]
    else:
        out["policy"] = torch.load(os.path.join(directory, "policy.pth"), map_location="cpu", weights_only=True)
    pkl, npz = os.path.join(directory, "vecnorm.pkl"), os.path.join(directory, "vecnorm.npz")
    if os.path.exists(pkl):
        out["vecnorm"] = read_vecnorm_pkl(pkl)
    elif os.path.exists(npz):
        from .ppo import import_vecnorm_npz
        out["vecnorm"] = import_vecnorm_npz(npz)
    return out
