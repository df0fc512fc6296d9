"""ctypes binding of libfwsim.so.  Fails loudly: there is no CPU or PyTorch fallback for the env step."""
from __future__ import annotations

import ctypes as C
import os

from .config import FwConfigC

_HERE = os.path.dirname(os.path.abspath(__file__))
# FWSIM_LIB=<path>: load an experiment build instead (A/B measurements; scripts/ab_build.py)
LIB_PATH = os.environ.get("FWSIM_LIB") or os.path.join(_HERE, "libfwsim.so")


class FwStateHostC(C.Structure):
    _fields_ = [
        ("pos", C.c_void_p), ("quat", C.c_void_p), ("vel", C.c_void_p), ("omega", C.c_void_p), ("act", C.c_void_p),
        ("targets", C.c_void_p), ("target_idx", C.c_void_p), ("step_count", C.c_void_p),
        ("physics_steps", C.c_void_p), ("episode", C.c_void_p), ("new_dist", C.c_void_p), ("wind", C.c_void_p),
        ("duck", C.c_void_p), ("obst", C.c_void_p), ("ol_f", C.c_void_p), ("ol_i", C.c_void_p),
        ("vis_hist", C.c_void_p),
    ]


class FwWindFieldC(C.Structure):
    """include/fwsim.h FwWindField (the host-side description of a gridded wind field, wind_mode 3)."""
    _fields_ = [
        ("values", C.c_void_p), ("nx", C.c_int32), ("ny", C.c_int32), ("nz", C.c_int32), ("nt", C.c_int32),
        ("origin", C.c_double * 3), ("spacing", C.c_double * 3), ("t_step", C.c_double),
        ("shift_lo", C.c_double * 3), ("shift_hi", C.c_double * 3), ("randomize_time", C.c_int32), ("_pad", C.c_int32),
    ]


class FwError(RuntimeError):
    pass


_lib = None

# every symbol include/fwsim.h and include/fwppo.h declare: (name, restype, argtypes)
_P = C.c_void_p
SYMBOLS = [
    ("fw_abi_version", C.c_int, []),
    ("fw_last_error", C.c_char_p, []),
    ("fw_config_size", C.c_int, []),
    ("fw_create", C.c_int, [C.POINTER(FwConfigC), C.c_int32, C.c_int32, C.c_uint64, C.c_uint32, C.POINTER(_P)]),
    ("fw_destroy", C.c_int, [_P]),
    ("fw_set_wind_field", C.c_int, [_P, C.POINTER(FwWindFieldC)]),
    ("fw_num_envs", C.c_int, [_P]),
    ("fw_obs_dim", C.c_int, [_P]),
    ("fw_act_dim", C.c_int, [_P]),
    ("fw_reset", C.c_int, [_P, _P, _P, _P]),
    ("fw_step", C.c_int, [_P, _P, _P, _P, _P, _P, _P]),
    ("fw_step_random", C.c_int, [_P, C.c_int32, _P, _P, _P]),
    ("fw_rollout_random", C.c_int, [C.POINTER(_P), C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P]),
    ("fw_step_host", C.c_int, [_P, _P, _P, _P, _P, _P]),
    ("fw_reset_host", C.c_int, [_P, _P]),
    ("fw_observe_host", C.c_int, [_P, _P]),
    ("fw_host_info_buffer", C.c_int, [_P, C.POINTER(_P)]),
    ("fw_targets_reached", C.c_int, [_P, _P, _P]),
    ("fw_render", C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    ("fw_set_obs_accumulator", C.c_int, [_P, _P]),
    ("fw_fault_count", C.c_int, [_P, C.POINTER(C.c_int64)]),
    ("fw_spare_stats", C.c_int, [_P, C.POINTER(C.c_int64)]),
    ("fw_host_buffers", C.c_int, [_P, C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), C.POINTER(_P)]),
    ("fw_set_state", C.c_int, [_P, C.POINTER(FwStateHostC)]),
    ("fw_get_state", C.c_int, [_P, C.POINTER(FwStateHostC)]),
    ("fw_episode_stats", C.c_int, [_P, C.POINTER(C.c_double)]),
    ("fw_launch_count", C.c_int64, [_P]),
    ("fw_measure_fp32_peak", C.c_int, [C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
]


ABI_VERSION = 11        # include/fwsim.h FW_ABI_VERSION this binding was written against


def load() -> C.CDLL:
    """Load libfwsim.so, (re)building it first when nvcc is present and a source is newer than the library
    (build.build() is a no-op otherwise).  A box without nvcc -- the GPU box -- uses the shipped library as it is."""
    global _lib
    if _lib is not None:
        return _lib
    from . import build as _build
    if os.environ.get("FWSIM_LIB"):
        pass
    elif _build.have_nvcc():
        _build.build()
    elif not os.path.exists(LIB_PATH):
        raise FwError(f"{LIB_PATH} is missing and nvcc is not available to build it; the env step has no CPU fallback")
    try:
        lib = C.CDLL(LIB_PATH)
    except OSError as e:
        raise FwError(f"cannot load {LIB_PATH}: {e}. Build it with `python -m pyflyt_drone_b200.build`; "
                      "the env step has no CPU fallback.") from e
    for name, res, args in SYMBOLS:
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    try:
        from ._ppo_lib import bind as _bind_ppo
        _bind_ppo(lib)
    except ImportError:
        pass
    if lib.fw_abi_version() != ABI_VERSION:
        raise FwError(f"libfwsim.so has ABI {lib.fw_abi_version()}, this package binds ABI {ABI_VERSION}: rebuild with "
                      "`python -m pyflyt_drone_b200.build --force`")
    if lib.fw_config_size() != C.sizeof(FwConfigC):
        raise FwError(f"FwConfig ABI mismatch: C {lib.fw_config_size()} bytes vs ctypes {C.sizeof(FwConfigC)}")
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().fw_last_error()
        raise FwError(f"libfwsim error {rc}: {msg.decode() if msg else '?'}")
