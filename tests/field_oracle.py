"""fp64 reference of the gridded wind field (wind_mode 3) for the tests -- TEST INFRASTRUCTURE ONLY.

The oracle of oracle/fw_oracle.c knows the uniform wind modes.  This module compiles a second library from an unmodified copy
of that source plus tests/field_oracle.c: the oracle's two wind entry points (`fwo_refresh_surface_vel`, `sample_wind`) are
renamed by an exact, checked text substitution of their definitions, and field_oracle.c provides them under their original
names -- the field for wind_mode 3, the renamed originals for every other mode.  Everything else (aerodynamics, rigid body,
tasks, camera) is the oracle's own code.  The library is built into a temporary directory (the tree may be read-only) and
keyed by the hash of both sources.

`FieldOracleVecEnv(cfg, n, ..., wind_field=WindField)` is `oracle.fw_oracle.OracleVecEnv` with the field installed.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import fw_oracle as fo

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE_DIR = os.path.join(os.path.dirname(_HERE), "oracle")
_RENAMES = [
    ("void fwo_refresh_surface_vel(const fwo_config* c, fwo_env* e, int stamp) {",
     "void fwo_refresh_surface_vel_uniform(const fwo_config* c, fwo_env* e, int stamp) {"),
    ("static void sample_wind(const fwo_config* c, fwo_env* e, uint64_t seed) {",
     "static void sample_wind(const fwo_config* c, fwo_env* e, uint64_t seed);\n"
     "static void sample_wind_uniform(const fwo_config* c, fwo_env* e, uint64_t seed) {"),
]
_D, _I = C.c_double, C.c_int32
_lib = None


class FieldC(C.Structure):
    """fwf_field (tests/field_oracle.c); the same layout as include/fwsim.h FwWindField."""
    _fields_ = [
        ("values", C.c_void_p), ("nx", _I), ("ny", _I), ("nz", _I), ("nt", _I),
        ("origin", _D * 3), ("spacing", _D * 3), ("t_step", _D), ("shift_lo", _D * 3), ("shift_hi", _D * 3),
        ("randomize_time", _I), ("_pad", _I),
    ]


def _source() -> str:
    src = open(os.path.join(_ORACLE_DIR, "fw_oracle.c")).read()
    for old, new in _RENAMES:
        if src.count(old) != 1:
            raise RuntimeError(f"oracle/fw_oracle.c no longer has exactly one `{old}`: update tests/field_oracle.py")
        src = src.replace(old, new)
    return src + "\n" + open(os.path.join(_HERE, "field_oracle.c")).read()


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    src = _source()
    key = hashlib.sha256((src + open(os.path.join(_ORACLE_DIR, "fw_oracle.h")).read()).encode()).hexdigest()[:16]
    d = os.path.join(tempfile.gettempdir(), f"fw_field_oracle_{os.getuid()}_{key}")
    so = os.path.join(d, "libfw_field_oracle.so")
    if not os.path.exists(so):
        os.makedirs(d, exist_ok=True)
        c_path = os.path.join(d, "fw_field_oracle.c")
        with open(c_path, "w") as f:
            f.write(src)
        tmp = so + f".{os.getpid()}"
        # the flags of oracle/Makefile
        r = subprocess.run(["gcc", "-O2", "-fPIC", "-Wall", "-std=c11", "-fno-fast-math", "-ffp-contract=off", "-I", _ORACLE_DIR,
                            "-shared", "-o", tmp, c_path, "-lm", "-lpthread"], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"field oracle build failed:\n{r.stdout}\n{r.stderr}")
        os.replace(tmp, so)
    L = C.CDLL(so)
    L.fwo_config_size.restype = C.c_int
    L.fwo_env_size.restype = C.c_int
    L.fwo_obs_dim.restype = C.c_int
    L.fwo_obs_dim.argtypes = [C.POINTER(fo.OConfig)]
    L.fwo_act_dim.restype = C.c_int
    L.fwo_act_dim.argtypes = [C.POINTER(fo.OConfig)]
    L.fwo_vec_reset.argtypes = [C.POINTER(fo.OConfig), C.POINTER(fo.OEnv), C.c_int, C.c_uint64, C.c_uint32, C.c_void_p, C.c_int]
    L.fwo_vec_step_info.argtypes = [C.POINTER(fo.OConfig), C.POINTER(fo.OEnv), C.c_int, C.c_uint64, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    L.fwo_refresh_surface_vel.argtypes = [C.POINTER(fo.OConfig), C.POINTER(fo.OEnv), C.c_int]
    L.fwf_set_field.argtypes = [C.c_void_p]
    L.fwf_set_field.restype = None
    L.fwf_wind_at.argtypes = [C.POINTER(FieldC), _D, C.POINTER(_D), C.POINTER(_D)]
    L.fwf_wind_at.restype = None
    if L.fwo_config_size() != C.sizeof(fo.OConfig) or L.fwo_env_size() != C.sizeof(fo.OEnv):
        raise RuntimeError("field oracle: struct sizes differ from the oracle's ctypes mirror")
    _lib = L
    return L


def make_field(wf) -> tuple[FieldC, np.ndarray]:
    """(descriptor, the float32 values it points to -- keep both alive) of a pyflyt_drone_b200.wind.WindField."""
    v = np.ascontiguousarray(wf.values, dtype=np.float32)
    f = FieldC()
    f.values = v.ctypes.data_as(C.c_void_p).value
    f.nt, f.nz, f.ny, f.nx = (int(s) for s in v.shape[:4])
    for k in range(3):
        f.origin[k], f.spacing[k] = float(wf.origin[k]), float(wf.spacing[k])
        f.shift_lo[k], f.shift_hi[k] = float(wf.shift_range[k, 0]), float(wf.shift_range[k, 1])
    f.t_step = float(wf.t_step)
    f.randomize_time = int(bool(wf.randomize_time))
    return f, v


def wind_at(field: tuple[FieldC, np.ndarray], t: float, x) -> np.ndarray:
    """The field's wind (fp64) at time t and field-frame point x."""
    xa = (C.c_double * 3)(*[float(v) for v in x])
    w = (C.c_double * 3)()
    lib().fwf_wind_at(C.byref(field[0]), float(t), xa, w)
    return np.array(w[:])


class FieldOracleVecEnv(fo.OracleVecEnv):
    """The oracle VecEnv flying a gridded wind field (wind_mode 3; the config's wind_randomize / wind_start_substep apply)."""

    def __init__(self, cfg: dict, n: int, seed: int = 0, env_id0: int = 0, nthreads: int = 1, wind_field=None):
        super().__init__(cfg, n, seed=seed, env_id0=env_id0, nthreads=nthreads)
        self.L = lib()
        self._field = make_field(wind_field)
        self.cfg.wind_mode = 3

    def _install(self) -> None:
        self.L.fwf_set_field(C.addressof(self._field[0]))

    def reset(self):
        self._install()
        return super().reset()

    def step(self, actions):
        self._install()
        return super().step(actions)

    def set_state(self, s: dict) -> None:
        self._install()
        super().set_state(s)
