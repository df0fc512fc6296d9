"""Gridded wind fields (wind_mode 3): the batched replacement for PyFlyt's ``Aviary.register_wind_field_function``.

The reference adds a custom wind with a Python closure ``f(time_s, positions[n, 3]) -> [n, 3]`` that PyFlyt evaluates at the
lifting surfaces on every physics step.  A closure cannot run inside the CUDA step, so a ``WindField`` samples it once on a
regular lattice over space and time (``WindField.from_function``); the step kernels interpolate that lattice at every lifting
surface's link CoM on every substep (include/fwsim.h ``FwWindField`` states the exact semantics: trilinear in space with
coordinates clamped to the box, linear and periodic in time, optional per-episode spatial shift and time offset).

    field = WindField.from_function(f, origin=(-100, -100, 0), spacing=2.0, shape=(101, 101, 51))
    env = FixedwingVecEnv(4096, preset="waypoints_v3", wind_field=field)
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, Sequence

import numpy as np


def _vec3(x, name: str) -> np.ndarray:
    a = np.asarray(x, dtype=np.float64)
    a = np.full(3, float(a)) if a.ndim == 0 else a.reshape(-1)
    if a.shape != (3,) or not np.all(np.isfinite(a)):
        raise ValueError(f"{name} must be a finite scalar or 3-vector, got {x!r}")
    return a


class WindField:
    """A world-frame (ENU) wind lattice: ``values[nt, nz, ny, nx, 3]`` float32 m/s at the points ``origin + (i, j, k) *
    spacing``, time slice ``s`` at ``s * t_step`` seconds (periodic with period ``nt * t_step``).

    shift_range: per-axis ``[(lo, hi)] * 3`` metres; with ``wind_randomize`` every reset draws a spatial shift from it (the
    field is sampled at ``position - shift``).  randomize_time: with ``wind_randomize`` every reset also draws a time offset
    from ``[0, nt * t_step)``."""

    def __init__(self, values, origin, spacing, t_step: float | None = None,
                 shift_range: Sequence[Sequence[float]] | None = None, randomize_time: bool = False):
        v = np.asarray(values)
        if v.ndim == 4:
            v = v[None]
        if v.ndim != 5 or v.shape[-1] != 3 or min(v.shape[:4]) < 1:
            raise ValueError(f"values must have shape [nt, nz, ny, nx, 3] (or [nz, ny, nx, 3]), got {np.shape(values)}")
        v = np.ascontiguousarray(v, dtype=np.float32)
        if not np.all(np.isfinite(v)):
            raise ValueError("wind field values must be finite")
        if v.size // 3 >= 2 ** 31:
            raise ValueError("a wind field holds fewer than 2^31 lattice points")
        self.values = v
        self.origin = _vec3(origin, "origin")
        self.spacing = _vec3(spacing, "spacing")
        if not np.all(self.spacing > 0):
            raise ValueError(f"spacing must be > 0, got {self.spacing.tolist()}")
        nt = v.shape[0]
        if t_step is None:
            if nt > 1:
                raise ValueError("a field with more than one time slice needs t_step")
            t_step = 1.0
        self.t_step = float(t_step)
        if not (np.isfinite(self.t_step) and self.t_step > 0):
            raise ValueError(f"t_step must be finite and > 0, got {t_step!r}")
        sr = np.zeros((3, 2)) if shift_range is None else np.asarray(shift_range, dtype=np.float64)
        if sr.shape != (3, 2) or not np.all(np.isfinite(sr)) or np.any(sr[:, 0] > sr[:, 1]):
            raise ValueError(f"shift_range must be [(lo, hi)] * 3 with lo <= hi, got {shift_range!r}")
        self.shift_range = sr
        self.randomize_time = bool(randomize_time)

    @property
    def shape(self) -> tuple[int, int, int]:
        """(nx, ny, nz)"""
        nt, nz, ny, nx, _ = self.values.shape
        return nx, ny, nz

    @property
    def n_slices(self) -> int:
        return int(self.values.shape[0])

    @property
    def device_bytes(self) -> int:
        """HBM the field occupies on the device (one float4 per lattice point)."""
        return int(self.values.size // 3 * 16)

    def lattice_points(self) -> np.ndarray:
        """World positions of the lattice points, [nz * ny * nx, 3] in the order of ``values``' spatial axes."""
        nx, ny, nz = self.shape
        z, y, x = np.meshgrid(np.arange(nz), np.arange(ny), np.arange(nx), indexing="ij")
        idx = np.stack([x, y, z], axis=-1).reshape(-1, 3).astype(np.float64)
        return self.origin + idx * self.spacing

    @classmethod
    def from_function(cls, f: Callable[[float, np.ndarray], np.ndarray], origin, spacing, shape: Sequence[int],
                      n_slices: int = 1, t_step: float | None = None, shift_range=None,
                      randomize_time: bool = False) -> "WindField":
        """Sample a PyFlyt-signature wind function ``f(time_s, positions[n, 3]) -> [n, 3]`` on the lattice of ``shape =
        (nx, ny, nz)`` points from ``origin`` with ``spacing``, at ``n_slices`` times ``0, t_step, ...`` (one call per slice)."""
        nx, ny, nz = (int(s) for s in shape)
        if min(nx, ny, nz) < 1 or int(n_slices) < 1:
            raise ValueError(f"shape and n_slices must be >= 1, got {tuple(shape)}, {n_slices}")
        if int(n_slices) > 1 and t_step is None:
            raise ValueError("a field with more than one time slice needs t_step")
        proto = cls(np.zeros((1, 1, 1, 1, 3), np.float32), origin, spacing)
        pts = cls(np.zeros((1, nz, ny, nx, 3), np.float32), proto.origin, proto.spacing).lattice_points()
        dt = 1.0 if t_step is None else float(t_step)
        out = np.empty((int(n_slices), nz, ny, nx, 3), np.float32)
        for s in range(int(n_slices)):
            w = np.asarray(f(s * dt, pts.copy()), dtype=np.float64)
            if w.shape != pts.shape:
                raise ValueError(f"the wind function returned shape {w.shape}, expected {pts.shape}")
            out[s] = w.reshape(nz, ny, nx, 3)
        return cls(out, proto.origin, proto.spacing, t_step=t_step, shift_range=shift_range, randomize_time=randomize_time)

    def to_c(self):
        """The ``FwWindField`` descriptor (its ``values`` pointer refers to this object's array: keep the object alive)."""
        from ._lib import FwWindFieldC
        nt, nz, ny, nx, _ = self.values.shape
        c = FwWindFieldC()
        c.values = self.values.ctypes.data_as(C.c_void_p).value
        c.nx, c.ny, c.nz, c.nt = nx, ny, nz, nt
        for k in range(3):
            c.origin[k] = float(self.origin[k])
            c.spacing[k] = float(self.spacing[k])
            c.shift_lo[k] = float(self.shift_range[k, 0])
            c.shift_hi[k] = float(self.shift_range[k, 1])
        c.t_step = self.t_step
        c.randomize_time = int(self.randomize_time)
        return c

    def __repr__(self) -> str:
        nx, ny, nz = self.shape
        return (f"WindField({nx}x{ny}x{nz} points x {self.n_slices} slices, origin={self.origin.tolist()}, "
                f"spacing={self.spacing.tolist()}, t_step={self.t_step})")
