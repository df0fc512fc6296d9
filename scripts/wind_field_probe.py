"""Cost of the gridded wind field (wind_mode 3) against the uniform winds, at 65,536 envs on one GPU.

For the physics-only and Waypoints tasks: wind off, `constant`, a static field of 101 x 101 x 51 points (2 m lattice over the
100 m dome, ~8 MB) and a 16-slice field of the same lattice (~133 MB, larger than the B200's 126 MB L2).  Each line times
`--launches` random-action env-step launches (fw_step_random: one launch per env-step) with CUDA events after a warm-up, and
reports env-steps/s, the field's bytes in HBM and the gather bytes the kernels request per env-step, computed from shapes:
substeps per env-step x 5 surfaces x 8 corners x 2 time slices x 16 B.  Card name and power limit are read in the same run.

    python scripts/wind_field_probe.py --out profiles/r3_wind_field_probe.jsonl
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import pyflyt_drone_b200 as fw  # noqa: E402
from pyflyt_drone_b200.vec_env import FixedwingVecEnv  # noqa: E402
from pyflyt_drone_b200.wind import WindField  # noqa: E402

NSURF, CORNERS, SLICES, POINT_BYTES = 5, 8, 2, 16


def dome_field(n_slices: int) -> WindField:
    """Shear plus a thermal on a 2 m lattice over the 100 m dome (x, y in [-100, 100], z in [0, 100])."""
    def f(t, x):
        z = np.maximum(x[:, 2], 0.0)
        r2 = (x[:, 0] - 20.0 - t) ** 2 + (x[:, 1] + 10.0) ** 2
        return np.stack([6.0 * (1.0 - np.exp(-z / 15.0)), 0.5 + 0.01 * x[:, 0],
                         2.5 * np.exp(-r2 / 300.0) * np.minimum(z / 10.0, 1.0)], axis=1)
    return WindField.from_function(f, origin=(-100.0, -100.0, 0.0), spacing=2.0, shape=(101, 101, 51), n_slices=n_slices,
                                   t_step=0.5 if n_slices > 1 else None, shift_range=[(-5, 5), (-5, 5), (0, 0)],
                                   randomize_time=n_slices > 1)


def card() -> dict:
    import torch
    out = {"device": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        out["nvidia_smi"] = r.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out["nvidia_smi"] = f"unavailable: {e}"
    return out


def measure(preset: str, wind: str, field: WindField | None, n_envs: int, launches: int, warmup: int) -> dict:
    import torch
    cfg = fw.make_config(preset)
    if wind == "constant":
        cfg = cfg.replace(wind_mode=1, wind_base=[3.0, -1.0, 0.2], wind_start_substep=0)
    elif field is not None:
        cfg = cfg.replace(wind_randomize=1, wind_start_substep=0)
    env = FixedwingVecEnv(n_envs, config=cfg, seed=1, wind_field=field)
    env.reset_tensor()
    env.step_random(warmup)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    env.step_random(launches)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    substeps = cfg.inner_per_step * cfg.substeps_per_inner
    line = dict(task=preset, wind=wind, n_envs=n_envs, launches=launches, ms=round(ms, 3),
                us_per_launch=round(1e3 * ms / launches, 2), env_steps_per_s=round(n_envs * launches / (ms * 1e-3)),
                field_bytes=field.device_bytes if field is not None else 0,
                field_shape=[*field.shape, field.n_slices] if field is not None else None,
                gather_bytes_per_env_step=substeps * NSURF * CORNERS * SLICES * POINT_BYTES if field is not None else 0,
                state_bytes_per_env_step=152)
    env.close()
    return line


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--launches", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    fields = {"field_static_8MB": dome_field(1), "field_16slice_133MB": dome_field(16)}
    lines = [dict(kind="card", **card())]
    print(json.dumps(lines[0]), flush=True)
    for preset in ("physics_only", "waypoints_v3"):
        for wind in ("off", "constant", *fields):
            ln = measure(preset, wind, fields.get(wind), a.envs, a.launches, a.warmup)
            lines.append(ln)
            print(json.dumps(ln), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
