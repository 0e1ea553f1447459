"""Timing of the gravitational acceleration (gradient_batch, gradient_at_positions) on the GPU, with CUDA events.

    python tools/time_gradient.py [--out FILE]

Prints one JSON line per case (and writes them to FILE):
  - GeographicGrid(0.5), N = 96, 240 epochs, both frames: the coefficient transform, the degree-97 synthesis of the 720
    sets and the rotation timed apart, next to one to_grid_batch of the same batch at N = 96 for scale;
  - 86 400 positions of a seeded near-polar circular orbit at R + 490 km, N = 96, 1 and 240 epochs.
The transform and the rotation are HBM-bound passes: their rates are the bytes they must move over their time.
Every input stays on the device; the 0.5 degree case moves 3 GB per rotation, far more than the 126 MB L2.
The GPU's name and power limit are read in the same run (nvidia-smi, read-only query).
"""
import ctypes
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import grates_b200 as gb
from grates_b200 import _lib, plan as gplan, utilities

N = 96
REPS = 20


def gpu_info():
    try:
        line = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
        name, power = (s.strip() for s in line.split(","))
    except (OSError, subprocess.CalledProcessError, IndexError, ValueError):
        name, power = torch.cuda.get_device_name(0), "unknown"
    return {"gpu": name, "power_limit": power}


def ev_ms(fn, reps=REPS, warm=3):
    """Median device time of fn over reps calls, each bracketed by its own events."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times))


def coefficients(E, seed):
    L = N + 1
    deg = np.arange(L)
    packed_degree = np.where(np.tril(np.ones((L, L), dtype=bool)), deg[:, None], deg[None, :])
    x = np.random.default_rng(seed).standard_normal((E, L, L)) / (packed_degree + 1.0)
    return torch.as_tensor(x).cuda()


def track(count, seed):
    """Earth-fixed positions of a near-polar (89 degree) circular orbit at R + 490 km, one per second."""
    rng = np.random.default_rng(seed)
    a, inc, node, u0 = gb.gravityfield.R_DEFAULT + 490e3, np.radians(89.0), rng.uniform(0, 2 * np.pi), rng.uniform(0, 2 * np.pi)
    t = np.arange(count, dtype=float)
    u = u0 + np.sqrt(gb.gravityfield.GM_DEFAULT / a ** 3) * t
    lam = node - 7.292115e-5 * t
    xo, yo, zo = np.cos(u), np.sin(u) * np.cos(inc), np.sin(u) * np.sin(inc)
    return a * np.stack((xo * np.cos(lam) - yo * np.sin(lam), xo * np.sin(lam) + yo * np.cos(lam), zo), axis=1)


def stages(x, p, npts, shape):
    """Times of the three steps of one gradient call on plan p, each alone."""
    lib, st = _lib.load(), gplan._stream_handle(p.device)
    E, L = x.shape[0], x.shape[-1]
    g = torch.empty((E, 3, L + 1, L + 1), dtype=torch.float64, device=x.device)
    res = torch.empty((E, 3) + shape, dtype=torch.float64, device=x.device)
    gview, rview = g.view(3 * E, L + 1, L + 1), res.view((3 * E,) + shape)

    def transform():
        _lib.check(lib.gb_gradient_coefficients(ctypes.c_void_p(x.data_ptr()), E, L - 1, ctypes.c_void_p(g.data_ptr()),
                                                p.device, st))

    def rotate():
        _lib.check(lib.gb_rotate_to_local(ctypes.c_void_p(res.data_ptr()), ctypes.c_void_p(p.frame.data_ptr()), E, npts,
                                          p.device, st))
    transform()
    t_tr = ev_ms(transform)
    t_syn = ev_ms(lambda: p.synthesis(gview, out=rview))
    t_rot = ev_ms(rotate)
    tr_bytes = 8 * (E * L * L + E * 3 * (L + 1) ** 2)          # read the input once, write the output once
    rot_bytes = 8 * (2 * E * 3 * npts + 4 * npts)             # read and write the values, read the frame
    return {"transform_ms": t_tr, "transform_GBps": tr_bytes / t_tr / 1e6, "synthesis_ms": t_syn,
            "rotation_ms": t_rot, "rotation_GBps": rot_bytes / t_rot / 1e6}


def grid_case():
    grid = gb.GeographicGrid(0.5)
    E = 240
    x = coefficients(E, 1)
    p = gb.get_gradient_plan(grid, N)
    shape = (p.nlat, p.nlon)
    out = {"case": "GeographicGrid(0.5) gradient", "N": N, "epochs": E, "sets": 3 * E, "octant": p.octant,
           "folded": p.folded}
    out.update(stages(x, p, p.nlat * p.nlon, shape))
    res = torch.empty((E, 3) + shape, dtype=torch.float64, device="cuda")
    out["gradient_batch_cartesian_ms"] = ev_ms(lambda: gb.gradient_batch(x, grid, out=res))
    out["gradient_batch_local_ms"] = ev_ms(lambda: gb.gradient_batch(x, grid, frame='local', out=res))
    vals = torch.empty((E,) + shape, dtype=torch.float64, device="cuda")
    out["to_grid_batch_ewh_ms"] = ev_ms(lambda: gb.to_grid_batch(x, grid, 'ewh', out=vals))
    return out


def orbit_cases():
    pos = track(86400, 2)
    rows = []
    for E in (1, 240):
        x = coefficients(E, 3)
        r, colat, lon = utilities.cartesian_to_spherical(pos)
        p = gb.get_gradient_points_plan(r, colat, lon, N)
        res = torch.empty((E, 3, pos.shape[0]), dtype=torch.float64, device="cuda")
        row = {"case": "orbit positions gradient", "N": N, "points": pos.shape[0], "epochs": E, "sets": 3 * E}
        row.update(stages(x, p, p.npts, (p.npts,)))
        row["gradient_at_positions_cartesian_ms"] = ev_ms(lambda: gb.gradient_at_positions(x, pos, out=res))
        row["gradient_at_positions_local_ms"] = ev_ms(lambda: gb.gradient_at_positions(x, pos, frame='local', out=res))
        rows.append(row)
    return rows


def main():
    if not torch.cuda.is_available():
        raise SystemExit("time_gradient.py needs a CUDA device")
    path = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    info = gpu_info()
    lines = []
    for row in [grid_case()] + orbit_cases():
        row.update(info)
        lines.append(json.dumps(row))
        print(lines[-1], flush=True)
    if path:
        with open(path, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
