"""Timing of the covariance of grad V (gb_points_gradient_covariance) on the GPU, with CUDA events.

    python tools/time_gradient_covariance.py [--out FILE]

Config 4's Sigma (oracle.synthetic_covariance, degree 96, K = 9409) at 86 400 positions of a seeded near-polar circular
orbit at R + 490 km and at the benchmark's 40 962 points.  One JSON line per case (also written to FILE):
  - the new call (3 x 3 covariances, Earth-fixed) and its rate: 2 (3P) K^2 algorithmic flops, 3 P K^2 executed (the
    lower triangle of the symmetric part), against the live DMMA peak of gb_probe_fp64_peak;
  - gb_points_covariance with a symmetric Sigma on the same points (P K^2 executed) and the ratio of the two times per
    design column (3P columns against P).
Every input stays on the device.  The GPU's name and power limit are read in the same run (nvidia-smi, read-only).
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
from oracle import sh_oracle as orc

N = 96


def gpu_info():
    try:
        line = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
        name, power = (s.strip() for s in line.split(","))
    except (OSError, subprocess.CalledProcessError, IndexError, ValueError):
        name, power = torch.cuda.get_device_name(0), "unknown"
    return {"gpu": name, "power_limit": power}


def ev_ms(fn, reps=3, warm=1):
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


def orbit(count, seed):
    """Earth-fixed positions of a seeded near-polar circular orbit at R + 490 km, one per second."""
    rng = np.random.default_rng(seed)
    a, inc, node, u0 = orc.R_DEFAULT + 490e3, np.radians(89.0), rng.uniform(0, 2 * np.pi), rng.uniform(0, 2 * np.pi)
    t = np.arange(count, dtype=float)
    u = u0 + np.sqrt(orc.GM_DEFAULT / a ** 3) * t
    lam = node - 7.292115e-5 * t
    xo, yo, zo = np.cos(u), np.sin(u) * np.cos(inc), np.sin(u) * np.sin(inc)
    return a * np.stack((xo * np.cos(lam) - yo * np.sin(lam), xo * np.sin(lam) + yo * np.cos(lam), zo), axis=1)


def main():
    out_path = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else os.path.join(
        os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "gradient_covariance.jsonl")
    info = gpu_info()
    lib = _lib.load()
    mma, fma = ctypes.c_double(0.0), ctypes.c_double(0.0)
    _lib.check(lib.gb_probe_fp64_peak(0, ctypes.byref(mma), ctypes.byref(fma)))
    K = (N + 1) ** 2
    sigma = torch.as_tensor(orc.synthetic_covariance(N)).cuda()
    rng = np.random.default_rng(7)                                   # as bench_configs.point_sets
    lon_b, lat_b = rng.uniform(-np.pi, np.pi, 40962), np.arcsin(rng.uniform(-1, 1, 40962))
    a, f = utilities.A_GRS80, utilities.F_GRS80
    cases = [("orbit, 86400 positions", utilities.cartesian_to_spherical(orbit(86400, 4))),
             ("benchmark points, 40962", (utilities.geocentric_radius(lat_b, a, f), utilities.colatitude(lat_b, a, f),
                                         lon_b))]
    lines = []
    for label, (r, colat, lon) in cases:
        P = r.size
        gp = gplan.get_gradient_points_plan(r, colat, lon, N)
        n = np.arange(N + 1)
        kn = np.power((orc.R_DEFAULT / r)[:, None], n + 1) * orc.GM_DEFAULT / orc.R_DEFAULT
        pp = gplan.PointsPlan(lon, 0.5 * np.pi - colat, a, f, N, degree_factors=kn, colatitude=colat)
        ms = ev_ms(lambda: gp.gradient_covariance(sigma, 0, 'cartesian', True))
        ms_local_std = ev_ms(lambda: gp.gradient_covariance(sigma, 0, 'local', False))
        ms_cov = ev_ms(lambda: pp.covariance_propagation(sigma, 0, take_sqrt=False, symmetric=True))
        executed, algorithmic = 3.0 * P * K ** 2, 2.0 * 3 * P * K ** 2
        rate = executed / (ms * 1e-3) / 1e12
        rate_cov = (1.0 * P * K ** 2) / (ms_cov * 1e-3) / 1e12
        res = dict(info, case=label, points=P, K=K, ms_gradient_covariance_full_cartesian=ms,
                   ms_gradient_covariance_std_local=ms_local_std, ms_points_covariance_symmetric=ms_cov,
                   tflop_algorithmic=algorithmic / 1e12, tflop_executed=executed / 1e12,
                   tflops_executed=rate, fraction_of_live_dmma_peak=rate / mma.value,
                   live_dmma_peak_tflops=mma.value, tflops_executed_points_covariance=rate_cov,
                   time_per_design_column_ratio=(ms / (3 * P)) / (ms_cov / P))
        print(json.dumps(res), flush=True)
        lines.append(res)
        del gp, pp
        gplan.clear_plan_cache()
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as fh:
        for res in lines:
            fh.write(json.dumps(res) + "\n")


if __name__ == "__main__":
    main()
