"""Timing of the normal equations of acceleration observations (gb_points_gradient_normals) on the GPU, with CUDA events.

    python tools/time_gradient_normals.py [--out FILE]

Degree 96 (K' = 9409) at the 86 400 positions of the seeded near-polar circular orbit at R + 490 km of
tools/time_gradient_covariance.py.  One JSON line (also written to FILE):
  - the normal matrix N = J~' J~ (PointsPlan.gradient_normals, Earth-fixed, unit weights) and the right-hand side
    J~' l of one observation set (PointsPlan.gradient_adjoint);
  - the flops executed, counted from the GEMM tiles actually contracted (the tiles that touch the upper triangle, with
    the zero-padded observation rows of each point block), and the algorithmic 3 P K'^2 of the symmetric product;
  - the executed rate against the live DMMA peak of gb_probe_fp64_peak.
Every input stays on the device.  The GPU's name and power limit are read in the same run (nvidia-smi, read-only).
"""
import ctypes
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from grates_b200 import _lib, plan as gplan, utilities
from time_gradient_covariance import ev_ms, gpu_info, orbit

N = 96
TM, TN, LDA = 128, 120, 132          # gbgemm tile shape and the A operand pitch (gb_common.cuh)


def executed_flops(P, K):
    """2 * 128 * 120 * rows per contracted tile, summed over the point blocks of gb_points_gradient_normals (the block
    size below restates the one of gb_points.cu: an A operand of about 512 MB, a multiple of 4 points, at most 16384)."""
    n_mt, n_nt = -(-K // TM), -(-K // TN)
    upper = sum(1 for mt in range(n_mt) for nt in range(n_nt) if (nt + 1) * TN > mt * TM)
    pb = (512 << 20) // (n_mt * LDA * 8) // 3 // 4 * 4
    pb = min(max(pb, 4), 16384, (P + 3) // 4 * 4)
    rows = sum((3 * min(pb, P - p0) + 3) // 4 * 4 for p0 in range(0, P, pb))
    return 2.0 * TM * TN * rows * upper, upper, n_mt * n_nt, pb


def main():
    out_path = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else os.path.join(
        os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "gradient_normals.jsonl")
    info = gpu_info()
    lib = _lib.load()
    mma, fma = ctypes.c_double(0.0), ctypes.c_double(0.0)
    _lib.check(lib.gb_probe_fp64_peak(0, ctypes.byref(mma), ctypes.byref(fma)))
    K = (N + 1) ** 2
    r, colat, lon = utilities.cartesian_to_spherical(orbit(86400, 4))
    P = r.size
    gp = gplan.gradient_points_plan(r, colat, lon, N)
    normals = torch.zeros((K, K), dtype=torch.float64, device="cuda")
    obs = torch.as_tensor(np.random.default_rng(5).standard_normal((1, 3, P)) * 1e-6).cuda()

    def run_normals():
        normals.zero_()
        gp.gradient_normals(normals, 0, 'cartesian')
    ms_normals = ev_ms(run_normals)
    ms_rhs = ev_ms(lambda: gp.gradient_adjoint(obs, 'cartesian'))
    executed, upper, tiles, pb = executed_flops(P, K)
    algorithmic = 3.0 * P * K ** 2
    rate = executed / (ms_normals * 1e-3) / 1e12
    res = dict(info, case="orbit, 86400 positions", points=P, K=K, ms_normals=ms_normals, ms_right_hand_side=ms_rhs,
               points_per_block=pb, tiles_contracted_per_block=upper, tiles_per_block=tiles,
               tflop_executed=executed / 1e12, tflop_algorithmic=algorithmic / 1e12, tflops_executed=rate,
               tflops_algorithmic=algorithmic / (ms_normals * 1e-3) / 1e12, fraction_of_live_dmma_peak=rate / mma.value,
               live_dmma_peak_tflops=mma.value)
    print(json.dumps(res), flush=True)
    gp.close()
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as fh:
        fh.write(json.dumps(res) + "\n")


if __name__ == "__main__":
    main()
