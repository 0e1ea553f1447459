"""Timing of the normal equations of gravity-gradient observations (gb_points_gravity_gradient_normals) on the GPU, with
CUDA events.

    python tools/time_gravity_gradient_normals.py [--out FILE] [--profile TRACE_DIR]

Degree 96 (K' = 9409) at the 86 400 positions of the seeded near-polar circular orbit at R + 490 km of
tools/time_gradient_covariance.py.  One JSON line per frame (also written to FILE):
  - the normal matrix N = J~' J~ (PointsPlan.gravity_gradient_normals, unit weights) and the right-hand side J~' l of
    one observation set (PointsPlan.gravity_gradient_adjoint);
  - the flops executed, counted from the GEMM tiles actually contracted (the tiles that touch the upper triangle, with
    the zero-padded observation rows of each point block), and the algorithmic 6 P K'^2 of the symmetric product;
  - the executed rate against the live DMMA peak of gb_probe_fp64_peak.
With --profile the run is a torch.profiler pass over one Earth-fixed call instead (tracing slows the host, so it is a
run of its own): one line with the device time per kernel and the row writer's share of the call.  Every input stays
on the device.  The GPU's name and power limit are read in the same run (nvidia-smi, read-only).
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
    """2 * 128 * 120 * rows per contracted tile, summed over the point blocks of gb_points_gravity_gradient_normals (the
    block size below restates the one of gb_points.cu: an A operand of about 512 MB at six rows per point, a multiple of
    4 points, at most 8192)."""
    n_mt, n_nt = -(-K // TM), -(-K // TN)
    upper = sum(1 for mt in range(n_mt) for nt in range(n_nt) if (nt + 1) * TN > mt * TM)
    pb = (512 << 20) // (n_mt * LDA * 8) // 6 // 4 * 4
    pb = min(max(pb, 4), 8192, (P + 3) // 4 * 4)
    rows = sum((6 * min(pb, P - p0) + 3) // 4 * 4 for p0 in range(0, P, pb))
    return 2.0 * TM * TN * rows * upper, upper, n_mt * n_nt, pb


def profile(gp, normals, trace_dir):
    """Device time per kernel of one Earth-fixed call, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile as tprofile
    normals.zero_()
    gp.gravity_gradient_normals(normals, 0, 'cartesian')
    torch.cuda.synchronize()
    with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
        normals.zero_()
        gp.gravity_gradient_normals(normals, 0, 'cartesian')
        torch.cuda.synchronize()
    if trace_dir:
        os.makedirs(trace_dir, exist_ok=True)
        prof.export_chrome_trace(os.path.join(trace_dir, "gravity_gradient_normals_trace.json"))
    per = {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            per[ev.name] = per.get(ev.name, 0.0) + ev.device_time_total / 1e3
    total = sum(per.values())
    writer = sum(v for k, v in per.items() if "gravity_gradient_normal_rows" in k)
    design = sum(v for k, v in per.items() if "design_rows" in k)
    top = sorted(per.items(), key=lambda kv: -kv[1])[:8]
    return dict(case="profile, cartesian", kernel_ms_total=total, row_writer_ms=writer, design_rows_ms=design,
                row_writer_share=writer / total, design_rows_share=design / total,
                kernels_ms={k[:80]: v for k, v in top})


def main():
    out_path = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else os.path.join(
        os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "gravity_gradient_normals.jsonl")
    trace_dir = sys.argv[sys.argv.index("--profile") + 1] if "--profile" in sys.argv else None
    info = gpu_info()
    lib = _lib.load()
    mma, fma = ctypes.c_double(0.0), ctypes.c_double(0.0)
    _lib.check(lib.gb_probe_fp64_peak(0, ctypes.byref(mma), ctypes.byref(fma)))
    K = (N + 1) ** 2
    r, colat, lon = utilities.cartesian_to_spherical(orbit(86400, 4))
    P = r.size
    gp = gplan.gravity_gradient_points_plan(r, colat, lon, N)
    normals = torch.zeros((K, K), dtype=torch.float64, device="cuda")
    obs = torch.as_tensor(np.random.default_rng(5).standard_normal((1, 6, P)) * 1e-9).cuda()
    executed, upper, tiles, pb = executed_flops(P, K)
    algorithmic = 6.0 * P * K ** 2
    lines = []
    for frame in () if "--profile" in sys.argv else ("cartesian", "local"):
        def run_normals():
            normals.zero_()
            gp.gravity_gradient_normals(normals, 0, frame)
        ms_normals = ev_ms(run_normals)
        ms_rhs = ev_ms(lambda: gp.gravity_gradient_adjoint(obs, frame))
        rate = executed / (ms_normals * 1e-3) / 1e12
        res = dict(info, case="orbit, 86400 positions, " + frame, points=P, K=K, ms_normals=ms_normals,
                   ms_right_hand_side=ms_rhs, points_per_block=pb, tiles_contracted_per_block=upper,
                   tiles_per_block=tiles, tflop_executed=executed / 1e12, tflop_algorithmic=algorithmic / 1e12,
                   tflops_executed=rate, tflops_algorithmic=algorithmic / (ms_normals * 1e-3) / 1e12,
                   fraction_of_live_dmma_peak=rate / mma.value, live_dmma_peak_tflops=mma.value)
        print(json.dumps(res), flush=True)
        lines.append(res)
    if "--profile" in sys.argv:
        res = dict(info, **profile(gp, normals, trace_dir))
        print(json.dumps(res), flush=True)
        lines.append(res)
    gp.close()
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as fh:
        fh.write("".join(json.dumps(res) + "\n" for res in lines))


if __name__ == "__main__":
    main()
