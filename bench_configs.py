#!/usr/bin/env python
"""Secondary benchmark: every BASELINE.json config (not only the headline config 2 of bench.py),
each with parity against the CPU oracle and the oracle (= reference algorithm) timed on a bounded
sample on this box's host cores.  One JSON line per config; `python bench_configs.py > file`.

Timing: CUDA events on the launch stream, 3 warm-ups, best of 5, inputs and outputs device resident.
"""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import grates_b200 as gb  # noqa: E402
from oracle import sh_oracle as orc  # noqa: E402


def ev_time(fn, reps=5, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return min(ts)


def err(a, b):
    return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))


def blas_threads():
    try:
        from threadpoolctl import threadpool_info
        return max([p["num_threads"] for p in threadpool_info() if p.get("user_api") == "blas"] or [os.cpu_count()])
    except Exception:
        return os.cpu_count()


def peak(device=0):
    import ctypes
    a, b = ctypes.c_double(0), ctypes.c_double(0)
    gb._lib.check(gb._lib.load().gb_probe_fp64_peak(int(device or 0), ctypes.byref(a), ctypes.byref(b)))
    return max(a.value, b.value)


def syn_flops(N, nlat, nlon, E):
    """SURVEY 8(d) contract flops of the direct two-stage synthesis."""
    L = N + 1
    return 2.0 * E * nlat * L * L + 2.0 * (2 * L - 1) * E * nlat * nlon


def syn_flops_executed(N, plan, E):
    """What the kernels execute: the symmetric stage 2 contracts one quadrant of meridians (one octant with the even
    orders split once more: 3/4 of that), the folded stage 1 the northern parallels."""
    L = N + 1
    s1 = 2.0 * E * plan.nlat * L * L / (2.0 if plan.folded else 1.0)
    s2 = 2.0 * (2 * L - 1) * E * plan.nlat * plan.nlon / (4.0 if plan.symmetric else 1.0) * (0.75 if plan.octant else 1.0)
    return s1 + s2


class Ctx:
    """Rank layout and collectives of one run (a single process when dist is None)."""

    def __init__(self, rank=0, world=1, dev=None, dist=None):
        self.rank, self.world, self.dist = rank, world, dist
        self.dev = dev if dev is not None else torch.device("cuda", torch.cuda.current_device())
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)      # > 126 MB L2

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max(self, x):
        t = torch.tensor([x], dtype=torch.float64, device=self.dev)
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def shard(self, count):
        return gb.distributed.shard_range(count, self.world, self.rank)

    def time(self, fn, reps=5, warm=3):
        """Device milliseconds of fn: CUDA events on the launch stream, L2 flushed before every repetition, mean of
        `reps` after `warm` warm-ups, max over ranks."""
        for _ in range(warm):
            fn()
        self.barrier()
        total = 0.0
        for _ in range(reps):
            self.flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            total += e0.elapsed_time(e1)
        return self.max(total / reps)


def _reference():
    """The unmodified reference package (baseline/_ref) or None; see bench.load_reference."""
    import bench
    return bench.load_reference()


def _ref_field(grates, anm):
    pc = grates.gravityfield.PotentialCoefficients(3.9860044150e+14, 6.3781363000e+06)
    pc.anm = anm
    return pc


def config1(pk, ctx=None, with_cpu=True):
    """Single coefficient set: no useful sharding, every rank is a replica (SURVEY 8e)."""
    ctx = ctx or Ctx()
    N, d = 60, 1.0
    grid, og = gb.GeographicGrid(d, d), orc.geographic_grid(d, d)
    anm = orc.synthetic_coefficients(N, 0)
    pc = gb.PotentialCoefficients()
    pc.anm = anm
    out = pc.to_grid(grid, "ewh")
    t0 = time.perf_counter()
    for _ in range(20):
        pc.to_grid(grid, "ewh")
    host_call = (time.perf_counter() - t0) / 20
    plan = gb.get_plan(grid, N, "ewh", device=ctx.dev.index)
    x = torch.as_tensor(anm[None]).to(ctx.dev)
    buf = torch.empty((1, 180, 360), dtype=torch.float64, device=ctx.dev)
    ms = ctx.time(lambda: plan.synthesis(x, out=buf))
    ref = orc.synthesis(anm, og, "ewh")
    res = {"config": "c1: single degree-60 set -> 1deg grid, ewh", "gpu_kernels_ms": ms,
           "gpu_to_grid_call_ms": host_call * 1e3, "grid_pts_per_s_device": 64800 / ms * 1e3,
           "grid_pts_per_s_call": 64800 / host_call, "parity_max_normalised": err(out.value_array, ref),
           "contract_flops": syn_flops(N, 180, 360, 1), "frac_fp64_peak_contract_flops": syn_flops(N, 180, 360, 1) / ms / 1e9 / pk,
           "sharding": "replicas only (one set)",
           "note": "latency bound: 19 MFLOP; the call time is plan lookup + 0.5 MB D2H"}
    if with_cpu and ctx.rank == 0:
        grates = _reference()
        if grates is not None:
            rg, rp = grates.grid.GeographicGrid(d, d), _ref_field(grates, anm)
            run, kind = (lambda: rp.to_grid(rg, "ewh")), "reference"
        else:
            run, kind = (lambda: orc.synthesis(anm, og, "ewh")), "port"
        run()
        t0 = time.perf_counter()
        for _ in range(5):
            run()
        cpu = (time.perf_counter() - t0) / 5
        res["cpu_baseline"] = {"s_per_call": cpu, "grid_pts_per_s": 64800 / cpu, "cores": blas_threads(), "kind": kind,
                               "sample": "5 full calls after warm-up"}
    return res


def config3(pk, ctx=None, with_cpu=True):
    ctx = ctx or Ctx()
    N, d, E_all = 180, 0.25, 120
    e0, e1 = ctx.shard(E_all)
    E = e1 - e0
    grid, og = gb.GeographicGrid(d, d), orc.geographic_grid(d, d)
    plan = gb.get_plan(grid, N, "ewh", device=ctx.dev.index)
    t0 = time.perf_counter()
    plan.set_analysis(0, grid.area.reshape(plan.nlat, plan.nlon))
    t_ops = time.perf_counter() - t0
    anm = np.stack([orc.synthetic_coefficients(N, e) for e in range(e0, e1)])
    x = torch.as_tensor(anm).to(ctx.dev)
    v = torch.empty((E, plan.nlat, plan.nlon), dtype=torch.float64, device=ctx.dev)
    back = torch.empty_like(x)
    ms_syn = ctx.time(lambda: plan.synthesis(x, out=v))
    ms_ana = ctx.time(lambda: plan.analysis(v, out=back))
    rt = float((back - x).abs().max() / x.abs().max())
    P = plan.nlat * plan.nlon
    res = {"config": "c3: degree-180 synthesis to 0.25deg + analysis round trip, 120 epochs",
           "epochs_per_gpu": E, "synthesis_ms": ms_syn, "analysis_ms": ms_ana, "analysis_operator_build_s_once": t_ops,
           "synthesis_grid_pts_epochs_per_s": E_all * P / ms_syn * 1e3, "analysis_grid_pts_epochs_per_s": E_all * P / ms_ana * 1e3,
           "contract_flops": syn_flops(N, plan.nlat, plan.nlon, E_all),
           "synthesis_contract_multiple_of_fp64_peak": syn_flops(N, plan.nlat, plan.nlon, E_all) / ms_syn / 1e9 / pk / ctx.world,
           "analysis_contract_multiple_of_fp64_peak": syn_flops(N, plan.nlat, plan.nlon, E_all) / ms_ana / 1e9 / pk / ctx.world,
           # executed: the four-fold meridian symmetry quarters the longitude stage of both directions, the equator fold
           # halves the Legendre stage of the synthesis
           "synthesis_frac_fp64_peak_executed_flops": syn_flops_executed(N, plan, E_all) / ms_syn / 1e9 / pk / ctx.world,
           "round_trip_max_normalised": rt}
    if ctx.rank == 0:
        # parity on a bounded sample: epoch 0 against the oracle (synthesis and analysis)
        ref0 = orc.synthesis(anm[0], og, "ewh")
        res["parity_synthesis"] = err(v[0].cpu().numpy(), ref0)
        res["parity_analysis_vs_oracle"] = err(back[0].cpu().numpy(), orc.analysis_separable(ref0, og, 0, N, "ewh"))
        if with_cpu:
            # CPU: synthesis through the reference on 2 epochs; analysis: per-order operator build + mat-vec for orders
            # 0, 90, 180 of ONE epoch, integrated over the orders (a full epoch is ~16 min and 6 GB in the reference,
            # grid.py:665-696)
            grates = _reference()
            if grates is not None:
                rg = grates.grid.GeographicGrid(d, d)
                run, kind = (lambda a: _ref_field(grates, a).to_grid(rg, "ewh")), "reference"
            else:
                run, kind = (lambda a: orc.synthesis(a, og, "ewh")), "port"
            t0 = time.perf_counter()
            run(anm[0])
            run(anm[1])
            cpu_syn = (time.perf_counter() - t0) / 2
            orders, secs = [0, 90, 180], []
            vals0 = ref0.ravel()
            for m in orders:
                t0 = time.perf_counter()
                ops = orc.analysis_operator_per_order(og, m, 0, N, "ewh")
                for op in (ops if isinstance(ops, tuple) else (ops,)):
                    op @ vals0
                secs.append(time.perf_counter() - t0)
            cpu_ana = float((np.trapezoid if hasattr(np, "trapezoid") else np.trapz)(secs, orders))
            res["cpu_baseline"] = {"synthesis_s_per_epoch": cpu_syn, "analysis_s_per_epoch_extrapolated": cpu_ana,
                                   "synthesis_grid_pts_epochs_per_s": P / cpu_syn, "analysis_grid_pts_epochs_per_s": P / cpu_ana,
                                   "cores": blas_threads(), "kind": kind + " (synthesis) / port (analysis)",
                                   "sample": "synthesis: 2 of 120 epochs; analysis: orders 0/90/180 of one epoch "
                                             "(%.1f/%.1f/%.1f s) integrated over 181 orders" % tuple(secs)}
    return res


def config4(pk, ctx=None, with_cpu=True, extras=True):
    ctx = ctx or Ctx()
    N, d = 96, 0.5
    grid, og = gb.GeographicGrid(d, d), orc.geographic_grid(d, d)
    plan = gb.get_plan(grid, N, "ewh", device=ctx.dev.index)
    sig_h = orc.synthetic_covariance(N)          # the same matrix on every rank: Sigma resident everywhere
    sigma = torch.as_tensor(sig_h).to(ctx.dev)
    # row blocks sharded over the GPUs: every rank takes a block of northern parallels and its mirror image
    # (GB_COV_MIRRORED: both halves share the first contraction); one GPU: the whole grid, which folds by itself
    r0, r1 = ctx.shard(plan.nlat // 2)
    mirrored = ctx.world > 1
    nloc = 2 * (r1 - r0)
    out = torch.empty((nloc, plan.nlon), dtype=torch.float64, device=ctx.dev)
    if mirrored:
        run = lambda o: plan.covariance_propagation(sigma, 0, r0, r1 - r0, out=o, mirrored=True)     # noqa: E731
        out_rows = list(range(r0, r1)) + list(range(plan.nlat - r1, plan.nlat - r0))
    else:
        run = lambda o: plan.covariance_propagation(sigma, 0, out=o)     # noqa: E731
        out_rows = list(range(plan.nlat))
    ms = ctx.time(lambda: run(out), reps=3, warm=1)
    again = torch.empty_like(out)
    run(again)
    K, P = (N + 1) ** 2, plan.nlat * plan.nlon
    contract = 2.0 * P * K * K + 2.0 * P * K
    # symmetric Sigma (detected by the host): only the order-block pairs k <= k' of H_i are formed; equator fold: the
    # first contraction runs for the northern parallels only
    # ... and the longitude form W = H T runs on the synthesis' Fourier stage (four-fold meridian symmetry: 1/4)
    executed = 0.5 * plan.nlat * K * K + 0.5 * P * (2 * N + 2) ** 2
    res = {"config": "c4: covariance propagation, degree 96 (K=9409) -> 0.5deg grid",
           "parallels_per_gpu": nloc, "ms": ms, "points_per_s": P / ms * 1e3,
           "bit_identical_across_two_runs": bool(torch.equal(out, again)),
           "contract_flops": contract, "executed_flops": executed,
           "contract_multiple_of_fp64_peak": contract / ms / 1e9 / pk / ctx.world,
           "frac_fp64_peak_executed_flops": executed / ms / 1e9 / pk / ctx.world,
           "declared_restructuring": "regular grid: F = U (x) T factors, H_i = U_i' Sigma U_i per parallel then a "
                                     "longitude quadratic form; 2 nlat K^2 + 2 P (2L)^2 flops instead of 2 P K^2; "
                                     "a symmetric Sigma (checked on a sample of entries) halves the first term, the "
                                     "equator fold (mirrored parallels share U up to the sign (-1)^(n-m)) halves it again; the longitude "
                                     "form runs on the synthesis' symmetric Fourier stage (1/4 of its multiply-adds)"}
    if ctx.dist is not None:
        # the broadcast a caller pays when Sigma originates on one rank (not part of `ms`)
        buf = torch.empty_like(sigma)
        ctx.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ctx.dist.broadcast(buf if ctx.rank else sigma, src=0)
        e1.record()
        e1.synchronize()
        res["sigma_broadcast_ms_not_in_ms"] = ctx.max(e0.elapsed_time(e1))
        del buf
    if ctx.rank == 0:
        pick = [0, nloc // 3, nloc - 1]               # positions in this rank's output
        rows = [out_rows[q] for q in pick]
        t0 = time.perf_counter()
        ref = orc.covariance_propagation(sig_h, og, 0, N, "ewh", rows=rows)
        cpu_row = (time.perf_counter() - t0) / len(rows)
        res["parity_max_normalised_3_parallels"] = err(out[pick].cpu().numpy(), ref)
        if with_cpu:
            res["cpu_baseline"] = {"s_per_parallel": cpu_row, "s_total_extrapolated": cpu_row * plan.nlat,
                                   "points_per_s": plan.nlon / cpu_row, "cores": blas_threads(), "kind": "port",
                                   "sample": "3 of 360 parallels of grid.py:833-835 (cost is identical per parallel: two dgemms)"}
    if extras and ctx.world == 1:
        ms_full = ctx.time(lambda: plan.covariance_propagation(sigma, 0, out=out, symmetric=False), reps=3, warm=1)
        res["ms_without_symmetry"] = ms_full
        res["executed_flops_without_symmetry"] = 1.0 * plan.nlat * K * K + 0.5 * P * (2 * N + 2) ** 2
        # the direct point kernel (no grid structure assumed) on a 4-parallel slice, for the contract-flop roofline
        sl = gb.IrregularGrid(grid.longitude[:4 * plan.nlon], grid.latitude[:4 * plan.nlon])
        pp = gb.get_points_plan(sl, N, "ewh")
        ms_direct = ctx.time(lambda: pp.covariance_propagation(sigma, 0, symmetric=False), reps=2, warm=1)
        ms_direct_sym = ctx.time(lambda: pp.covariance_propagation(sigma, 0, symmetric=True), reps=2, warm=1)
        direct_flops = 2.0 * sl.point_count * K * K
        res["direct_point_kernel"] = {"points": sl.point_count, "ms": ms_direct, "flops": direct_flops,
                                      "frac_fp64_peak": direct_flops / ms_direct / 1e9 / pk,
                                      "ms_upper_triangle_of_symmetric_sigma": ms_direct_sym,
                                      "note": "gbgemm::kernel<PointQuadForm>: blocked diag(F Sigma F') on DMMA, no grid structure assumed"}
    return res


def config5(pk, ctx=None, with_cpu=True):
    ctx = ctx or Ctx()
    N, d, E_all = 120, 0.25, 500
    e0, e1 = ctx.shard(E_all)
    E = e1 - e0
    grid, og = gb.GeographicGrid(d, d), orc.geographic_grid(d, d)
    blocks = orc.synthetic_filter_blocks(N)
    flt = gb.OrderWiseFilter(blocks)
    plan = gb.get_plan(grid, N, "ewh", device=ctx.dev.index)
    anm = np.stack([orc.synthetic_coefficients(N, e) for e in range(e0, e1)])
    x = torch.as_tensor(anm).to(ctx.dev)
    y = torch.empty_like(x)
    v = torch.empty((E, plan.nlat, plan.nlon), dtype=torch.float64, device=ctx.dev)
    ms_f = ctx.time(lambda: flt.filter_batch(x, out=y))
    ms_two = ctx.time(lambda: plan.synthesis(flt.filter_batch(x, out=y), out=v), reps=3, warm=1)
    v2 = v.clone()
    # the shipped path: the filter writes straight into the synthesis workspace (no unpack / second pack)
    ms_all = ctx.time(lambda: plan.synthesis(x, out=v, orderwise_filter=flt), reps=3, warm=1)
    fused_identical = bool(torch.equal(v, v2))
    P = plan.nlat * plan.nlon
    fbytes = 2.0 * x.numel() * 8 + sum(b.size for b in blocks) * 8
    hbm = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"] if os.path.exists(
        os.path.join(ROOT, "MEASURED_PEAKS.json")) else None
    res = {"config": "c5: order-wise block filter + synthesis, 500 epochs, degree 120 -> 0.25deg grid",
           "epochs_per_gpu": E, "filter_ms": ms_f, "filter_gbs_algorithmic": fbytes / ms_f / 1e6,
           "filter_frac_hbm_peak": (fbytes / ms_f / 1e6 / hbm) if hbm else None,
           "filter_plus_synthesis_ms": ms_all, "filter_then_synthesis_two_calls_ms": ms_two,
           "fused_bit_identical_to_two_calls": fused_identical, "grid_pts_epochs_per_s": E_all * P / ms_all * 1e3,
           "contract_flops": syn_flops(N, plan.nlat, plan.nlon, E_all),
           "contract_multiple_of_fp64_peak": syn_flops(N, plan.nlat, plan.nlon, E_all) / ms_all / 1e9 / pk / ctx.world,
           "frac_fp64_peak_executed_flops": syn_flops_executed(N, plan, E_all) / ms_all / 1e9 / pk / ctx.world}
    if ctx.rank == 0:
        picks = (0, E - 1)
        refs = [orc.synthesis(orc.orderwise_filter(blocks, anm[e]), og, "ewh") for e in picks]
        res["parity_max_normalised_2_epochs"] = max(err(v[e].cpu().numpy(), r) for e, r in zip(picks, refs))
        if with_cpu:
            grates = _reference()
            if grates is not None:
                rg, rf = grates.grid.GeographicGrid(d, d), grates.filter.OrderWiseFilter(blocks)
                run, kind = (lambda a: rf.filter(_ref_field(grates, a)).to_grid(rg, "ewh")), "reference"
            else:
                run, kind = (lambda a: orc.synthesis(orc.orderwise_filter(blocks, a), og, "ewh")), "port"
            t0 = time.perf_counter()
            for e in picks:
                run(anm[e])
            cpu = (time.perf_counter() - t0) / 2
            res["cpu_baseline"] = {"s_per_epoch": cpu, "grid_pts_epochs_per_s": P / cpu, "cores": blas_threads(), "kind": kind,
                                   "sample": "2 of 500 epochs (OrderWiseFilter.filter + to_grid, cost linear in epochs)"}
    return res


def run_all(rank, world, dev, dist, with_cpu=True):
    """BASELINE configs 1, 3, 4, 5 for bench.py's `configs` block: every rank takes part (epoch shards for c3 / c5, row
    blocks with Sigma resident on every rank for c4, replicas for c1), times are max over ranks; parity and the CPU
    arms (N=1 only) on rank 0.  Returns a dict on every rank."""
    ctx = Ctx(rank, world, dev, dist)
    pk = peak(dev.index)
    res = {"fp64_peak_tflops_measured_live": pk, "n_gpus": world,
           "timing": "CUDA events, L2 flushed before every repetition, mean of 3-5 repetitions, max over ranks"}
    for name, fn in (("c1", config1), ("c3", config3), ("c4", lambda p, c, w: config4(p, c, w, extras=False)), ("c5", config5)):
        res[name] = fn(pk, ctx, with_cpu)
        gb.clear_plan_cache()
        torch.cuda.empty_cache()
    return res


def widened(pk):
    """Rows of SURVEY 8(f) built so far, at config-2 / config-4 sizes: isotropic filter fused into the synthesis,
    device-resident consumers, filtered covariance propagation, basin variances."""
    N, d, E = 96, 0.5, 240
    grid, og = gb.GeographicGrid(d, d), orc.geographic_grid(d, d)
    plan = gb.get_plan(grid, N, "ewh")
    P = plan.nlat * plan.nlon
    anm = np.stack([orc.synthetic_coefficients(N, e) for e in range(E)])
    x = torch.as_tensor(anm).cuda()
    v = torch.empty((E, plan.nlat, plan.nlon), dtype=torch.float64, device="cuda")
    flt = gb.Gaussian(300.0)
    w = torch.as_tensor(flt.degree_weights(N)).cuda()
    ms_plain = ev_time(lambda: plan.synthesis(x, out=v))
    ms_fused = ev_time(lambda: plan.synthesis(x, out=v, degree_weights=w))
    t0 = time.perf_counter()
    ref = orc.synthesis(orc.degreewise_filter(anm[3], orc.gauss_weights(300.0, N), 2), og, "ewh")
    cpu_syn = time.perf_counter() - t0
    par_fused = err(v[3].cpu().numpy(), ref)
    # consumers on the device
    mask = np.random.default_rng(2).uniform(size=P) < 0.2
    mask_d = torch.as_tensor(mask).cuda()
    ms_stats = ev_time(lambda: gb.grid_statistics(v, grid, mask_d), reps=3, warm=1)
    st = gb.grid_statistics(v, grid, mask)
    g1 = grid.copy()
    g1.values = v[5].cpu().numpy().ravel()
    t0 = time.perf_counter()
    cpu_stats = (g1.mean(mask), g1.rms(mask), g1.std(mask))
    cpu_stats_s = time.perf_counter() - t0
    par_stats = max(abs(st["mean"][5] - cpu_stats[0]), abs(st["rms"][5] - cpu_stats[1]), abs(st["std"][5] - cpu_stats[2])) / abs(cpu_stats[1])
    rms = torch.empty(P, dtype=torch.float64, device="cuda")
    import ctypes
    lib = gb._lib.load()
    vv = v.reshape(E, -1)
    ms_rms = ev_time(lambda: gb._lib.check(lib.gb_temporal_rms(ctypes.c_void_p(vv.data_ptr()), E, P, ctypes.c_void_p(rms.data_ptr()),
                                                               0, gb.plan._stream_handle(0))))
    hbm = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"] if os.path.exists(
        os.path.join(ROOT, "MEASURED_PEAKS.json")) else None
    # covariance side
    sig_h = orc.synthetic_covariance(N)
    sigma = torch.as_tensor(sig_h).cuda()
    out = torch.empty((plan.nlat, plan.nlon), dtype=torch.float64, device="cuda")
    blocks = orc.synthetic_filter_blocks(N)
    of = gb.OrderWiseFilter(blocks)
    ms_cov = ev_time(lambda: plan.covariance_propagation(sigma, 0, out=out), reps=3, warm=1)
    ms_cov_f = ev_time(lambda: plan.covariance_propagation(sigma, 0, out=out, spatial_filter=of), reps=3, warm=1)
    masks = np.random.default_rng(3).uniform(size=(16, P)) < 0.05
    t0 = time.perf_counter()
    gb.basin_variances(sigma, grid, masks, 0, N, "ewh")           # builds the adjoint operators (host, once)
    first_call = time.perf_counter() - t0
    t0 = time.perf_counter()
    std = gb.basin_variances(sigma, grid, masks, 0, N, "ewh")
    basin_s = time.perf_counter() - t0
    K = (N + 1) ** 2
    return {"config": "f-rows at config-2/4 sizes (N=96, 0.5deg, 240 epochs / K=9409)",
            "synthesis_ms": ms_plain, "synthesis_with_fused_gaussian_ms": ms_fused,
            "parity_fused_gaussian": par_fused,
            "grid_statistics_ms_3_moments_240_epochs": ms_stats,
            "grid_statistics_gbs": 2.0 * E * P * 8 / ms_stats / 1e6,
            "grid_statistics_parity_vs_host_formulas": par_stats,
            "temporal_rms_ms": ms_rms, "temporal_rms_gbs": E * P * 8 / ms_rms / 1e6,
            "temporal_rms_frac_hbm_peak": (E * P * 8 / ms_rms / 1e6 / hbm) if hbm else None,
            "covprop_ms": ms_cov, "covprop_with_orderwise_filter_ms": ms_cov_f,
            "reference_way_for_filtered_covprop": "F Sigma F' dense: 2 * 2 K^3 = %.1f TFLOP before the propagation" % (4.0 * K ** 3 / 1e12),
            "basin_variances_16_basins_s": basin_s, "basin_variances_first_call_s_incl_operator_build": first_call,
            "basin_std_range": [float(std.min()), float(std.max())],
            "cpu_baseline": {"synthesis_one_epoch_s": cpu_syn, "grid_statistics_one_epoch_s": cpu_stats_s,
                             "cores": blas_threads(), "kind": "port"}}


def point_sets(pk):
    """Rows a6 / a13 / f1 of SURVEY 8 at degree 96 on 40 962 scattered points: batched synthesis, the direct
    diag(F Sigma F'), and the adjoint (RadialBasisFunctions.to_potential_coefficients)."""
    N, P, E = 96, 40962, 240
    rng = np.random.default_rng(7)
    lon, lat = rng.uniform(-np.pi, np.pi, P), np.arcsin(rng.uniform(-1, 1, P))
    pts = gb.IrregularGrid(lon, lat)
    pp = gb.get_points_plan(pts, N, "ewh")
    K = (N + 1) ** 2
    anm = np.stack([orc.synthetic_coefficients(N, e) for e in range(E)])
    x = torch.as_tensor(anm).cuda()
    out = torch.empty((E, P), dtype=torch.float64, device="cuda")
    ms_syn = ev_time(lambda: pp.synthesis(x, out=out), reps=3, warm=1)
    sub = np.arange(0, P, P // 512)[:512]          # every 80th point: the sample reaches every block of points
    t0 = time.perf_counter()
    ref = orc.synthesis_points(anm[7], lon[sub], lat[sub], "ewh")
    cpu_syn = (time.perf_counter() - t0) * P / 512
    par_syn = err(out[7].cpu().numpy()[sub], ref)
    sig_h = orc.synthetic_covariance(N)
    sigma = torch.as_tensor(sig_h).cuda()
    ms_cov = ev_time(lambda: pp.covariance_propagation(sigma, 0, symmetric=True), reps=2, warm=1)
    ms_cov_full = ev_time(lambda: pp.covariance_propagation(sigma, 0, symmetric=False), reps=2, warm=1)
    std = pp.covariance_propagation(sigma, 0).cpu().numpy()
    t0 = time.perf_counter()
    ref_std = orc.covariance_propagation_points(sig_h, lon[sub], lat[sub], 0, N, "ewh")
    cpu_cov = (time.perf_counter() - t0) * P / 512
    par_cov = err(std[sub], ref_std)
    Kf = np.ones((N + 1, N + 1))
    rbf = gb.RadialBasisFunctions(pts, Kf, 0, N)
    v1 = torch.as_tensor(rng.standard_normal((1, P))).cuda()
    vE = torch.as_tensor(rng.standard_normal((E, P))).cuda()
    plan = rbf._points_plan()
    ms_adj1 = ev_time(lambda: plan.adjoint(v1), reps=3, warm=1)
    ms_adjE = ev_time(lambda: plan.adjoint(vE), reps=3, warm=1)
    got = rbf.to_potential_coefficients_batch(v1)[0].cpu().numpy()
    n_cpu = 2048
    cpu_pts = np.arange(0, P, P // n_cpu)[:n_cpu]    # every 20th point, spread over the whole set
    t0 = time.perf_counter()
    part = orc.radial_basis_to_coefficients(Kf, v1[0, cpu_pts].cpu().numpy(), lon[cpu_pts], lat[cpu_pts], N)
    cpu_adj = (time.perf_counter() - t0) * P / n_cpu
    small = gb.RadialBasisFunctions(gb.IrregularGrid(lon[cpu_pts], lat[cpu_pts]), Kf, 0, N)
    par_adj = err(small.to_potential_coefficients_batch(v1[:, cpu_pts].contiguous())[0].cpu().numpy(), part)
    del got
    return {"config": "point sets: N=96, 40962 scattered points, 240 epochs / K=9409",
            "synthesis_ms": ms_syn, "synthesis_tflops": 2.0 * P * K * E / ms_syn / 1e9, "synthesis_parity": par_syn,
            "covariance_symmetric_ms": ms_cov, "covariance_general_ms": ms_cov_full,
            "covariance_general_tflops": 2.0 * P * K * K / ms_cov_full / 1e9,
            "covariance_general_frac_fp64_peak": 2.0 * P * K * K / ms_cov_full / 1e9 / pk,
            "covariance_parity": par_cov,
            "adjoint_one_value_set_ms": ms_adj1, "adjoint_240_value_sets_ms": ms_adjE,
            "adjoint_240_tflops": 2.0 * P * K * E / ms_adjE / 1e9, "adjoint_parity_2048_points": par_adj,
            "cpu_baseline": {"synthesis_one_epoch_s_extrapolated_from_512_points": cpu_syn,
                             "covariance_s_extrapolated_from_512_points": cpu_cov,
                             "adjoint_one_value_set_s_extrapolated_from_2048_points": cpu_adj,
                             "cores": blas_threads(), "kind": "port"}}


def main():
    torch.cuda.set_device(0)
    pk = peak()
    which = sys.argv[1:] or ["c1", "c3", "c4", "c5", "f", "pts"]
    fns = {"c1": config1, "c3": config3, "c4": config4, "c5": config5, "f": widened, "pts": point_sets}
    for name in which:
        line = fns[name](pk)
        line["fp64_peak_tflops_measured_live"] = pk
        print(json.dumps(line), flush=True)
        gb.clear_plan_cache()
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
