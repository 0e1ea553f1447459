#!/usr/bin/env python
"""Benchmark of the B200 spherical-harmonic synthesis path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--scaling strong|weak]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

A step is one pass of the hot path over one batch: BASELINE config 2, synthesis of 240 epochs of
degree-96 coefficients onto the 0.5 degree geographic grid with the water-height kernel
(62.2 M grid-points x epochs).  The 240 epochs are split over the ranks ("strong" scaling, the north
star's partition: 30 epochs per GPU at N=8, no data-path collective); `--scaling weak` gives every
rank the whole batch instead, and a short weak measurement is reported beside the strong one.

Output: one JSON line (rank 0).
  value         device-resident throughput of the whole job (all ranks' units / max-over-ranks time)
  e2e           the same through the host-buffer C-ABI call (pinned host memory, H2D + D2H inside the
                timed region), with the measured D2H copy ceiling of this box beside it
  roofline      the dominant kernel (FP64 tensor-core longitude contraction): executed flops / its
                CUDA-event time against the live-measured FP64 DMMA peak
  cpu_baseline  the UNMODIFIED reference (baseline/_ref, PotentialCoefficients.to_grid) on this box's
                host cores on a bounded sample (N=1 only)
  configs       BASELINE configs 1, 3, 4, 5: device time, parity on a bounded sample, roofline, CPU arm

`--impl reference` times the reference's own CPU implementation (baseline/_ref when present, else the
numpy oracle port) on the same config, metric and unit; rank 0 only.

`--dump-outputs DIR` writes a fixed sample of the grid values of the last timed step to DIR (see dump_outputs); the
inputs are seeded, so runs with the same arguments on two builds can be compared output for output.
"""
import os
import sys

# torchrun exports OMP_NUM_THREADS=1; the CPU arms get every host core (set before numpy loads its BLAS)
if "reference" in sys.argv or int(os.environ.get("WORLD_SIZE", "1")) == 1:
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        if os.environ.get(_v) == "1":
            os.environ.pop(_v)

import argparse  # noqa: E402
import json  # noqa: E402
import statistics  # noqa: E402
import threading  # noqa: E402
import time  # noqa: E402

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NMAX, DGRID, EPOCHS, KERNEL = 96, 0.5, 240, "ewh"
METRIC = "sh_synthesis_grid_points_x_epochs_per_s"
UNIT = "grid-pts*epochs/s"


def config_dict():
    """Identical in both arms (the driver compares them key by key)."""
    return {"workload": "config2: degree-96 synthesis of 240 epochs -> 0.5deg GeographicGrid, ewh",
            "nmax": NMAX, "grid": "geographic 0.5deg (360x720)", "epochs": EPOCHS, "kernel": KERNEL}


def algorithmic_flops(nmax, nlat, nlon, epochs):
    """SURVEY 8(d) contract figure: direct two-stage synthesis, no symmetry / FFT credit."""
    L = nmax + 1
    K = L * L
    stage1 = 2.0 * epochs * nlat * K
    stage2 = 2.0 * (2 * L - 1) * epochs * nlat * nlon
    legendre = 5.0 * nlat * L * (L + 1) / 2
    return stage1, stage2, legendre


def synthetic_batch(nmax, epochs, first_epoch=0):
    from oracle import sh_oracle  # input generator only (shared with the tests)
    return np.stack([sh_oracle.synthetic_coefficients(nmax, first_epoch + e) for e in range(epochs)])


DUMP_EPOCHS, DUMP_VALUES, DUMP_SEED = 8, 1 << 20, 20240


def dump_outputs(directory, out, first_epoch, total_epochs, dist=None, rank=0):
    """Write a fixed sample of the job's grid values to `directory` as .npy files, so that the outputs of two builds
    can be compared value for value.  `out` [epochs, nlat, nlon] (float64) holds this rank's epochs first_epoch, ...
    of the job's total_epochs.  The whole batch of config 2 is 498 MB; the sample is about 34 MB: the first, the last
    and six seeded whole epochs, and 2^20 seeded single values of the job, each beside the indices it was taken at
    (epoch numbers, and flat indices into the [total_epochs, nlat, nlon] values), stored as float64.  The sample is
    drawn over the whole job and collected on rank 0, which writes it: the same files for any number of GPUs."""
    import torch
    epochs, nlat, nlon = out.shape
    points = nlat * nlon
    rng = np.random.default_rng(DUMP_SEED)
    inner = np.arange(1, max(total_epochs - 1, 1))
    pick = np.unique(np.concatenate(([0, total_epochs - 1], rng.choice(inner, min(DUMP_EPOCHS - 2, inner.size), replace=False))))
    flat = np.sort(rng.choice(total_epochs * points, min(DUMP_VALUES, total_epochs * points), replace=False))

    def share(index, per_epoch, source):
        """The entries of the sample at `index` that this rank holds; the others stay zero."""
        held = (index >= first_epoch * per_epoch) & (index < (first_epoch + epochs) * per_epoch)
        dst = torch.zeros((index.size,) + source.shape[1:], dtype=torch.float64, device=out.device)
        dst[torch.as_tensor(np.flatnonzero(held), device=out.device)] = \
            source[torch.as_tensor(index[held] - first_epoch * per_epoch, device=out.device)]
        return dst

    whole, values = share(pick, 1, out), share(flat, points, out.reshape(-1))
    if dist is not None:
        for t in (whole, values):       # one rank holds each entry: the integer sum of the bit patterns is exact
            dist.reduce(t.view(torch.int64), dst=0, op=dist.ReduceOp.SUM)
    if rank != 0:
        return
    os.makedirs(directory, exist_ok=True)
    arrays = {
        "grid_values_epochs": whole.cpu().numpy(),
        "grid_values_epochs_index": pick.astype(np.float64),
        "grid_values_sample": values.cpu().numpy(),
        "grid_values_sample_index": flat.astype(np.float64),
    }
    for name, array in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), array)


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index, period=0.01):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as exc:  # NVML missing: report that instead of inventing numbers
            self.err = str(exc)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake_slowdown",
        }
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "no NVML samples"}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def gpu_local_cpus(index):
    """Host cores NVML lists as local to GPU `index` (empty set if unknown)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w in range(words) for b in range(64) if (int(mask[w]) >> b) & 1}
        return cpus & os.sched_getaffinity(0)
    except Exception:
        return set()


def blas_threads():
    try:
        from threadpoolctl import threadpool_info
        blas = [p["num_threads"] for p in threadpool_info() if p.get("user_api") == "blas"]
        return max(blas) if blas else os.cpu_count()
    except Exception:
        return os.cpu_count()


def load_reference():
    """The unmodified reference package from baseline/_ref (git-ignored; __graft_entry__.install_reference puts it
    there when a reference checkout is present); netCDF4 / h5py are unused on this path (grates/__init__.py:48 ->
    io.py:18-19), so they are stubbed.  Returns the module or None."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "grates")):
        return None
    import types
    import warnings
    warnings.filterwarnings("ignore")
    nc = types.ModuleType("netCDF4")
    nc.Dataset = object
    sys.modules.setdefault("netCDF4", nc)
    sys.modules.setdefault("h5py", types.ModuleType("h5py"))
    if ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    try:
        import grates
        return grates
    except Exception:
        return None


def cpu_reference_rate(epochs_sample, warm=1):
    """The reference's to_grid (gravityfield.py:331-368) per epoch on the host cores: the real package when
    baseline/_ref is present (kind "reference"), else the numpy oracle port of the same algorithm (kind "port").
    Returns (grid-pts*epochs/s, seconds, BLAS threads, kind)."""
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(os.cpu_count())
    except Exception:
        pass
    batch = synthetic_batch(NMAX, epochs_sample + warm)
    grates = load_reference()
    if grates is not None:
        grid = grates.grid.GeographicGrid(DGRID, DGRID)
        fields = []
        for a in batch:
            pc = grates.gravityfield.PotentialCoefficients(3.9860044150e+14, 6.3781363000e+06)
            pc.anm = a
            fields.append(pc)
        run = lambda i: fields[i].to_grid(grid, KERNEL)     # noqa: E731
        nlat, nlon = grid.parallels.size, grid.meridians.size
        kind = "reference"
    else:
        from oracle import sh_oracle as orc
        grid = orc.geographic_grid(DGRID, DGRID)
        run = lambda i: orc.synthesis(batch[i], grid, KERNEL)     # noqa: E731
        nlat, nlon = grid.shape
        kind = "port"
    for e in range(warm):
        run(e)
    t0 = time.perf_counter()
    for e in range(warm, warm + epochs_sample):
        run(e)
    dt = time.perf_counter() - t0
    return epochs_sample * nlat * nlon / dt, dt, blas_threads(), kind


def run_reference(args, rank):
    """--impl reference: the reference's own CPU implementation on the same config, metric and unit.  A step is a
    bounded sample of the 240-epoch workload (the reference has no cross-epoch reuse: cost is linear in epochs)."""
    if rank != 0:
        return
    try:
        os.sched_setaffinity(0, range(os.cpu_count()))     # every host core, whatever the launcher bound us to
    except Exception:
        pass
    sample = max(1, min(8, 120 // max(args.steps, 1)))
    for _ in range(min(max(args.warmup, 0), 3)):
        cpu_reference_rate(1, warm=1)
    times, kind, threads = [], "port", 1
    for _ in range(max(args.steps, 1)):
        _, dt, threads, kind = cpu_reference_rate(sample, warm=0)
        times.append(dt)
    nlat, nlon = int(180 / DGRID), int(360 / DGRID)
    total_time = sum(times)
    value = len(times) * sample * nlat * nlon / total_time
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total_time / len(times),          # measured: one step = `sample` epochs
        "units_per_step": sample * nlat * nlon,
        "ms_per_full_workload_extrapolated": 1e3 * total_time / len(times) * (EPOCHS / sample),
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_dict(),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind,
                         "sample": "%d of 240 epochs per step (cost is linear in epochs: no cross-epoch reuse in the "
                                   "reference), %s, numpy/OpenBLAS threads=%d of %d host cores; ~3/4 of the time is "
                                   "single-threaded numpy table building"
                                   % (sample, "unmodified grates.PotentialCoefficients.to_grid from baseline/_ref"
                                      if kind == "reference" else "numpy oracle port (baseline/_ref missing)",
                                      threads, os.cpu_count())},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"])
    ap.add_argument("--e2e-steps", type=int, default=None, help="steps of the host-buffer loop (default min(steps, 30))")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the BASELINE configs 1/3/4/5 block")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed sample of the grid values of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    import grates_b200 as gb

    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d does not match WORLD_SIZE %d" % (args.gpus, world))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    distributed = world > 1
    full_affinity = os.sched_getaffinity(0)
    local_cpus = gpu_local_cpus(local_rank)
    if local_cpus:
        os.sched_setaffinity(0, local_cpus)    # pinned host buffers of the e2e loop land next to the GPU (first touch)
    if distributed:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if distributed:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def reduce_sum(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if distributed:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---- workload ---------------------------------------------------------------------------------
    if args.scaling == "weak":
        epochs, first = EPOCHS, rank * EPOCHS
    else:
        first, stop = gb.distributed.shard_range(EPOCHS, world, rank)
        epochs = stop - first
    grid = gb.GeographicGrid(DGRID, DGRID)
    torch.cuda.synchronize()
    t_plan = time.perf_counter()
    plan = gb.get_plan(grid, NMAX, KERNEL, device=local_rank)      # host tables + upload, once per (grid, degree, kernel)
    torch.cuda.synchronize()
    t_plan = time.perf_counter() - t_plan
    nlat, nlon = plan.nlat, plan.nlon
    anm_host = synthetic_batch(NMAX, epochs, first)
    anm = torch.as_tensor(anm_host).to(dev)
    out = torch.empty((epochs, nlat, nlon), dtype=torch.float64, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # > 126 MB L2
    units_per_step = epochs * nlat * nlon
    lib = gb._lib.load()
    warmup = max(args.warmup, 3)
    sym, folded, octant = plan.symmetric, plan.folded, plan.octant     # (the configs block below clears the plan cache)

    def timed_steps(x, y, steps):
        """K steps, device resident, L2 flushed between steps; returns the per-step CUDA-event times (ms)."""
        ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        ev1 = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        for s in range(steps):
            flush.zero_()                         # L2 flush between steps (not part of the step time)
            ev0[s].record()
            plan.synthesis(x, out=y)
            ev1[s].record()
        barrier()
        return [a.elapsed_time(b) for a, b in zip(ev0, ev1)]

    # ---- warm-up --------------------------------------------------------------------------------------
    for _ in range(warmup):
        plan.synthesis(anm, out=out)
    torch.cuda.synchronize()

    # ---- timed region: K steps, device-resident (the kernels chain with programmatic dependent launch) --------
    sampler = ClockSampler(local_rank)
    lib.gb_launch_count(1)
    barrier()
    sampler.start()
    t_wall0 = time.perf_counter()
    step_ms = timed_steps(anm, out, args.steps)
    t_wall = time.perf_counter() - t_wall0
    launches = int(lib.gb_launch_count(1))
    my_time = sum(step_ms) * 1e-3
    max_time = reduce_max(my_time)
    total_units = reduce_sum(float(units_per_step))
    value = total_units * args.steps / max_time
    if args.dump_outputs is not None:          # `out` holds the last timed step's result until the pass below
        dump_outputs(args.dump_outputs, out, first, int(round(total_units / (nlat * nlon))),
                     dist if distributed else None, rank)

    # ---- the same K steps with an event pair around every kernel (per-kernel times for the roofline; the extra
    #      stream operations between the kernels switch the launch chaining off, so this pass is not the headline) ----
    plan.set_profiling(args.steps)
    barrier()
    prof_step_ms = timed_steps(anm, out, args.steps)
    stages = plan.stage_times(args.steps)     # [steps, 3] pack / stage 1 / stage 2
    plan.set_profiling(0)

    # ---- weak figure beside the strong one (every rank runs all 240 epochs) -----------------------------------
    weak = None
    if distributed and args.scaling == "strong":
        w_steps = min(args.steps, 10)
        anm_w = torch.as_tensor(synthetic_batch(NMAX, EPOCHS, rank * EPOCHS)).to(dev)
        out_w = torch.empty((EPOCHS, nlat, nlon), dtype=torch.float64, device=dev)
        for _ in range(3):
            plan.synthesis(anm_w, out=out_w)
        barrier()
        w_time = reduce_max(sum(timed_steps(anm_w, out_w, w_steps)) * 1e-3)
        weak = {"value": world * EPOCHS * nlat * nlon * w_steps / w_time, "unit": UNIT, "steps": w_steps,
                "ms_per_step": 1e3 * w_time / w_steps, "epochs_per_gpu": EPOCHS,
                "note": "every rank runs the whole 240-epoch batch on its own epochs (independent replicas)"}
        del anm_w, out_w

    # ---- end to end: host buffers through gb_synthesis_host ----------------------------------------
    e2e_steps = args.e2e_steps if args.e2e_steps is not None else min(args.steps, 30)
    pin_in = gb.PinnedArray(anm_host.shape)
    pin_in.array[...] = anm_host
    pin_out = gb.PinnedArray((epochs, nlat, nlon))
    pin_out.array[...] = 0.0                      # first touch under the NUMA binding
    for _ in range(2):
        plan.synthesis_host(pin_in.array, out=pin_out.array)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        plan.synthesis_host(pin_in.array, out=pin_out.array)
    torch.cuda.synchronize()
    e2e_time = reduce_max(time.perf_counter() - t0)
    sampler.stop()
    e2e_value = total_units * e2e_steps / e2e_time
    checksum = float(np.abs(pin_out.array[0]).max()) if epochs else 0.0

    # ---- copy ceiling of this box: every rank copies its result shard device -> pinned host, nothing else ----------
    def d2h_rate(host_array, reps=5):
        src = out.reshape(-1)
        dst = torch.from_numpy(host_array.reshape(-1))
        for _ in range(2):
            dst.copy_(src, non_blocking=True)
        barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
        dt = reduce_max(time.perf_counter() - t0)
        return reduce_sum(float(src.numel() * 8)) * reps / dt / 1e9

    ceiling_bound = d2h_rate(pin_out.array)
    os.sched_setaffinity(0, full_affinity)
    pin_free = gb.PinnedArray((epochs, nlat, nlon))
    pin_free.array[...] = 0.0                     # first touch without a binding
    ceiling_unbound = d2h_rate(pin_free.array)
    pin_free.free()
    e2e_bytes = float(anm_host.nbytes + pin_out.nbytes)
    e2e_gbs = reduce_sum(e2e_bytes) * e2e_steps / e2e_time / 1e9

    # ---- BASELINE configs 1, 3, 4, 5 (every rank takes part: shards + max-over-ranks times) ---------------------
    configs = None
    if not args.no_configs:
        import bench_configs
        del out, anm
        torch.cuda.empty_cache()
        configs = bench_configs.run_all(rank, world, dev, dist if distributed else None,
                                        with_cpu=(world == 1 and not args.no_cpu_baseline))

    if rank == 0:
        # ---- roofline of the dominant kernel (Fourier stage 2, FP64 tensor pipe) ----------------------
        import ctypes
        c_mma, c_fma = ctypes.c_double(0), ctypes.c_double(0)
        gb._lib.check(lib.gb_probe_fp64_peak(local_rank, ctypes.byref(c_mma), ctypes.byref(c_fma)))
        peak = max(c_mma.value, c_fma.value)
        f1, f2, fl = algorithmic_flops(NMAX, nlat, nlon, epochs)
        s2_ms = float(np.mean(stages[:, 2])) if len(stages) else float("nan")
        s1_ms = float(np.mean(stages[:, 1])) if len(stages) else float("nan")
        pk_ms = float(np.mean(stages[:, 0])) if len(stages) else float("nan")
        # executed multiply-adds of the dominant kernel: the symmetric path contracts one quadrant of meridians
        # (the octant kernel: the even orders split once more under mu -> pi/2 - mu, 3/4 of the quadrant kernel's work)
        f2_exec = f2 / 4.0 * (0.75 if octant else 1.0) if sym else f2
        # the folded Legendre stage contracts the northern parallels only
        f1_exec = f1 / 2.0 if folded else f1
        step_mean_ms = 1e3 * my_time / args.steps
        traffic, traffic_src = None, None
        tfile = os.path.join(ROOT, "profiles", "stage2_traffic.json")
        if os.path.exists(tfile):
            try:
                tj = json.load(open(tfile))
                if int(tj.get("epochs", -1)) == epochs:      # a capture of this launch shape only
                    traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
            except Exception:
                traffic = None
        peaks_file = os.path.join(ROOT, "MEASURED_PEAKS.json")
        hbm = json.load(open(peaks_file)).get("hbm_gbs") if os.path.exists(peaks_file) else None
        bytes_step = 8.0 * units_per_step + 8.0 * epochs * (NMAX + 1) ** 2
        executed_tf = f2_exec / (s2_ms * 1e-3) / 1e12
        roofline = {
            "bound": "tensor",
            "kernel": ("gb_fourier_stage2_oct" if octant else "gb_fourier_stage2_sym" if sym else "gbgemm::kernel<RowMajorStore>")
                      + " (FP64 DMMA.8x8x4)",
            "achieved": executed_tf, "peak": peak, "unit": "TFLOP/s", "frac": executed_tf / peak,
            "traffic": traffic, "traffic_source": traffic_src,
            "peak_source": "live gb_probe_fp64_peak on this GPU (DMMA %.2f / DFMA %.2f TFLOP/s); MEASURED_PEAKS.json "
                           "has no FP64 figure" % (c_mma.value, c_fma.value),
            "flops_per_launch": f2_exec, "kernel_ms": s2_ms,
            "kernel_ms_source": "CUDA events around every kernel, second pass of the same K steps",
            "contract_flops_per_launch": f2, "contract_achieved": f2 / (s2_ms * 1e-3) / 1e12,
            "contract_multiple": f2 / (s2_ms * 1e-3) / 1e12 / peak,
            "note": ("`achieved` / `frac` count the multiply-adds the tensor pipe executes. Declared algorithmic shortcut: "
                     "four-fold longitude symmetry of the grid (meridians symmetric about 0 and under a half turn) -> the "
                     "kernel executes 1/4 of the SURVEY 8(d) contract multiply-adds (direct contraction, no symmetry "
                     "credit)" + ("; eight-fold here (the first quadrant mirrors about pi/4: the even orders split by order mod 4, "
                                  "the odd orders are contracted with two table rows per coefficient fragment) -> 3/16"
                                  if octant else "") + "; `contract_*` divide the contract flops by the same time, so `contract_multiple` is not a "
                     "utilisation. GB_NO_SYMMETRY=1 runs the direct contraction. Second declared shortcut (Legendre stage): "
                     "parallels mirrored about the equator share one table row, gated on a measured hemisphere asymmetry "
                     "of the reference's tables (GB_NO_FOLD=1 disables)."
                     if sym else "direct contraction (no symmetry shortcut active)"),
            "step": {"ms": step_mean_ms, "ms_with_kernel_events": float(np.mean(prof_step_ms)),
                     "executed_flops": f1_exec + f2_exec, "contract_flops": f1 + f2 + fl,
                     "frac_of_fp64_peak": (f1_exec + f2_exec) / (step_mean_ms * 1e-3) / 1e12 / peak,
                     "contract_multiple": (f1 + f2 + fl) / (step_mean_ms * 1e-3) / 1e12 / peak,
                     "legendre_stage_folded_about_equator": bool(folded),
                     "kernel_ms": {"pack": pk_ms, "legendre_stage1": s1_ms, "fourier_stage2": s2_ms}},
            "hbm": {"algorithmic_bytes_per_step": bytes_step, "peak_gbs": hbm,
                    "achieved_gbs": bytes_step / (step_mean_ms * 1e-3) / 1e9,
                    "frac": (bytes_step / (step_mean_ms * 1e-3) / 1e9 / hbm) if hbm else None},
        }
        if args.no_cpu_baseline or world > 1:
            cpu = None
        else:
            os.sched_setaffinity(0, full_affinity)     # the CPU arm gets every host core
            rate, dt, threads, kind = cpu_reference_rate(24)
            cpu = {"value": rate, "unit": UNIT, "cores": threads, "kind": kind,
                   "sample": "24 of 240 epochs after 1 warm-up call, %.1f s; %s (numpy+OpenBLAS, %d threads of %d host "
                             "cores; the reference has no cross-epoch reuse so cost is linear in epochs)"
                             % (dt, "unmodified grates.PotentialCoefficients.to_grid from baseline/_ref"
                                if kind == "reference" else "numpy oracle port of to_grid (baseline/_ref missing)",
                                threads, os.cpu_count())}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": 1e3 * max_time / args.steps, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(),
            "run": {"epochs_per_gpu": epochs, "epochs_total": int(round(total_units / (nlat * nlon))),
                    "parallelism": "epochs sharded over %d GPU(s), no data-path collective" % world,
                    "l2": "256 MiB memset between steps (outside the step's events)",
                    "timing": "CUDA events per step on the launch stream, max over ranks of the summed step times",
                    "plan_create_s": t_plan},
            "clocks": sampler.summary(),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(anm_host.nbytes),
                    "d2h_bytes_per_step": int(pin_out.nbytes), "steps": e2e_steps,
                    "path": "SHPlan.synthesis_host -> gb_synthesis_host (pinned host buffers, chunked D2H overlap)",
                    "result_check_max_abs": checksum,
                    "achieved_gbs": e2e_gbs, "copy_ceiling_gbs": max(ceiling_bound, ceiling_unbound),
                    "copy_ceiling_numa_bound_gbs": ceiling_bound, "copy_ceiling_unbound_gbs": ceiling_unbound,
                    "frac_of_copy_ceiling": e2e_gbs / max(ceiling_bound, ceiling_unbound),
                    "copy_ceiling_note": "all ranks copy their result shard device -> pinned host at the same time, nothing "
                                         "else running; pinned buffer first-touched on the GPU's NUMA node / without a binding"},
            "gpu_launches": launches,
            "wall_s_timed_region": t_wall,
            "roofline": roofline,
            "cpu_baseline": cpu,
        }
        if weak is not None:
            line["weak_scaling"] = weak
        if configs is not None:
            line["configs"] = configs
        print(json.dumps(line))
    pin_in.free()
    pin_out.free()
    if distributed:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
