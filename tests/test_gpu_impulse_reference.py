"""Every coefficient of the regular-grid synthesis and analysis at production size against an exact impulse reference.

Synthesis is linear, and on a regular grid the field of one coefficient k is a rank-one product: with the Legendre
factors U[i, k] (the fully normalised P_nm of parallel i times its degree factor) and the trigonometric factors
T[j, k] (cos or sin of m lon_j),

    ref[e, i, j] = a_e U[i, k_e] T[j, k_e]

for epoch e of a batch whose only nonzero coefficient is k_e, with amplitude a_e.  Each value is two correctly rounded
products, so the reference is exact to rounding for every coefficient and can be formed on the device.  U and T are
the oracle's float64 tables (never the plan's: a wrong table entry would otherwise be invisible).  A seeded
permutation of all (n, m, cos / sin) spreads the coefficients over the epoch columns, so every column of every stage-1
tile sees every degree band; amplitudes are drawn from +-[0.5, 2) without powers of two, so a kernel that squares,
drops or double-counts a coefficient cannot pass by accident.

The error of an impulse is max |got - ref| / max |ref| over its own grid: every coefficient is judged against its own
size, not against the largest coefficient of a Kaula field.  With an order-wise filter fused into the synthesis the
field of an impulse is still rank one, (U_m B_m)[:, n - m] T[:, k], with B_m the filter block of its order and
trigonometric function.  Analysis is fed the exact impulse grids (not the GPU synthesis) and must return a_e e_k: its
error is max over all coefficients of |back - a_e e_k| / |a_e|, one column of (analysis o synthesis - I).

What impulses cannot see, accumulation across K chunks and order pairs, is covered by one dense check at the
headline shape (D1) against a separable float64 reference, itself guarded by 64 entries in extended precision.  The
reference is checked against the oracle's own synthesis, filter and analysis at degree 12 (test_impulse_reference_
matches_oracle, no GPU).
"""
import subprocess
import time

import numpy as np
import pytest

from oracle import sh_oracle as orc
from test_gpu_full_size_reference import _Checks, _plan_state

EXACT_TOL = 1e-14          # float64 dense reference against its extended-precision recomputation

# Largest error each sweep may show, never more than 1e-12.  The folded Legendre stage reuses the northern recursion for
# the southern parallels, which the plan's fold gate admits up to 2e-13 of a degree's largest value; the float64 oracle
# analysis of exact impulse fields at degree 96 on the 0.5 degree grid errs by up to 2.3e-14.  The errors a B200 shows
# have not been recorded here yet: once they are, each bound becomes ten times the largest of them (capped at 1e-12).
TOL_SYN = 1e-12            # synthesis impulses, per impulse against its own maximum
TOL_FILT = 1e-12           # synthesis impulses with the fused order-wise filter
TOL_ANA = 1e-12            # analysis of impulse grids, against the impulse's amplitude
TOL_DENSE = 1e-12          # dense config-2 batch, per (epoch, parallel) against the row maximum of the reference


@pytest.fixture(scope="module")
def gb():
    import grates_b200
    import torch
    grates_b200._lib.require_device()
    dev = torch.cuda.current_device()
    try:
        card = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        card = ""
    print("\ndevice %d: %s" % (dev, card or torch.cuda.get_device_name(dev) + ", power limit unknown"))
    return grates_b200


@pytest.fixture(scope="module")
def tables():
    """(U, T) of the oracle for a grid and degree, host and device copies, cached for the module."""
    import torch
    cache = {}

    def get(grid, N):
        key = (grid.parallels.tobytes(), grid.meridians.tobytes(), N)
        if key not in cache:
            U, T = _tables(grid.parallels, grid.meridians, grid.semimajor_axis, grid.flattening, N)
            cache[key] = (U, T, torch.as_tensor(U).cuda(), torch.as_tensor(T).cuda())
        return cache[key]
    return get


# ------------------------------------------------------------------------------ reference
def _tables(parallels, meridians, a, f, N):
    """Packed Legendre factors U [nlat, L, L] (P_nm times the ewh degree factors of each parallel) and trigonometric
    factors T [nlon, L, L]: the oracle's float64 definition."""
    colat, kn = orc.kn_table("ewh", N, parallels, a, f)
    return orc._scale_packed_by_degree(orc.legendre_functions(N, colat), kn), orc.trigonometric_functions(N, meridians)


def _impulses(N, nmin, seed):
    """Packed (row, col) of every coefficient of degree nmin..N (C_nm at [n, m], S_nm at [m - 1, n]) in a seeded random
    order, and an amplitude for each: uniform in +-[0.5, 2), never a power of two."""
    rows, cols = orc._degreewise_index(nmin, N)
    rng = np.random.default_rng(seed)
    perm = rng.permutation(rows.size)
    amp = rng.uniform(0.5, 2.0, rows.size)
    amp[np.isin(amp, (0.5, 1.0))] = 1.5
    amp *= rng.choice((-1.0, 1.0), rows.size)
    return rows[perm], cols[perm], amp


def _name(r, c):
    """'C(n,m)' or 'S(n,m)' of the packed entry [r, c]."""
    return "C(%d,%d)" % (r, c) if c <= r else "S(%d,%d)" % (c, r + 1)


def _order(r, c):
    return int(c) if c <= r else int(r) + 1


def _impulse_grids(U, T, rows, cols, amp):
    """ref[e, i, j] = (amp_e U[i, k_e]) T[j, k_e] for k_e = (rows_e, cols_e): [E, nlat, nlon].  numpy or torch."""
    u = U[:, rows, cols].T * amp[:, None]
    return u[:, :, None] * T[:, rows, cols].T[:, None, :]


def _filtered_legendre(U, blocks):
    """UF [nlat, L, L] with UF[:, k] the Legendre factor of the order-wise filtered impulse k: per order m and
    trigonometric function U_m B, U_m [nlat, N + 1 - m] the factors of the order and B the leading block of the filter,
    whose rows of degrees 0 and 1 are the identity (orc.orderwise_filter passes those degrees through)."""
    N = U.shape[1] - 1
    UF = np.empty_like(U)
    for m in range(N + 1):
        k = N + 1 - m
        for cs in ((0,) if m == 0 else (0, 1)):
            B = blocks[0 if m == 0 else 2 * m - 1 + cs][:k, :k].copy()
            for r in range(max(0, 2 - m)):
                B[r] = 0.0
                B[r, r] = 1.0
            if cs == 0:
                UF[:, m:, m] = U[:, m:, m] @ B
            else:
                UF[:, m - 1, m:] = U[:, m - 1, m:] @ B
    return UF


def _separable_synthesis(X, U, T):
    """Dense reference [E, nlat, nlon] of packed coefficients X [E, L, L]: per order m the products U_m X_m of the
    cosine and sine coefficients, then one product with the cos / sin (m lon) rows."""
    E, L = X.shape[0], X.shape[-1]
    Gc, Gs = np.zeros((E, U.shape[0], L)), np.zeros((E, U.shape[0], L))
    for m in range(L):
        Gc[:, :, m] = X[:, m:, m] @ U[:, m:, m].T
        if m:
            Gs[:, :, m] = X[:, m - 1, m:] @ U[:, m - 1, m:].T
    m = np.arange(L)
    cos_m = T[:, m, m].T                                           # T[:, m, m] = cos(m lon)
    sin_m = np.zeros_like(cos_m)
    sin_m[1:] = T[:, m[:-1], m[1:]].T                              # T[:, m - 1, m] = sin(m lon)
    return (Gc.reshape(-1, L) @ cos_m + Gs.reshape(-1, L) @ sin_m).reshape(E, U.shape[0], -1)


def _equal_power(N, E, seed):
    """Packed coefficients [E, L, L] whose degrees contribute equally to the ewh field: standard deviation
    1 / (kn(n) sqrt(2n + 1)) with the degree factor kn at the equator."""
    _, kn = orc.kn_table("ewh", N, np.zeros(1))
    L = N + 1
    deg = np.maximum(np.arange(L)[:, None], np.arange(L)[None, :])      # degree of packed entry [r, c]
    sd = 1.0 / (kn[0][deg] * np.sqrt(2.0 * deg + 1.0))
    return np.random.default_rng(seed).standard_normal((E, L, L)) * sd


def _dense_guard(X, U, T, ref, rowmax, seed):
    """Largest difference between the dense float64 reference and 64 entries recomputed in extended precision,
    relative to the row maximum."""
    rng = np.random.default_rng(seed)
    es, rs, js = (rng.integers(0, n, 64) for n in ref.shape)
    rs[:2], js[:2] = (0, ref.shape[1] - 1), (0, ref.shape[2] - 1)
    ld = np.longdouble
    return max(float(abs(ref[e, i, j] - np.sum(X[e].astype(ld) * U[i].astype(ld) * T[j].astype(ld))) / rowmax[e, i])
               for e, i, j in zip(es, rs, js))


# ------------------------------------------------------------------------------ sweeps
class _Worst:
    """Worst impulse of a sweep, where it was, and the orders with an impulse over tolerance."""

    def __init__(self, tol):
        self.tol, self.err, self.where, self.orders, self.count = tol, -1.0, "", set(), 0

    def add(self, err, rows, cols, locate):
        """err: per-impulse errors of a batch (CUDA tensor, inf where not finite); locate(e) -> text for impulse e."""
        e = int(err.argmax())
        v = float(err[e])
        if v > self.err or self.count == 0:
            self.err, self.where = v, locate(e)
        for b in (~(err <= self.tol)).nonzero().flatten().tolist():
            self.orders.add(_order(rows[b], cols[b]))
        self.count += err.numel()

    def report(self, checks, label):
        print("%s %s: %d impulses, worst %s" % (checks.case, label, self.count, self.where))
        checks.err(label, self.err, self.tol)
        checks.state(label + ", orders with an impulse over tolerance", sorted(self.orders), [])


def _synthesis_sweep(checks, label, synth, U, T, rows, cols, amp, width, tol):
    """Synthesize every impulse in batches of `width` (the last one ragged) and compare each with its rank-one field."""
    import torch
    dev, L, nlon = U.device, U.shape[1], T.shape[0]
    R, C, A = (torch.as_tensor(v, device=dev) for v in (rows, cols, amp))
    worst = _Worst(tol)
    t0 = time.perf_counter()
    for b0 in range(0, rows.size, width):
        E = min(width, rows.size - b0)
        sl = slice(b0, b0 + E)
        x = torch.zeros((E, L, L), dtype=torch.float64, device=dev)
        x[torch.arange(E, device=dev), R[sl], C[sl]] = A[sl]
        got = synth(x)
        ref = _impulse_grids(U, T, R[sl], C[sl], A[sl])
        d = (got - ref).abs()
        err = d.flatten(1).amax(1) / ref.abs().flatten(1).amax(1)
        err[~torch.isfinite(got).flatten(1).all(1)] = float("inf")

        def locate(e):
            i, j = divmod(int(d[e].argmax()), nlon)
            return "%.3e at %s, epoch column %d of a %d-epoch batch, parallel %d, meridian %d" % (
                float(err[e]), _name(rows[b0 + e], cols[b0 + e]), e, E, i, j)
        worst.add(err, rows[sl], cols[sl], locate)
        del got, ref, d
    torch.cuda.synchronize()
    print("%s %s: %.1f s" % (checks.case, label, time.perf_counter() - t0))
    worst.report(checks, label)


def _analysis_sweep(checks, label, analyse, U, T, rows, cols, amp, width, tol):
    """Analyse the exact field of every impulse in batches of `width`; each must return a_e e_k."""
    import torch
    dev, L = U.device, U.shape[1]
    R, C, A = (torch.as_tensor(v, device=dev) for v in (rows, cols, amp))
    worst = _Worst(tol)
    t0 = time.perf_counter()
    for b0 in range(0, rows.size, width):
        E = min(width, rows.size - b0)
        sl = slice(b0, b0 + E)
        back = analyse(_impulse_grids(U, T, R[sl], C[sl], A[sl]).contiguous())
        fin = torch.isfinite(back).flatten(1).all(1)
        back[torch.arange(E, device=dev), R[sl], C[sl]] -= A[sl]
        d = back.abs().flatten(1)
        err = d.amax(1) / A[sl].abs()
        err[~fin] = float("inf")

        def locate(e):
            r, c = divmod(int(d[e].argmax()), L)
            return "%.3e for %s, epoch column %d of a %d-epoch batch, largest in %s" % (
                float(err[e]), _name(rows[b0 + e], cols[b0 + e]), e, E, _name(r, c))
        worst.add(err, rows[sl], cols[sl], locate)
        del back, d
    torch.cuda.synchronize()
    print("%s %s: %.1f s" % (checks.case, label, time.perf_counter() - t0))
    worst.report(checks, label)


# ------------------------------------------------------------------------------ the reference itself (no GPU)
def test_impulse_reference_matches_oracle():
    """At degree 12 on a 10 degree grid and a small ragged grid (odd meridian count, uneven parallels): the rank-one
    impulse fields equal orc.synthesis of the same impulse, also behind an order-wise filter (of higher degree than the
    data, as orc.orderwise_filter truncates it); orc.analysis_separable of every impulse field returns a e_k, from
    degree 0 and from degree 2; the separable dense reference equals orc.synthesis."""
    N = 12
    dlon = 2 * np.pi / 31                  # whole circle, equally spaced: the separable analysis needs both
    ragged = orc.OracleGrid(np.linspace(-np.pi + dlon / 2, np.pi - dlon / 2, 31),
                            np.array([1.45, 1.3, 1.1, 0.95, 0.7, 0.6, 0.4, 0.1, -0.05, -0.3, -0.5, -0.75, -0.9, -1.15, -1.5]))
    blocks = orc.synthetic_filter_blocks(N + 3)
    for og in (orc.geographic_grid(10.0, 10.0), ragged):
        U, T = _tables(og.parallels, og.meridians, og.a, og.f, N)
        UF = _filtered_legendre(U, blocks)
        rows, cols, amp = _impulses(N, 0, 3)
        ref = _impulse_grids(U, T, rows, cols, amp)
        filt = _impulse_grids(UF, T, rows, cols, amp)
        for e, (r, c, a) in enumerate(zip(rows, cols, amp)):
            x = np.zeros((N + 1, N + 1))
            x[r, c] = a
            syn = orc.synthesis(x, og, "ewh")
            assert np.max(np.abs(ref[e] - syn)) <= 1e-15 * np.max(np.abs(syn)), _name(r, c)
            syn = orc.synthesis(orc.orderwise_filter(blocks, x), og, "ewh")
            assert np.max(np.abs(filt[e] - syn)) <= 1e-15 * np.max(np.abs(syn)), _name(r, c)
        for nmin in (0, 2):
            keep = np.maximum(rows, cols) >= nmin
            back = orc.analysis_separable(ref[keep], og, nmin, N, "ewh")
            back[np.arange(keep.sum()), rows[keep], cols[keep]] -= amp[keep]
            assert np.max(np.abs(back).reshape(keep.sum(), -1).max(axis=1) / np.abs(amp[keep])) < 1e-12, nmin
        X = _equal_power(N, 4, 9)
        dense = _separable_synthesis(X, U, T)
        for e in range(X.shape[0]):
            syn = orc.synthesis(X[e], og, "ewh")
            assert np.max(np.abs(dense[e] - syn)) <= 1e-14 * np.max(np.abs(syn))


# ------------------------------------------------------------------------------ synthesis
@pytest.mark.gpu
def test_s1_config2_every_coefficient(gb, tables):
    """GeographicGrid(0.5, 0.5), degree 96 (config 2, the benchmark path): octant Fourier stage, folded table-fed Legendre
    stage; all 9 409 coefficients in 39 batches of 240 epochs (240-column tiling) and the ragged remainder of 49
    (120-column tiling)."""
    checks = _Checks("S1")
    grid = gb.GeographicGrid(0.5, 0.5)
    plan = gb.get_plan(grid, 96, "ewh")
    _plan_state(gb, checks, plan, True, True, 1)
    _, _, U, T = tables(grid, 96)
    rows, cols, amp = _impulses(96, 0, 101)
    _synthesis_sweep(checks, "batches of 240", plan.synthesis, U, T, rows, cols, amp, 240, TOL_SYN)
    checks.done()


@pytest.mark.gpu
def test_s2_config2_shard_widths(gb, tables):
    """S1 in batches of 30 epochs (64-column items spread over the SMs: the 8-GPU shard of config 2) and of 70 epochs
    (80-column tiling)."""
    checks = _Checks("S2")
    grid = gb.GeographicGrid(0.5, 0.5)
    plan = gb.get_plan(grid, 96, "ewh")
    _plan_state(gb, checks, plan, True, True, 1)
    _, _, U, T = tables(grid, 96)
    for width, seed in ((30, 102), (70, 103)):
        rows, cols, amp = _impulses(96, 0, seed)
        _synthesis_sweep(checks, "batches of %d" % width, plan.synthesis, U, T, rows, cols, amp, width, TOL_SYN)
    checks.done()


@pytest.mark.gpu
def test_s3_config2_legendre_recursion_in_kernel(gb, tables, monkeypatch):
    """S1 with GB_S1_ONTHEFLY=1: the Legendre stage runs the recursion inside the kernel instead of reading the plan's
    table (what a plan over its table budget does), at production size."""
    checks = _Checks("S3")
    grid = gb.GeographicGrid(0.5, 0.5)
    plan = gb.get_plan(grid, 96, "ewh")
    _plan_state(gb, checks, plan, True, True, 1)
    _, _, U, T = tables(grid, 96)
    rows, cols, amp = _impulses(96, 0, 104)
    monkeypatch.setenv("GB_S1_ONTHEFLY", "1")
    _synthesis_sweep(checks, "batches of 240, recursion", plan.synthesis, U, T, rows, cols, amp, 240, TOL_SYN)
    checks.done()


@pytest.mark.gpu
def test_s4_config3_every_coefficient(gb, tables):
    """GeographicGrid(0.25, 0.25), degree 180 (config 3): all 32 761 coefficients in batches of 120 epochs; octant Fourier
    stage, folded Legendre stage with one 32-parallel polar-cap tile per pole left to the unfolded stage
    (gb_plan_is_folded == 2)."""
    checks = _Checks("S4")
    grid = gb.GeographicGrid(0.25, 0.25)
    plan = gb.get_plan(grid, 180, "ewh")
    _plan_state(gb, checks, plan, True, True, 2)
    _, _, U, T = tables(grid, 180)
    rows, cols, amp = _impulses(180, 0, 105)
    _synthesis_sweep(checks, "batches of 120", plan.synthesis, U, T, rows, cols, amp, 120, TOL_SYN)
    checks.done()


@pytest.mark.gpu
def test_s5_quadrant_fourier_stage(gb, tables):
    """GeographicGrid(1.0, 1.0), degree 96: 360 meridians are a multiple of 8 but not of 16, so the Fourier stage is the
    four-fold (quadrant) one; folded without polar caps."""
    checks = _Checks("S5")
    grid = gb.GeographicGrid(1.0, 1.0)
    plan = gb.get_plan(grid, 96, "ewh")
    _plan_state(gb, checks, plan, False, True, 1)
    _, _, U, T = tables(grid, 96)
    rows, cols, amp = _impulses(96, 0, 106)
    _synthesis_sweep(checks, "batches of 240", plan.synthesis, U, T, rows, cols, amp, 240, TOL_SYN)
    checks.done()


@pytest.mark.gpu
def test_s6_general_fourier_stage_unfolded(gb, tables):
    """359 parallels (the 0.5 degree parallels without the southernmost: not mirror images, so unfolded) and 721
    meridians (not a multiple of 4: the general GEMM Fourier stage), degree 96."""
    checks = _Checks("S6")
    dlon = 2 * np.pi / 721
    grid = gb.RegularGrid(np.linspace(-np.pi + dlon / 2, np.pi - dlon / 2, 721), gb.GeographicGrid(0.5, 0.5).parallels[:-1])
    plan = gb.get_plan(grid, 96, "ewh")
    _plan_state(gb, checks, plan, False, False, 0)
    _, _, U, T = tables(grid, 96)
    rows, cols, amp = _impulses(96, 0, 107)
    _synthesis_sweep(checks, "batches of 240", plan.synthesis, U, T, rows, cols, amp, 240, TOL_SYN)
    checks.done()


@pytest.mark.gpu
def test_s7_config5_fused_orderwise_filter(gb, tables):
    """GeographicGrid(0.25, 0.25), degree 120 with the order-wise filter fused into the synthesis (config 5: the filter's
    epilogue writes X in the Legendre stage's layout): all 14 641 coefficients in batches of 500 epochs."""
    import torch
    checks = _Checks("S7")
    grid = gb.GeographicGrid(0.25, 0.25)
    plan = gb.get_plan(grid, 120, "ewh")
    _plan_state(gb, checks, plan, True, True, 2)
    blocks = orc.synthetic_filter_blocks(120)
    flt = gb.OrderWiseFilter(blocks)
    U, _, _, T = tables(grid, 120)
    UF = torch.as_tensor(_filtered_legendre(U, blocks)).cuda()
    rows, cols, amp = _impulses(120, 0, 108)
    _synthesis_sweep(checks, "batches of 500, filtered", lambda x: plan.synthesis(x, orderwise_filter=flt), UF, T,
                     rows, cols, amp, 500, TOL_FILT)
    checks.done()


# ------------------------------------------------------------------------------ analysis
@pytest.mark.gpu
def test_a1_config2_analysis_every_coefficient(gb, tables):
    """Analysis on GeographicGrid(0.5, 0.5) to degree 96 of every impulse field, from degree 0 and from degree 2 (impulses
    of degree 2 and higher), in batches of 240."""
    checks = _Checks("A1")
    grid = gb.GeographicGrid(0.5, 0.5)
    _, _, U, T = tables(grid, 96)
    for nmin, seed in ((0, 109), (2, 110)):
        rows, cols, amp = _impulses(96, nmin, seed)
        _analysis_sweep(checks, "min_degree %d, batches of 240" % nmin,
                        lambda v: gb.analysis_batch(v, grid, nmin, 96, "ewh", device_output=True),
                        U, T, rows, cols, amp, 240, TOL_ANA)
    checks.done()


@pytest.mark.gpu
def test_a2_config3_analysis_every_coefficient(gb, tables):
    """Analysis on GeographicGrid(0.25, 0.25) to degree 180 (config 3, latitude operators from the device Cholesky path) of
    every impulse field, in batches of 120."""
    checks = _Checks("A2")
    grid = gb.GeographicGrid(0.25, 0.25)
    _, _, U, T = tables(grid, 180)
    rows, cols, amp = _impulses(180, 0, 111)
    _analysis_sweep(checks, "min_degree 0, batches of 120",
                    lambda v: gb.analysis_batch(v, grid, 0, 180, "ewh", device_output=True),
                    U, T, rows, cols, amp, 120, TOL_ANA)
    checks.done()


# ------------------------------------------------------------------------------ dense
@pytest.mark.gpu
def test_d1_config2_dense_batch(gb, tables):
    """All 240 epochs of config 2 with equal power per degree against the separable float64 reference: accumulation
    across K chunks and order pairs, which single impulses do not exercise.  Error per (epoch, parallel) against the
    row maximum of the reference."""
    import torch
    checks = _Checks("D1")
    grid = gb.GeographicGrid(0.5, 0.5)
    plan = gb.get_plan(grid, 96, "ewh")
    U, T, _, _ = tables(grid, 96)
    X = _equal_power(96, 240, 112)
    ref = _separable_synthesis(X, U, T)
    rowmax = np.abs(ref).max(axis=2)
    checks.err("reference vs extended precision", _dense_guard(X, U, T, ref, rowmax, 113), EXACT_TOL)
    got = plan.synthesis(torch.as_tensor(X).cuda()).cpu().numpy()
    err = np.abs(got - ref).max(axis=2) / rowmax
    e, i = np.unravel_index(np.argmax(err), err.shape)
    print("D1 worst row: epoch %d, parallel %d" % (e, i))
    checks.err("240 epochs, per (epoch, parallel)", float(err.max()) if np.all(np.isfinite(got)) else float("nan"),
               TOL_DENSE)
    checks.done()
