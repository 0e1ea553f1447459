"""Covariance propagation and the point-set kernels at production size against an exact reference.

The regular-grid covariance diag(A Sigma A') (config 4: degree 96, K = 9409) and the three point-set kernels (the point
sets row of the README: degree 96, 40 962 points, 240 epochs) take paths only at full size that no small case reaches:
several blocks of points, two spectral row tiles of the LonEpilogue GEMM, polar caps of the fold, the N = 96 instances of
the quadratic form.  A dense oracle costs minutes per thousand points at this size, so Sigma is built with a closed-form
variance instead:

    Sigma = G G' + diag(d),   G [K', 32] and d > 0 scaled by 1 / (n + 1) per degree n,
    var_p = ||(F G)_p||^2 + (F o F)_p d   for the synthesis row F_p of output point p,

which is strictly positive, so variances are compared point by point (max |got - ref| / ref): an error confined to
small-variance points or high-degree tiles cannot hide behind the largest value.  A dense antisymmetric part leaves
every variance unchanged and sends the propagation down its general (non-symmetric) path.  On a regular grid
F[(i, j), a] = U_i[a] T_j[a] (Legendre factor times trigonometric factor), and a spatial filter that only couples
coefficients of one order and trigonometric function (order-wise blocks, degree weights) acts on U_i alone.

The reference itself is guarded twice: against the dense oracle at degree 12 (test_reference_matches_dense_oracle, no
GPU), and in every GPU case by 64 sampled entries recomputed in extended precision.
"""
import numpy as np
import pytest

from conftest import maxnorm_err

N = 96
RANK = 32
NPTS = 40962               # the benchmark's point set (bench_configs.point_sets)
CHUNK = 2048               # points per chunk of the point-set reference
EXACT_TOL = 1e-14          # float64 reference against its extended-precision recomputation

# Largest error each comparison may show: ten times the largest error an NVIDIA B200 (1000 W power limit) showed for it.
# The general-Sigma cases contract a dense antisymmetric part (10 % of max|Sigma| at every degree, while Sigma itself
# falls off as 1/(n+1)^2) that cancels only in exact arithmetic: up to 4.3e-11 on the octant and quadrant grids, so
# their tolerance is held at 1e-10 with less headroom; the inputs are seeded and the propagation is bit-reproducible.
TOL_SYM = 3e-12            # variances, symmetric Sigma, point by point (observed up to 2.8e-13)
TOL_GEN = 1e-10            # variances, general Sigma, point by point (observed up to 4.3e-11)
TOL_LOC = 2e-12            # localized Sigma, relative to the row maximum of the reference (1.7e-13)
TOL_STD = 1e-12            # standard deviations, point by point (8.9e-14)
TOL_SYN = 2e-12            # point synthesis, relative to each epoch's maximum (1.5e-13)
TOL_ADJ = 3e-13            # point adjoint, relative to each value set's maximum (2.0e-14)


@pytest.fixture(scope="module")
def gb():
    import grates_b200
    grates_b200._lib.require_device()
    return grates_b200


@pytest.fixture(scope="module")
def orc():
    from oracle import sh_oracle
    return sh_oracle


# ------------------------------------------------------------------------------ reference
def _degrees(nmin, nmax):
    """Degree of every coefficient in degree-wise order (per degree n: C_n0, then C_nm, S_nm for m = 1..n)."""
    n = np.arange(nmin, nmax + 1)
    return np.repeat(n, 2 * n + 1)


def _orders(nmin, nmax):
    return np.concatenate([np.concatenate(([0], np.repeat(np.arange(1, n + 1), 2))) for n in range(nmin, nmax + 1)])


def _factors(nmax, seed, support=None):
    """G [K, RANK] and d [K] of Sigma = G G' + diag(d) from degree 0; Sigma from min_degree nmin is the trailing block
    (G[nmin^2:], d[nmin^2:]).  support: coefficients Sigma is restricted to (rows of G and entries of d elsewhere 0)."""
    prof = 1.0 / (_degrees(0, nmax) + 1.0)        # high degrees still contribute visibly
    rng = np.random.default_rng(seed)
    G = rng.standard_normal((prof.size, RANK)) * prof[:, None]
    d = rng.uniform(0.5, 1.5, prof.size) * prof ** 2
    if support is not None:
        G[~support] = 0.0
        d[~support] = 0.0
    return G, d


def _grid_tables(orc, parallels, meridians, nmin, nmax, kernel="ewh"):
    """U [nlat, K'] (Legendre functions times degree factors) and T [nlon, K'] (cos / sin of m lon), degree-wise."""
    colat, kn = orc.kn_table(kernel, nmax, parallels)
    U = orc.ravel_coefficients(orc._scale_packed_by_degree(orc.legendre_functions(nmax, colat), kn), nmin, nmax)
    T = orc.ravel_coefficients(orc.trigonometric_functions(nmax, meridians), nmin, nmax)
    return U, T


def _orderwise_apply(U, blocks, nmin, nmax):
    """U F for the order-wise filter matrix F of ``blocks`` (orc.orderwise_filter_matrix(blocks, nmin, nmax)), one
    block of (order, trigonometric function) at a time; works in U's precision."""
    out = np.zeros_like(U)
    base = np.arange(nmax + 1) ** 2 - nmin * nmin
    for m in range(nmax + 1):
        n = np.arange(max(m, nmin), nmax + 1)
        for cs in ((0,) if m == 0 else (0, 1)):
            idx = base[n] + (0 if m == 0 else 2 * m - 1 + cs)
            sub = blocks[0 if m == 0 else 2 * m - 1 + cs][np.ix_(n - m, n - m)]
            out[..., idx] = U[..., idx] @ sub
    return out


def _grid_variances(U, T, G, d, chunk=45):
    """var[i, j] = sum_r (T (U_i o g_r))_j^2 + ((T o T)(U_i^2 o d))_j: [nlat, nlon]."""
    nlat, K = U.shape
    out = np.empty((nlat, T.shape[0]))
    T2 = T * T
    for i0 in range(0, nlat, chunk):
        Ui = U[i0:i0 + chunk]
        M = (Ui.T[:, :, None] * G[:, None, :]).reshape(K, -1)           # [K, rows * RANK]
        W = (T @ M).reshape(T.shape[0], Ui.shape[0], G.shape[1])
        out[i0:i0 + chunk] = np.einsum("jir,jir->ij", W, W) + (T2 @ (Ui * Ui * d).T).T
    return out


def _point_variances(F, G, d):
    y = F @ G
    return np.einsum("pr,pr->p", y, y) + (F * F) @ d


def _exact_variance(f, G_ld, d_ld):
    """f' Sigma f in extended precision for one synthesis row f."""
    f = np.asarray(f, dtype=np.longdouble)
    y = f @ G_ld
    return y @ y + (f * f) @ d_ld


def _grid_guard(U, T, G, d, ref, scale, seed, filt=None):
    """Largest relative difference between the float64 reference and 64 entries recomputed in extended precision.
    U: the unfiltered Legendre factors; filt: the filter applied to them (any precision)."""
    rng = np.random.default_rng(seed)
    rows = rng.integers(0, U.shape[0], 64)
    cols = rng.integers(0, T.shape[0], 64)
    rows[:2], cols[:2] = (0, U.shape[0] - 1), (0, T.shape[0] - 1)
    G_ld, d_ld = G.astype(np.longdouble), d.astype(np.longdouble)
    worst = 0.0
    for i, j in zip(rows, cols):
        u = U[i].astype(np.longdouble)
        if filt is not None:
            u = filt(u[None])[0]
        exact = _exact_variance(T[j].astype(np.longdouble) * u, G_ld, d_ld)
        worst = max(worst, float(abs(ref[i, j] - exact) / scale[i, j]))
    return worst


def _rel(got, ref):
    """max |got - ref| / ref over all points (ref > 0); NaN if anything is not finite."""
    got, ref = np.asarray(got, dtype=float), np.asarray(ref, dtype=float)
    if not np.all(np.isfinite(got)):
        return float("nan")
    return float(np.max(np.abs(got - ref) / ref))


def _rel_rowmax(got, ref):
    """max |got - ref| / (maximum of the reference's row): for references that may be zero."""
    got, ref = np.asarray(got, dtype=float), np.asarray(ref, dtype=float)
    if not np.all(np.isfinite(got)):
        return float("nan")
    return float(np.max(np.abs(got - ref) / np.max(np.abs(ref), axis=-1, keepdims=True)))


class _Checks:
    """Records every comparison of a case (printed, so that a run shows the observed errors beside their tolerances)
    and fails once at the end with all of them that are out of tolerance."""

    def __init__(self, case):
        self.case, self.bad = case, []

    def err(self, label, err, tol):
        print("%s %-44s %.3e  (tol %.0e)" % (self.case, label, err, tol))
        if not err <= tol:
            self.bad.append("%s: %.3e > %.0e" % (label, err, tol))

    def equal(self, label, ok):
        print("%s %-44s %s" % (self.case, label, "equal" if ok else "DIFFERENT"))
        if not ok:
            self.bad.append(label + ": not bit-identical")

    def state(self, label, got, want):
        if got != want:
            self.bad.append("%s is %r, expected %r" % (label, got, want))

    def done(self):
        assert not self.bad, "%s: %s" % (self.case, "; ".join(self.bad))


def _sigma(torch, G, d):
    """Sigma = G G' + diag(d) on the device, exactly symmetric."""
    g = torch.as_tensor(G).cuda()
    s = g @ g.T
    s = 0.5 * (s + s.T)
    s.diagonal().add_(torch.as_tensor(d).cuda())
    return s


def _antisymmetric(torch, K, scale, seed):
    """B - B' with entries up to 0.1 scale: changes no variance, but Sigma + (B - B') is visibly not symmetric."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    b = torch.rand((K, K), generator=gen, dtype=torch.float64, device="cuda") - 0.5
    return (b - b.T) * (0.1 * scale)


def _plan_state(gb, checks, plan, octant, symmetric, folded):
    lib = gb._lib.load()
    checks.state("octant", plan.octant, octant)
    checks.state("symmetric", plan.symmetric, symmetric)
    checks.state("gb_plan_is_folded", lib.gb_plan_is_folded(plan._handle), folded)


def _grid_var(plan, s, nmin, **kwargs):
    return plan.covariance_propagation(s, nmin, take_sqrt=False, **kwargs).cpu().numpy()


def _two_cap_grid(gb):
    """0.5 degree parallels (1 degree meridians) with parallel 40 moved by 1e-9: it fails the fold gate, so the first
    two tiles of 32 parallels per hemisphere stay unfolded (gb_plan_is_folded == 3)."""
    base = gb.GeographicGrid(1.0, 0.5)
    par = base.parallels.copy()
    par[40] += 1e-9
    return gb.RegularGrid(base.meridians, par)


def _symmetric_and_general(gb, torch, checks, plan, G, d, nmin, ref, label=""):
    """Symmetric Sigma and Sigma plus an antisymmetric part, both left to the automatic detection."""
    from grates_b200 import plan as gplan
    s = _sigma(torch, G[nmin * nmin:], d[nmin * nmin:])
    checks.state("symmetric Sigma detected" + label, gplan._looks_symmetric(s), True)
    checks.err("variances, symmetric Sigma" + label, _rel(_grid_var(plan, s, nmin), ref), TOL_SYM)
    s += _antisymmetric(torch, s.shape[0], float(s.abs().max()), 17)
    checks.state("general Sigma detected" + label, gplan._looks_symmetric(s), False)
    checks.err("variances, general Sigma" + label, _rel(_grid_var(plan, s, nmin), ref), TOL_GEN)


# ------------------------------------------------------------------------------ the reference itself (no GPU)
def test_reference_matches_dense_oracle(orc):
    """The closed-form reference against the dense oracle at degree 12: min_degree 2, an order-wise filter and an
    antisymmetric part, on a regular grid and at scattered points; and degree weights on the grid."""
    nmax, nmin = 12, 2
    G, d = _factors(nmax, 3)
    G, d = G[nmin * nmin:], d[nmin * nmin:]
    S = G @ G.T + np.diag(d)
    rng = np.random.default_rng(4)
    B = rng.uniform(-0.5, 0.5, S.shape)
    S_gen = S + (B - B.T) * 0.1 * np.abs(S).max()
    blocks = orc.synthetic_filter_blocks(nmax)
    F = orc.orderwise_filter_matrix(blocks, nmin, nmax)
    og = orc.geographic_grid(15.0, 10.0)
    U, T = _grid_tables(orc, og.parallels, og.meridians, nmin, nmax)
    ref = orc.covariance_propagation(F @ S_gen @ F.T, og, nmin, nmax, "ewh") ** 2
    mine = _grid_variances(_orderwise_apply(U, blocks, nmin, nmax), T, G, d)
    assert _rel(mine.ravel(), ref) < 1e-13
    w = orc.gauss_weights(1000.0, nmax)[_degrees(nmin, nmax)]
    ref = orc.covariance_propagation(w[:, None] * S_gen * w[None, :], og, nmin, nmax, "ewh") ** 2
    assert _rel(_grid_variances(U * w, T, G, d).ravel(), ref) < 1e-13
    lon, lat = rng.uniform(-np.pi, np.pi, 300), np.arcsin(rng.uniform(-1, 1, 300))
    Fp = orc.synthesis_matrix_points(lon, lat, nmin, nmax, "ewh")
    ref = orc.covariance_propagation_points(F @ S_gen @ F.T, lon, lat, nmin, nmax, "ewh") ** 2
    assert _rel(_point_variances(_orderwise_apply(Fp, blocks, nmin, nmax), G, d), ref) < 1e-13


# ------------------------------------------------------------------------------ regular grids
@pytest.mark.gpu
def test_r1_config4_symmetric_general_localized_and_row_blocks(gb, orc):
    """Config 4 (0.5 x 0.5 degree, 360 x 720): octant Fourier stage, folded, 180 representative parallels (quadratic
    form <3,4>).  Whole grid with symmetric, general and two localized Sigma; one standard-deviation output; eight row
    blocks of 45; a mirrored block bit-identical to the whole-grid rows."""
    import torch
    checks = _Checks("R1")
    grid = gb.GeographicGrid(0.5, 0.5)
    plan = gb.get_plan(grid, N, "ewh")
    _plan_state(gb, checks, plan, True, True, 1)
    G, d = _factors(N, 1)
    U, T = _grid_tables(orc, grid.parallels, grid.meridians, 0, N)
    ref = _grid_variances(U, T, G, d)
    checks.err("reference vs extended precision", _grid_guard(U, T, G, d, ref, ref, 1), EXACT_TOL)
    _symmetric_and_general(gb, torch, checks, plan, G, d, 0, ref)
    s = _sigma(torch, G, d)
    whole = plan.covariance_propagation(s, 0, take_sqrt=False)
    std = plan.covariance_propagation(s, 0).cpu().numpy()
    checks.err("standard deviations", _rel(std, np.sqrt(ref)), TOL_STD)
    blocks = np.concatenate([_grid_var(plan, s, 0, row0=r0, nrows=45) for r0 in range(0, 360, 45)])
    checks.err("8 row blocks of 45", _rel(blocks, ref), TOL_SYM)
    both = plan.covariance_propagation(s, 0, 7, 60, take_sqrt=False, mirrored=True)
    checks.equal("mirrored block 7 + 60, northern rows", torch.equal(both[:60], whole[7:67]))
    checks.equal("mirrored block 7 + 60, southern rows", torch.equal(both[60:], whole[293:353]))
    del s, whole
    # Sigma on degrees 90-96 only; on orders {0, 1} and {95, 96} together (k < k' pairs of the first and last row tile)
    for label, support in (("degrees 90-96", _degrees(0, N) >= 90),
                           ("orders 0, 1, 95, 96", np.isin(_orders(0, N), (0, 1, 95, 96)))):
        Gl, dl = _factors(N, 2, support)
        ref = _grid_variances(U, T, Gl, dl)
        rowmax = np.broadcast_to(ref.max(axis=1, keepdims=True), ref.shape)
        checks.err("reference vs extended precision, " + label, _grid_guard(U, T, Gl, dl, ref, rowmax, 2), EXACT_TOL)
        checks.err("localized Sigma, " + label, _rel_rowmax(_grid_var(plan, _sigma(torch, Gl, dl), 0), ref), TOL_LOC)
    checks.done()


@pytest.mark.gpu
def test_r2_octant_with_120_representatives(gb, orc):
    """0.75 x 0.75 degree (240 x 480): octant Fourier stage, folded, 120 representatives (quadratic form <5,3>)."""
    import torch
    checks = _Checks("R2")
    grid = gb.GeographicGrid(0.75, 0.75)
    plan = gb.get_plan(grid, N, "ewh")
    _plan_state(gb, checks, plan, True, True, 1)
    G, d = _factors(N, 5)
    U, T = _grid_tables(orc, grid.parallels, grid.meridians, 0, N)
    ref = _grid_variances(U, T, G, d)
    checks.err("reference vs extended precision", _grid_guard(U, T, G, d, ref, ref, 5), EXACT_TOL)
    _symmetric_and_general(gb, torch, checks, plan, G, d, 0, ref)
    checks.done()


@pytest.mark.gpu
def test_r3_lon_epilogue_with_two_row_tiles(gb, orc):
    """2 x 2 degree (90 x 180): 180 meridians are not a multiple of 8, so the longitude contraction is the LonEpilogue
    GEMM instead of the symmetric Fourier stage, with two spectral row tiles at degree 96 (kpad = 196) and, for symmetric Sigma,
    row tile 1 starting at k = 128; 45 representatives (quadratic form <3,3>).  min_degree 0 and 2."""
    import torch
    checks = _Checks("R3")
    grid = gb.GeographicGrid(2.0, 2.0)
    plan = gb.get_plan(grid, N, "ewh")
    _plan_state(gb, checks, plan, False, False, 1)
    G, d = _factors(N, 6)
    for nmin in (0, 2):
        Gn, dn = G[nmin * nmin:], d[nmin * nmin:]
        U, T = _grid_tables(orc, grid.parallels, grid.meridians, nmin, N)
        ref = _grid_variances(U, T, Gn, dn)
        label = ", min_degree %d" % nmin
        checks.err("reference vs extended precision" + label, _grid_guard(U, T, Gn, dn, ref, ref, 6), EXACT_TOL)
        _symmetric_and_general(gb, torch, checks, plan, G, d, nmin, ref, label)
    checks.done()


@pytest.mark.gpu
def test_r4_fold_with_polar_caps(gb, orc):
    """The two-cap grid (1 x 0.5 degree, parallel 40 moved by 1e-9): the covariance fold leaves the 64 parallels next to
    each pole unfolded (fold_cap = 64); four-fold but not eight-fold Fourier stage."""
    import torch
    checks = _Checks("R4")
    grid = _two_cap_grid(gb)
    plan = gb.get_plan(grid, N, "ewh")
    _plan_state(gb, checks, plan, False, True, 3)
    G, d = _factors(N, 7)
    U, T = _grid_tables(orc, grid.parallels, grid.meridians, 0, N)
    ref = _grid_variances(U, T, G, d)
    checks.err("reference vs extended precision", _grid_guard(U, T, G, d, ref, ref, 7), EXACT_TOL)
    _symmetric_and_general(gb, torch, checks, plan, G, d, 0, ref)
    checks.done()


@pytest.mark.gpu
def test_r5_odd_gauss_grid(gb, orc):
    """GaussGrid(97): an odd parallel count (the equator is its own mirror image), left unfolded by the fold gate, and
    194 meridians (LonEpilogue)."""
    import torch
    checks = _Checks("R5")
    grid = gb.GaussGrid(97)
    plan = gb.get_plan(grid, N, "ewh")
    _plan_state(gb, checks, plan, False, False, 0)
    G, d = _factors(N, 8)
    U, T = _grid_tables(orc, grid.parallels, grid.meridians, 0, N)
    ref = _grid_variances(U, T, G, d)
    checks.err("reference vs extended precision", _grid_guard(U, T, G, d, ref, ref, 8), EXACT_TOL)
    _symmetric_and_general(gb, torch, checks, plan, G, d, 0, ref)
    checks.done()


@pytest.mark.gpu
def test_r6_filtered_propagation_at_degree_96(gb, orc):
    """Spatial filters at degree 96: order-wise blocks (gb_cov_apply_blocks, unfolded) on the config-4 grid and on the
    LonEpilogue grid; Gaussian degree weights (the wn factor of gb_cov_legendre, folded) on the config-4 grid."""
    import torch
    checks = _Checks("R6")
    G, d = _factors(N, 9)
    s = _sigma(torch, G, d)
    blocks = orc.synthetic_filter_blocks(100)
    flt = gb.OrderWiseFilter(blocks)
    w = orc.gauss_weights(300.0, N)
    np.testing.assert_allclose(w, gb.Gaussian(300.0)._weights(N), rtol=1e-14, atol=0)
    wk = w[_degrees(0, N)]
    cases = ((gb.GeographicGrid(0.5, 0.5), flt, lambda u: _orderwise_apply(u, blocks, 0, N), "0.5 deg, order-wise"),
             (gb.GeographicGrid(2.0, 2.0), flt, lambda u: _orderwise_apply(u, blocks, 0, N), "2 deg, order-wise"),
             (gb.GeographicGrid(0.5, 0.5), gb.Gaussian(300.0), lambda u: u * wk, "0.5 deg, Gaussian 300 km"))
    for seed, (grid, spatial_filter, apply, label) in enumerate(cases):
        plan = gb.get_plan(grid, N, "ewh")
        U, T = _grid_tables(orc, grid.parallels, grid.meridians, 0, N)
        ref = _grid_variances(apply(U), T, G, d)
        checks.err("reference vs extended precision, " + label, _grid_guard(U, T, G, d, ref, ref, seed, apply), EXACT_TOL)
        got = _grid_var(plan, s, 0, spatial_filter=spatial_filter)
        checks.err("variances, " + label, _rel(got, ref), TOL_SYM)
    checks.done()


# ------------------------------------------------------------------------------ point sets
@pytest.fixture(scope="module")
def points(gb, orc):
    """The benchmark's point set at degree 96 with every reference of the point-set cases, computed in one pass over
    chunks of the dense synthesis matrix; plus rows and columns of that matrix at sampled points and coefficients for
    the extended-precision recomputation."""
    rng = np.random.default_rng(7)                                   # as bench_configs.point_sets
    lon, lat = rng.uniform(-np.pi, np.pi, NPTS), np.arcsin(rng.uniform(-1, 1, NPTS))
    L, K = N + 1, (N + 1) ** 2
    rng = np.random.default_rng(11)
    deg = np.arange(L)
    packed_degree = np.where(np.tril(np.ones((L, L), dtype=bool)), deg[:, None], deg[None, :])
    X = rng.standard_normal((240, L, L)) / (packed_degree + 1.0)
    V = rng.standard_normal((130, NPTS))
    G, d = _factors(N, 12)
    Xd = orc.ravel_coefficients(X)
    syn, adj = np.empty((240, NPTS)), np.zeros((130, K))
    var = {0: np.empty(NPTS), 2: np.empty(NPTS)}
    sp = np.sort(np.concatenate((rng.choice(NPTS - 1, 63, replace=False), [NPTS - 1])))   # sampled points
    sa = rng.integers(0, K, 64)                                                             # sampled coefficients
    rows, cols = np.empty((sp.size, K)), np.empty((NPTS, sa.size))
    for c0 in range(0, NPTS, CHUNK):
        c1 = min(c0 + CHUNK, NPTS)
        F = orc.synthesis_matrix_points(lon[c0:c1], lat[c0:c1], 0, N, "ewh")
        syn[:, c0:c1] = Xd @ F.T
        adj += V[:, c0:c1] @ F
        for nmin in (0, 2):
            var[nmin][c0:c1] = _point_variances(F[:, nmin * nmin:], G[nmin * nmin:], d[nmin * nmin:])
        inside = (sp >= c0) & (sp < c1)
        rows[inside] = F[sp[inside] - c0]
        cols[c0:c1] = F[:, sa]
    # extended-precision recomputation of sampled entries of every reference
    se = rng.integers(0, 240, sp.size)
    exact = {"synthesis": max(float(abs(syn[e, p] - rows[i].astype(np.longdouble) @ Xd[e].astype(np.longdouble))
                                    / np.abs(syn[e]).max()) for i, (e, p) in enumerate(zip(se, sp))),
             "adjoint": max(float(abs(adj[e, a] - cols[:, j].astype(np.longdouble) @ V[e].astype(np.longdouble))
                                  / np.abs(adj[e]).max()) for j, (e, a) in enumerate(zip(se % 130, sa)))}
    for nmin in (0, 2):
        G_ld, d_ld = G[nmin * nmin:].astype(np.longdouble), d[nmin * nmin:].astype(np.longdouble)
        exact["covariance, min_degree %d" % nmin] = max(
            float(abs(var[nmin][p] - _exact_variance(rows[i, nmin * nmin:], G_ld, d_ld)) / var[nmin][p])
            for i, p in enumerate(sp))
    plan = gb.get_points_plan(gb.IrregularGrid(lon, lat), N, "ewh")
    adj_packed = orc.unravel_coefficients(adj, 0, N)
    return {"plan": plan, "X": X, "V": V, "G": G, "d": d, "syn": syn, "adj": adj_packed, "var": var, "exact": exact}


def _launches(gb, fn):
    """Kernel launches of one library call (gb_launch_count, reset before the call) and its result."""
    lib = gb._lib.load()
    lib.gb_launch_count(1)
    out = fn()
    return int(lib.gb_launch_count(0)), out


@pytest.mark.gpu
def test_p1_point_synthesis_over_several_blocks(gb, points):
    """Batched point synthesis on the DMMA GEMM, 240 and 17 epochs: every point and every epoch against F X."""
    import torch
    checks = _Checks("P1")
    checks.err("reference vs extended precision", points["exact"]["synthesis"], EXACT_TOL)
    pp, X = points["plan"], torch.as_tensor(points["X"]).cuda()
    for E in (240, 17):
        out = torch.full((E, NPTS), float("nan"), dtype=torch.float64, device="cuda")
        n, _ = _launches(gb, lambda: pp.synthesis(X[:E], out=out))
        # 1 + 2B launches for B blocks of points: the coefficient tiles once, then design tiles and GEMM per block
        checks.state("launches of the %d-epoch synthesis (1 + 2B, B >= 2)" % E, (n - 1) % 2 == 0 and n >= 5, True)
        checks.err("%d epochs, max over epochs of max|d| / max|ref|" % E,
                   max(maxnorm_err(o, r) for o, r in zip(out.cpu().numpy(), points["syn"][:E])), TOL_SYN)
    checks.done()


@pytest.mark.gpu
def test_p2_point_adjoint_accumulates_every_block(gb, points):
    """Adjoint of the point synthesis with 1, 30 and 130 value sets (column fragments NI = 1, 2, 5): the blocks of
    points accumulate into the coefficients."""
    import torch
    checks = _Checks("P2")
    checks.err("reference vs extended precision", points["exact"]["adjoint"], EXACT_TOL)
    pp, V = points["plan"], torch.as_tensor(points["V"]).cuda()
    for E in (1, 30, 130):
        n, out = _launches(gb, lambda: pp.adjoint(V[:E].contiguous()))
        # 3B launches for B blocks of points: design tiles, value tiles and the accumulating GEMM per block
        checks.state("launches of the adjoint of %d value sets (3B, B >= 2)" % E, n % 3 == 0 and n >= 6, True)
        checks.err("%d value sets, max over sets of max|d| / max|ref|" % E,
                   max(maxnorm_err(o, r) for o, r in zip(out.cpu().numpy(), points["adj"][:E])), TOL_ADJ)
    checks.done()


@pytest.mark.gpu
def test_p3_point_covariance_over_several_blocks(gb, points):
    """diag(F Sigma F') at the benchmark's points: lower-triangle (symmetric) path, full path, automatic detection of a
    non-symmetric Sigma; min_degree 0 and 2; point by point."""
    import torch
    from grates_b200 import plan as gplan
    checks = _Checks("P3")
    pp = points["plan"]
    for nmin in (0, 2):
        checks.err("reference vs extended precision, min_degree %d" % nmin,
                   points["exact"]["covariance, min_degree %d" % nmin], EXACT_TOL)
        ref = points["var"][nmin]
        s = _sigma(torch, points["G"][nmin * nmin:], points["d"][nmin * nmin:])
        gen = s + _antisymmetric(torch, s.shape[0], float(s.abs().max()), 23)
        checks.state("general Sigma detected", gplan._looks_symmetric(gen), False)
        for label, sigma, symmetric in (("symmetric", s, True), ("general", gen, False), ("auto-detected", gen, None)):
            n, out = _launches(gb, lambda: pp.covariance_propagation(sigma, nmin, take_sqrt=False, symmetric=symmetric))
            # 1 + 3B launches for B blocks of points: Sigma tiles once, then design tiles, GEMM and finish per block
            checks.state("launches, %s, min_degree %d (1 + 3B, B >= 2)" % (label, nmin), (n - 1) % 3 == 0 and n >= 7, True)
            checks.err("variances, %s Sigma, min_degree %d" % (label, nmin), _rel(out.cpu().numpy(), ref),
                       TOL_SYM if symmetric else TOL_GEN)
        std = pp.covariance_propagation(s, nmin).cpu().numpy()
        checks.err("standard deviations, min_degree %d" % nmin, _rel(std, np.sqrt(ref)), TOL_STD)
        del s, gen
    checks.done()
