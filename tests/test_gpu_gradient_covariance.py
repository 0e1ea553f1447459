"""Covariance of the gravitational acceleration (gradient_covariance_propagation, gradient_covariance_at_positions):
C_p = J_p sym(Sigma) J_p' with the Jacobian J_p = F'_p T of grad V, T Cunningham's transform and F'_p the point's
degree-(N+1) synthesis row with the factors GM/R^2 (R/r)^(n'+1).

The host restatement of J reuses the numpy restatement of the transform and of the gradient in test_gpu_gradient.py
(T as sparse matrices, built by applying gradient_coefficients to unit vectors) and the oracle's degree-(N+1) Legendre
and trigonometric tables; without a GPU it is tied to the restated gradient, J_p x = grad V(p).  On the GPU:

  - low rank, Sigma = G G' with G [K', 32]: C_p = sum_r g_r(p) g_r(p)' where g_r is the merged acceleration path
    (gradient_at_positions / gradient_batch) of the 32 columns of G, a reference that shares no code with the new
    kernels; errors entry by entry as |dC_cc'| / sqrt(C_cc C_c'c') (cross terms cross zero);
  - full rank, Sigma = G G' + diag(d) (the closed form of test_gpu_full_size_reference.py): variances at 64 sampled
    points against the restated J rows in extended precision;
  - up against gb_points_covariance with the radial-derivative degree factors -(n+1)/r GM/R (R/r)^(n+1);
  - a known answer (variance on C00 only), the local frame against Q C Q' on the host, and the edges: min_degree 2,
    point counts that are not a multiple of 40 over several point blocks, an antisymmetric part, repeated calls.
"""
import numpy as np
import pytest

from test_gpu_gradient import _track, gradient, gradient_coefficients
from test_gpu_full_size_reference import _antisymmetric, _exact_variance, _factors, _sigma

N = 96
NPTS = 40962               # the benchmark's point set (bench_configs.point_sets)
CHUNK = 256                # unit vectors per pass of the transform restatement

# Largest error each comparison may show: ten times the largest error an NVIDIA B200 (1000 W power limit) showed for it.
TOL_LOW = 1.2e-12          # low rank against the merged gradient path, |dC| / sqrt(C_cc C_c'c') (observed up to 1.2e-13)
TOL_FULL = 3e-14           # full rank against the restated Jacobian in extended precision, variances (2.5e-15)
TOL_UP = 2e-13             # up variance against gb_points_covariance with radial-derivative factors (1.5e-14)
TOL_C00 = 8e-15            # known answer: std(up) relative to s GM / r^2, east and north over (s GM / r^2)^2 (7.8e-16)
TOL_FRAME = 1e-14          # local frame against Q C Q' of the Cartesian result on the host (8.3e-16)
TOL_ANTI = 2e-13           # Sigma plus a dense antisymmetric part against the low-rank reference (1.6e-14)
EXACT_TOL = 1e-14          # float64 restated Jacobian rows against their extended-precision contraction


@pytest.fixture(scope="module")
def orc():
    from oracle import sh_oracle
    return sh_oracle


# ------------------------------------------------------------------------------ host restatement of the Jacobian
def _transform_matrices(orc, nmax):
    """T_c [(N+2)^2, K] (scipy CSR) for c = x, y, z, degree-wise on both sides from degree 0: column a is the
    degree-wise ravel of gradient_coefficients(e_a).  Sigma from min_degree nmin uses the columns nmin^2 .. K - 1."""
    from scipy import sparse
    K, Lo = (nmax + 1) ** 2, nmax + 2
    rows, cols, vals = [[], [], []], [[], [], []], [[], [], []]
    for a0 in range(0, K, CHUNK):
        a1 = min(a0 + CHUNK, K)
        unit = np.zeros((a1 - a0, K))
        unit[np.arange(a1 - a0), np.arange(a0, a1)] = 1.0
        g = gradient_coefficients(orc.unravel_coefficients(unit, 0, nmax))          # [B, 3, Lo, Lo]
        flat = orc.ravel_coefficients(g.reshape(-1, Lo, Lo)).reshape(a1 - a0, 3, Lo * Lo)
        for c in range(3):
            b, r = np.nonzero(flat[:, c])
            rows[c].append(r)
            cols[c].append(b + a0)
            vals[c].append(flat[b, c, r])
    return [sparse.csr_matrix((np.concatenate(vals[c]), (np.concatenate(rows[c]), np.concatenate(cols[c]))),
                              shape=(Lo * Lo, K)) for c in range(3)]


def _jacobian(orc, T, r, colat, lon, nmin, GM=None, R=None):
    """J [P, 3, K'] of grad V at geocentric (r, colat, lon): the oracle's degree-(N+1) synthesis rows F' with the factors
    GM/R^2 (R/r)^(n'+1), times T_c (columns from nmin^2 on)."""
    GM = orc.GM_DEFAULT if GM is None else GM
    R = orc.R_DEFAULT if R is None else R
    Lo = int(round(np.sqrt(T[0].shape[0])))
    kn = np.power((R / r)[:, None], np.arange(Lo, dtype=int) + 1) * (GM / R ** 2)
    kn[:, 0] = 0.0
    F = orc.ravel_coefficients(orc._scale_packed_by_degree(orc.spherical_harmonics(Lo - 1, colat, lon), kn))
    return np.stack([(T[c].T @ F.T).T[:, nmin * nmin:] for c in range(3)], axis=1)


def _to_local_matrix(colat, lon):
    """Q [P, 3, 3]: rows east, north, up of the geocentric spherical frame."""
    ct, st, cl, sl = np.cos(colat), np.sin(colat), np.cos(lon), np.sin(lon)
    z = np.zeros_like(ct)
    return np.stack((np.stack((-sl, cl, z), -1), np.stack((-ct * cl, -ct * sl, st), -1),
                     np.stack((st * cl, st * sl, ct), -1)), axis=1)


def _cov_err(got, ref):
    """max over points and entries of |got - ref| / sqrt(ref_cc ref_c'c') for [P, 3, 3] arrays (numpy or torch)."""
    import torch
    got, ref = torch.as_tensor(got), torch.as_tensor(ref).to(torch.as_tensor(got).device)
    if not bool(torch.isfinite(got).all()):
        return float("nan")
    d = torch.diagonal(ref, dim1=1, dim2=2).sqrt()
    return float(((got - ref).abs() / (d[:, :, None] * d[:, None, :])).max())


# ------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("nmin", [0, 2])
def test_restated_jacobian_reproduces_the_gradient(orc, nmin):
    """J_p x = grad V(p) for random x at N = 12, from the surface to 500 km, with two points within 1e-6 rad of the
    poles; the restated Jacobian is the reference of the GPU cases."""
    nmax = 12
    rng = np.random.default_rng(nmin)
    P = 40
    r = orc.R_DEFAULT + rng.uniform(0.0, 500e3, P)
    colat = np.arccos(rng.uniform(-1.0, 1.0, P))
    lon = rng.uniform(-np.pi, np.pi, P)
    colat[0], colat[1] = 3e-7, np.pi - 5e-7
    degrees = np.arange(nmin, nmax + 1)
    x = rng.standard_normal((nmax + 1) ** 2 - nmin ** 2) / (np.repeat(degrees, 2 * degrees + 1) + 1.0)
    J = _jacobian(orc, _transform_matrices(orc, nmax), r, colat, lon, nmin)
    g = gradient(orc, orc.unravel_coefficients(x, nmin, nmax), r, colat, lon)
    got = np.einsum("pca,a->cp", J, x)
    for c in range(3):
        assert np.max(np.abs(got[c] - g[c])) <= 1e-14 * np.max(np.abs(g[c])), c


def test_argument_errors_come_before_any_device_call(monkeypatch):
    import grates_b200 as gb
    from grates_b200 import plan

    def no_device(*args, **kwargs):
        raise AssertionError("a device was requested before the arguments were checked")
    monkeypatch.setattr(plan, "_current_device", no_device)
    pos = np.array([[7e6, 0.0, 0.0], [0.0, 7e6, 0.0]])
    s = np.zeros((25, 25))                                  # degrees 0..4
    grid = gb.GeographicGrid(30.0)
    for call in (lambda *a, **k: gb.gradient_covariance_at_positions(a[0], pos, *a[1:], **k),
                 lambda *a, **k: gb.gradient_covariance_propagation(a[0], grid, *a[1:], **k)):
        with pytest.raises(ValueError, match="shape"):
            call(np.zeros((24, 24)), 0, 4)
        with pytest.raises(ValueError, match="shape"):
            call(s, 2, 4)                                   # 21 coefficients from degree 2
        with pytest.raises(ValueError, match="degree range"):
            call(s, 5, 4)
        with pytest.raises(ValueError, match="degree range"):
            call(s, -1, 4)
        with pytest.raises(ValueError, match="frame"):
            call(s, 0, 4, frame='enu')
        with pytest.raises(ValueError, match="full"):
            call(s, 0, 4, full='yes')
    for bad in (np.zeros((1, 3)), np.array([[np.nan, 0.0, 1.0]]), np.zeros((4, 2))):
        with pytest.raises(ValueError, match="positions"):
            gb.gradient_covariance_at_positions(s, bad, 0, 4)


def test_c_abi_refuses_a_null_point_set():
    import ctypes
    from grates_b200 import _lib
    lib = _lib.load()
    for flags in (0, 1, 2):
        assert lib.gb_points_gradient_covariance(None, None, 0, None, None, flags, None) == _lib.GB_ERR_ARGUMENT
    assert b"NULL" in lib.gb_last_error()
    assert ctypes.sizeof(ctypes.c_void_p) == 8


# ------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def gb():
    import grates_b200
    grates_b200._lib.require_device()
    return grates_b200


@pytest.fixture(scope="module")
def low_rank(gb, orc):
    """G [K, 32] and its 32 columns as packed coefficient sets on the device (degrees below nmin zeroed per case)."""
    import torch
    G, d = _factors(N, 31)
    return {"G": G, "d": d, "X": torch.as_tensor(orc.unravel_coefficients(G.T.copy(), 0, N)).cuda()}


def _outer(g):
    """[R, 3, ...points] -> [P, 3, 3] sum over r of g_r g_r'."""
    g = g.reshape(g.shape[0], 3, -1)
    return __import__("torch").einsum("rcp,rdp->pcd", g, g)


def _benchmark_points():
    rng = np.random.default_rng(7)                                   # as bench_configs.point_sets
    return rng.uniform(-np.pi, np.pi, NPTS), np.arcsin(rng.uniform(-1, 1, NPTS))


@pytest.mark.gpu
def test_low_rank_against_the_gradient_path(gb, low_rank):
    """Sigma = G G' at the 86 402 orbit positions (both frames), the benchmark's 40 962 points and the 1 degree grid."""
    import torch
    s = _sigma(torch, low_rank["G"], np.zeros(low_rank["G"].shape[0]))
    X = low_rank["X"]
    pos = _track(86400, 4)
    worst = {}
    for frame in ("cartesian", "local"):
        ref = _outer(gb.gradient_at_positions(X, pos, frame=frame))
        got = gb.gradient_covariance_at_positions(s, pos, 0, N, frame=frame, full=True, device_output=True)
        assert tuple(got.shape) == (pos.shape[0], 3, 3)
        worst["orbit " + frame] = _cov_err(got, ref)
    lon, lat = _benchmark_points()
    grid = gb.IrregularGrid(lon, lat)
    ref = _outer(gb.gradient_batch(X, grid))
    got = gb.gradient_covariance_propagation(s, grid, 0, N, full=True, device_output=True)
    worst["benchmark points"] = _cov_err(got, ref)
    grid = gb.GeographicGrid(1.0, 1.0)
    ref = _outer(gb.gradient_batch(X, grid, frame='local'))
    got = gb.gradient_covariance_propagation(s, grid, 0, N, frame='local', full=True)
    assert isinstance(got, np.ndarray) and got.shape == (180, 360, 3, 3)
    worst["1 degree grid local"] = _cov_err(got.reshape(-1, 3, 3), ref.cpu())
    std = gb.gradient_covariance_propagation(s, grid, 0, N, frame='local')
    assert std.shape == (3, 180, 360)
    assert np.array_equal(std, np.sqrt(np.moveaxis(np.diagonal(got, axis1=2, axis2=3), -1, 0)))
    for label, err in worst.items():
        print("GRADCOV low rank %-22s %.3e" % (label, err))
    assert max(worst.values()) <= TOL_LOW, worst


@pytest.mark.gpu
def test_full_rank_against_the_restated_jacobian_and_up(gb, orc):
    """Sigma = G G' + diag(d) at the benchmark's points, min_degree 0 and 2: variances at 64 sampled points against the
    restated J rows in extended precision; the up variance at every point against gb_points_covariance with the
    radial-derivative degree factors; the local frame against Q C Q' and its standard deviations."""
    import torch
    from grates_b200 import utilities
    lon, lat = _benchmark_points()
    grid = gb.IrregularGrid(lon, lat)
    a, f = grid.semimajor_axis, grid.flattening
    r, colat = utilities.geocentric_radius(lat, a, f), utilities.colatitude(lat, a, f)
    G, d = _factors(N, 12)
    T = _transform_matrices(orc, N)
    sp = np.sort(np.concatenate((np.random.default_rng(3).choice(NPTS - 1, 63, replace=False), [NPTS - 1])))
    GM, R = gb.gravityfield.GM_DEFAULT, gb.gravityfield.R_DEFAULT
    n = np.arange(N + 1)
    up_factors = -(n + 1) / r[:, None] * np.power((R / r)[:, None], n + 1) * GM / R
    up_plan = gb.PointsPlan(lon, 0.5 * np.pi - colat, a, f, N, degree_factors=up_factors, colatitude=colat)
    Q = _to_local_matrix(colat, lon)
    errs = {}
    for nmin in (0, 2):
        Gn, dn = G[nmin * nmin:], d[nmin * nmin:]
        s = _sigma(torch, Gn, dn)
        cart = gb.gradient_covariance_propagation(s, grid, nmin, N, full=True)
        local = gb.gradient_covariance_propagation(s, grid, nmin, N, frame='local', full=True)
        J = _jacobian(orc, T, r[sp], colat[sp], lon[sp], nmin)
        G_ld, d_ld = Gn.astype(np.longdouble), dn.astype(np.longdouble)
        y = J @ Gn
        ref = np.einsum("pcr,pcr->pc", y, y) + (J * J) @ dn
        exact = np.array([[_exact_variance(J[i, c], G_ld, d_ld) for c in range(3)] for i in range(sp.size)])
        errs["restated vs extended precision, min_degree %d" % nmin] = (float(np.max(np.abs(ref - exact) / exact)),
                                                                       EXACT_TOL)
        got = np.diagonal(cart[sp], axis1=1, axis2=2)
        errs["variances, min_degree %d" % nmin] = (float(np.max(np.abs(got - exact) / exact)), TOL_FULL)
        up = up_plan.covariance_propagation(s, nmin, take_sqrt=False, symmetric=True).cpu().numpy()
        errs["up vs gb_points_covariance, min_degree %d" % nmin] = (float(np.max(np.abs(local[:, 2, 2] - up) / up)),
                                                                   TOL_UP)
        rotated = np.einsum("pij,pjk,plk->pil", Q, cart, Q)
        errs["local vs Q C Q', min_degree %d" % nmin] = (_cov_err(local, rotated), TOL_FRAME)
        std = gb.gradient_covariance_propagation(s, grid, nmin, N, frame='local')
        assert std.shape == (3, NPTS)
        assert np.array_equal(std, np.sqrt(np.diagonal(local, axis1=1, axis2=2).T)), nmin
        del s
    for label, (err, tol) in errs.items():
        print("GRADCOV full rank %-44s %.3e (tol %.0e)" % (label, err, tol))
    assert all(err <= tol for err, tol in errs.values()), errs


@pytest.mark.gpu
def test_variance_of_c00_alone(gb):
    """Variance s^2 on C00 only: std(up) = s GM / r^2 along the orbit, east and north vanish to rounding."""
    import torch
    from grates_b200 import utilities
    pos = _track(86400, 4)
    K = (N + 1) ** 2
    s2 = 4.0e-18
    sigma = torch.zeros((K, K), dtype=torch.float64, device="cuda")
    sigma[0, 0] = s2
    std = gb.gradient_covariance_at_positions(sigma, pos, 0, N, frame='local')
    full = gb.gradient_covariance_at_positions(sigma, pos, 0, N, frame='local', full=True)
    scale = np.sqrt(s2) * gb.gravityfield.GM_DEFAULT / utilities.cartesian_to_spherical(pos)[0] ** 2
    err_up = float(np.max(np.abs(std[2] - scale) / scale))
    err_en = float(np.max(np.abs(full[:, :2, :]) / scale[:, None, None] ** 2))
    print("GRADCOV C00 up %.3e east/north %.3e" % (err_up, err_en))
    assert err_up <= TOL_C00 and err_en <= TOL_C00


@pytest.mark.gpu
def test_edges_antisymmetric_part_partial_tiles_and_repeats(gb, low_rank):
    """Sigma plus a dense antisymmetric part gives the low-rank result; 7 and 1 001 points (a partial tile, two point
    blocks) equal the same points of the 86 402-point call; two identical calls are bit-identical; min_degree 2 on the
    orbit; flags other than GB_COV_SQRT are refused."""
    import ctypes
    import torch
    G = low_rank["G"]
    s = _sigma(torch, G, np.zeros(G.shape[0]))
    pos = _track(86400, 4)
    ref = _outer(gb.gradient_at_positions(low_rank["X"], pos))
    whole = gb.gradient_covariance_at_positions(s, pos, 0, N, full=True, device_output=True)
    again = gb.gradient_covariance_at_positions(s, pos, 0, N, full=True, device_output=True)
    assert torch.equal(whole, again)
    parts_equal = []
    for count in (7, 1001):
        part = gb.gradient_covariance_at_positions(s, pos[:count], 0, N, full=True, device_output=True)
        parts_equal.append(torch.equal(part, whole[:count]))
        assert _cov_err(part, whole[:count]) <= 1e-15, count
    print("GRADCOV partial point sets bit-identical to the whole call: %s" % parts_equal)
    anti = s + _antisymmetric(torch, s.shape[0], float(s.abs().max()), 29)
    err_anti = _cov_err(gb.gradient_covariance_at_positions(anti, pos, 0, N, full=True, device_output=True), ref)
    X2 = low_rank["X"].clone()
    X2[:, :2, :2] = 0.0
    ref2 = _outer(gb.gradient_at_positions(X2, pos))
    s2 = _sigma(torch, G[4:], np.zeros(G.shape[0] - 4))
    err_nmin = _cov_err(gb.gradient_covariance_at_positions(s2, pos, 2, N, full=True, device_output=True), ref2)
    print("GRADCOV antisymmetric part %.3e, min_degree 2 %.3e" % (err_anti, err_nmin))
    assert err_anti <= TOL_ANTI and err_nmin <= TOL_LOW
    from grates_b200 import plan as gplan, utilities
    p = gplan.get_gradient_points_plan(*utilities.cartesian_to_spherical(pos), N)
    out = torch.empty((3, p.npts), dtype=torch.float64, device="cuda")
    lib = gb._lib.load()
    for flags in (2, 4, 3):
        rc = lib.gb_points_gradient_covariance(p._handle, ctypes.c_void_p(s.data_ptr()), 0, None,
                                               ctypes.c_void_p(out.data_ptr()), flags, None)
        assert rc == gb._lib.GB_ERR_ARGUMENT, flags
