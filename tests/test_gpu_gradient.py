"""Gravitational acceleration (gradient_batch, gradient_at_positions): the coefficient transform of Cunningham's
relation, the degree-(N+1) synthesis of its 3E sets and the rotation to (east, north, up).

The numpy restatement below (gradient_coefficients, gradient: the oracle's Legendre and trigonometric tables at degree
N + 1; kept here so that the pinned oracle module stays as it is) is tied to the reference twice without a GPU: to
central differences of the oracle's potential, and to the reference's own zonal gradient behind GRS80 normal gravity
(oracle.normal_gravity, pinned by tests/golden/kernels.npz through the obp kernel).  On the GPU every path of the
synthesis that the 3E sets can take is compared with that restatement, and the whole 0.5 degree grid is checked once
more through the existing scalar synthesis with radial and longitudinal derivative factors, a path that shares no code
with the transform or the rotation.
"""
import numpy as np
import pytest

from conftest import maxnorm_err

N = 96
NPTS = 40962               # the benchmark's point set (bench_configs.point_sets)
# Largest max-normalised error per component a comparison with the restatement or the scalar-synthesis path may show:
# ten times the largest error an NVIDIA B200 (1000 W power limit) showed, 6.9e-14 on the 0.5 degree grid.
TOL = 7e-13


@pytest.fixture(scope="module")
def orc():
    from oracle import sh_oracle
    return sh_oracle


def _coefficients(E, nmax, seed):
    """Random sets with a 1/(n+1) spectrum and no dominant degree 0, so that every degree shows in the gradient."""
    L = nmax + 1
    deg = np.arange(L)
    packed_degree = np.where(np.tril(np.ones((L, L), dtype=bool)), deg[:, None], deg[None, :])
    return np.random.default_rng(seed).standard_normal((E, L, L)) / (packed_degree + 1.0)


def _to_cartesian(r, colat, lon):
    return np.stack((r * np.sin(colat) * np.cos(lon), r * np.sin(colat) * np.sin(lon), r * np.cos(colat)), axis=1)


def _to_local(g, colat, lon):
    """[.., 3, P] Cartesian -> (east, north, up) of the geocentric spherical frame, on the host."""
    ct, st, cl, sl = np.cos(colat), np.sin(colat), np.cos(lon), np.sin(lon)
    gx, gy, gz = g[..., 0, :], g[..., 1, :], g[..., 2, :]
    return np.stack((-sl * gx + cl * gy, -ct * cl * gx - ct * sl * gy + st * gz, st * cl * gx + st * sl * gy + ct * gz),
                    axis=-2)


def gradient_coefficients(anm):
    """numpy restatement of the transform: packed [..., L, L] -> [..., 3, L+1, L+1] (x, y, z).  With q = (2n+1)/(2n+3),
    (C_nm, S_nm) goes to Z[n+1, m] -sqrt((n-m+1)(n+m+1) q) (C, S);  X[n+1, m+1] -fp (C, S), Y[n+1, m+1] (fp S, -fp C);
    X[n+1, m-1] fm (C, S), Y[n+1, m-1] (fm S, -fm C) for m >= 1;  fp = sqrt((n+m+1)(n+m+2) q) / 2 (x sqrt 2 at m = 0),
    fm = sqrt((n-m+1)(n-m+2) q) / 2 (x sqrt 2 at m = 1).  Factors and sums in the order of gb_gradient_coefficients: an
    output of order m' adds its fp term (source order m' - 1) before its fm term (source order m' + 1)."""
    anm = np.asarray(anm, dtype=float)
    L = anm.shape[-1]
    lead = anm.shape[:-2]
    C = np.zeros(lead + (L, L))
    S = np.zeros(lead + (L, L))
    for m in range(L):
        C[..., m:, m] = anm[..., m:, m]
        if m > 0:
            S[..., m:, m] = anm[..., m - 1, m:]
    Lo = L + 1
    gc = np.zeros(lead + (3, Lo, Lo))                  # [.., component, n', m'] cosines
    gs = np.zeros(lead + (3, Lo, Lo))                  # sines
    sqrt2 = np.sqrt(2.0)
    for n in range(L):
        q = (2.0 * n + 1.0) / (2.0 * n + 3.0)
        for m in range(n + 1):
            c, s = C[..., n, m], S[..., n, m]
            fz = np.sqrt(float((n - m + 1) * (n + m + 1)) * q)
            gc[..., 2, n + 1, m] = -fz * c
            gs[..., 2, n + 1, m] = -fz * s
            fp = np.sqrt(float((n + m + 1) * (n + m + 2)) * q) * 0.5
            fp = fp * sqrt2 if m == 0 else fp
            gc[..., 0, n + 1, m + 1] += -fp * c
            gs[..., 0, n + 1, m + 1] += -fp * s
            gc[..., 1, n + 1, m + 1] += fp * s
            gs[..., 1, n + 1, m + 1] += -fp * c
        for m in range(1, n + 1):
            c, s = C[..., n, m], S[..., n, m]
            fm = np.sqrt(float((n - m + 1) * (n - m + 2)) * q) * 0.5
            fm = fm * sqrt2 if m == 1 else fm
            gc[..., 0, n + 1, m - 1] += fm * c
            gs[..., 0, n + 1, m - 1] += fm * s
            gc[..., 1, n + 1, m - 1] += fm * s
            gs[..., 1, n + 1, m - 1] += -fm * c
    out = np.zeros(lead + (3, Lo, Lo))
    for m in range(Lo):
        out[..., m:, m] = gc[..., m:, m]
        if m > 0:
            out[..., m - 1, m:] = gs[..., m:, m]
    return out


def gradient(orc, anm, r, colat, lon, GM=None, R=None):
    """grad V at geocentric (r, colat, lon), Earth-fixed Cartesian: [3, P] for anm [L, L], [E, 3, P] for [E, L, L].  Each
    component is the degree-(N+1) synthesis of gradient_coefficients with the degree factors GM/R^2 (R/r)^(n'+1), from
    the oracle's Legendre functions (legendre_functions(N + 1, .)) and trigonometric tables, 512 points at a time."""
    GM = orc.GM_DEFAULT if GM is None else GM
    R = orc.R_DEFAULT if R is None else R
    anm = np.asarray(anm, dtype=float)
    single = anm.ndim == 2
    G = gradient_coefficients(anm[None] if single else anm)
    E, Lo = G.shape[0], G.shape[-1]
    r, colat, lon = (np.atleast_1d(np.asarray(v, dtype=float)) for v in (r, colat, lon))
    flat = G.reshape(E * 3, Lo * Lo)
    out = np.empty((E * 3, r.size))
    for i1 in range(0, r.size, 512):
        i2 = min(i1 + 512, r.size)
        kn = np.power((R / r[i1:i2])[:, None], np.arange(Lo, dtype=int) + 1) * (GM / R ** 2)
        kn[:, 0] = 0.0
        Y = orc._scale_packed_by_degree(orc.spherical_harmonics(Lo - 1, colat[i1:i2], lon[i1:i2]), kn)
        out[:, i1:i2] = flat @ Y.reshape(i2 - i1, Lo * Lo).T
    out = out.reshape(E, 3, r.size)
    return out[0] if single else out


def _worst(got, ref):
    """Largest max-normalised error over epochs and components of [E, 3, ...] arrays."""
    return max(maxnorm_err(got[e, c], ref[e, c]) for e in range(ref.shape[0]) for c in range(3))


# ------------------------------------------------------------------------------ CPU: the oracle and the host side
def _potential(orc, anm, r, colat, lon):
    L = anm.shape[0]
    kn = np.power((orc.R_DEFAULT / r)[:, None], np.arange(L) + 1) * (orc.GM_DEFAULT / orc.R_DEFAULT)
    Y = orc._scale_packed_by_degree(orc.spherical_harmonics(L - 1, colat, lon), kn)
    return Y.reshape(r.size, -1) @ anm.reshape(-1)


@pytest.mark.parametrize("nmax", [12, 30])
def test_oracle_gradient_matches_finite_differences(orc, nmax):
    """Central differences (10 m steps) of the oracle's potential along x, y and z, from the surface to 500 km, with
    two points within 1e-6 rad of the poles."""
    from grates_b200 import utilities
    rng = np.random.default_rng(nmax)
    anm = _coefficients(1, nmax, nmax)[0]
    P = 40
    r = orc.R_DEFAULT + rng.uniform(0.0, 500e3, P)
    colat = np.arccos(rng.uniform(-1.0, 1.0, P))
    lon = rng.uniform(-np.pi, np.pi, P)
    colat[0], colat[1] = 3e-7, np.pi - 5e-7
    g = gradient(orc, anm, r, colat, lon)
    x = _to_cartesian(r, colat, lon)
    h = 10.0
    for k in range(3):
        step = np.zeros(3)
        step[k] = h
        fd = (_potential(orc, anm, *utilities.cartesian_to_spherical(x + step)) -
              _potential(orc, anm, *utilities.cartesian_to_spherical(x - step))) / (2 * h)
        assert maxnorm_err(g[k], fd) < 2e-9, (k, maxnorm_err(g[k], fd))      # the differences reach 3e-10


def _bowring_latitude(x, z, a, flat):
    """Geodetic latitude of (x, 0, z) by the iteration of oracle.normal_gravity (reference grid.py:1991-2006)."""
    e2 = 2 * flat - flat ** 2
    p2 = x ** 2
    h0 = 0
    k = (1 - e2) ** -1
    for _ in range(10):
        c = np.power(p2 + (1 - e2) * z ** 2 * k ** 2, 1.5) / (a * e2)
        k = 1 + (p2 + (1 - e2) * z ** 2 * k ** 3) / (c - p2)
        h = (k ** -1 - (1 - e2)) * np.sqrt(p2 + z ** 2 * k ** 2) / e2
        if np.max(np.abs(h - h0)) < 1e-6:
            break
        h0 = h
    return np.arctan2(k * z, np.sqrt(p2))


def test_oracle_gradient_reproduces_grs80_normal_gravity(orc):
    """The GRS80 zonal field as C_n0 with R = a: the oracle gradient plus the centrifugal term, projected on the Bowring
    latitude, is the reference's normal gravity (sign, normalisation and the sqrt 2 of order 0), from 20 km below to
    320 km above the ellipsoid."""
    GM, omega, a, flat, zonal = orc._grs80_field()
    anm = np.zeros((zonal.size, zonal.size))
    anm[:, 0] = zonal
    rng = np.random.default_rng(3)
    lat = rng.uniform(-0.5 * np.pi, 0.5 * np.pi, 50)
    colat = orc.colatitude(lat)
    r = orc.geocentric_radius(lat) + rng.uniform(-20e3, 320e3, 50)
    g = gradient(orc, anm, r, colat, np.zeros(50), GM, a)
    x, z = r * np.sin(colat), r * np.cos(colat)
    phi = _bowring_latitude(x, z, a, flat)
    gamma = -np.cos(phi) * (g[0] + omega ** 2 * x) - np.sin(phi) * g[2]
    ref = orc.normal_gravity(r, colat)
    assert np.max(np.abs(gamma - ref) / np.abs(ref)) < 1e-14
    assert np.max(np.abs(g[1])) == 0.0


def test_cartesian_to_spherical():
    from grates_b200 import utilities
    R = 7e6
    pts = np.array([[R, 0, 0], [0, R, 0], [-R, 0, 0], [0, 0, R], [0, 0, -R], [-0.0, 0.0, R], [-0.0, -0.0, -R],
                    [1.0, 1.0, np.sqrt(2.0)]])
    r, colat, lon = utilities.cartesian_to_spherical(pts)
    np.testing.assert_allclose(r, [R] * 7 + [2.0], rtol=1e-15)
    np.testing.assert_allclose(colat, [np.pi / 2, np.pi / 2, np.pi / 2, 0, np.pi, 0, np.pi, np.pi / 4], rtol=1e-15)
    np.testing.assert_allclose(lon, [0, np.pi / 2, np.pi, 0, 0, 0, 0, np.pi / 4], rtol=1e-15)
    assert np.all(lon[3:7] == 0.0) and colat[3] == 0.0 and colat[4] == np.pi
    rng = np.random.default_rng(1)
    x = rng.standard_normal((100, 3)) * 7e6
    np.testing.assert_allclose(_to_cartesian(*utilities.cartesian_to_spherical(x)), x, rtol=0, atol=1e-8)
    for bad in ([[0.0, 0.0, 0.0]], [[np.nan, 0, 1]], [[np.inf, 0, 1]], np.zeros((3, 2)), np.zeros(3)):
        with pytest.raises(ValueError):
            utilities.cartesian_to_spherical(np.asarray(bad, dtype=float))


def test_argument_errors_come_before_any_device_call(monkeypatch):
    import torch
    import grates_b200 as gb
    from grates_b200 import plan

    def no_device(*args, **kwargs):
        raise AssertionError("a device was requested before the arguments were checked")
    monkeypatch.setattr(plan, "_current_device", no_device)
    anm = np.zeros((2, 5, 5))
    pos = np.array([[7e6, 0.0, 0.0]])
    with pytest.raises(ValueError, match="frame"):
        gb.gradient_batch(anm, frame='enu')
    with pytest.raises(ValueError, match="frame"):
        gb.gradient_at_positions(anm, pos, frame='ellipsoidal')
    for bad in (np.zeros((5, 5)), np.zeros((2, 5, 4))):
        with pytest.raises(ValueError, match="shape"):
            gb.gradient_batch(bad)
        with pytest.raises(ValueError, match="shape"):
            gb.gradient_at_positions(bad, pos)
    with pytest.raises(ValueError, match="float64 CUDA"):
        gb.gradient_batch(torch.zeros((2, 5, 5), dtype=torch.float64))
    with pytest.raises(ValueError, match="float64 CUDA"):
        gb.gradient_at_positions(torch.zeros((2, 5, 5), dtype=torch.float32), pos)
    for bad in (np.zeros((1, 3)), np.array([[np.nan, 0.0, 1.0]]), np.zeros((4, 2))):
        with pytest.raises(ValueError, match="positions"):
            gb.gradient_at_positions(anm, bad)


# ------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def gb():
    import grates_b200
    grates_b200._lib.require_device()
    return grates_b200


def _sample_rows(nlat, seed):
    """Both polar rows, the row(s) at the equator and 13 random rows."""
    eq = [nlat // 2] if nlat % 2 else [nlat // 2 - 1, nlat // 2]
    rest = np.setdiff1d(np.arange(nlat), [0, nlat - 1] + eq)
    return np.sort(np.concatenate(([0, nlat - 1], eq, np.random.default_rng(seed).choice(rest, 13, replace=False))))


def _grid_reference(orc, grid, X, rows):
    """Oracle gradient (Cartesian) on the sampled rows of a regular grid: [E, 3, rows, nlon], with (colat, lon) per point."""
    lat = np.asarray(grid.parallels)[rows]
    lon = np.asarray(grid.meridians)
    colat = np.repeat(orc.colatitude(lat), lon.size)
    r = np.repeat(orc.geocentric_radius(lat), lon.size)
    lon_p = np.tile(lon, lat.size)
    ref = gradient(orc, X, r, colat, lon_p)
    return ref.reshape(X.shape[0], 3, lat.size, lon.size), colat, lon_p


def _launches(gb, fn):
    lib = gb._lib.load()
    lib.gb_launch_count(1)
    out = fn()
    return int(lib.gb_launch_count(0)), out


@pytest.fixture(scope="module")
def half(gb, orc):
    """GeographicGrid(0.5), N = 96, 240 epochs: both frames on the device, the oracle on the sampled rows."""
    import torch
    grid = gb.GeographicGrid(0.5)
    X = _coefficients(240, N, 21)
    x = torch.as_tensor(X).cuda()
    cart = gb.gradient_batch(x, grid)
    local = gb.gradient_batch(x, grid, frame='local')
    rows = _sample_rows(grid.parallels.size, 5)
    ref, colat, lon = _grid_reference(orc, grid, X, rows)
    return {"grid": grid, "X": X, "x": x, "cart": cart, "local": local, "rows": rows, "ref": ref, "colat": colat,
            "lon": lon}


@pytest.mark.gpu
def test_transform_matches_oracle_bit_for_bit(gb, orc):
    import ctypes
    import torch
    lib = gb._lib.load()
    for nmax, E in ((N, 3), (1, 2), (0, 1)):
        X = _coefficients(E, nmax, 2)
        x = torch.as_tensor(X).cuda()
        g = torch.full((E, 3, nmax + 2, nmax + 2), float("nan"), dtype=torch.float64, device="cuda")
        gb._lib.check(lib.gb_gradient_coefficients(ctypes.c_void_p(x.data_ptr()), E, nmax, ctypes.c_void_p(g.data_ptr()),
                                                   0, None))
        assert torch.equal(g.cpu(), torch.as_tensor(gradient_coefficients(X))), nmax


@pytest.mark.gpu
def test_half_degree_grid_against_oracle(gb, half):
    """Production paths: the octant Fourier stage and the folded Legendre stage, 720 sets at degree 97."""
    p = gb.get_gradient_plan(half["grid"], N)
    assert p.octant and p.folded and p.max_degree == N + 1
    rows = half["rows"]
    cart = half["cart"][:, :, rows].cpu().numpy()
    err = _worst(cart, half["ref"])
    print("GRADERR half cartesian %.3e" % err)
    assert err < TOL
    E = half["X"].shape[0]
    ref_local = _to_local(half["ref"].reshape(E, 3, -1), half["colat"], half["lon"])
    err = _worst(half["local"][:, :, rows].cpu().numpy().reshape(E, 3, -1), ref_local)
    print("GRADERR half local %.3e" % err)
    assert err < TOL


@pytest.mark.gpu
def test_one_degree_and_gauss_grids_against_oracle(gb, orc):
    """The four-fold (not octant) Fourier stage on GeographicGrid(1.0), and GaussGrid(97); numpy in, numpy out."""
    import torch
    X = _coefficients(5, N, 8)
    for grid, octant in ((gb.GeographicGrid(1.0), False), (gb.GaussGrid(97), None)):
        p = gb.get_gradient_plan(grid, N)
        if octant is not None:
            assert p.symmetric and p.octant == octant
        rows = _sample_rows(grid.parallels.size, 6)
        ref, colat, lon = _grid_reference(orc, grid, X, rows)
        got = gb.gradient_batch(X, grid)
        assert isinstance(got, np.ndarray) and got.shape == (5, 3, grid.parallels.size, grid.meridians.size)
        err = _worst(got[:, :, rows], ref)
        print("GRADERR %s cartesian %.3e" % (type(grid).__name__, err))
        assert err < TOL
        out = np.empty((5, 3, grid.parallels.size, grid.meridians.size))
        local = gb.gradient_batch(X, grid, frame='local', out=out)
        assert local is out
        err = _worst(local[:, :, rows].reshape(5, 3, -1), _to_local(ref.reshape(5, 3, -1), colat, lon))
        print("GRADERR %s local %.3e" % (type(grid).__name__, err))
        assert err < TOL
        dev = gb.gradient_batch(torch.as_tensor(X).cuda(), grid)
        assert dev.is_cuda and np.array_equal(dev.cpu().numpy(), got)


@pytest.mark.gpu
def test_point_set_per_point_kernel_and_gemm(gb, orc):
    """The benchmark's 40 962 points: 1 epoch (3 sets, per-point kernel) and 17 epochs (51 sets, design-tile GEMM)."""
    import torch
    rng = np.random.default_rng(7)                                   # as bench_configs.point_sets
    lon, lat = rng.uniform(-np.pi, np.pi, NPTS), np.arcsin(rng.uniform(-1, 1, NPTS))
    grid = gb.IrregularGrid(lon, lat)
    sub = np.sort(np.concatenate((rng.choice(NPTS - 1, 1023, replace=False), [NPTS - 1])))
    colat, r = orc.colatitude(lat[sub]), orc.geocentric_radius(lat[sub])
    X = _coefficients(17, N, 9)
    ref = gradient(orc, X, r, colat, lon[sub])
    x = torch.as_tensor(X).cuda()
    gb.gradient_batch(x[:1], grid)                                   # plan creation outside the counted calls
    for E in (1, 17):
        n, got = _launches(gb, lambda: gb.gradient_batch(x[:E], grid))
        if E == 1:
            assert n == 2, n            # transform + the per-point synthesis kernel
        else:
            assert n >= 6 and n % 2 == 0, n      # transform + coefficient tiles + (design tiles, GEMM) per block, B >= 2
        assert got.shape == (E, 3, NPTS)
        err = _worst(got[:, :, sub].cpu().numpy(), ref[:E])
        print("GRADERR points E=%d cartesian %.3e" % (E, err))
        assert err < TOL
        n, got = _launches(gb, lambda: gb.gradient_batch(x[:E], grid, frame='local'))
        assert (n == 3) if E == 1 else (n >= 7 and n % 2 == 1), n
        err = _worst(got[:, :, sub].cpu().numpy(), _to_local(ref[:E], colat, lon[sub]))
        print("GRADERR points E=%d local %.3e" % (E, err))
        assert err < TOL


def _track(count, seed):
    """Earth-fixed positions of a seeded near-polar circular orbit at R + 490 km, one per second, and the two poles."""
    from oracle.sh_oracle import GM_DEFAULT, R_DEFAULT
    rng = np.random.default_rng(seed)
    a, inc, node, u0 = R_DEFAULT + 490e3, np.radians(89.0), rng.uniform(0, 2 * np.pi), rng.uniform(0, 2 * np.pi)
    t = np.arange(count, dtype=float)
    u = u0 + np.sqrt(GM_DEFAULT / a ** 3) * t
    lam = node - 7.292115e-5 * t                                     # node in the Earth-fixed frame
    xo, yo, zo = np.cos(u), np.sin(u) * np.cos(inc), np.sin(u) * np.sin(inc)
    pos = a * np.stack((xo * np.cos(lam) - yo * np.sin(lam), xo * np.sin(lam) + yo * np.cos(lam), zo), axis=1)
    return np.concatenate((pos, [[0.0, 0.0, a], [0.0, 0.0, -a]]))


@pytest.mark.gpu
def test_positions_on_an_orbit_against_oracle(gb, orc):
    import torch
    from grates_b200 import utilities
    pos = _track(86400, 4)
    P = pos.shape[0]
    r, colat, lon = utilities.cartesian_to_spherical(pos)
    assert colat[-2] == 0.0 and colat[-1] == np.pi and lon[-1] == 0.0
    sub = np.sort(np.concatenate((np.random.default_rng(5).choice(P - 2, 1022, replace=False), [P - 2, P - 1])))
    X = _coefficients(6, N, 10)
    ref = gradient(orc, X, r[sub], colat[sub], lon[sub])
    for E in (1, 6):
        for frame in ('cartesian', 'local'):
            got = gb.gradient_at_positions(torch.as_tensor(X[:E]).cuda(), pos, frame=frame)
            assert got.shape == (E, 3, P)
            want = ref[:E] if frame == 'cartesian' else _to_local(ref[:E], colat[sub], lon[sub])
            err = _worst(got[:, :, sub].cpu().numpy(), want)
            print("GRADERR orbit E=%d %s %.3e" % (E, frame, err))
            assert err < TOL


@pytest.mark.gpu
def test_up_and_east_equal_scalar_syntheses_over_the_whole_grid(gb, half):
    """up = dV/dr and east = dV/dlon / (r sin theta) through SHPlan syntheses of degree N with derivative degree factors,
    over every point of the 0.5 degree grid and all 240 epochs."""
    import torch
    from grates_b200 import utilities
    grid, X, local = half["grid"], half["X"], half["local"]
    a, f, GM, R = grid.semimajor_axis, grid.flattening, gb.gravityfield.GM_DEFAULT, gb.gravityfield.R_DEFAULT
    r = utilities.geocentric_radius(grid.parallels, a, f)
    colat = utilities.colatitude(grid.parallels, a, f)
    n = np.arange(N + 1)
    kn = np.power((R / r)[:, None], n + 1) * GM / R
    up_plan = gb.SHPlan(grid.meridians, grid.parallels, a, f, N, degree_factors=-(n + 1) / r[:, None] * kn)
    east_plan = gb.SHPlan(grid.meridians, grid.parallels, a, f, N, degree_factors=kn / (r * np.sin(colat))[:, None])
    L = N + 1
    Xe = np.zeros_like(X)
    for m in range(1, L):
        Xe[:, m:, m] = m * X[:, m - 1, m:]          # C' = m S
        Xe[:, m - 1, m:] = -m * X[:, m:, m]         # S' = -m C
    up = up_plan.synthesis(half["x"]).cpu().numpy()
    east = east_plan.synthesis(torch.as_tensor(Xe).cuda()).cpu().numpy()
    err_up = max(maxnorm_err(local[e, 2].cpu().numpy(), up[e]) for e in range(240))
    err_east = max(maxnorm_err(local[e, 0].cpu().numpy(), east[e]) for e in range(240))
    print("GRADERR full grid up %.3e east %.3e" % (err_up, err_east))
    assert err_up < TOL and err_east < TOL


@pytest.mark.gpu
def test_point_mass(gb):
    """C00 = 1 at N = 96: up = -GM/r^2, east = north = 0, on the 0.5 degree grid and along the orbit."""
    from grates_b200 import utilities
    GM = gb.gravityfield.GM_DEFAULT
    X = np.zeros((1, N + 1, N + 1))
    X[0, 0, 0] = 1.0
    grid = gb.GeographicGrid(0.5)
    g = gb.gradient_batch(X, grid, frame='local')[0]
    r = utilities.geocentric_radius(grid.parallels, grid.semimajor_axis, grid.flattening)[:, None]
    scale = GM / r ** 2
    assert np.max(np.abs(g[2] + scale) / scale) < 1e-14
    assert np.max(np.abs(g[:2]) / scale) < 1e-14
    pos = _track(86400, 4)
    g = gb.gradient_at_positions(X, pos, frame='local')[0]
    scale = GM / utilities.cartesian_to_spherical(pos)[0] ** 2
    assert np.max(np.abs(g[2] + scale) / scale) < 1e-14
    assert np.max(np.abs(g[:2]) / scale) < 1e-14


@pytest.mark.gpu
def test_epoch_slices_are_bit_identical_on_a_regular_grid(gb, half):
    """Rows [lo, hi) of the 240-epoch result equal a call on that slice bit for bit (the grid synthesis is
    batch-independent; transform and rotation are element-wise)."""
    import torch
    for lo, hi in ((100, 101), (57, 94)):
        for frame in ('cartesian', 'local'):
            part = gb.gradient_batch(half["x"][lo:hi], half["grid"], frame=frame)
            assert torch.equal(part, half[frame if frame == 'local' else 'cart'][lo:hi]), (lo, hi, frame)


@pytest.mark.gpu
def test_local_frame_rotates_back_to_cartesian(gb, half):
    """The local result rotated back with the transposed frame on the host equals the Cartesian result."""
    grid = half["grid"]
    from grates_b200 import utilities
    colat = utilities.colatitude(grid.parallels, grid.semimajor_axis, grid.flattening)[:, None]
    lon = np.asarray(grid.meridians)[None, :]
    ct, st, cl, sl = np.cos(colat), np.sin(colat), np.cos(lon), np.sin(lon)
    for e in (0, 119, 239):
        east, north, up = half["local"][e].cpu().numpy()
        back = np.stack((-sl * east - ct * cl * north + st * cl * up, cl * east - ct * sl * north + st * sl * up,
                         st * north + ct * up))
        cart = half["cart"][e].cpu().numpy()
        for c in range(3):
            assert maxnorm_err(back[c], cart[c]) < 1e-15, (e, c, maxnorm_err(back[c], cart[c]))


@pytest.mark.gpu
def test_gradient_plans_are_their_own_cache_entries(gb):
    grid = gb.GeographicGrid(2.0)
    g = gb.get_gradient_plan(grid, 30)
    assert g is gb.get_gradient_plan(grid, 30)
    assert g is not gb.get_plan(grid, 31, 'potential') and g is not gb.get_plan(grid, 30, 'potential')
    assert g.max_degree == 31 and tuple(g.frame.shape) == (4, grid.parallels.size * grid.meridians.size)
    assert g.kn[:, 0].max() == 0.0
