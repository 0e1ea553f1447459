"""Gravity gradient tensor (gravity_gradient_batch, gravity_gradient_at_positions): the coefficient transform of
Cunningham's relation applied twice, the degree-(N+2) synthesis of its 6E sets and the rotation Q V Q' to
(east, north, up).

The restatement is the one of test_gpu_gradient (gradient_coefficients) applied twice: component (a, b) is T_a(T_b(C)).
Without a GPU it is tied to the reference through that file's acceleration, which is tied to the oracle's potential and
to the reference's normal gravity: the tensor must be symmetric and trace-free coefficient by coefficient, equal central
differences of the restated acceleration, and give the point-mass tensor for C00 = 1.  Its local frame is tied to two
scalar syntheses of degree N (second radial derivative, radial derivative of the longitude derivative), which share no
code with the transform or the rotation; on the GPU those two run over every point and epoch of the 0.5 degree grid.
"""
import ctypes

import numpy as np
import pytest

from conftest import maxnorm_err
from test_gpu_gradient import (_coefficients, _launches, _sample_rows, _to_cartesian, _to_local, _track,
                               gradient, gradient_coefficients)

N = 96
NPTS = 40962               # the benchmark's point set (bench_configs.point_sets)
PAIRS = ((0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2))      # (a, b) of the six components xx, xy, xz, yy, yz, zz
# Largest max-normalised error per component a comparison with the restatement or the scalar syntheses may show: ten
# times the largest error an NVIDIA B200 (1000 W power limit) showed, 6.7e-14 (the 0.5 degree grid, local frame).
TOL = 7e-13
# Largest |trace| / max |V_zz| (|V_uu| in the local frame): ten times the largest the B200 showed, 8.9e-16.
TRACE_TOL = 1e-14
# Point mass, relative to GM / r^3: ten times the largest the B200 showed, 7.3e-15.
POINT_MASS_TOL = 8e-14


@pytest.fixture(scope="module")
def orc():
    from oracle import sh_oracle
    return sh_oracle


def tensor_coefficients(anm):
    """Restated transform: packed [..., L, L] -> [..., 6, L+2, L+2], component (a, b) = T_a(T_b(anm)) with T the
    restated acceleration transform (test_gpu_gradient.gradient_coefficients)."""
    h = gradient_coefficients(gradient_coefficients(anm))     # [..., b, a, L+2, L+2]
    return np.stack([h[..., b, a, :, :] for a, b in PAIRS], axis=-3)


def tensor(orc, anm, r, colat, lon, GM=None, R=None):
    """Restated tensor at geocentric (r, colat, lon), Earth-fixed: [E, 6, P] for anm [E, L, L].  Each component is the
    degree-(N+2) synthesis of tensor_coefficients with degree factors GM/R^3 (R/r)^(n''+1), from the oracle's tables,
    512 points at a time."""
    GM = orc.GM_DEFAULT if GM is None else GM
    R = orc.R_DEFAULT if R is None else R
    G = tensor_coefficients(np.asarray(anm, dtype=float))
    E, Lo = G.shape[0], G.shape[-1]
    r, colat, lon = (np.atleast_1d(np.asarray(v, dtype=float)) for v in (r, colat, lon))
    flat = G.reshape(E * 6, Lo * Lo)
    out = np.empty((E * 6, r.size))
    for i1 in range(0, r.size, 512):
        i2 = min(i1 + 512, r.size)
        kn = np.power((R / r[i1:i2])[:, None], np.arange(Lo, dtype=int) + 1) * (GM / R ** 3)
        kn[:, :2] = 0.0
        Y = orc._scale_packed_by_degree(orc.spherical_harmonics(Lo - 1, colat[i1:i2], lon[i1:i2]), kn)
        out[:, i1:i2] = flat @ Y.reshape(i2 - i1, Lo * Lo).T
    return out.reshape(E, 6, r.size)


def full_matrix(v):
    """[..., 6, P] upper triangle -> [..., 3, 3, P]"""
    xx, xy, xz, yy, yz, zz = (v[..., k, :] for k in range(6))
    return np.stack((np.stack((xx, xy, xz), -2), np.stack((xy, yy, yz), -2), np.stack((xz, yz, zz), -2)), -3)


def to_local(v, colat, lon):
    """Q V Q' of [..., 6, P] on the host in the operation order of gb_rotate_tensor_to_local: the rotation of
    test_gpu_gradient._to_local (the arithmetic of gb_rotate_to_local) on the three columns of V, then on the three rows
    of the result; the upper triangle (ee, en, eu, nn, nu, uu)."""
    M = full_matrix(v)                                         # [..., i, j, P]
    W = _to_local(np.swapaxes(M, -3, -2), colat, lon)          # columns: [..., j, i', P] = (Q V)[i', j]
    Z = _to_local(np.swapaxes(W, -3, -2), colat, lon)          # rows:    [..., i', j', P] = (Q V Q')[i', j']
    return np.stack([Z[..., a, b, :] for a, b in PAIRS], axis=-2)


def _worst(got, ref):
    """Largest max-normalised error over epochs and components of [E, 6, ...] arrays."""
    return max(maxnorm_err(got[e, c], ref[e, c]) for e in range(ref.shape[0]) for c in range(6))


def _trace(v):
    return v[:, 0] + v[:, 3] + v[:, 5]


# ------------------------------------------------------------------------------ CPU: the restatement and the host side
@pytest.mark.parametrize("nmax", [12, 40])
def test_restated_coefficients_are_symmetric_and_trace_free(nmax):
    """T_a T_b = T_b T_a and T_x T_x + T_y T_y + T_z T_z = 0 (Laplace), coefficient by coefficient."""
    anm = _coefficients(2, nmax, nmax)
    h = gradient_coefficients(gradient_coefficients(anm))
    scale = np.abs(h).max()
    for a in range(3):
        for b in range(3):
            assert np.abs(h[:, b, a] - h[:, a, b]).max() / scale < 2e-15, (a, b)
    assert np.abs(h[:, 0, 0] + h[:, 1, 1] + h[:, 2, 2]).max() / scale < 2e-15
    assert np.all(h[..., :2, :2] == 0.0)                      # degrees 0 and 1


@pytest.mark.parametrize("nmax", [12, 40])
def test_restated_tensor_matches_finite_differences_of_the_acceleration(orc, nmax):
    """Central differences (10 m steps) of the restated acceleration along x, y and z, from the surface to 500 km, with
    two points within 1e-6 rad of the poles."""
    from grates_b200 import utilities
    rng = np.random.default_rng(nmax + 1)
    anm = _coefficients(1, nmax, nmax)
    P = 40
    r = orc.R_DEFAULT + rng.uniform(0.0, 500e3, P)
    colat = np.arccos(rng.uniform(-1.0, 1.0, P))
    lon = rng.uniform(-np.pi, np.pi, P)
    colat[0], colat[1] = 3e-7, np.pi - 5e-7
    V = full_matrix(tensor(orc, anm, r, colat, lon))[0]
    x = _to_cartesian(r, colat, lon)
    h = 10.0
    for k in range(3):
        step = np.zeros(3)
        step[k] = h
        fd = (gradient(orc, anm[0], *utilities.cartesian_to_spherical(x + step)) -
              gradient(orc, anm[0], *utilities.cartesian_to_spherical(x - step))) / (2 * h)
        for a in range(3):
            assert maxnorm_err(V[k, a], fd[a]) < 1e-8, (k, a, maxnorm_err(V[k, a], fd[a]))   # 1.2e-9 at most


def _point_mass_reference(GM, pos):
    r = np.linalg.norm(pos, axis=1)
    x = pos.T
    return GM * (3 * x[:, None] * x[None, :] - r ** 2 * np.eye(3)[:, :, None]) / r ** 5, GM / r ** 3


def test_restated_point_mass_is_the_closed_form(orc):
    """C00 = 1: V = GM (3 x x' - r^2 I) / r^5."""
    from grates_b200 import utilities
    anm = np.zeros((1, 5, 5))
    anm[0, 0, 0] = 1.0
    rng = np.random.default_rng(2)
    pos = _to_cartesian(orc.R_DEFAULT + rng.uniform(0, 500e3, 30), np.arccos(rng.uniform(-1, 1, 30)),
                        rng.uniform(-np.pi, np.pi, 30))
    V = full_matrix(tensor(orc, anm, *utilities.cartesian_to_spherical(pos)))[0]
    ref, scale = _point_mass_reference(orc.GM_DEFAULT, pos)
    assert np.max(np.abs(V - ref) / scale) < 1e-14


def _radial_syntheses(orc, anm, r, colat, degree_synthesis):
    """V_uu = sum (n+1)(n+2)/r^2 kn V_n and V_eu = -sum (n+2) kn / (r^2 sin theta) dV_n/dlon, kn = GM/R (R/r)^(n+1),
    through degree_synthesis(coefficients, factors [P, L]) of degree N."""
    GM, R = orc.GM_DEFAULT, orc.R_DEFAULT
    n = np.arange(anm.shape[-1])
    kn = np.power((R / r)[:, None], n + 1) * GM / R
    Xe = np.zeros_like(anm)
    for m in range(1, anm.shape[-1]):
        Xe[..., m:, m] = m * anm[..., m - 1, m:]      # C' = m S
        Xe[..., m - 1, m:] = -m * anm[..., m:, m]     # S' = -m C
    uu = degree_synthesis(anm, (n + 1) * (n + 2) / r[:, None] ** 2 * kn)
    eu = degree_synthesis(Xe, -(n + 2) * kn / (r ** 2 * np.sin(colat))[:, None])
    return uu, eu


def test_restated_local_frame_matches_radial_syntheses(orc):
    """V_uu and V_eu of the restated tensor rotated on the host against the two scalar syntheses of degree N."""
    rng = np.random.default_rng(4)
    P, nmax = 50, 40
    anm = _coefficients(2, nmax, 3)
    r = orc.R_DEFAULT + rng.uniform(0, 500e3, P)
    colat, lon = np.arccos(rng.uniform(-1, 1, P)), rng.uniform(-np.pi, np.pi, P)
    local = to_local(tensor(orc, anm, r, colat, lon), colat, lon)

    def synth(X, factors):
        Y = orc._scale_packed_by_degree(orc.spherical_harmonics(nmax, colat, lon), factors)
        return X.reshape(X.shape[0], -1) @ Y.reshape(P, -1).T
    uu, eu = _radial_syntheses(orc, anm, r, colat, synth)
    for e in range(2):
        assert maxnorm_err(local[e, 5], uu[e]) < 1e-13
        assert maxnorm_err(local[e, 2], eu[e]) < 1e-13
        assert np.abs(_trace(local)[e]).max() / np.abs(local[e, 5]).max() < 1e-14


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
        gb.gravity_gradient_batch(anm, frame='enu')
    with pytest.raises(ValueError, match="frame"):
        gb.gravity_gradient_at_positions(anm, pos, frame='lnof')
    for bad in (np.zeros((5, 5)), np.zeros((2, 5, 4))):
        with pytest.raises(ValueError, match="shape"):
            gb.gravity_gradient_batch(bad)
        with pytest.raises(ValueError, match="shape"):
            gb.gravity_gradient_at_positions(bad, pos)
    with pytest.raises(ValueError, match="float64 CUDA"):
        gb.gravity_gradient_batch(torch.zeros((2, 5, 5), dtype=torch.float64))
    with pytest.raises(ValueError, match="float64 CUDA"):
        gb.gravity_gradient_at_positions(torch.zeros((2, 5, 5), dtype=torch.float32), pos)
    with pytest.raises(TypeError, match="grid"):
        gb.gravity_gradient_batch(anm, grid=object())
    for bad in (np.zeros((1, 3)), np.array([[np.nan, 0.0, 1.0]]), np.array([[np.inf, 0.0, 1.0]]), np.zeros((4, 2))):
        with pytest.raises(ValueError, match="positions"):
            gb.gravity_gradient_at_positions(anm, bad)


# ------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def gb():
    import grates_b200
    grates_b200._lib.require_device()
    return grates_b200


def _call(lib, name, *args):
    from grates_b200 import _lib
    _lib.check(getattr(lib, name)(*args))


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


@pytest.mark.gpu
def test_transform_is_the_two_call_composition_bit_for_bit(gb):
    """gb_gravity_gradient_coefficients against gb_gradient_coefficients applied twice (element [b][a] of the second
    call's [3E][3] output), bit for bit, and against the numpy restatement; NaN-filled outputs show every element is
    written."""
    import torch
    lib = gb._lib.load()
    for nmax, E in ((N, 11), (1, 2), (0, 1)):
        X = _coefficients(E, nmax, 2)
        x = torch.as_tensor(X).cuda()
        L = nmax + 1
        g1 = torch.full((E, 3, L + 1, L + 1), float("nan"), dtype=torch.float64, device="cuda")
        g2 = torch.full((E, 3, 3, L + 2, L + 2), float("nan"), dtype=torch.float64, device="cuda")
        out = torch.full((E, 6, L + 2, L + 2), float("nan"), dtype=torch.float64, device="cuda")
        _call(lib, "gb_gradient_coefficients", _ptr(x), E, nmax, _ptr(g1), 0, None)
        _call(lib, "gb_gradient_coefficients", _ptr(g1), 3 * E, nmax + 1, _ptr(g2), 0, None)
        _call(lib, "gb_gravity_gradient_coefficients", _ptr(x), E, nmax, _ptr(out), 0, None)
        composed = torch.stack([g2[:, b, a] for a, b in PAIRS], dim=1)
        assert torch.equal(out.view(torch.int64), composed.view(torch.int64)), nmax
        assert torch.equal(out.cpu(), torch.as_tensor(tensor_coefficients(X))), nmax
        assert torch.all(out[:, :, :2, :2] == 0.0)


@pytest.mark.gpu
def test_transform_argument_checks(gb):
    import torch
    lib = gb._lib.load()
    x = torch.zeros((1, 4, 4), dtype=torch.float64, device="cuda")
    out = torch.zeros((1, 6, 6, 6), dtype=torch.float64, device="cuda")
    assert lib.gb_gravity_gradient_coefficients(_ptr(x), 0, 3, None, 0, None) == 0          # 0 sets: no-op
    for args in ((_ptr(x), -1, 3, _ptr(out)), (_ptr(x), 1, -1, _ptr(out)), (None, 1, 3, _ptr(out)),
                 (_ptr(x), 1, 3, None), (_ptr(x), 1, 8192, _ptr(out)), (_ptr(x), 65535 * 8 + 1, 3, _ptr(out))):
        assert lib.gb_gravity_gradient_coefficients(*args, 0, None) == gb._lib.GB_ERR_ARGUMENT, args
    frame = torch.zeros((4, 6), dtype=torch.float64, device="cuda")
    v = torch.zeros((1, 6, 6), dtype=torch.float64, device="cuda")
    assert lib.gb_rotate_tensor_to_local(_ptr(v), _ptr(frame), 0, 6, 0, None) == 0
    for args in ((_ptr(v), _ptr(frame), -1, 6), (_ptr(v), _ptr(frame), 1, -6), (None, _ptr(frame), 1, 6),
                 (_ptr(v), None, 1, 6)):
        assert lib.gb_rotate_tensor_to_local(*args, 0, None) == gb._lib.GB_ERR_ARGUMENT, args


def _grid_reference(orc, grid, X, rows):
    """Restated tensor (Cartesian) on the sampled rows of a regular grid: [E, 6, rows * nlon], with (colat, lon)."""
    lat = np.asarray(grid.parallels)[rows]
    lon = np.asarray(grid.meridians)
    colat = np.repeat(orc.colatitude(lat), lon.size)
    r = np.repeat(orc.geocentric_radius(lat), lon.size)
    lon_p = np.tile(lon, lat.size)
    return tensor(orc, X, r, colat, lon_p), colat, lon_p


@pytest.fixture(scope="module")
def half(gb, orc):
    """GeographicGrid(0.5), N = 96, 240 epochs (1440 sets at degree 98): both frames on the device, the restatement on
    the sampled rows."""
    import torch
    grid = gb.GeographicGrid(0.5)
    X = _coefficients(240, N, 31)
    x = torch.as_tensor(X).cuda()
    cart = gb.gravity_gradient_batch(x, grid)
    local = gb.gravity_gradient_batch(x, grid, frame='local')
    rows = _sample_rows(grid.parallels.size, 7)
    ref, colat, lon = _grid_reference(orc, grid, X, rows)
    return {"grid": grid, "X": X, "x": x, "cart": cart, "local": local, "rows": rows, "ref": ref, "colat": colat,
            "lon": lon}


def _rows(v, rows):
    E = v.shape[0]
    return v[:, :, rows].cpu().numpy().reshape(E, 6, -1)


@pytest.mark.gpu
def test_half_degree_grid_against_restatement(gb, half):
    """Production paths: the octant Fourier stage and the folded Legendre stage, 1440 sets at degree 98."""
    p = gb.get_gravity_gradient_plan(half["grid"], N)
    assert p.octant and p.folded and p.max_degree == N + 2
    assert half["cart"].shape == (240, 6, half["grid"].parallels.size, half["grid"].meridians.size)
    err = _worst(_rows(half["cart"], half["rows"]), half["ref"])
    print("GGERR half cartesian %.3e" % err)
    assert err < TOL
    err = _worst(_rows(half["local"], half["rows"]), to_local(half["ref"], half["colat"], half["lon"]))
    print("GGERR half local %.3e" % err)
    assert err < TOL


@pytest.mark.gpu
def test_rotation_is_the_restated_operation_order_bit_for_bit(gb, half):
    """The local result equals the Cartesian one rotated on the host in the kernel's operation order, bit for bit, on
    the sampled rows; rotated back with Q' on the host it equals the Cartesian result to rounding.  An odd point count
    takes the one-point-per-thread kernel."""
    import torch
    E = 240
    cart, local = _rows(half["cart"], half["rows"]), _rows(half["local"], half["rows"])
    assert np.array_equal(to_local(cart, half["colat"], half["lon"]), local)
    ct, st, cl, sl = (f(v) for f, v in ((np.cos, half["colat"]), (np.sin, half["colat"]), (np.cos, half["lon"]),
                                        (np.sin, half["lon"])))
    Q = np.array([[-sl, cl, 0 * sl], [-ct * cl, -ct * sl, st], [st * cl, st * sl, ct]])
    back = np.einsum('kip,eklp,ljp->eijp', Q, full_matrix(local), Q)
    ref = full_matrix(cart)
    for e in (0, 119, 239):
        for a, b in PAIRS:
            assert maxnorm_err(back[e, a, b], ref[e, a, b]) < 1e-14, (e, a, b)
    # the scalar kernel: 1001 points, and a value pointer that is not 16-byte aligned
    lib = gb._lib.load()
    rng = np.random.default_rng(3)
    P = 1001
    colat, lon = np.arccos(rng.uniform(-1, 1, P)), rng.uniform(-np.pi, np.pi, P)
    frame = torch.as_tensor(np.stack((np.cos(colat), np.sin(colat), np.cos(lon), np.sin(lon)))).cuda()
    V = rng.standard_normal((9, 6, P))
    for offset in (0, 1):
        buf = torch.as_tensor(np.concatenate((np.zeros(offset), V.ravel()))).cuda()
        v = buf[offset:]
        _call(lib, "gb_rotate_tensor_to_local", _ptr(v), _ptr(frame), 9, P, 0, None)
        assert np.array_equal(v.cpu().numpy().reshape(9, 6, P), to_local(V, colat, lon)), offset
    # the two-point kernel on an even count outside the grid
    v = torch.as_tensor(V[:, :, :1000].copy()).cuda()
    fr = torch.as_tensor(np.ascontiguousarray(frame.cpu().numpy()[:, :1000])).cuda()
    _call(lib, "gb_rotate_tensor_to_local", _ptr(v), _ptr(fr), 9, 1000, 0, None)
    assert np.array_equal(v.cpu().numpy(), to_local(V[:, :, :1000], colat[:1000], lon[:1000]))


@pytest.mark.gpu
def test_uu_and_eu_equal_scalar_syntheses_over_the_whole_grid(gb, half):
    """V_uu and V_eu through SHPlan syntheses of degree N with derivative degree factors, over every point of the
    0.5 degree grid and all 240 epochs; the trace in both frames relative to max |V_zz| / |V_uu|."""
    import torch
    from grates_b200 import utilities
    from oracle import sh_oracle as orc
    grid, X, local, cart = half["grid"], half["X"], half["local"], half["cart"]
    a, f = grid.semimajor_axis, grid.flattening
    r = utilities.geocentric_radius(grid.parallels, a, f)
    colat = utilities.colatitude(grid.parallels, a, f)

    def synth(C, factors):
        plan = gb.SHPlan(grid.meridians, grid.parallels, a, f, N, degree_factors=factors)
        return plan.synthesis(torch.as_tensor(C).cuda())
    uu, eu = _radial_syntheses(orc, X, r, colat, synth)

    def err(got, ref):
        d = (got - ref).abs().amax(dim=(1, 2)) / ref.abs().amax(dim=(1, 2))
        return float(d.max())
    err_uu, err_eu = err(local[:, 5], uu), err(local[:, 2], eu)
    print("GGERR full grid uu %.3e eu %.3e" % (err_uu, err_eu))
    assert err_uu < TOL and err_eu < TOL
    for name, v, ref in (("cartesian", cart, cart[:, 5]), ("local", local, local[:, 5])):
        tr = float(((v[:, 0] + v[:, 3] + v[:, 5]).abs().amax(dim=(1, 2)) / ref.abs().amax(dim=(1, 2))).max())
        print("GGERR full grid trace %s %.3e" % (name, tr))
        assert tr < TRACE_TOL


@pytest.mark.gpu
def test_epoch_slices_are_bit_identical_on_a_regular_grid(gb, half):
    import torch
    for lo, hi in ((100, 101), (57, 94)):
        for frame in ('cartesian', 'local'):
            part = gb.gravity_gradient_batch(half["x"][lo:hi], half["grid"], frame=frame)
            assert torch.equal(part, half["local" if frame == 'local' else "cart"][lo:hi]), (lo, hi, frame)


@pytest.mark.gpu
def test_one_degree_and_gauss_grids_against_restatement(gb, orc):
    """The four-fold (not octant) Fourier stage on GeographicGrid(1.0), and GaussGrid(97); numpy in, numpy out, out=."""
    import torch
    X = _coefficients(5, N, 8)
    for grid, octant in ((gb.GeographicGrid(1.0), False), (gb.GaussGrid(97), None)):
        p = gb.get_gravity_gradient_plan(grid, N)
        if octant is not None:
            assert p.symmetric and p.octant == octant
        shape = (5, 6, grid.parallels.size, grid.meridians.size)
        rows = _sample_rows(grid.parallels.size, 6)
        ref, colat, lon = _grid_reference(orc, grid, X, rows)
        got = gb.gravity_gradient_batch(X, grid)
        assert isinstance(got, np.ndarray) and got.shape == shape
        err = _worst(got[:, :, rows].reshape(5, 6, -1), ref)
        print("GGERR %s cartesian %.3e" % (type(grid).__name__, err))
        assert err < TOL
        out = np.empty(shape)
        local = gb.gravity_gradient_batch(X, grid, frame='local', out=out)
        assert local is out
        err = _worst(local[:, :, rows].reshape(5, 6, -1), to_local(ref, colat, lon))
        print("GGERR %s local %.3e" % (type(grid).__name__, err))
        assert err < TOL
        dev = gb.gravity_gradient_batch(torch.as_tensor(X).cuda(), grid)
        assert dev.is_cuda and np.array_equal(dev.cpu().numpy(), got)
        res = torch.empty(shape, dtype=torch.float64, device="cuda")
        assert gb.gravity_gradient_batch(X, grid, device_output=True, out=res) is res
        assert np.array_equal(res.cpu().numpy(), got)
        with pytest.raises(ValueError):
            gb.gravity_gradient_batch(X, grid, out=np.empty((5, 3) + shape[2:]))


@pytest.mark.gpu
def test_point_set_per_point_kernel_and_gemm(gb, orc):
    """The benchmark's 40 962 points: 1 epoch (6 sets, per-point kernel) and 17 epochs (102 sets, design-tile GEMM);
    each call is the transform, one synthesis of the 6E sets and, for the local frame, one rotation."""
    import torch
    from grates_b200 import utilities
    rng = np.random.default_rng(7)                                   # as bench_configs.point_sets
    lon, lat = rng.uniform(-np.pi, np.pi, NPTS), np.arcsin(rng.uniform(-1, 1, NPTS))
    grid = gb.IrregularGrid(lon, lat)
    sub = np.sort(np.concatenate((rng.choice(NPTS - 1, 1023, replace=False), [NPTS - 1])))
    colat, r = orc.colatitude(lat[sub]), orc.geocentric_radius(lat[sub])
    X = _coefficients(17, N, 9)
    ref = tensor(orc, X, r, colat, lon[sub])
    x = torch.as_tensor(X).cuda()
    gb.gravity_gradient_batch(x[:1], grid)                           # plan creation outside the counted calls
    a, f = grid.semimajor_axis, grid.flattening
    p = gb.get_gravity_gradient_points_plan(utilities.geocentric_radius(lat, a, f), utilities.colatitude(lat, a, f), lon,
                                            N)                      # the plan of the call, from the cache
    for E in (1, 17):
        sets = torch.zeros((6 * E, N + 3, N + 3), dtype=torch.float64, device="cuda")
        n_syn, _ = _launches(gb, lambda: p.synthesis(sets))
        n, got = _launches(gb, lambda: gb.gravity_gradient_batch(x[:E], grid))
        assert n == n_syn + 1, (E, n, n_syn)
        if E == 1:
            assert n_syn == 1
        assert got.shape == (E, 6, NPTS)
        err = _worst(got[:, :, sub].cpu().numpy(), ref[:E])
        print("GGERR points E=%d cartesian %.3e" % (E, err))
        assert err < TOL
        n, got = _launches(gb, lambda: gb.gravity_gradient_batch(x[:E], grid, frame='local'))
        assert n == n_syn + 2, (E, n, n_syn)
        err = _worst(got[:, :, sub].cpu().numpy(), to_local(ref[:E], colat, lon[sub]))
        print("GGERR points E=%d local %.3e" % (E, err))
        assert err < TOL


@pytest.mark.gpu
def test_launch_counts_on_the_half_degree_grid(gb, half):
    """Cartesian: one synthesis of the 6E sets on the plan plus the transform; local: plus the rotation."""
    import torch
    p = gb.get_gravity_gradient_plan(half["grid"], N)
    x = half["x"][:30]
    sets = torch.zeros((180, N + 3, N + 3), dtype=torch.float64, device="cuda")
    n_syn, _ = _launches(gb, lambda: p.synthesis(sets))
    n_cart, _ = _launches(gb, lambda: gb.gravity_gradient_batch(x, half["grid"]))
    n_local, _ = _launches(gb, lambda: gb.gravity_gradient_batch(x, half["grid"], frame='local'))
    assert n_cart == n_syn + 1 and n_local == n_cart + 1, (n_syn, n_cart, n_local)


@pytest.mark.gpu
def test_positions_on_an_orbit_against_restatement(gb, orc):
    import torch
    from grates_b200 import utilities
    pos = _track(86400, 4)
    P = pos.shape[0]
    r, colat, lon = utilities.cartesian_to_spherical(pos)
    assert colat[-2] == 0.0 and colat[-1] == np.pi
    sub = np.sort(np.concatenate((np.random.default_rng(5).choice(P - 2, 1022, replace=False), [P - 2, P - 1])))
    X = _coefficients(6, N, 10)
    ref = tensor(orc, X, r[sub], colat[sub], lon[sub])
    for E in (1, 6):
        for frame in ('cartesian', 'local'):
            got = gb.gravity_gradient_at_positions(torch.as_tensor(X[:E]).cuda(), pos, frame=frame)
            assert got.shape == (E, 6, P)
            want = ref[:E] if frame == 'cartesian' else to_local(ref[:E], colat[sub], lon[sub])
            err = _worst(got[:, :, sub].cpu().numpy(), want)
            print("GGERR orbit E=%d %s %.3e" % (E, frame, err))
            assert err < TOL


@pytest.mark.gpu
def test_point_mass(gb):
    """C00 = 1 at N = 96: uu = 2GM/r^3, ee = nn = -GM/r^3, off-diagonal 0, on the 0.5 degree grid and along the orbit;
    Cartesian against GM (3 x x' - r^2 I) / r^5 along the orbit."""
    from grates_b200 import utilities
    GM = gb.gravityfield.GM_DEFAULT
    X = np.zeros((1, N + 1, N + 1))
    X[0, 0, 0] = 1.0

    def check(v, r):
        s = GM / r ** 3
        errs = (np.max(np.abs(v[5] - 2 * s) / s), np.max(np.abs(v[0] + s) / s), np.max(np.abs(v[3] + s) / s),
                max(np.max(np.abs(v[k]) / s) for k in (1, 2, 4)))
        print("GGERR point mass uu %.3e ee %.3e nn %.3e off-diagonal %.3e" % errs)
        assert max(errs) < POINT_MASS_TOL
    grid = gb.GeographicGrid(0.5)
    check(gb.gravity_gradient_batch(X, grid, frame='local')[0],
          utilities.geocentric_radius(grid.parallels, grid.semimajor_axis, grid.flattening)[:, None])
    pos = _track(86400, 4)
    r = utilities.cartesian_to_spherical(pos)[0]
    check(gb.gravity_gradient_at_positions(X, pos, frame='local')[0], r)
    cart = full_matrix(gb.gravity_gradient_at_positions(X, pos))
    ref, scale = _point_mass_reference(GM, pos)
    err = np.max(np.abs(cart[0] - ref) / scale)
    print("GGERR point mass orbit cartesian %.3e" % err)
    assert err < POINT_MASS_TOL


@pytest.mark.gpu
def test_gravity_gradient_plans_are_their_own_cache_entries(gb):
    grid = gb.GeographicGrid(2.0)
    g = gb.get_gravity_gradient_plan(grid, 30)
    assert g is gb.get_gravity_gradient_plan(grid, 30)
    assert g is not gb.get_gradient_plan(grid, 31) and g.max_degree == gb.get_gradient_plan(grid, 31).max_degree
    assert g is not gb.get_plan(grid, 32, 'potential') and g is not gb.get_plan(grid, 30, 'potential')
    assert g.max_degree == 32 and tuple(g.frame.shape) == (4, grid.parallels.size * grid.meridians.size)
    assert np.all(g.kn[:, :2] == 0.0) and np.all(g.kn[:, 2:] > 0.0)
    rng = np.random.default_rng(1)
    r, colat, lon = 7e6 + rng.uniform(0, 1e5, 10), rng.uniform(0, np.pi, 10), rng.uniform(-np.pi, np.pi, 10)
    pp = gb.get_gravity_gradient_points_plan(r, colat, lon, 30)
    assert pp is gb.get_gravity_gradient_points_plan(r, colat, lon, 30)
    assert pp is not gb.get_gradient_points_plan(r, colat, lon, 31)
    assert pp.max_degree == 32 and tuple(pp.frame.shape) == (4, 10) and np.all(pp.kn[:, :2] == 0.0)
