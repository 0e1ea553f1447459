"""Normal equations and adjoint of gravity-gradient observations at orbit positions
(gravity_gradient_normal_equations_at_positions, gravity_gradient_adjoint_at_positions): N = J~' W J~, n = J~' W l and
the transpose of ``gravity_gradient_at_positions``, with J~_p the Jacobian of the six components V_ab = F''_p T_a T_b x
of the tensor in the observations' frame.

The references reuse the host restatements of test_gpu_gravity_gradient.py (the tensor, its rotation to the local
frame), test_gpu_gradient_covariance.py (the transform T as sparse matrices) and test_gpu_gradient_normals.py.  Without a
GPU the Jacobian rows F''_p T_a^(N+1) T_b^(N) are tied to the restated tensor, the restated composed transpose to the
dense transpose of the sparse transforms, and the restated transposed rotation to the forward rotation through the
dot-product identity.  On the GPU:

  - the dot-product identity <G x, y> = <x, G' y> at 86 402 orbit positions, degree 96, both frames, 1 and 6 sets;
  - gb_gravity_gradient_coefficients_adjoint and gb_rotate_tensor_from_local bit for bit against their restatements;
  - Laplace's equation through the transpose: the adjoint of V_xx = V_yy = V_zz = y is zero to rounding;
  - N, n, l'Wl and the count against the restated Jacobian (degree 30, 2 000 positions, random weights with zeros,
    both frames, min_degree 0 and 2);
  - a closed loop at degree 96: noiseless observations of a Kaula-scaled field at 20 000 positions are solved back, and
    the forward operator applied to the columns of L^-T (N = L L') gives sum_pc w_pc (J~_pc L^-T)^2 = K';
  - invariants and edges: the frames agree for weights w_p (1, 2, 2, 1, 2, 1), N is exactly symmetric, two point blocks
    in one C call equal two calls, the chunked Python path agrees with one chunk, repeated calls are bit-identical, and
    the C ABI refuses bad arguments without writing.
"""
import ctypes

import numpy as np
import pytest

from test_gpu_gradient import _coefficients, _track
from test_gpu_gradient_covariance import _transform_matrices
from test_gpu_gradient_normals import _kaula, _positions, _sym_err
from test_gpu_gravity_gradient import PAIRS, full_matrix, tensor, to_local

N = 96
# Largest error each comparison may show: ten times the largest error an NVIDIA B200 (1000 W power limit) showed for it.
TOL_DOT = 1.9e-16          # |<G x, y> - <x, G' y>| / (|G x| |y|) (observed up to 1.8e-17)
TOL_LAPLACE = 2.9e-15      # |G'(y, 0, 0, y, 0, y)| / max (|G'_xx y| + |G'_yy y| + |G'_zz y|) (2.8e-16)
TOL_N = 9.4e-14            # N against the restated Jacobian, |dN_ab| / sqrt(N_aa N_bb) (9.3e-15)
TOL_RHS = 7.4e-16          # n against the restated Jacobian, |dn_a| / sqrt(N_aa l'Wl) (7.3e-17)
TOL_LPL = 1.6e-15          # l'Wl, relative (1.59e-16)
TOL_SOLVE = 2.4e-14        # closed loop: recovered coefficients, max-normalised (2.4e-15)
TOL_TRACE = 1.9e-15        # closed loop: sum_pc w_pc (J~_pc L^-T)^2 against K', relative (1.9e-16)
TOL_FRAME = 2.4e-13        # N local against N cartesian for weights w_p (1, 2, 2, 1, 2, 1) (2.4e-14)
TOL_CHUNK_N = 8.8e-14      # chunked against one chunk: N as for TOL_N (8.7e-15)
TOL_CHUNK = 1.9e-15        # chunked against one chunk: n as for TOL_RHS, l'Wl relative (1.8e-16)
EXACT_TOL = 1e-14          # float64 restated N entries against their extended-precision sums
BLOCK_30 = 8192            # points per block of gb_points_gravity_gradient_normals at degree 30 (at most 8192)


@pytest.fixture(scope="module")
def orc():
    from oracle import sh_oracle
    return sh_oracle


# ------------------------------------------------------------------------------ host restatements
def _terms(c, n, m, s):
    """gbgrad::grad_terms: the outputs (f, m', s') at degree n + 1 that component c of the input (n, m, s) reaches, the
    fp / fz term first, with the factors of the kernel in its expression order."""
    q = (2.0 * n + 1.0) / (2.0 * n + 3.0)
    if c == 2:
        return [(-np.sqrt(float((n - m + 1) * (n + m + 1)) * q), m, s)]
    fp = np.sqrt(float((n + m + 1) * (n + m + 2)) * q) * 0.5
    fp = fp * np.sqrt(2.0) if m == 0 else fp

    def fm():
        f = np.sqrt(float((n - m + 1) * (n - m + 2)) * q) * 0.5
        return f * np.sqrt(2.0) if m == 1 else f
    if c == 0:
        return [(-fp, m + 1, s)] + ([(fm(), m - 1, s)] if m >= 1 and (s == 0 or m >= 2) else [])
    if s == 0:
        return [(-fp, m + 1, 1)] + ([(-fm(), m - 1, 1)] if m >= 2 else [])
    return [(fp, m + 1, 0), (fm(), m - 1, 0)]


def _apply(terms, x):
    """gbgrad::apply: f1 x1 (+ f2 x2), each product and sum rounded on its own."""
    v = terms[0][0] * x(*terms[0][1:])
    if len(terms) > 1:
        v = v + terms[1][0] * x(*terms[1][1:])
    return v


def _apply_pair(a, b, n, m, s, x):
    """gbgrad::apply_pair: the terms of T_b at degree n, each of them the terms of T_a at degree n + 1 of x at n + 2."""
    return _apply(_terms(b, n, m, s), lambda mp, sp: _apply(_terms(a, n + 1, mp, sp), x))


def gravity_gradient_coefficients_adjoint(g):
    """numpy restatement of gb_gravity_gradient_coefficients_adjoint: [..., 6, L+2, L+2] (xx .. zz) -> [..., L, L]
    packed; per input (n, m, s) the composed terms of each pair read degree n + 2, added in the order xx .. zz."""
    g = np.asarray(g, dtype=float)
    L = g.shape[-1] - 2
    out = np.zeros(g.shape[:-3] + (L, L))
    for n in range(L):
        for m in range(n + 1):
            for s in ((0, 1) if m > 0 else (0,)):
                v = np.zeros(g.shape[:-3])
                for k, (a, b) in enumerate(PAIRS):
                    v = v + _apply_pair(a, b, n, m, s, lambda mp, sp, k=k: g[..., k, mp - 1, n + 2] if sp else
                                        g[..., k, n + 2, mp])
                if s:
                    out[..., m - 1, n] = v
                else:
                    out[..., n, m] = v
    return out


def _from_local(g, colat, lon):
    """[.., 3, P] (east, north, up) -> Q' g, the arithmetic of gbgrad::rotate_back, on the host."""
    ct, st, cl, sl = np.cos(colat), np.sin(colat), np.cos(lon), np.sin(lon)
    e, n, u = g[..., 0, :], g[..., 1, :], g[..., 2, :]
    return np.stack((-sl * e + -ct * cl * n + st * cl * u, cl * e + -ct * sl * n + st * sl * u, st * n + ct * u),
                    axis=-2)


def from_local(v, colat, lon):
    """numpy restatement of gb_rotate_tensor_from_local on [..., 6, P], the transpose of to_local on 6-vectors: the
    off-diagonal inputs halved, Q' on the three columns of the symmetric matrix, then on the three rows of the result,
    and the off-diagonal entries of the upper triangle doubled."""
    h = np.array(v, dtype=float, copy=True)
    h[..., (1, 2, 4), :] *= 0.5
    M = full_matrix(h)
    W = _from_local(np.swapaxes(M, -3, -2), colat, lon)
    Z = _from_local(np.swapaxes(W, -3, -2), colat, lon)
    out = np.stack([Z[..., a, b, :] for a, b in PAIRS], axis=-2)
    out[..., (1, 2, 4), :] *= 2.0
    return out


def _composed(T0, T1):
    """The six dense products T_a^(N+1) T_b^(N) [(N+3)^2, (N+1)^2], degree-wise, in the order xx .. zz."""
    return [(T1[a] @ T0[b]).toarray() for a, b in PAIRS]


def _jacobian(orc, TT, r, colat, lon, nmin, GM=None, R=None):
    """J [P, 6, K'] of the tensor at geocentric (r, colat, lon), Earth-fixed: the oracle's degree-(N+2) synthesis rows F''
    with the factors GM/R^3 (R/r)^(n''+1), times T_a T_b (columns from nmin^2 on)."""
    GM = orc.GM_DEFAULT if GM is None else GM
    R = orc.R_DEFAULT if R is None else R
    Lo = int(round(np.sqrt(TT[0].shape[0])))
    kn = np.power((R / r)[:, None], np.arange(Lo, dtype=int) + 1) * (GM / R ** 3)
    kn[:, :2] = 0.0
    F = orc.ravel_coefficients(orc._scale_packed_by_degree(orc.spherical_harmonics(Lo - 1, colat, lon), kn))
    return np.stack([(F @ TT[k])[:, nmin * nmin:] for k in range(6)], axis=1)


# ------------------------------------------------------------------------------ CPU
def test_restated_jacobian_reproduces_the_restated_tensor(orc):
    """F''_p T_a^(N+1) T_b^(N) x equals the restated tensor for random x at N = 12, at points from the surface to 500 km
    including points next to the poles."""
    from grates_b200 import utilities
    nmax = 12
    TT = _composed(_transform_matrices(orc, nmax), _transform_matrices(orc, nmax + 1))
    pos = np.concatenate((_positions(200, 3, 0.0, 500e3), [[1.0, 2.0, 6.5e6], [-3.0, 0.5, -6.8e6]]))
    r, colat, lon = utilities.cartesian_to_spherical(pos)
    x = _coefficients(2, nmax, 4)
    J = _jacobian(orc, TT, r, colat, lon, 0)
    got = np.einsum("pck,ek->ecp", J, orc.ravel_coefficients(x))
    ref = tensor(orc, x, r, colat, lon)
    err = float(np.max(np.abs(got - ref)) / np.max(np.abs(ref)))
    assert err <= 1e-13, err


def test_restated_adjoint_is_the_transpose_of_the_composed_transform(orc):
    """The restated composed transpose equals sum_ab (T_a^(N+1) T_b^(N))' g_ab for random g (every packed entry) at
    N = 12, and <G x, g> = <x, G' g> with the restated forward transform of test_gpu_gravity_gradient."""
    from test_gpu_gravity_gradient import tensor_coefficients
    nmax = 12
    Lo = nmax + 3
    TT = _composed(_transform_matrices(orc, nmax), _transform_matrices(orc, nmax + 1))
    rng = np.random.default_rng(5)
    g = rng.standard_normal((2, 6, Lo, Lo))
    got = gravity_gradient_coefficients_adjoint(g)
    for e in range(2):
        ref = sum(TT[k].T @ orc.ravel_coefficients(g[e, k]) for k in range(6))
        vec = orc.ravel_coefficients(got[e])
        assert np.max(np.abs(vec - ref)) <= 1e-15 * np.max(np.abs(ref)), e
    x = rng.standard_normal((2, nmax + 1, nmax + 1))
    Gx = tensor_coefficients(x)
    assert abs(np.sum(Gx * g) - np.sum(x * got)) <= 1e-14 * np.sqrt(np.sum(Gx ** 2) * np.sum(g ** 2))


def test_restated_rotation_transpose_satisfies_the_dot_product_identity():
    """<A v, w> = <v, A' w> for the rotation of the upper triangle (to_local) and the restated gb_rotate_tensor_from_local;
    the plain inverse rotation (Q' W Q of the stored upper triangle) does not satisfy it."""
    rng = np.random.default_rng(6)
    P = 500
    colat, lon = np.arccos(rng.uniform(-1, 1, P)), rng.uniform(-np.pi, np.pi, P)
    v, w = rng.standard_normal((3, 6, P)), rng.standard_normal((3, 6, P))
    Av, Atw = to_local(v, colat, lon), from_local(w, colat, lon)
    lhs, rhs = np.sum(Av * w, axis=(1, 2)), np.sum(v * Atw, axis=(1, 2))
    scale = np.sqrt(np.sum(Av ** 2, axis=(1, 2)) * np.sum(w ** 2, axis=(1, 2)))
    assert np.all(np.abs(lhs - rhs) <= 1e-14 * scale), (lhs - rhs) / scale
    # the inverse rotation is not the transpose on these 6-vectors
    M = full_matrix(w)
    W = _from_local(np.swapaxes(M, -3, -2), colat, lon)
    Z = _from_local(np.swapaxes(W, -3, -2), colat, lon)
    inverse = np.stack([Z[..., a, b, :] for a, b in PAIRS], axis=-2)
    assert np.all(np.abs(lhs - np.sum(v * inverse, axis=(1, 2))) > 1e-3 * scale)
    # and the forward rotation is orthogonal for the weights (1, 2, 2, 1, 2, 1)
    D = np.array([1.0, 2.0, 2.0, 1.0, 2.0, 1.0])[:, None]
    assert np.allclose(np.sum(D * Av ** 2, axis=(1, 2)), np.sum(D * v ** 2, axis=(1, 2)), rtol=1e-14, atol=0)


def test_argument_errors_come_before_any_device_call(monkeypatch):
    import torch
    import grates_b200 as gb
    from grates_b200 import plan
    from grates_b200.plan import PointsPlan

    def no_device(*args, **kwargs):
        raise AssertionError("a device was requested before the arguments were checked")
    monkeypatch.setattr(plan, "_current_device", no_device)
    pos = np.array([[7e6, 0.0, 0.0], [0.0, 7e6, 0.0]])
    obs = np.zeros((6, 2))
    normals = gb.gravity_gradient_normal_equations_at_positions
    with pytest.raises(ValueError, match="frame"):
        normals(obs, pos, 0, 4, frame='enu')
    with pytest.raises(ValueError, match="degree range"):
        normals(obs, pos, 5, 4)
    with pytest.raises(ValueError, match="degree range"):
        normals(obs, pos, -1, 4)
    for bad in (np.zeros((3, 2)), np.zeros((6, 3)), np.zeros((2, 3, 2)), np.zeros((0, 6, 2)), np.zeros(12)):
        with pytest.raises(ValueError, match="shape"):
            normals(bad, pos, 0, 4)
    for bad in (np.ones((3, 2)), np.ones(2), np.ones((6, 3))):
        with pytest.raises(ValueError, match="shape"):
            normals(obs, pos, 0, 4, weights=bad)
    for bad in (np.where(np.arange(12).reshape(6, 2) == 5, np.nan, 1.0), np.full((6, 2), np.inf),
                np.where(np.arange(12).reshape(6, 2) == 7, -1e-30, 1.0)):
        with pytest.raises(ValueError, match="finite and non-negative"):
            normals(obs, pos, 0, 4, weights=bad)
    for bad in (np.where(np.arange(12).reshape(6, 2) == 3, np.nan, 0.0), np.full((2, 6, 2), -np.inf)):
        with pytest.raises(ValueError, match="observations must be finite"):
            normals(bad, pos, 0, 4, weights=np.zeros((6, 2)))
    with pytest.raises(ValueError, match="float64 CUDA"):
        normals(torch.zeros((6, 2), dtype=torch.float64), pos, 0, 4)
    with pytest.raises(ValueError, match="block_size"):
        normals(obs, pos, 0, 4, block_size=0)
    with pytest.raises(ValueError, match="positions_per_chunk"):
        normals(obs, pos, 0, 4, positions_per_chunk=0)
    adjoint = gb.gravity_gradient_adjoint_at_positions
    with pytest.raises(ValueError, match="frame"):
        adjoint(obs[None], pos, 4, frame='ellipsoidal')
    for bad in (obs, np.zeros((1, 3, 2)), np.zeros((1, 6, 3))):
        with pytest.raises(ValueError, match="shape"):
            adjoint(bad, pos, 4)
    with pytest.raises(ValueError, match="max_degree"):
        adjoint(obs[None], pos, -1)
    for bad in (np.zeros((1, 3)), np.array([[np.nan, 0.0, 1.0]]), np.zeros((4, 2))):
        with pytest.raises(ValueError, match="positions"):
            normals(np.zeros((6, bad.shape[0])), bad, 0, 4)
        with pytest.raises(ValueError, match="positions"):
            adjoint(np.zeros((1, 6, bad.shape[0])), bad, 4)
    # the plan-order guard, both directions: a plan of the other order (or none) is refused before anything else
    for order, wrong in ((1, ("gravity_gradient_normals", "gravity_gradient_adjoint")),
                         (2, ("gradient_normals", "gradient_adjoint", "gradient_covariance")),
                         (None, ("gradient_normals", "gravity_gradient_normals", "gravity_gradient_adjoint"))):
        p = PointsPlan.__new__(PointsPlan)
        p.max_degree, p.npts = 8, 2
        if order is not None:
            p.derivative_order = order
        for name in wrong:
            with pytest.raises(ValueError, match="needs a .*gradient point plan"):
                if name.endswith("adjoint"):
                    getattr(p, name)(None)
                else:
                    getattr(p, name)(None, 0)


def test_c_abi_refuses_a_null_point_set():
    from grates_b200 import _lib
    lib = _lib.load()
    assert lib.gb_points_gravity_gradient_normals(None, 0, None, None, None, None) == _lib.GB_ERR_ARGUMENT
    assert b"NULL" in lib.gb_last_error()
    assert lib.gb_gravity_gradient_coefficients_adjoint(None, 1, 4, None, 0, None) == _lib.GB_ERR_ARGUMENT
    assert lib.gb_gravity_gradient_coefficients_adjoint(None, -1, 4, None, 0, None) == _lib.GB_ERR_ARGUMENT
    assert lib.gb_gravity_gradient_coefficients_adjoint(None, 1, -1, None, 0, None) == _lib.GB_ERR_ARGUMENT
    assert lib.gb_rotate_tensor_from_local(None, None, 1, 4, 0, None) == _lib.GB_ERR_ARGUMENT
    assert lib.gb_rotate_tensor_from_local(None, None, 1, -4, 0, None) == _lib.GB_ERR_ARGUMENT


# ------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def gb():
    import grates_b200
    grates_b200._lib.require_device()
    return grates_b200


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


@pytest.mark.gpu
def test_adjoint_dot_product_identity(gb):
    """<gravity_gradient_at_positions(X), Y> = <X, gravity_gradient_adjoint_at_positions(Y)> at degree 96 on the 86 402
    orbit positions, both frames, 1 and 6 sets; a numpy input gives a numpy result equal to the device path."""
    import torch
    pos = _track(86400, 4)
    P = pos.shape[0]
    worst = {}
    for E in (1, 6):
        X = torch.as_tensor(_coefficients(E, N, 50 + E)).cuda()
        Y = torch.as_tensor(np.random.default_rng(E).standard_normal((E, 6, P))).cuda()
        for frame in ("cartesian", "local"):
            GX = gb.gravity_gradient_at_positions(X, pos, frame=frame)
            GtY = gb.gravity_gradient_adjoint_at_positions(Y, pos, N, frame=frame)
            assert tuple(GtY.shape) == (E, N + 1, N + 1) and GtY.is_cuda
            lhs = (GX * Y).sum(dim=(1, 2))
            rhs = (X * GtY).sum(dim=(1, 2))
            scale = GX.norm(dim=(1, 2)) * Y.norm(dim=(1, 2))
            worst["E=%d %s" % (E, frame)] = float(((lhs - rhs).abs() / scale).max())
            if E == 1:
                host = gb.gravity_gradient_adjoint_at_positions(Y.cpu().numpy(), pos, N, frame=frame)
                assert isinstance(host, np.ndarray) and np.array_equal(host, GtY.cpu().numpy())
    for label, err in worst.items():
        print("GGNORMALS dot product %-14s %.3e" % (label, err))
    assert max(worst.values()) <= TOL_DOT, worst


@pytest.mark.gpu
def test_adjoint_kernels_bit_for_bit(gb):
    """gb_gravity_gradient_coefficients_adjoint against the restated composed transpose (degrees 96, 1, 0; 11 sets: a
    partial batch of eight) and gb_rotate_tensor_from_local against its restatement (the two-point kernel, and the
    one-point kernel on an odd count and a misaligned pointer), bit for bit."""
    import torch
    lib = gb._lib.load()
    rng = np.random.default_rng(9)
    for nmax, E in ((N, 11), (1, 2), (0, 1)):
        G = rng.standard_normal((E, 6, nmax + 3, nmax + 3))
        g = torch.as_tensor(G).cuda()
        out = torch.full((E, nmax + 1, nmax + 1), float("nan"), dtype=torch.float64, device="cuda")
        gb._lib.check(lib.gb_gravity_gradient_coefficients_adjoint(_ptr(g), E, nmax, _ptr(out), 0, None))
        assert np.array_equal(out.cpu().numpy(), gravity_gradient_coefficients_adjoint(G)), nmax
    P = 1001
    colat, lon = np.arccos(rng.uniform(-1, 1, P)), rng.uniform(-np.pi, np.pi, P)
    frame = torch.as_tensor(np.stack((np.cos(colat), np.sin(colat), np.cos(lon), np.sin(lon)))).cuda()
    V = rng.standard_normal((9, 6, P))
    for offset in (0, 1):
        buf = torch.as_tensor(np.concatenate((np.zeros(offset), V.ravel()))).cuda()
        v = buf[offset:]
        gb._lib.check(lib.gb_rotate_tensor_from_local(_ptr(v), _ptr(frame), 9, P, 0, None))
        assert np.array_equal(v.cpu().numpy().reshape(9, 6, P), from_local(V, colat, lon)), offset
    v = torch.as_tensor(V[:, :, :1000].copy()).cuda()
    fr = torch.as_tensor(np.ascontiguousarray(frame.cpu().numpy()[:, :1000])).cuda()
    gb._lib.check(lib.gb_rotate_tensor_from_local(_ptr(v), _ptr(fr), 9, 1000, 0, None))
    assert np.array_equal(v.cpu().numpy(), from_local(V[:, :, :1000], colat[:1000], lon[:1000]))


@pytest.mark.gpu
def test_laplace_equation_through_the_adjoint(gb):
    """The adjoint of V_xx = V_yy = V_zz = y (off-diagonals zero) is zero to rounding against the sum of the three
    single-component adjoints, coefficient by coefficient over the largest; the same for ee, nn, uu in the local frame
    (degree 96, 86 402 orbit positions)."""
    import torch
    pos = _track(86400, 7)
    P = pos.shape[0]
    y = torch.as_tensor(np.random.default_rng(8).standard_normal(P)).cuda()
    errs = {}
    for frame in ("cartesian", "local"):
        parts = []
        for k in (0, 3, 5):
            Y = torch.zeros((1, 6, P), dtype=torch.float64, device="cuda")
            Y[0, k] = y
            parts.append(gb.gravity_gradient_adjoint_at_positions(Y, pos, N, frame=frame))
        Y = torch.zeros((1, 6, P), dtype=torch.float64, device="cuda")
        Y[0, 0] = Y[0, 3] = Y[0, 5] = y
        whole = gb.gravity_gradient_adjoint_at_positions(Y, pos, N, frame=frame)
        scale = sum(p.abs() for p in parts).max()
        errs[frame] = float(whole.abs().max() / scale)
    for label, err in errs.items():
        print("GGNORMALS Laplace %-10s %.3e" % (label, err))
    assert max(errs.values()) <= TOL_LAPLACE, errs


def _restated(orc, TT, pos, nmin, frame, weights, obs):
    """Rows sqrt(w) J~ [6P, K'] of the restated Jacobian, and the extended-precision n = J~' W l [K', E] and l'Wl [E]."""
    from grates_b200 import utilities
    r, colat, lon = utilities.cartesian_to_spherical(pos)
    J = _jacobian(orc, TT, r, colat, lon, nmin)                                  # [P, 6, K']
    if frame == 'local':
        J = np.transpose(to_local(np.transpose(J, (2, 1, 0)), colat, lon), (2, 1, 0))
    sw = np.sqrt(weights.T)[:, :, None]                                          # [P, 6, 1]
    rows = (J * sw).reshape(-1, J.shape[-1])
    wl = (obs * weights[None]).transpose(0, 2, 1).reshape(obs.shape[0], -1).astype(np.longdouble)   # [E, 6P]
    n = (J.reshape(-1, J.shape[-1]).astype(np.longdouble).T @ wl.T)
    lpl = np.sum(wl * obs.transpose(0, 2, 1).reshape(obs.shape[0], -1), axis=1)
    return rows, n.astype(float), lpl.astype(float)


@pytest.mark.gpu
def test_normals_against_the_restated_jacobian(gb, orc):
    """Degree 30, 2 000 positions between 0 and 500 km, random weights of which about 10 % are zero, two observation
    sets, both frames, min_degree 0 and 2: N, n, l'Wl and the count against the restated Jacobian (N in float64 from
    the restated rows, checked on 256 entries in extended precision; n and l'Wl in extended precision)."""
    nmax, P, E = 30, 2000, 2
    pos = _positions(P, 11, 0.0, 500e3)
    rng = np.random.default_rng(12)
    TT = _composed(_transform_matrices(orc, nmax), _transform_matrices(orc, nmax + 1))
    obs = rng.standard_normal((E, 6, P)) * 1e-9
    weights = rng.uniform(0.25, 4.0, (6, P)) * 1e18 * (rng.uniform(0.0, 1.0, (6, P)) >= 0.1)
    positive = int(np.count_nonzero(weights))
    assert 0.85 * 6 * P < positive < 0.95 * 6 * P
    errs = {}
    for nmin in (0, 2):
        for frame in ("cartesian", "local"):
            ne = gb.gravity_gradient_normal_equations_at_positions(obs, pos, nmin, nmax, frame=frame, weights=weights,
                                                                   block_size=400)
            kp = (nmax + 1) ** 2 - nmin ** 2
            got = ne.matrix.to_tensor()
            assert tuple(got.shape) == (kp, kp) and ne.matrix.shape == (3, 3)
            rows, n_ref, lpl_ref = _restated(orc, TT, pos, nmin, frame, weights, obs)
            N_ref = rows.T @ rows
            sample = np.random.default_rng(nmin).integers(0, kp, (256, 2))
            rows_ld = rows.astype(np.longdouble)
            exact = np.array([np.sum(rows_ld[:, a] * rows_ld[:, b]) for a, b in sample])
            d = np.sqrt(np.diagonal(N_ref))
            label = "min_degree %d %s" % (nmin, frame)
            errs["restated N vs extended precision, " + label] = (
                float(np.max(np.abs(N_ref[sample[:, 0], sample[:, 1]] - exact) / (d[sample[:, 0]] * d[sample[:, 1]]))),
                EXACT_TOL)
            errs["N, " + label] = (_sym_err(got.cpu().numpy(), N_ref), TOL_N)
            rhs = ne.right_hand_side
            assert tuple(rhs.shape) == (kp, E) and rhs.is_cuda
            errs["n, " + label] = (float(np.max(np.abs(rhs.cpu().numpy() - n_ref) / (d[:, None] * np.sqrt(lpl_ref)))),
                                   TOL_RHS)
            errs["l'Wl, " + label] = (float(np.max(np.abs(ne.observation_square_sum - lpl_ref) / lpl_ref)), TOL_LPL)
            assert ne.observation_count == positive
            assert ne.observation_square_sum.shape == (E,)
    for label, (err, tol) in errs.items():
        print("GGNORMALS %-52s %.3e (tol %.0e)" % (label, err, tol))
    assert all(err <= tol for err, tol in errs.values()), errs


def _packed_index(nmax, nmin):
    """Flat packed positions [K'] of the degree-wise coefficients from nmin: C_nm at [n][m], S_nm at [m - 1][n]."""
    L = nmax + 1
    idx = []
    for n in range(nmin, nmax + 1):
        idx.append(n * L)
        for m in range(1, n + 1):
            idx += [n * L + m, (m - 1) * L + n]
    return np.array(idx)


@pytest.mark.gpu
def test_closed_loop_at_production_size(gb):
    """Degree 96, 20 000 seeded positions between 200 and 300 km: noiseless observations of a Kaula-scaled field from
    gravity_gradient_at_positions are solved back (NormalEquations.solve), and with N = L L' the forward operator applied
    to the K' coefficient sets of the columns of L^-T gives sum_pc w_pc (J~_pc L^-T)^2 = trace(L^-1 N L^-T) = K': unit
    weights in the Cartesian frame, random weights with the xy and yz components left out in the local frame."""
    import torch
    nmin = 2
    pos = _positions(20000, 41, 200e3, 300e3)
    P = pos.shape[0]
    kp = (N + 1) ** 2 - nmin ** 2
    X = torch.as_tensor(_kaula(N, nmin, 42)).cuda()
    x_ref = gb.ravel_batch(X, nmin)[0]
    idx = torch.as_tensor(_packed_index(N, nmin)).cuda()
    rng = np.random.default_rng(43)
    local_w = rng.uniform(0.5, 2.0, (6, P)) * np.array([[1.0], [0.0], [1.0], [1.0], [0.0], [0.25]])
    errs = {}
    for frame, weights in (("cartesian", None), ("local", local_w)):
        obs = gb.gravity_gradient_at_positions(X, pos, frame=frame)[0]                  # [6, P] on the device
        ne = gb.gravity_gradient_normal_equations_at_positions(obs, pos, nmin, N, frame=frame, weights=weights)
        assert ne.observation_count == (6 * P if weights is None else int(np.count_nonzero(weights)))
        normals = ne.matrix.to_tensor()                                              # solve() factors in place
        x = ne.solve()
        assert tuple(x.shape) == (kp, 1)
        errs["solve, " + frame] = (float((x[:, 0] - x_ref).abs().max() / x_ref.abs().max()), TOL_SOLVE)
        del ne
        Lc = torch.linalg.cholesky(normals)
        del normals
        Linv = torch.linalg.solve_triangular(Lc, torch.eye(kp, dtype=torch.float64, device="cuda"), upper=False)
        del Lc
        w = torch.ones((6, P), dtype=torch.float64, device="cuda") if weights is None else torch.as_tensor(weights).cuda()
        total = 0.0
        for k0 in range(0, kp, 512):
            rows = Linv[k0:k0 + 512]                                                   # columns of L^-T
            sets = torch.zeros((rows.shape[0], (N + 1) ** 2), dtype=torch.float64, device="cuda")
            sets[:, idx] = rows
            G = gb.gravity_gradient_at_positions(sets.view(-1, N + 1, N + 1), pos, frame=frame)
            total += float((w[None] * G * G).sum())
            del G, sets
        del Linv
        errs["trace, " + frame] = (abs(total - kp) / kp, TOL_TRACE)
    for label, (err, tol) in errs.items():
        print("GGNORMALS closed loop %-18s %.3e (tol %.0e)" % (label, err, tol))
    assert all(err <= tol for err, tol in errs.values()), errs


@pytest.mark.gpu
def test_invariants_and_edges(gb):
    """Degree 30: weights w_p (1, 2, 2, 1, 2, 1) give the same N in both frames; N is exactly symmetric; 9 191 positions
    (a full block of 8 192 and a partial one) in one C call equal two calls on the two blocks, bit for bit, and repeat
    bit for bit; the Python path in chunks of 700 positions agrees with one chunk; the C ABI refuses an out-of-range
    min_degree, a point set of degree 1 and a NULL matrix, and writes nothing."""
    import torch
    from grates_b200 import plan as gplan, utilities
    nmax = 30
    kp = (nmax + 1) ** 2
    rng = np.random.default_rng(51)
    pos = _positions(BLOCK_30 + 999, 52, 200e3, 500e3)
    P = pos.shape[0]
    weights = rng.uniform(0.5, 2.0, (1, P)) * np.array([[1.0], [2.0], [2.0], [1.0], [2.0], [1.0]])
    w = torch.as_tensor(weights).cuda()
    r, colat, lon = utilities.cartesian_to_spherical(pos)
    whole = gplan.gravity_gradient_points_plan(r, colat, lon, nmax)
    assert whole.derivative_order == 2
    zeros = lambda: torch.zeros((kp, kp), dtype=torch.float64, device="cuda")     # noqa: E731
    cart = whole.gravity_gradient_normals(zeros(), 0, 'cartesian', w)
    local = whole.gravity_gradient_normals(zeros(), 0, 'local', w)
    again = whole.gravity_gradient_normals(zeros(), 0, 'local', w)
    assert torch.equal(local, again)
    assert torch.equal(cart, cart.T) and torch.equal(local, local.T)
    err_frame = _sym_err(local, cart)
    halves = zeros()
    for p0, p1 in ((0, BLOCK_30), (BLOCK_30, P)):
        part = gplan.gravity_gradient_points_plan(r[p0:p1], colat[p0:p1], lon[p0:p1], nmax)
        part.gravity_gradient_normals(halves, 0, 'local', w[:, p0:p1].contiguous())
        part.close()
    assert torch.equal(halves, local)
    lib = gb._lib.load()
    ptr = _ptr(halves)
    for nmin in (-1, nmax + 1):
        assert lib.gb_points_gravity_gradient_normals(whole._handle, nmin, None, None, ptr, None) == \
            gb._lib.GB_ERR_ARGUMENT
    assert lib.gb_points_gravity_gradient_normals(whole._handle, 0, None, None, None, None) == gb._lib.GB_ERR_ARGUMENT
    low = gb.PointsPlan(lon[:4], 0.5 * np.pi - colat[:4], utilities.A_GRS80, utilities.F_GRS80, 1)
    assert lib.gb_points_gravity_gradient_normals(low._handle, 0, None, None, ptr, None) == gb._lib.GB_ERR_ARGUMENT
    assert b"degree" in lib.gb_last_error()
    torch.cuda.synchronize()
    assert torch.equal(halves, local)                                # nothing was written by the refused calls
    whole.close()
    low.close()
    obs = rng.standard_normal((3, 6, 2000)) * 1e-9
    wts = rng.uniform(0.5, 2.0, (6, 2000)) * 1e18
    wts[1] = wts[4] = 0.0
    one = gb.gravity_gradient_normal_equations_at_positions(obs, pos[:2000], 2, nmax, frame='local', weights=wts)
    chunked = gb.gravity_gradient_normal_equations_at_positions(obs, pos[:2000], 2, nmax, frame='local', weights=wts,
                                                                positions_per_chunk=700)
    assert one.observation_count == chunked.observation_count == 4 * 2000
    N1, N2 = one.matrix.to_tensor(), chunked.matrix.to_tensor()
    d = torch.diagonal(N1).sqrt()
    lpl = torch.as_tensor(one.observation_square_sum).cuda()
    errs = {"frames for weights w (1, 2, 2, 1, 2, 1)": (err_frame, TOL_FRAME),
            "chunked N": (_sym_err(N2, N1), TOL_CHUNK_N),
            "chunked n": (float(((chunked.right_hand_side - one.right_hand_side).abs() /
                                 (d[:, None] * lpl.sqrt()[None, :])).max()), TOL_CHUNK),
            "chunked l'Wl": (float(np.max(np.abs(chunked.observation_square_sum - one.observation_square_sum) /
                                          one.observation_square_sum)), TOL_CHUNK)}
    for label, (err, tol) in errs.items():
        print("GGNORMALS %-40s %.3e (tol %.0e)" % (label, err, tol))
    assert all(err <= tol for err, tol in errs.values()), errs
