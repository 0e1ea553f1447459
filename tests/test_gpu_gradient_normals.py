"""Normal equations and adjoint of gravitational-acceleration observations at orbit positions
(gradient_normal_equations_at_positions, gradient_adjoint_at_positions): N = J~' W J~, n = J~' W l and the transpose J'
of ``gradient_at_positions``, with J~_p = Q_p J_p the Jacobian of grad V in the observations' frame.

The references reuse the host restatements of test_gpu_gradient.py (the transform T and the gradient) and of
test_gpu_gradient_covariance.py (T as sparse matrices, the Jacobian rows J_p = F'_p T from the oracle's degree-(N+1)
tables, the rotation Q).  Without a GPU the restated transpose T' below is tied to those sparse matrices.  On the GPU:

  - the dot-product identity <J x, y> = <x, J' y> at 86 402 orbit positions, degree 96, both frames, 1 and 6 sets;
  - gb_gradient_coefficients_adjoint bit for bit against the restated T' and to rounding against the sparse T_c';
  - N, n, l'Wl and the count against the restated Jacobian (degree 30, 2 000 positions, random weights, both frames,
    min_degree 0 and 2);
  - a closed loop at degree 96: noiseless observations of a Kaula-scaled field at 20 000 positions are solved back, and
    the covariance N^-1 propagated to the same positions is consistent with the weights (sum_p tr(W_p J~_p Sigma J~_p')
    = K');
  - invariants and edges: the frames agree for equal weights per position, N is exactly symmetric, several point blocks
    and two C calls on two halves equal one call, the chunked Python path agrees with one chunk, repeated calls are
    bit-identical, and the C ABI refuses bad arguments.
"""
import ctypes

import numpy as np
import pytest

from test_gpu_gradient import _coefficients, _track, gradient_coefficients
from test_gpu_gradient_covariance import _jacobian, _to_local_matrix, _transform_matrices

N = 96
# Largest error each comparison may show: ten times the largest error an NVIDIA B200 (1000 W power limit) showed for it.
TOL_DOT = 2e-16            # |<J x, y> - <x, J' y>| / (|J x| |y|) (observed up to 1.9e-17)
TOL_T = 1e-15              # T' on the device against the sparse T_c' products, max-normalised (observed 0)
TOL_N = 8e-14              # N against the restated Jacobian, |dN_ab| / sqrt(N_aa N_bb) (7.4e-15)
TOL_RHS = 1.1e-15          # n against the restated Jacobian, |dn_a| / sqrt(N_aa l'Wl) (1.07e-16)
TOL_LPL = 1.5e-15          # l'Wl, relative (1.44e-16)
TOL_SOLVE = 2.4e-14        # closed loop: recovered coefficients, max-normalised (2.3e-15)
TOL_TRACE = 8e-15          # closed loop: sum_p tr(W_p J~_p Sigma J~_p') against K', relative (7.7e-16)
TOL_FRAME = 2.6e-13        # N local against N cartesian for equal weights per position (2.6e-14)
TOL_CHUNK_N = 7e-14        # chunked against one chunk: N as for TOL_N (7.0e-15)
TOL_CHUNK = 1.3e-15        # chunked against one chunk: n as for TOL_RHS, l'Wl relative (1.2e-16)
EXACT_TOL = 1e-14          # float64 restated N entries against their extended-precision sums
BLOCK_30 = 16384           # points per block of gb_points_gradient_normals at degree 30 (at most 16384)


@pytest.fixture(scope="module")
def orc():
    from oracle import sh_oracle
    return sh_oracle


def gradient_coefficients_adjoint(g):
    """numpy restatement of T' summed over the components: [..., 3, L+1, L+1] (x, y, z) -> [..., L, L] packed.  The
    input (n, m, s) reads the outputs it feeds at degree n + 1 (the table of gbgrad::grad_terms): z -fz (m, s); x -fp
    (m+1, s) + fm (m-1, s) for m >= 1 and not the sine of order 0; y of a cosine -fp (m+1, S) - fm (m-1, S) for m >= 2,
    of a sine +fp (m+1, C) + fm (m-1, C).  Factors, products and sums in the order of gb_gradient_coefficients_adjoint:
    per component f1 x1 (+ f2 x2), added to the sum in the order x, y, z."""
    g = np.asarray(g, dtype=float)
    Lo = g.shape[-1]
    L = Lo - 1
    out = np.zeros(g.shape[:-3] + (L, L))
    sqrt2 = np.sqrt(2.0)
    for n in range(L):
        q = (2.0 * n + 1.0) / (2.0 * n + 3.0)

        def x(c, mp, sp):
            return g[..., c, mp - 1, n + 1] if sp else g[..., c, n + 1, mp]
        for m in range(n + 1):
            fz = np.sqrt(float((n - m + 1) * (n + m + 1)) * q)
            fp = np.sqrt(float((n + m + 1) * (n + m + 2)) * q) * 0.5
            fp = fp * sqrt2 if m == 0 else fp
            fm = None
            if m >= 1:
                fm = np.sqrt(float((n - m + 1) * (n - m + 2)) * q) * 0.5
                fm = fm * sqrt2 if m == 1 else fm
            for s in ((0, 1) if m > 0 else (0,)):
                terms = [[(-fp, m + 1, s)], [], [(-fz, m, s)]]
                if m >= 1 and (s == 0 or m >= 2):
                    terms[0].append((fm, m - 1, s))
                if s == 0:
                    terms[1].append((-fp, m + 1, 1))
                    if m >= 2:
                        terms[1].append((-fm, m - 1, 1))
                else:
                    terms[1] += [(fp, m + 1, 0), (fm, m - 1, 0)]
                v = 0.0
                for c in range(3):
                    t = terms[c][0][0] * x(c, *terms[c][0][1:])
                    if len(terms[c]) > 1:
                        t = t + terms[c][1][0] * x(c, *terms[c][1][1:])
                    v = v + t
                if s:
                    out[..., m - 1, n] = v
                else:
                    out[..., n, m] = v
    return out


def _positions(count, seed, low=0.0, high=300e3):
    """Seeded Earth-fixed positions [P, 3], uniform over the sphere at R + U(low, high) metres."""
    from oracle.sh_oracle import R_DEFAULT
    rng = np.random.default_rng(seed)
    r = R_DEFAULT + rng.uniform(low, high, count)
    colat = np.arccos(rng.uniform(-1.0, 1.0, count))
    lon = rng.uniform(-np.pi, np.pi, count)
    return np.stack((r * np.sin(colat) * np.cos(lon), r * np.sin(colat) * np.sin(lon), r * np.cos(colat)), axis=1)


def _sym_err(got, ref):
    """max |got - ref|_ab / sqrt(ref_aa ref_bb) for symmetric positive matrices (numpy or torch)."""
    import torch
    got, ref = torch.as_tensor(got), torch.as_tensor(ref).to(torch.as_tensor(got).device)
    d = torch.diagonal(ref).sqrt()
    return float(((got - ref).abs() / (d[:, None] * d[None, :])).max())


# ------------------------------------------------------------------------------ CPU
def test_restated_adjoint_is_the_transpose_of_the_restated_transform(orc):
    """sum_c T_c' g_c for the sparse T of test_gpu_gradient_covariance.py equals the restated T' at N = 12, for random
    g (every packed entry, degree 0 included), and <T x, g> = <x, T' g> through gradient_coefficients."""
    nmax = 12
    Lo = nmax + 2
    rng = np.random.default_rng(5)
    g = rng.standard_normal((2, 3, Lo, Lo))
    T = _transform_matrices(orc, nmax)
    got = gradient_coefficients_adjoint(g)
    for e in range(2):
        ref = sum(T[c].T @ orc.ravel_coefficients(g[e, c]) for c in range(3))
        vec = orc.ravel_coefficients(got[e])
        assert np.max(np.abs(vec - ref)) <= 1e-15 * np.max(np.abs(ref)), e
    x = rng.standard_normal((2, nmax + 1, nmax + 1))
    lhs = np.sum(gradient_coefficients(x) * g)
    rhs = np.sum(x * got)
    assert abs(lhs - rhs) <= 1e-14 * np.sqrt(np.sum(gradient_coefficients(x) ** 2) * np.sum(g ** 2))


def test_argument_errors_come_before_any_device_call(monkeypatch):
    import torch
    import grates_b200 as gb
    from grates_b200 import plan

    def no_device(*args, **kwargs):
        raise AssertionError("a device was requested before the arguments were checked")
    monkeypatch.setattr(plan, "_current_device", no_device)
    pos = np.array([[7e6, 0.0, 0.0], [0.0, 7e6, 0.0]])
    obs = np.zeros((3, 2))
    normals = gb.gradient_normal_equations_at_positions
    with pytest.raises(ValueError, match="frame"):
        normals(obs, pos, 0, 4, frame='enu')
    with pytest.raises(ValueError, match="degree range"):
        normals(obs, pos, 5, 4)
    with pytest.raises(ValueError, match="degree range"):
        normals(obs, pos, -1, 4)
    for bad in (np.zeros((3, 3)), np.zeros((2, 2)), np.zeros((2, 4, 2)), np.zeros((0, 3, 2)), np.zeros(6)):
        with pytest.raises(ValueError, match="shape"):
            normals(bad, pos, 0, 4)
    for bad in (np.ones((3, 3)), np.ones(2), np.ones((2, 3))):
        with pytest.raises(ValueError, match="shape"):
            normals(obs, pos, 0, 4, weights=bad)
    for bad in (np.array([[1.0, 1.0], [1.0, np.nan], [1.0, 1.0]]), np.array([[1.0, np.inf]] * 3),
                np.array([[1.0, 0.0]] * 3), np.array([[1.0, -2.0]] * 3)):
        with pytest.raises(ValueError, match="finite and positive"):
            normals(obs, pos, 0, 4, weights=bad)
    with pytest.raises(ValueError, match="float64 CUDA"):
        normals(torch.zeros((3, 2), dtype=torch.float64), pos, 0, 4)
    with pytest.raises(ValueError, match="block_size"):
        normals(obs, pos, 0, 4, block_size=0)
    with pytest.raises(ValueError, match="positions_per_chunk"):
        normals(obs, pos, 0, 4, positions_per_chunk=0)
    adjoint = gb.gradient_adjoint_at_positions
    with pytest.raises(ValueError, match="frame"):
        adjoint(obs[None], pos, 4, frame='ellipsoidal')
    for bad in (obs, np.zeros((1, 3, 3)), np.zeros((1, 2, 2))):
        with pytest.raises(ValueError, match="shape"):
            adjoint(bad, pos, 4)
    with pytest.raises(ValueError, match="max_degree"):
        adjoint(obs[None], pos, -1)
    for bad in (np.zeros((1, 3)), np.array([[np.nan, 0.0, 1.0]]), np.zeros((4, 2))):
        with pytest.raises(ValueError, match="positions"):
            normals(np.zeros((3, bad.shape[0])), bad, 0, 4)
        with pytest.raises(ValueError, match="positions"):
            adjoint(np.zeros((1, 3, bad.shape[0])), bad, 4)


def test_c_abi_refuses_a_null_point_set():
    from grates_b200 import _lib
    lib = _lib.load()
    assert lib.gb_points_gradient_normals(None, 0, None, None, None, None) == _lib.GB_ERR_ARGUMENT
    assert b"NULL" in lib.gb_last_error()
    assert lib.gb_gradient_coefficients_adjoint(None, 1, 4, None, 0, None) == _lib.GB_ERR_ARGUMENT
    assert lib.gb_gradient_coefficients_adjoint(None, -1, 4, None, 0, None) == _lib.GB_ERR_ARGUMENT
    assert lib.gb_rotate_from_local(None, None, 1, 4, 0, None) == _lib.GB_ERR_ARGUMENT
    assert lib.gb_rotate_from_local(None, None, 1, -4, 0, None) == _lib.GB_ERR_ARGUMENT


# ------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def gb():
    import grates_b200
    grates_b200._lib.require_device()
    return grates_b200


@pytest.mark.gpu
def test_adjoint_dot_product_identity(gb):
    """<gradient_at_positions(X), Y> = <X, gradient_adjoint_at_positions(Y)> at degree 96 on the 86 402 orbit positions,
    both frames, 1 and 6 sets; a numpy input gives a numpy result equal to the device path."""
    import torch
    pos = _track(86400, 4)
    P = pos.shape[0]
    worst = {}
    for E in (1, 6):
        X = torch.as_tensor(_coefficients(E, N, 40 + E)).cuda()
        Y = torch.as_tensor(np.random.default_rng(E).standard_normal((E, 3, P))).cuda()
        for frame in ("cartesian", "local"):
            JX = gb.gradient_at_positions(X, pos, frame=frame)
            JtY = gb.gradient_adjoint_at_positions(Y, pos, N, frame=frame)
            assert tuple(JtY.shape) == (E, N + 1, N + 1) and JtY.is_cuda
            lhs = (JX * Y).sum(dim=(1, 2))
            rhs = (X * JtY).sum(dim=(1, 2))
            scale = JX.norm(dim=(1, 2)) * Y.norm(dim=(1, 2))
            worst["E=%d %s" % (E, frame)] = float(((lhs - rhs).abs() / scale).max())
            if E == 1:
                host = gb.gradient_adjoint_at_positions(Y.cpu().numpy(), pos, N, frame=frame)
                assert isinstance(host, np.ndarray) and np.array_equal(host, JtY.cpu().numpy())
    for label, err in worst.items():
        print("GRADNORMALS dot product %-14s %.3e" % (label, err))
    assert max(worst.values()) <= TOL_DOT, worst


@pytest.mark.gpu
def test_coefficients_adjoint_against_the_host(gb, orc):
    """gb_gradient_coefficients_adjoint bit for bit against the restated T' (degrees 96, 1, 0; 11 sets: a partial batch
    of eight), and to rounding against the sparse products sum_c T_c' g_c at degree 30."""
    import torch
    lib = gb._lib.load()
    rng = np.random.default_rng(9)

    def device_adjoint(G, nmax):
        g = torch.as_tensor(G).cuda()
        out = torch.full((G.shape[0], nmax + 1, nmax + 1), float("nan"), dtype=torch.float64, device="cuda")
        gb._lib.check(lib.gb_gradient_coefficients_adjoint(ctypes.c_void_p(g.data_ptr()), G.shape[0], nmax,
                                                           ctypes.c_void_p(out.data_ptr()), 0, None))
        return out.cpu().numpy()
    for nmax, E in ((N, 11), (1, 2), (0, 1)):
        G = rng.standard_normal((E, 3, nmax + 2, nmax + 2))
        assert np.array_equal(device_adjoint(G, nmax), gradient_coefficients_adjoint(G)), nmax
    nmax = 30
    T = _transform_matrices(orc, nmax)
    G = rng.standard_normal((3, 3, nmax + 2, nmax + 2))
    got = device_adjoint(G, nmax)
    err = 0.0
    for e in range(3):
        ref = sum(T[c].T @ orc.ravel_coefficients(G[e, c]) for c in range(3))
        err = max(err, float(np.max(np.abs(orc.ravel_coefficients(got[e]) - ref)) / np.max(np.abs(ref))))
    print("GRADNORMALS T' against sparse T_c' %.3e" % err)
    assert err <= TOL_T


def _restated(orc, T, pos, nmin, frame, weights, obs):
    """Rows sqrt(w) J~ [3P, K'] of the restated Jacobian, and the extended-precision n = J~' W l [K', E] and l'Wl [E]."""
    from grates_b200 import utilities
    r, colat, lon = utilities.cartesian_to_spherical(pos)
    J = _jacobian(orc, T, r, colat, lon, nmin)                                   # [P, 3, K']
    if frame == 'local':
        J = np.einsum("pij,pjk->pik", _to_local_matrix(colat, lon), J)
    sw = np.sqrt(weights.T)[:, :, None]                                          # [P, 3, 1]
    rows = (J * sw).reshape(-1, J.shape[-1])
    wl = (obs * weights[None]).transpose(0, 2, 1).reshape(obs.shape[0], -1).astype(np.longdouble)   # [E, 3P]
    n = (J.reshape(-1, J.shape[-1]).astype(np.longdouble).T @ wl.T)
    lpl = np.sum(wl * obs.transpose(0, 2, 1).reshape(obs.shape[0], -1), axis=1)
    return rows, n.astype(float), lpl.astype(float)


@pytest.mark.gpu
def test_normals_against_the_restated_jacobian(gb, orc):
    """Degree 30, 2 000 positions between 0 and 500 km, random weights, two observation sets, both frames, min_degree 0
    and 2: N, n, l'Wl and the count against the restated Jacobian (N in float64 from the restated rows, checked on 256
    entries in extended precision; n and l'Wl in extended precision)."""
    nmax, P, E = 30, 2000, 2
    pos = _positions(P, 11, 0.0, 500e3)
    rng = np.random.default_rng(12)
    T = _transform_matrices(orc, nmax)
    obs = rng.standard_normal((E, 3, P)) * 1e-6
    weights = rng.uniform(0.25, 4.0, (3, P)) * 1e12
    errs = {}
    for nmin in (0, 2):
        for frame in ("cartesian", "local"):
            ne = gb.gradient_normal_equations_at_positions(obs, pos, nmin, nmax, frame=frame, weights=weights,
                                                           block_size=400)
            kp = (nmax + 1) ** 2 - nmin ** 2
            got = ne.matrix.to_tensor()
            assert tuple(got.shape) == (kp, kp) and ne.matrix.shape == (3, 3)
            rows, n_ref, lpl_ref = _restated(orc, T, pos, nmin, frame, weights, obs)
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
            assert ne.observation_count == 3 * P
            assert ne.observation_square_sum.shape == (E,)
    for label, (err, tol) in errs.items():
        print("GRADNORMALS %-52s %.3e (tol %.0e)" % (label, err, tol))
    assert all(err <= tol for err, tol in errs.values()), errs


def _kaula(nmax, nmin, seed):
    """One packed set [1, L, L] with a Kaula-scaled spectrum 1e-5 / n^2, zero below nmin."""
    L = nmax + 1
    deg = np.arange(L, dtype=float)
    packed_degree = np.where(np.tril(np.ones((L, L), dtype=bool)), deg[:, None], deg[None, :])
    x = np.random.default_rng(seed).standard_normal((1, L, L)) * 1e-5 / np.maximum(packed_degree, 1.0) ** 2
    x[:, packed_degree < nmin] = 0.0
    return x


@pytest.mark.gpu
def test_closed_loop_at_production_size(gb):
    """Degree 96, 20 000 seeded positions between 0 and 300 km: noiseless observations of a Kaula-scaled field from
    gradient_at_positions are solved back (NormalEquations.solve), and Sigma = N^-1 (compute_covariance(sparse=False))
    propagated with gradient_covariance_at_positions to the same positions gives sum_p tr(W_p J~_p Sigma J~_p') = K':
    unit weights in the Cartesian frame, random weights in the local frame."""
    import torch
    nmin = 2
    pos = _positions(20000, 21)
    P = pos.shape[0]
    kp = (N + 1) ** 2 - nmin ** 2
    X = torch.as_tensor(_kaula(N, nmin, 22)).cuda()
    x_ref = gb.ravel_batch(X, nmin)[0]
    rng = np.random.default_rng(23)
    errs = {}
    for frame, weights in (("cartesian", None), ("local", rng.uniform(0.5, 2.0, (3, P)) * np.array([[1.0], [1.0], [0.25]]))):
        obs = gb.gradient_at_positions(X, pos, frame=frame)[0]                      # [3, P] on the device
        ne = gb.gradient_normal_equations_at_positions(obs, pos, nmin, N, frame=frame, weights=weights)
        x = ne.solve()
        assert tuple(x.shape) == (kp, 1)
        errs["solve, " + frame] = (float((x[:, 0] - x_ref).abs().max() / x_ref.abs().max()), TOL_SOLVE)
        ne.compute_covariance(sparse=False)
        sigma = ne.matrix.symmetrize().to_tensor()
        cov = gb.gradient_covariance_at_positions(sigma, pos, nmin, N, frame=frame, full=True, device_output=True)
        var = torch.diagonal(cov, dim1=1, dim2=2)                                  # [P, 3]
        w = torch.ones_like(var) if weights is None else torch.as_tensor(weights.T).cuda()
        trace = float((w * var).sum())
        errs["trace, " + frame] = (abs(trace - kp) / kp, TOL_TRACE)
        del ne, sigma, cov
    for label, (err, tol) in errs.items():
        print("GRADNORMALS closed loop %-18s %.3e (tol %.0e)" % (label, err, tol))
    assert all(err <= tol for err, tol in errs.values()), errs


@pytest.mark.gpu
def test_invariants_and_edges(gb):
    """Degree 30: equal weights per position give the same N in both frames; N is exactly symmetric; 17 383 positions
    (a full block of 16 384 and a partial one) in one C call equal two calls on the two blocks, bit for bit, and repeat
    bit for bit; the Python path in chunks of 700 positions agrees with one chunk; the C ABI refuses an out-of-range
    min_degree, a point set of degree 0 and a NULL matrix."""
    import torch
    from grates_b200 import plan as gplan, utilities
    nmax = 30
    kp = (nmax + 1) ** 2
    rng = np.random.default_rng(31)
    pos = _positions(BLOCK_30 + 999, 32, 200e3, 500e3)
    P = pos.shape[0]
    weights = np.repeat(rng.uniform(0.5, 2.0, (1, P)), 3, axis=0)
    w = torch.as_tensor(weights).cuda()
    r, colat, lon = utilities.cartesian_to_spherical(pos)
    whole = gplan.gradient_points_plan(r, colat, lon, nmax)
    cart = whole.gradient_normals(torch.zeros((kp, kp), dtype=torch.float64, device="cuda"), 0, 'cartesian', w)
    local = whole.gradient_normals(torch.zeros((kp, kp), dtype=torch.float64, device="cuda"), 0, 'local', w)
    again = whole.gradient_normals(torch.zeros((kp, kp), dtype=torch.float64, device="cuda"), 0, 'local', w)
    assert torch.equal(local, again)
    assert torch.equal(cart, cart.T) and torch.equal(local, local.T)
    err_frame = _sym_err(local, cart)
    halves = torch.zeros((kp, kp), dtype=torch.float64, device="cuda")
    for p0, p1 in ((0, BLOCK_30), (BLOCK_30, P)):
        part = gplan.gradient_points_plan(r[p0:p1], colat[p0:p1], lon[p0:p1], nmax)
        part.gradient_normals(halves, 0, 'local', w[:, p0:p1].contiguous())
        part.close()
    assert torch.equal(halves, local)
    lib = gb._lib.load()
    ptr = ctypes.c_void_p(halves.data_ptr())
    for nmin in (-1, nmax + 1):
        assert lib.gb_points_gradient_normals(whole._handle, nmin, None, None, ptr, None) == gb._lib.GB_ERR_ARGUMENT
    assert lib.gb_points_gradient_normals(whole._handle, 0, None, None, None, None) == gb._lib.GB_ERR_ARGUMENT
    scalar = gb.PointsPlan(lon[:4], 0.5 * np.pi - colat[:4], utilities.A_GRS80, utilities.F_GRS80, 0)
    assert lib.gb_points_gradient_normals(scalar._handle, 0, None, None, ptr, None) == gb._lib.GB_ERR_ARGUMENT
    assert torch.equal(halves, local)                                # nothing was written by the refused calls
    whole.close()
    scalar.close()
    obs = rng.standard_normal((3, 3, 2000)) * 1e-6
    wts = rng.uniform(0.5, 2.0, (3, 2000)) * 1e12
    one = gb.gradient_normal_equations_at_positions(obs, pos[:2000], 2, nmax, frame='local', weights=wts)
    chunked = gb.gradient_normal_equations_at_positions(obs, pos[:2000], 2, nmax, frame='local', weights=wts,
                                                        positions_per_chunk=700)
    N1, N2 = one.matrix.to_tensor(), chunked.matrix.to_tensor()
    d = torch.diagonal(N1).sqrt()
    lpl = torch.as_tensor(one.observation_square_sum).cuda()
    errs = {"frames for equal weights": (err_frame, TOL_FRAME),
            "chunked N": (_sym_err(N2, N1), TOL_CHUNK_N),
            "chunked n": (float(((chunked.right_hand_side - one.right_hand_side).abs() /
                                 (d[:, None] * lpl.sqrt()[None, :])).max()), TOL_CHUNK),
            "chunked l'Wl": (float(np.max(np.abs(chunked.observation_square_sum - one.observation_square_sum) /
                                          one.observation_square_sum)), TOL_CHUNK)}
    for label, (err, tol) in errs.items():
        print("GRADNORMALS %-26s %.3e (tol %.0e)" % (label, err, tol))
    assert all(err <= tol for err, tol in errs.values()), errs
