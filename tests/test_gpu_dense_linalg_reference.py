"""The dense FP64 kernels of gb_linalg.cu (gb_dpotrf_upper, gb_dtrsm_upper, gb_dgemm) and the algorithms built on them
(lstsq.BlockMatrix / NormalEquations with blocks of 2048, grid.covariance_from_normals) at the production size of the
degree-96 normal equations, K' = 9405 (min_degree 2) and 9409 (min_degree 0).

Exact reference.  W = I + U is a unit upper-triangular integer matrix whose U has entries in {-1, 0, 1} on even rows and
odd columns above the diagonal only, so U^2 = 0 and W^-1 = I - U; D holds per-column powers of two.  Then
N = (WD)'(WD) has the Cholesky factor WD, N^-1 = D^-1 (I - U)(I - U)' D^-1, and every value the factorisation, the
triangular solves and the inverses produce is an integer times a power of two: each trailing entry (i, j) is d_i d_j
times an integer of magnitude <= n, each pivot is d_j^2, each division is by a power of two.  That holds in any
summation order, the DMMA tiles' included, so the device results are compared with torch.equal, dense, at every tile
and panel edge.  The references are built from the integer matrices with torch.matmul (cuBLAS, independent of gb_dgemm)
and D applied elementwise.  The right-hand sides are W x and D W' y for integer x, y, whose solutions x / D and y are
exact whatever the spread of D.

Rounding.  The exact reference cannot see a loss of precision, so the factorisation and the solve also run on the real
normal matrix of 20 000 orbit positions at degree 96 (as in test_gpu_gradient_normals.py): their backward errors, in
extended precision, are bounded by a small multiple of LAPACK's on the same matrix.

Edges of gb_dgemm: beta = 0 never reads C, k = 0 scales C, upper_only leaves the tiles below the diagonal untouched,
a contraction of 100 003 terms, and element offsets beyond 2^31.  gb_dpotrf_upper refuses n > 65535 before it writes.
"""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

KP = (9405, 9409)          # unknowns of the degree-96 normal equations for min_degree 2 and 0
BLOCK = 2048               # block size of gradient_normal_equations_at_positions
NAN_BITS = 0x7FF8000000000000
# Bounds of the rounding tests.  Observed on an NVIDIA B200 (1000 W power limit), LAPACK on its host.
RATIO_CHOLESKY = 5.0       # device Cholesky backward error over LAPACK's on the same N (2.26 for both paths: 1.37e-15
                           # against 6.06e-16)
RATIO_SOLVE = 5.0          # device solve backward error over LAPACK's (1.77 block, 2.02 dense: 1.15e-18 / 1.31e-18
                           # against 6.49e-19)
TOL_LONG_K = 2.5e-15       # k = 100 003 contraction against extended precision, over |row| |column|: ten times the
                           # observed 2.48e-16


@pytest.fixture(scope="module")
def gb():
    import grates_b200
    grates_b200._lib.require_device()
    return grates_b200


@pytest.fixture(scope="module")
def ops(gb):
    from grates_b200.lstsq import _Ops
    return _Ops(None)


def _exact(n, seed, spread=20, blocks=None, device="cuda"):
    """W = I + U (U in {-1, 0, 1} on even rows and odd columns above the diagonal; with blocks: only in the diagonal
    and first super-diagonal blocks and block (0, 3)), d = 2^e with e in [-spread, spread], and from them exactly:
    F = W D, N = F'F, F^-1 = D^-1 (I - U) and Sigma = N^-1 = F^-1 F^-T."""
    g = torch.Generator(device=device).manual_seed(seed)
    i = torch.arange(n, device=device)
    mask = (i[:, None] % 2 == 0) & (i[None, :] % 2 == 1) & (i[:, None] < i[None, :])
    if blocks is not None:
        bi = i // blocks
        mask &= (bi[None, :] - bi[:, None] <= 1) | ((bi[:, None] == 0) & (bi[None, :] == 3))
    U = torch.randint(-1, 2, (n, n), generator=g, device=device).to(torch.float64) * mask
    del mask
    e = np.random.default_rng(seed).integers(-spread, spread + 1, n)
    d = torch.as_tensor(np.ldexp(1.0, e)).to(device)
    eye = torch.eye(n, dtype=torch.float64, device=device)
    W, V = eye + U, eye - U
    del U, eye
    return {"W": W, "d": d, "F": W * d[None, :], "N": (W.T @ W) * d[:, None] * d[None, :], "Finv": V / d[:, None],
            "Sigma": (V @ V.T) / d[:, None] / d[None, :]}


def _framed(a, top=1, left=2, bottom=2, right=3):
    """a copied into a NaN-filled buffer with margins on every side: (buffer, view); the view's leading dimension is
    larger than its width."""
    m, n = a.shape
    buf = torch.full((top + m + bottom, left + n + right), float("nan"), dtype=torch.float64, device=a.device)
    view = buf[top:top + m, left:left + n]
    view.copy_(a)
    return buf, view


def _frame_intact(buf, view):
    """Every element of buf outside view still holds the NaN sentinel, bit for bit."""
    top, left = divmod((view.data_ptr() - buf.data_ptr()) // 8, buf.stride(0))
    outside = torch.ones(buf.shape, dtype=torch.bool, device=buf.device)
    outside[top:top + view.shape[0], left:left + view.shape[1]] = False
    return bool((buf.view(torch.int64)[outside] == NAN_BITS).all())


def _block_mask(index, pattern):
    """Dense boolean mask of the blocks (i, j) for which pattern(i, j) holds."""
    n = int(index[-1])
    mask = torch.zeros((n, n), dtype=torch.bool, device="cuda")
    for i in range(len(index) - 1):
        for j in range(len(index) - 1):
            if pattern(i, j):
                mask[index[i]:index[i + 1], index[j]:index[j + 1]] = True
    return mask


@pytest.fixture(scope="module")
def ref9409():
    return _exact(9409, 1)


# ------------------------------------------------------------------------------ exact: dense path
@pytest.mark.parametrize("n, spread", [(9409, 20), (9408, 20), (9405, 20), (9409, 200)])
def test_dense_factor_and_inverse_are_exact(gb, ops, n, spread):
    """_Ops.cholesky_upper on a strided view (last panel of 1, 64 and 61 rows) returns W D with a zeroed strict lower
    triangle and writes nothing outside the view; inv_triangular, inv_gram and covariance_from_normals return
    D^-1 (I - U) and Sigma exactly; D spans 2^[-200, 200] in the last case, so no scaling step may be missing."""
    ref = _exact(n, n + spread, spread)
    buf, w = _framed(ref["N"])
    ops.cholesky_upper(w)
    assert torch.equal(w, ref["F"])
    assert _frame_intact(buf, w)
    assert torch.equal(ops.inv_triangular(w), ref["Finv"])
    assert torch.equal(ops.inv_gram(w), ref["Sigma"])
    del buf, w
    sigma = gb.covariance_from_normals(ref["N"])
    assert sigma.is_cuda and torch.equal(sigma, ref["Sigma"])


@pytest.mark.parametrize("m", [1, 63, 64, 65, 9409])
def test_triangular_solves_are_exact_in_strided_views(ops, ref9409, m):
    """gb_dtrsm_upper at n = 9409 with m right-hand sides, both directions: W D y = W x gives x / D and (W D)' y =
    D W' x gives x.  W and B are views (leading dimensions n + 5 and m + 5) framed by NaN sentinels; the strict lower
    triangle of W holds NaN too, since it must not be referenced.  W and every sentinel come back bit-identical."""
    ref = ref9409
    n = ref["F"].shape[0]
    lower = torch.ones((n, n), dtype=torch.bool, device="cuda").tril_(-1)
    wbuf, w = _framed(ref["F"].masked_fill(lower, float("nan")))
    del lower
    wbits = wbuf.view(torch.int64).clone()
    x = torch.randint(-3, 4, (n, m), generator=torch.Generator(device="cuda").manual_seed(m), device="cuda").double()
    d = ref["d"][:, None]
    for trans, b, want in ((False, ref["W"] @ x, x / d), (True, d * (ref["W"].T @ x), x)):
        bbuf, bv = _framed(b)
        ops.solve_triangular(w, bv, trans=trans)
        assert torch.equal(bv, want), trans
        assert _frame_intact(bbuf, bv), trans
    assert torch.equal(wbuf.view(torch.int64), wbits)


# ------------------------------------------------------------------------------ exact: block path
@pytest.mark.parametrize("kp", KP)
def test_block_matrix_is_exact_with_2048_blocks(gb, kp):
    """BlockMatrix with blocks of 2048 (last blocks of 1213 and 1217 rows, whose diagonal updates run with upper_only)
    on a block-bidiagonal W plus the far block (0, 3), which makes the factor's block (1, 3) structurally nonzero but
    numerically zero: multiply_symmetric, cholesky and its block pattern, solve_triangular and multiply_triangular in
    both directions, NormalEquations.solve, inverse (upper blocks and symmetrised) and sparse_inverse (Sigma on the
    pattern, zero elsewhere), all exact."""
    ref = _exact(kp, kp, 20, blocks=BLOCK)
    W, d, F, Sigma = ref["W"], ref["d"][:, None], ref["F"], ref["Sigma"]
    index, _ = gb.BlockMatrix.compute_block_index((kp, kp), BLOCK)
    nb = len(index) - 1
    upper = _block_mask(index, lambda i, j: i <= j)

    def upper_part(bm):
        return torch.where(upper, bm.to_tensor(), 0.0)

    bm = gb.BlockMatrix.from_array(ref["N"], index, index)
    z = torch.randint(-3, 4, (kp, 3), generator=torch.Generator(device="cuda").manual_seed(kp), device="cuda").double()
    rhs = d * (W.T @ (W @ z))                                        # N (z / D)
    assert torch.equal(bm.multiply_symmetric(z / d), rhs)
    chol = bm.copy()
    chol.cholesky()
    assert torch.equal(upper_part(chol), F)
    for i in range(nb):
        for j in range(i, nb):
            if bool(F[index[i]:index[i + 1], index[j]:index[j + 1]].any()):
                assert chol.is_nonzero(i, j), (i, j)
    assert chol.is_nonzero(1, 3) and not bool(F[index[1]:index[2], index[3]:index[4]].any())
    assert not chol.is_nonzero(0, 2)
    assert torch.equal(chol.solve_triangular(W @ z), z / d)
    assert torch.equal(chol.solve_triangular(d * (W.T @ z), transpose=True), z)
    assert torch.equal(chol.multiply_triangular(z / d), W @ z)
    assert torch.equal(chol.multiply_triangular(z, transpose=True), d * (W.T @ z))
    ne = gb.NormalEquations(bm.copy(), rhs, 1.0, kp)
    assert torch.equal(ne.solve(), z / d)
    del ne, bm
    full = chol.copy()
    full.inverse()
    assert torch.equal(upper_part(full), torch.where(upper, Sigma, 0.0))
    assert torch.equal(full.symmetrize().to_tensor(), Sigma)
    del full
    sparse = chol.copy()
    sparse.sparse_inverse()
    pattern = _block_mask(index, lambda i, j: i <= j and sparse.is_nonzero(i, j))
    assert torch.equal(upper_part(sparse), torch.where(pattern, Sigma, 0.0))


def test_pivot_failures_name_the_leading_minor(gb, ops, ref9409):
    """N[p, p] - d_p^2 at p = 4100 makes that pivot exactly zero: the dense path raises LinAlgError for leading minor
    4101, BlockMatrix.cholesky for minor 5 of block 2 (numbered within the block, as scipy.linalg.cholesky of the
    reference's block loop numbers it).  A NaN on the diagonal raises too, at its own index."""
    N, d = ref9409["N"], ref9409["d"]
    index, _ = gb.BlockMatrix.compute_block_index(tuple(N.shape), BLOCK)
    p = 4100
    bad = N.clone()
    bad[p, p] -= d[p] ** 2
    with pytest.raises(np.linalg.LinAlgError, match=r"^4101-th leading minor"):
        gb.covariance_from_normals(bad)
    with pytest.raises(np.linalg.LinAlgError, match=r"^4101-th leading minor"):
        ops.cholesky_upper(bad.clone())
    with pytest.raises(np.linalg.LinAlgError, match=r"^5-th leading minor"):
        gb.BlockMatrix.from_array(bad, index, index).cholesky()
    bad = N.clone()
    bad[7000, 7000] = float("nan")
    with pytest.raises(np.linalg.LinAlgError, match=r"^7001-th leading minor"):
        ops.cholesky_upper(bad.clone())
    with pytest.raises(np.linalg.LinAlgError, match=r"^857-th leading minor"):
        gb.BlockMatrix.from_array(bad, index, index).cholesky()


# ------------------------------------------------------------------------------ rounding on a production matrix
@pytest.fixture(scope="module")
def production(gb):
    """N = J~' J~ of 20 000 seeded positions between 0 and 300 km at degree 96, min_degree 2 (K' = 9405), as a
    BlockMatrix with blocks of 2048."""
    from test_gpu_gradient_normals import _positions
    pos = _positions(20000, 21)
    obs = np.random.default_rng(24).standard_normal((3, pos.shape[0])) * 1e-6
    return gb.gradient_normal_equations_at_positions(obs, pos, 2, 96).matrix


def _samples(n, rng, count=4096):
    """Entries (a <= b): the diagonals of the first and last blocks of 2048, three entries at every 64-row boundary
    (the 2048-row boundaries among them), the rest random."""
    last = ((n - 1) // BLOCK) * BLOCK
    diag = np.concatenate([np.arange(BLOCK), np.arange(last, n)])
    b = np.arange(64, n, 64)
    pairs = [np.stack([diag, diag], 1), np.stack([b - 1, b], 1), np.stack([b, rng.integers(b, n)], 1),
             np.stack([rng.integers(0, b), b], 1)]
    have = sum(len(p) for p in pairs)
    pairs.append(np.sort(rng.integers(0, n, (count - have, 2)), axis=1))
    return np.concatenate(pairs)


def _cholesky_backward_error(w, N, samples):
    """max |(W'W - N)_ab| / sqrt(N_aa N_bb) over the sampled entries, W'W in extended precision."""
    dn = np.sqrt(np.diagonal(N))
    err = 0.0
    for s in range(0, len(samples), 256):
        a, b = samples[s:s + 256, 0], samples[s:s + 256, 1]
        wtw = np.sum(w[:, a].astype(np.longdouble) * w[:, b].astype(np.longdouble), axis=0)
        err = max(err, float(np.max(np.abs(wtw - N[a, b]) / (dn[a] * dn[b]))))
    return err


def _solve_backward_errors(N, xs, rhs):
    """Normwise backward error |n - N x|_inf / (|N|_inf |x|_inf + |n|_inf) per solution and column, N x in extended
    precision; the largest per solution."""
    X = np.concatenate(xs, axis=1).astype(np.longdouble)
    NX = np.empty(X.shape, dtype=np.longdouble)
    for r in range(0, N.shape[0], 1024):
        NX[r:r + 1024] = N[r:r + 1024].astype(np.longdouble) @ X
    R = np.tile(rhs, (1, len(xs))) - NX
    norm_n = np.max(np.sum(np.abs(N), axis=1))
    be = np.max(np.abs(R), axis=0) / (norm_n * np.max(np.abs(X), axis=0) + np.tile(np.max(np.abs(rhs), axis=0), len(xs)))
    return [float(v) for v in np.max(be.astype(float).reshape(len(xs), -1), axis=1)]


def test_production_factorisation_and_solve_against_lapack(gb, ops, production):
    """The block path (BlockMatrix.cholesky, NormalEquations.solve) and the dense path (_Ops.cholesky_upper and two
    solve_triangular) on the production N against scipy.linalg.cholesky / cho_solve of the same N on the host:
    Cholesky backward error on 4096 sampled entries, normwise solve backward error for four random right-hand sides,
    each at most a small multiple of LAPACK's.  Two factorisations of the same N are bit-identical."""
    import scipy.linalg as sla
    N = production.to_tensor()
    kp = N.shape[0]
    rng = np.random.default_rng(25)
    rhs = rng.standard_normal((kp, 4))
    rhs_d = torch.as_tensor(rhs).cuda()
    ne = gb.NormalEquations(production.copy(), rhs_d, 0.0, 0)
    x_block = ne.solve().cpu().numpy()
    w_block = torch.triu(ne.matrix.to_tensor())
    again = production.copy()
    again.cholesky()
    repeat_block = torch.equal(torch.triu(again.to_tensor()), w_block)
    del again, ne
    w_dense = ops.cholesky_upper(N.clone())
    repeat_dense = torch.equal(ops.cholesky_upper(N.clone()), w_dense)
    x_dense = ops.solve_triangular(w_dense, ops.solve_triangular(w_dense, rhs_d.clone(), trans=True)).cpu().numpy()
    Nh = N.cpu().numpy()
    w_lapack = sla.cholesky(Nh, lower=False)
    x_lapack = sla.cho_solve((w_lapack, False), rhs)
    samples = _samples(kp, rng)
    chol = {"block": _cholesky_backward_error(w_block.cpu().numpy(), Nh, samples),
            "dense": _cholesky_backward_error(w_dense.cpu().numpy(), Nh, samples),
            "LAPACK": _cholesky_backward_error(w_lapack, Nh, samples)}
    solve = dict(zip(("block", "dense", "LAPACK"), _solve_backward_errors(Nh, [x_block, x_dense, x_lapack], rhs)))
    for label in ("block", "dense", "LAPACK"):
        print("DENSELA production K' = %d, Cholesky backward error, %-6s %.3e (%.2f x LAPACK, bound %.0f x)"
              % (kp, label, chol[label], chol[label] / chol["LAPACK"], RATIO_CHOLESKY))
    for label in ("block", "dense", "LAPACK"):
        print("DENSELA production K' = %d, solve backward error, %-6s    %.3e (%.2f x LAPACK, bound %.0f x)"
              % (kp, label, solve[label], solve[label] / solve["LAPACK"], RATIO_SOLVE))
    print("DENSELA production repeat factorisation bit-identical: block %s, dense %s" % (repeat_block, repeat_dense))
    assert repeat_block and repeat_dense
    assert all(chol[p] <= RATIO_CHOLESKY * chol["LAPACK"] for p in ("block", "dense")), chol
    assert all(solve[p] <= RATIO_SOLVE * solve["LAPACK"] for p in ("block", "dense")), solve


# ------------------------------------------------------------------------------ gb_dgemm edges
def _ints(shape, seed, low=-8, high=9):
    return torch.randint(low, high, shape, generator=torch.Generator(device="cuda").manual_seed(seed),
                         device="cuda").double()


def test_gemm_beta_zero_never_reads_c(ops):
    """beta = 0 with C full of NaN gives alpha op(A) op(B) exactly (integer data, all four transposes, ragged shapes);
    A, B and C are views framed by NaN sentinels that come back bit-identical."""
    for (m, n, k) in ((1, 1, 1), (130, 70, 33), (64, 64, 16), (65, 129, 100)):
        for ta in (False, True):
            for tb in (False, True):
                a = _ints((k, m) if ta else (m, k), m + k)
                b = _ints((n, k) if tb else (k, n), n + 2 * k)
                (abuf, av), (bbuf, bv) = _framed(a), _framed(b)
                cbuf = torch.full((m + 3, n + 5), float("nan"), dtype=torch.float64, device="cuda")
                cv = cbuf[1:1 + m, 2:2 + n]
                ops.gemm(av, bv, cv, alpha=-0.5, beta=0.0, trans_a=ta, trans_b=tb)
                want = -0.5 * ((a.T if ta else a) @ (b.T if tb else b))
                label = (m, n, k, ta, tb)
                assert torch.equal(cv, want), label
                assert _frame_intact(cbuf, cv) and _frame_intact(abuf, av) and _frame_intact(bbuf, bv), label


def test_gemm_empty_contraction_scales_c(ops):
    """k = 0: C = beta C (beta = 0.5 exactly, beta = 0 clears a NaN-filled C)."""
    a = torch.empty((70, 0), dtype=torch.float64, device="cuda")
    b = torch.empty((0, 130), dtype=torch.float64, device="cuda")
    c = torch.randn((70, 130), dtype=torch.float64, device="cuda")
    want = 0.5 * c
    assert torch.equal(ops.gemm(a, b, c, alpha=3.0, beta=0.5), want)
    c = torch.full((70, 130), float("nan"), dtype=torch.float64, device="cuda")
    assert torch.equal(ops.gemm(a, b, c, alpha=3.0, beta=0.0), torch.zeros_like(c))


@pytest.mark.parametrize("n", [65, 1213, 1217])
def test_gemm_upper_only_leaves_the_tiles_below_the_diagonal(ops, n):
    """upper_only through the C entry point on square C: the tiles on and above the diagonal hold the product (beta = 0
    over NaN, and the trailing update C - A'A of gb_dpotrf_upper with beta = 1), every tile strictly below the diagonal
    keeps its sentinel bit for bit."""
    t = torch.arange(n, device="cuda") // 64
    below = t[:, None] > t[None, :]
    a, b = _ints((n, 100), n), _ints((100, n), n + 1)
    c = torch.full((n, n), float("nan"), dtype=torch.float64, device="cuda")
    ops.gemm(a, b, c, upper_only=True)
    assert torch.equal(c[~below], (a @ b)[~below])
    assert bool((c.view(torch.int64)[below] == NAN_BITS).all())
    panel = _ints((64, n), n + 2)
    c0 = _ints((n, n), n + 3, -1000, 1001)
    c = c0.clone()
    ops.gemm(panel, panel, c, alpha=-1.0, beta=1.0, trans_a=True, upper_only=True)
    assert torch.equal(c[~below], (c0 - panel.T @ panel)[~below])
    assert torch.equal(c.view(torch.int64)[below], c0.view(torch.int64)[below])


def test_gemm_long_contraction_against_extended_precision(ops):
    """k = 100 003 at m = n = 130, all four transposes: |C - A B| / (|A_i| |B^j|) against extended-precision dot
    products.  The tiles reach shared memory in one layout whatever the transposition, so the four results are
    bit-identical."""
    m = n = 130
    k = 100003
    rng = np.random.default_rng(26)
    a, bt = rng.standard_normal((m, k)), rng.standard_normal((n, k))          # logical A [m, k] and B' [n, k]
    ref = a.astype(np.longdouble) @ bt.astype(np.longdouble).T
    scale = np.linalg.norm(a, axis=1)[:, None] * np.linalg.norm(bt, axis=1)[None, :]
    ad, btd = torch.as_tensor(a).cuda(), torch.as_tensor(bt).cuda()
    errs, results = {}, []
    for ta in (False, True):
        for tb in (False, True):
            c = torch.empty((m, n), dtype=torch.float64, device="cuda")
            ops.gemm(ad.T.contiguous() if ta else ad, btd if tb else btd.T.contiguous(), c, trans_a=ta, trans_b=tb)
            results.append(c)
            errs[(ta, tb)] = float(np.max(np.abs(c.cpu().numpy() - ref) / scale))
    for (ta, tb), err in errs.items():
        print("DENSELA gemm k = %d, trans_a %d trans_b %d %.3e (tol %.1e)" % (k, ta, tb, err, TOL_LONG_K))
    assert all(torch.equal(c, results[0]) for c in results[1:])
    assert max(errs.values()) <= TOL_LONG_K, errs


def test_gemm_offsets_beyond_two_to_the_31(ops):
    """Operands and result in a [40 000, 65 536] buffer (21 GB) of which the products use 16-column slices: element
    offsets row * ld + column reach 2.6e9 in the k-contiguous and the x-contiguous fetches and in the epilogue.
    Integer data, exact against torch.matmul; the columns next to the written slice keep their sentinels."""
    rows, ld = 40000, 65536
    free, _ = torch.cuda.mem_get_info()
    if free < 8.0 * rows * ld + 4e9:
        pytest.skip("needs 25 GB of free device memory")
    z = torch.empty((rows, ld), dtype=torch.float64, device="cuda")
    a, b, c, guard = z[:, 0:16], z[:, 16:32], z[:, 32:48], z[:, 48:64]
    a.copy_(_ints((rows, 16), 1))
    b.copy_(_ints((rows, 16), 2))
    guard.fill_(float("nan"))
    assert (rows - 1) * ld > 2**31
    s = _ints((16, 16), 3)
    small = ops.gemm(a, b, torch.empty((16, 16), dtype=torch.float64, device="cuda"), trans_a=True)
    assert torch.equal(small, a.T @ b)
    ops.gemm(a, s, c)
    assert torch.equal(c, a @ s)
    wide = ops.gemm(s, b, torch.empty((16, rows), dtype=torch.float64, device="cuda"), trans_b=True)
    assert torch.equal(wide, s @ b.T)
    assert bool((guard.contiguous().view(torch.int64) == NAN_BITS).all())
    del z, a, b, c, guard
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------ argument check before any write
def test_potrf_refuses_more_than_65535_rows_before_writing(gb):
    """gb_dpotrf_upper with n = 65 536 (an uninitialised 34 GB matrix) returns GB_ERR_ARGUMENT and leaves the matrix
    and *d_info as they were."""
    n = 65536
    free, _ = torch.cuda.mem_get_info()
    if free < 8.0 * n * n + 4e9:
        pytest.skip("needs 39 GB of free device memory")
    a = torch.empty((n, n), dtype=torch.float64, device="cuda")
    spots = ((0, 0), (1, 0), (0, 1), (64, 64), (40000, 123), (123, 40000), (n - 1, n - 1))
    for v, (i, j) in enumerate(spots):
        a[i, j] = -1.5 - v
    info = torch.full((1,), 7, dtype=torch.int32, device="cuda")
    lib = gb._lib.load()
    torch.cuda.synchronize()
    rc = lib.gb_dpotrf_upper(ctypes.c_void_p(a.data_ptr()), n, n, ctypes.c_void_p(info.data_ptr()),
                             torch.cuda.current_device(), None)
    assert rc == gb._lib.GB_ERR_ARGUMENT and b"65535" in lib.gb_last_error()
    torch.cuda.synchronize()
    assert [float(a[i, j]) for i, j in spots] == [-1.5 - v for v in range(len(spots))]
    assert int(info.item()) == 7
    del a
    torch.cuda.empty_cache()
