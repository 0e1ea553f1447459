"""The filters, the device reductions and the basin variances at production size against exact references.

Every kernel tested here is a linear or bilinear contraction, a permutation or a sum, so most cases use data that makes
the reference exact rather than merely more precise: dyadic integers, small integers times a power of two
(_dyadic), sized so that every partial sum of every contraction stays below 2^52.  Any float64 summation order, BLAS
with FMA included, then gives the same bits, and the GPU result must equal the numpy reference bit for bit at every
entry (compared as int64 views, so -0 / +0 and NaN are seen).  No tolerance is involved and an error in a small entry
cannot hide behind the largest one.  The data operand of each contraction needs more than 24 significant bits, so an
FP32 intermediate anywhere fails.  A mismatch names its first differing entry: epoch, basin, C(n,m) / S(n,m).

Exact data cannot show a precision downgrade that only rounds, so each GEMM-like kernel also has one realistic float
case, compared with a float64 reference that is itself checked at 64 entries in extended precision (np.longdouble).

  A  order-wise filter (gb_filter.cu with the pack / unpack of gb_pack.cu) and the degree weights (gb_scale_by_degree)
  B  dense filter matrices (gb_densefilter.cu and the UnravelStore epilogue of the shared DMMA GEMM)
  C  device reductions (gb_reduce.cu): temporal RMS, weighted moments, ravel, quadratic forms
  D  basin variances: the adjoint synthesis run through the analysis kernels, then ravel and quadratic forms

The adjoint of a one-point grid e_(i,j) is the synthesis row U[i, :] o T[j, :] (Legendre factor of parallel i times the
trigonometric factor of meridian j), so every row of A' is checked against a rank-one product, as in the impulse suite.
The basin functional a_b = A' w_b is separable, a_b[k] = sum_i U[i, k] (W_b T)[i, k], and its variance under
Sigma = G G' + diag(d) is ||G' a_b||^2 + (a_b o a_b) . d.  The references themselves are checked against the oracle
without a GPU (section E).

The module's GPU cases run in about 25 s on an NVIDIA B200 (1000 W power limit); the host references (the K' = 9405
dense filter product, the 1.7 GB of filter blocks at degree 687, the basin functionals) take most of it.
"""
import ctypes
import datetime
import subprocess
import time

import numpy as np
import pytest

from test_gpu_full_size_reference import _Checks, _factors, _grid_tables, _sigma
from test_gpu_impulse_reference import _name

N = 96

# Largest error each realistic comparison may show: ten times the largest error an NVIDIA B200 (1000 W power limit)
# showed for it, never more than 1e-12.  The inputs are seeded, so the observed values are reproducible.  The rows of
# A' on the folded 0.5 degree grid differ from the rank-one products by up to 1.1e-13 (at S(96,96)): the folded
# longitude stage takes +-sin(96 lon) of the quadrant meridian for the mirrored ones, whose own sine differs in the last
# bits; the unfolded grid matched exactly.  The global basin from degree 2 is a small residual of large cancelling
# terms (5.1e-13).
EXACT_TOL = 1e-14          # float64 reference against its extended-precision recomputation
TOL_ORDERWISE = 3e-14      # order-wise filter, per (epoch, order, cos | sin) block against its output maximum (2.2e-15)
TOL_DENSE = 2e-13          # dense filter, per (epoch, degree) against that degree's output maximum (1.7e-14)
TOL_QF = 3e-14             # quadratic forms, per vector (2.9e-15)
TOL_STATS = 7e-15          # grid_statistics, per epoch, relative (6.8e-16)
TOL_ADJ = 1e-12            # rows of A', per point against the row maximum (1.1e-13)
TOL_BASIN = 1e-12          # basin variances, per basin (5.1e-13)


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
def orc():
    from oracle import sh_oracle
    return sh_oracle


# ------------------------------------------------------------------------------ exact data and comparison
def _dyadic(rng, shape, bits, scale_exp):
    """Uniform integers in +-[0, 2^bits), times 2^scale_exp (the exponent only moves values to realistic magnitudes)."""
    return np.ldexp(rng.integers(-(2 ** bits - 1), 2 ** bits, size=shape).astype(np.float64), scale_exp)


def _dyadic_rows(rng, rows, cols, bits, scale_exp, chunk=1024):
    """A large dyadic matrix generated in row chunks (no int64 copy of the whole matrix)."""
    out = np.empty((rows, cols))
    for r0 in range(0, rows, chunk):
        out[r0:r0 + chunk] = _dyadic(rng, (min(chunk, rows - r0), cols), bits, scale_exp)
    return out


def _first_diff(got, ref):
    """Index of the first entry whose bits differ, or None."""
    g = np.ascontiguousarray(got, dtype=np.float64).view(np.int64)
    r = np.ascontiguousarray(ref, dtype=np.float64).view(np.int64)
    bad = np.flatnonzero(g != r)
    return None if bad.size == 0 else np.unravel_index(bad[0], g.shape)


def _same(checks, label, got, ref, where=str):
    """Bit-for-bit comparison; a mismatch is reported at its first entry, named by ``where(index)``."""
    got, ref = np.asarray(got), np.asarray(ref)
    if got.shape != ref.shape:
        checks.equal("%s (shape %s, expected %s)" % (label, got.shape, ref.shape), False)
        return
    idx = _first_diff(got, ref)
    if idx is not None:
        label += ", first at %s: %r, expected %r" % (where(idx), float(got[idx]), float(ref[idx]))
    checks.equal(label, idx is None)


def _packed(idx):
    """'epoch e, C(n,m)' of an index into a packed batch [E, L, L]."""
    return "epoch %d, %s" % (idx[0], _name(idx[1], idx[2]))


def _raveled(nmin, nmax, what="set"):
    rows, cols = _degreewise(nmin, nmax)
    return lambda idx: "%s %d, %s" % (what, idx[0], _name(rows[idx[1]], cols[idx[1]]))


def _degreewise(nmin, nmax):
    from oracle import sh_oracle
    return sh_oracle._degreewise_index(nmin, nmax)


def _torch(x):
    import torch
    return torch.as_tensor(x).cuda()


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def _stream():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _coefficients(orc, nmax, E, first=0):
    return np.stack([orc.synthetic_coefficients(nmax, first + e) for e in range(E)])


# ------------------------------------------------------------------------------ references
def _dense_reference(W, nmin, nmax, X):
    """orc.dense_filter of every epoch of X [E, Lin, Lin] as one product (exact on dyadic data)."""
    from oracle import sh_oracle as orc
    Lin = X.shape[-1]
    max_degree = min(Lin - 1, nmax)
    k_out = (max_degree + 1) ** 2 - nmin ** 2 if max_degree >= nmin else 0
    k_in = max(min(Lin, nmax + 1) ** 2 - nmin ** 2, 0)
    x = orc.ravel_coefficients(X, nmin, nmax)[:, :k_in]
    out = orc.unravel_coefficients(x @ W[:k_out, :k_in].T if k_out else np.zeros((X.shape[0], 0)), nmin, max_degree)
    out[:, 0:nmin, 0:nmin] = X[:, 0:nmin, 0:nmin]
    return out


def _kaula(nmin, nmax, scale, power):
    return np.concatenate([np.full(2 * n + 1, scale * float(n) ** power) for n in range(nmin, nmax + 1)])


def _vdk_low_rank(G, d, kaula):
    """orc.vdk_matrix of the normal matrix G G' + diag(d): (N + D)^-1 N = I - (N + D)^-1 D with D = diag(kaula), the
    inverse by the Woodbury identity (a K^2 r product instead of a dense K^3 solve)."""
    m = 1.0 / (d + kaula)
    MG = G * m[:, None]
    C = np.eye(G.shape[1]) + G.T @ MG
    W = MG @ np.linalg.solve(C, MG.T * kaula[None, :])
    W.flat[::W.shape[0] + 1] += 1.0 - m * kaula
    return W


def _per_order_tables(orc, parallels, meridians, nmin, nmax):
    """U [nlat, K'] from the per-order Legendre functions (the s = sqrt(1 - t^2) variant of the reference's
    synthesis_matrix_per_order and adjoint operators) times the ewh degree factors, and T [nlon, K'] (cos / sin of
    m lon), both degree-wise from nmin."""
    colat, kn = orc.kn_table("ewh", nmax, parallels)
    U = np.empty((parallels.size, (nmax + 1) ** 2 - nmin ** 2))
    for m in range(nmax + 1):
        P = (orc.legendre_functions_per_order(nmax, m, colat) * kn[:, m:])[:, max(nmin - m, 0):]
        n = np.arange(max(m, nmin), nmax + 1)
        base = n * n - nmin * nmin
        if m == 0:
            U[:, base] = P
        else:
            U[:, base + 2 * m - 1] = P
            U[:, base + 2 * m] = P
    _, T = _grid_tables(orc, parallels, meridians, nmin, nmax)
    return U, T


def _functionals(U, T, W):
    """a_b[k] = sum_i U[i, k] (W_b T)[i, k] for weights W [B, nlat, nlon]: [B, K'].  T has only 2L - 1 distinct
    columns (one per order and trigonometric function), so W_b T costs nlat nlon (2L - 1)."""
    Tu, inv = np.unique(T, axis=1, return_inverse=True)
    inv = inv.ravel()
    out = np.empty((W.shape[0], U.shape[1]))
    for b in range(W.shape[0]):
        out[b] = np.einsum("ik,ik->k", U, (W[b] @ Tu)[:, inv])
    return out


def _functional_guard(U, T, W, a, seed):
    """Largest difference between a [B, K'] and 64 of its entries recomputed in extended precision, relative to the
    maximum of each functional."""
    rng = np.random.default_rng(seed)
    worst = 0.0
    for b, k in zip(rng.integers(0, W.shape[0], 64), rng.integers(0, U.shape[1], 64)):
        Wb = W[b].astype(np.longdouble)
        exact = U[:, k].astype(np.longdouble) @ (Wb @ T[:, k].astype(np.longdouble))
        worst = max(worst, float(abs(a[b, k] - exact) / np.abs(a[b]).max()))
    return worst


def _basin_weights(masks, area):
    """w_b = mask_b * area / sum(mask_b * area), as basin_variances forms them."""
    w = masks.astype(float) * np.asarray(area, dtype=float).reshape(1, -1)
    return w / w.sum(axis=1, keepdims=True)


# ------------------------------------------------------------------------------ E. the references themselves (no GPU)
def test_dyadic_products_are_exact():
    """A float64 GEMM of dyadic data sized as in this file equals the same product in Python integers, entry for
    entry; so does an FP32 rounding of the data operand not (it needs more than 24 significant bits)."""
    rng = np.random.default_rng(1)
    k, bits_a, bits_x = 9405, 12, 26                 # the dense-filter case: 2^12 2^26 k < 2^52
    A = _dyadic(rng, (5, k), bits_a, -17)
    X = _dyadic(rng, (k, 3), bits_x, -60)
    got = A @ X
    Ai = [[int(v) for v in row] for row in np.ldexp(A, 17).astype(np.int64)]
    Xi = [[int(v) for v in row] for row in np.ldexp(X, 60).astype(np.int64)]
    for r in range(5):
        for c in range(3):
            exact = sum(Ai[r][i] * Xi[i][c] for i in range(k))
            assert got[r, c] == np.ldexp(float(exact), -77) and abs(exact) < 2 ** 53
    assert not np.array_equal(A @ X.astype(np.float32).astype(np.float64), got)
    # the reductions: the quadratic form a' S a with 25-bit S and ternary a, the weighted second moment
    S = _dyadic(rng, (40, 40), 25, -30)
    a = _dyadic(rng, 40, 1, -3)
    Si = np.ldexp(S, 30).astype(np.int64)
    ai = [int(v) for v in np.ldexp(a, 3).astype(np.int64)]
    exact = sum(ai[r] * sum(int(Si[r, c]) * ai[c] for c in range(40)) for r in range(40))
    assert a @ (S @ a) == np.ldexp(float(exact), -36)


def test_batched_references_match_the_oracle(orc):
    """The batched dense-filter reference equals orc.dense_filter epoch by epoch on dyadic data, for input degrees at,
    below and above the filter's and below min_degree; orc.orderwise_filter passes degrees 0 and 1 of dyadic data
    through; the low-rank VDK matrix equals orc.vdk_matrix."""
    rng = np.random.default_rng(2)
    nmin, nmax = 2, 12
    K = (nmax + 1) ** 2 - nmin ** 2
    W = _dyadic(rng, (K, K), 12, -17)
    for lin in (13, 9, 16, 2):
        X = _dyadic(rng, (3, lin, lin), 26, -60)
        ref = _dense_reference(W, nmin, nmax, X)
        for e in range(3):
            assert np.array_equal(ref[e], orc.dense_filter(W, nmin, nmax, X[e])), lin
    blocks = [_dyadic(rng, (nmax + 1 - (g + 1) // 2,) * 2, 16, -17) for g in range(2 * nmax + 1)]
    X = _dyadic(rng, (nmax + 1, nmax + 1), 26, -60)
    out = orc.orderwise_filter(blocks, X)
    assert np.array_equal(out[0:2, 0:2], X[0:2, 0:2]) and not np.array_equal(out[2:, 0], X[2:, 0])
    G, d = _factors(nmax, 3)
    G, d = G[nmin * nmin:] * 1e3, d[nmin * nmin:] * 1e8
    kaula = _kaula(nmin, nmax, 1e-2, 4.0)
    ref = orc.vdk_matrix(G @ G.T + np.diag(d), nmin, nmax, 1e-2, 4.0)
    assert np.max(np.abs(_vdk_low_rank(G, d, kaula) - ref)) < 1e-13 * np.max(np.abs(ref))


def test_per_order_tables_match_the_oracle(orc):
    """U o T of the per-order tables equals the columns of orc.synthesis_matrix_per_order, bit for bit, from degree 0
    and 2; and agrees with the packed Legendre tables of _grid_tables to rounding."""
    nmax = 12
    og = orc.geographic_grid(10.0, 10.0)
    for nmin in (0, 2):
        U, T = _per_order_tables(orc, og.parallels, og.meridians, nmin, nmax)
        A = (U[:, None, :] * T[None, :, :]).reshape(-1, U.shape[1])
        for m in range(nmax + 1):
            n = np.arange(max(m, nmin), nmax + 1)
            base = n * n - nmin * nmin
            mats = orc.synthesis_matrix_per_order(og, m, nmin, nmax, "ewh")
            if m == 0:
                assert np.array_equal(A[:, base], mats), m
            else:
                assert np.array_equal(A[:, base + 2 * m - 1], mats[0]), m
                assert np.array_equal(A[:, base + 2 * m], mats[1]), m
        Up, _ = _grid_tables(orc, og.parallels, og.meridians, nmin, nmax)
        assert np.max(np.abs(U - Up)) < 1e-14 * np.max(np.abs(Up))


def test_separable_basin_functional_matches_the_oracle(orc):
    """The separable functional a_b equals the dense w @ A of orc.basin_variances (A from unit-coefficient syntheses)
    at degree 12 on the 10 degree grid and on a ragged grid, from degree 0 and 2, and the closed-form variance equals
    orc.basin_variances."""
    nmax = 12
    dlon = 2 * np.pi / 31
    ragged = orc.OracleGrid(np.linspace(-np.pi + dlon / 2, np.pi - dlon / 2, 31),
                            np.array([1.45, 1.3, 1.1, 0.95, 0.7, 0.6, 0.4, 0.1, -0.05, -0.3, -0.5, -0.75, -0.9, -1.15, -1.5]))
    rng = np.random.default_rng(4)
    for og in (orc.geographic_grid(10.0, 10.0), ragged):
        P = og.parallels.size * og.meridians.size
        masks = np.vstack((rng.uniform(size=(2, P)) < 0.3, np.ones((1, P)), rng.uniform(size=(1, P))))
        masks[0, :] = False
        masks[0, 7] = True                                                  # single point
        w = _basin_weights(masks, og.areas)
        for nmin in (0, 2):
            K = (nmax + 1) ** 2 - nmin ** 2
            A = np.empty((P, K))
            for c in range(K):
                unit = np.zeros(K)
                unit[c] = 1.0
                A[:, c] = orc.synthesis(orc.unravel_coefficients(unit, nmin, nmax), og, "ewh").ravel()
            U, T = _per_order_tables(orc, og.parallels, og.meridians, nmin, nmax)
            a = _functionals(U, T, w.reshape(-1, *og.shape))
            f = w @ A
            assert np.max(np.abs(a - f) / np.abs(f).max(axis=1, keepdims=True)) < 1e-13, nmin
            G, d = _factors(nmax, 5)
            G, d = G[nmin * nmin:], d[nmin * nmin:]
            var = np.einsum("br,br->b", a @ G, a @ G) + (a * a) @ d
            ref = orc.basin_variances(G @ G.T + np.diag(d), og, masks, nmin, nmax, "ewh")
            assert np.max(np.abs(var - ref) / ref) < 1e-13, nmin


# ------------------------------------------------------------------------------ A. order-wise filter
def _filter_blocks(rng, nf):
    """Dyadic order-wise blocks of degree nf: 16 bits (2^16 2^26 k < 2^52 for k <= 688); the rows of degrees 0 and 1
    are not the identity, so a kernel that multiplies them instead of passing them through fails."""
    return [_dyadic(rng, (nf + 1 - (g + 1) // 2,) * 2, 16, -17) for g in range(2 * nf + 1)]


def _orderwise(orc, blocks, X):
    return np.stack([orc.orderwise_filter(blocks, x) for x in X])


@pytest.mark.gpu
def test_a1_orderwise_filter_config5_and_epoch_tiles(gb, orc):
    """Config 5 (N = nf = 120, 500 epochs) bit for bit; epoch counts around the pack kernel's switch from 8 to 32
    epochs per CTA (E <= 64) and the filter's 32-epoch tiles; filters of higher degree than the data (block leading
    dimension kf != k): nf = 180 and nf = N + 3."""
    checks = _Checks("A1")
    rng = np.random.default_rng(11)
    X = _dyadic(rng, (500, 121, 121), 26, -60)                # 26 bits: an FP32 copy of the data cannot pass
    blocks = _filter_blocks(rng, 120)
    flt = gb.OrderWiseFilter(blocks)
    ref = _orderwise(orc, blocks, X)
    Xd = _torch(X)
    _same(checks, "N = nf = 120, 500 epochs", flt.filter_batch(Xd).cpu().numpy(), ref, _packed)
    for E in (1, 31, 32, 33, 64, 65):
        _same(checks, "N = nf = 120, %d epochs" % E, flt.filter_batch(Xd[:E].contiguous()).cpu().numpy(), ref[:E], _packed)
    for nf, E in ((180, 65), (123, 33)):
        blocks = _filter_blocks(rng, nf)
        _same(checks, "nf = %d, N = 120, %d epochs" % (nf, E),
              gb.OrderWiseFilter(blocks).filter_batch(Xd[:E].contiguous()).cpu().numpy(),
              _orderwise(orc, blocks, X[:E]), _packed)
    checks.done()


@pytest.mark.gpu
def test_a2_orderwise_filter_high_degree_and_shared_memory_bound(gb, orc):
    """N = 360 (three 128-row passes); N = 687, the largest degree the shared-memory tile of the filter admits, with
    L = 688 > 512 taking the second column chunk of pack and unpack (about 1.7 GB of blocks); degree 688 refused with
    GB_ERR_ARGUMENT by the shared-memory check of filter_packed, which runs before any launch or read of the buffers."""
    import torch
    checks = _Checks("A2")
    rng = np.random.default_rng(12)
    for nf in (360, 687):
        t0 = time.perf_counter()
        X = _dyadic(rng, (2, nf + 1, nf + 1), 26, -60)
        blocks = _filter_blocks(rng, nf)
        flt = gb.OrderWiseFilter(blocks)
        got = flt.filter_batch(_torch(X)).cpu().numpy()
        _same(checks, "N = nf = %d, 2 epochs" % nf, got, _orderwise(orc, blocks, X), _packed)
        del flt, blocks
        print("A2 N = %d: %.1f s" % (nf, time.perf_counter() - t0))
    torch.cuda.empty_cache()
    lib = gb._lib.load()
    dummy_in = torch.zeros(4, dtype=torch.float64, device="cuda")
    dummy_out = torch.zeros(4, dtype=torch.float64, device="cuda")
    offsets = np.zeros(1, dtype=np.int64)
    rc = lib.gb_orderwise_filter(_ptr(dummy_in), offsets.ctypes.data_as(ctypes.c_void_p), 688, _ptr(dummy_in), 1, 688,
                                 _ptr(dummy_out), torch.cuda.current_device(), _stream())
    msg = lib.gb_last_error().decode()
    print("A2 max_degree 688: rc %d, %s" % (rc, msg))
    checks.state("gb_orderwise_filter at max_degree 688", rc, gb._lib.GB_ERR_ARGUMENT)
    checks.state("refused by the shared-memory bound", "shared-memory" in msg, True)
    checks.done()


@pytest.mark.gpu
def test_a3_degree_weights_and_realistic_orderwise_filter(gb, orc):
    """gb_scale_by_degree with Gaussian and Butterworth weights at config-5 size bit for bit against
    anm * w[max(r, c)]; the order-wise filter on Kaula-like data with orc.synthetic_filter_blocks(120), 500 epochs,
    per (epoch, order, cos | sin) block against the block's own output maximum."""
    checks = _Checks("A3")
    X = _coefficients(orc, 120, 500)
    Xd = _torch(X)
    deg = np.maximum(np.arange(121)[:, None], np.arange(121)[None, :])
    for label, flt in (("Gaussian 300 km", gb.Gaussian(300.0)), ("Butterworth 4 / 60", gb.Butterworth(4, 60))):
        w = flt.degree_weights(120)
        _same(checks, "degree weights, " + label, flt.filter_batch(Xd).cpu().numpy(), X * w[deg], _packed)
    blocks = orc.synthetic_filter_blocks(120)
    got = gb.OrderWiseFilter(blocks).filter_batch(Xd).cpu().numpy()
    ref = _orderwise(orc, blocks, X)
    rng = np.random.default_rng(13)
    worst = 0.0
    for e, r, c in zip(rng.integers(0, 500, 64), rng.integers(0, 121, 64), rng.integers(0, 121, 64)):
        m, n = (c, r) if c <= r else (r + 1, c)
        if n < 2:                                   # passed through, not filtered
            continue
        B = blocks[0 if m == 0 else 2 * m - 1 + (c > r)]
        vec = X[e, m:, m] if c <= r else X[e, m - 1, m:]
        exact = B[n - m, :121 - m].astype(np.longdouble) @ vec.astype(np.longdouble)
        col = ref[e, m:, m] if c <= r else ref[e, m - 1, m:]
        worst = max(worst, float(abs(ref[e, r, c] - exact) / np.abs(col).max()))
    checks.err("reference vs extended precision", worst, EXACT_TOL)
    err, where = 0.0, ""
    for m in range(121):
        for sine in ((False,) if m == 0 else (False, True)):
            g, f = (got[:, m - 1, m:], ref[:, m - 1, m:]) if sine else (got[:, m:, m], ref[:, m:, m])
            rel = np.abs(g - f).max(axis=1) / np.abs(f).max(axis=1)
            if not np.all(np.isfinite(g)):
                rel = np.full(rel.shape, np.inf)
            if rel.max() > err or not np.isfinite(rel.max()):
                err, where = float(rel.max()), "epoch %d, order %d %s" % (int(rel.argmax()), m, "sin" if sine else "cos")
    checks.err("realistic, per block (worst: %s)" % where, err, TOL_ORDERWISE)
    checks.done()


# ------------------------------------------------------------------------------ B. dense filter
@pytest.mark.gpu
def test_b1_dense_filter_vdk_size(gb, orc):
    """A dyadic non-symmetric W of the VDK size (min_degree 2, max_degree 96, K = 9405: 74 row tiles of 128), bit for
    bit on every epoch: 1, 121 and 241 epochs (one, two and three 120-column epoch tiles, the last ragged); input
    degree 60 (zero beyond it, output degree 60) and 120 (output truncated to 96); input degree 1 below min_degree
    (output: the passed-through corner only).  Every output starts NaN-filled."""
    import torch
    checks = _Checks("B1")
    nmin, nmax = 2, N
    K = (nmax + 1) ** 2 - nmin ** 2
    rng = np.random.default_rng(21)
    t0 = time.perf_counter()
    W = _dyadic_rows(rng, K, K, 12, -13)                      # 2^12 2^26 K < 2^52
    checks.state("W is not symmetric", bool(W[0, 1] != W[1, 0] or W[5, 9] != W[9, 5]), True)
    flt = gb.GeneralMatrix(W, nmin, nmax)
    X = _dyadic(rng, (241, nmax + 1, nmax + 1), 26, -60)
    ref = _dense_reference(W, nmin, nmax, X)
    print("B1 reference, degree 96: %.1f s" % (time.perf_counter() - t0))

    def run(x):
        lout = min(x.shape[-1], nmax + 1)
        out = torch.full((x.shape[0], lout, lout), float("nan"), dtype=torch.float64, device="cuda")
        res = flt.filter_batch(_torch(x), out=out)
        checks.state("out= buffer returned", res.data_ptr() == out.data_ptr(), True)
        return out.cpu().numpy()

    for E in (1, 121, 241):
        _same(checks, "input degree 96, %d epochs" % E, run(X[:E]), ref[:E], _packed)
    for lin, E in ((61, 121), (121, 130), (2, 5)):
        Xl = _dyadic(rng, (E, lin, lin), 26, -60)
        _same(checks, "input degree %d, %d epochs" % (lin - 1, E), run(Xl), _dense_reference(W, nmin, nmax, Xl), _packed)
    checks.done()


@pytest.mark.gpu
def test_b2_dense_filter_realistic_vdk(gb, orc):
    """The VDK matrix of a synthetic SPD normal matrix at degree 96 (min_degree 2) on Kaula-like data, 130 epochs,
    against float64 per (epoch, degree) relative to that degree's output maximum, with a longdouble guard."""
    checks = _Checks("B2")
    nmin, nmax = 2, N
    G, d = _factors(nmax, 22)
    G, d = G[nmin * nmin:] * 1e3, d[nmin * nmin:] * 1e9
    W = _vdk_low_rank(G, d, _kaula(nmin, nmax, 1e-2, 4.0))
    X = _coefficients(orc, nmax, 130, 200)
    x = orc.ravel_coefficients(X, nmin, nmax)
    Y = x @ W.T
    rng = np.random.default_rng(23)
    worst = 0.0
    for e, k in zip(rng.integers(0, 130, 64), rng.integers(0, W.shape[0], 64)):
        exact = W[k].astype(np.longdouble) @ x[e].astype(np.longdouble)
        worst = max(worst, float(abs(Y[e, k] - exact) / np.abs(Y[e]).max()))
    checks.err("reference vs extended precision", worst, EXACT_TOL)
    got = orc.ravel_coefficients(gb.GeneralMatrix(W, nmin, nmax).filter_batch(_torch(X)).cpu().numpy(), nmin, nmax)
    err, where = 0.0, ""
    for n in range(nmin, nmax + 1):
        sl = slice(n * n - nmin * nmin, (n + 1) ** 2 - nmin * nmin)
        rel = np.abs(got[:, sl] - Y[:, sl]).max(axis=1) / np.abs(Y[:, sl]).max(axis=1)
        if not np.all(np.isfinite(got[:, sl])):
            rel[:] = np.inf
        if not rel.max() <= err:
            err, where = float(rel.max()), "epoch %d, degree %d" % (int(rel.argmax()), n)
    checks.err("realistic VDK, per degree (worst: %s)" % where, err, TOL_DENSE)
    checks.done()


# ------------------------------------------------------------------------------ C. device reductions
def _rms_loop(v):
    """The reference's accumulation (gravityfield.py:1143-1172): s = s + v[e] * v[e] in epoch order, sqrt(s / E)."""
    s = np.zeros(v.shape[1])
    for e in range(v.shape[0]):
        s = s + v[e] * v[e]
    return np.sqrt(s / v.shape[0])


def _temporal_rms(gb, v):
    import torch
    out = torch.full((v.shape[1],), float("nan"), dtype=torch.float64, device="cuda")
    gb._lib.check(gb._lib.load().gb_temporal_rms(_ptr(v), v.shape[0], v.shape[1], _ptr(out), torch.cuda.current_device(),
                                                 _stream()))
    return out.cpu().numpy()


@pytest.mark.gpu
def test_c1_temporal_rms_bit_identical_to_the_reference_loop(gb, orc):
    """gb_temporal_rms on realistic float data is bit-identical to the reference's loop: 240 epochs on the 0.5 degree
    grid, 500 epochs on the 0.25 degree grid, one epoch, 1001 points; and gridded_rms end to end on the 0.5 degree
    grid equals that loop over the grids to_grid_batch returns for the same TimeSeries."""
    import torch
    checks = _Checks("C1")
    gen = torch.Generator(device="cuda").manual_seed(31)
    for E, P in ((240, 259200), (500, 1036800), (1, 259200), (240, 1001)):
        v = torch.randn((E, P), generator=gen, dtype=torch.float64, device="cuda") * 0.05 + 0.01
        got = _temporal_rms(gb, v)
        _same(checks, "%d epochs x %d points" % (E, P), got, _rms_loop(v.cpu().numpy()), lambda i: "point %d" % i[0])
        del v
    grid = gb.GeographicGrid(0.5, 0.5)
    data = []
    for e in range(48):
        pc = gb.PotentialCoefficients()
        pc.anm = orc.synthetic_coefficients(N, 300 + e)
        pc.epoch = datetime.datetime(2002, 4, 15) + datetime.timedelta(days=30.4375 * e)
        data.append(pc)
    ts = gb.TimeSeries(data)
    rms = gb.gridded_rms(ts, ts.epochs(), "ewh", grid)
    packed = np.stack([ts.evaluate_at(t).anm for t in ts.epochs()])
    vals = gb.to_grid_batch(packed, grid, "ewh", data[0].GM, data[0].R, device_output=True).reshape(48, -1).cpu().numpy()
    _same(checks, "gridded_rms, 48 epochs at degree 96", rms.values, _rms_loop(vals), lambda i: "point %d" % i[0])
    checks.done()


def _moments(gb, v, w, shift, E, P):
    import torch
    out = torch.full((max(E, 1), 2), float("nan"), dtype=torch.float64, device="cuda")
    rc = gb._lib.load().gb_weighted_moments(_ptr(v), _ptr(w), _ptr(shift) if shift is not None else None, E, P, _ptr(out),
                                            torch.cuda.current_device(), _stream())
    return rc, out.cpu().numpy()


def _moment_case(rng, E, P, zero_weights=0.0):
    """Values v = c_e + u (c_e an integer near 2^30: v needs 31 bits) with 9-bit u, 12-bit weights, shift c_e; the sums
    sum_p w u and sum_p w u^2 in exact integer arithmetic (below 2^50 at a million points).  A share of the points
    gets weight +0 or -0 and a NaN or +-Inf value."""
    import torch
    u = rng.integers(-511, 512, size=(E, P), dtype=np.int16)
    wi = rng.integers(1, 4096, size=P)
    c = rng.integers(2 ** 29, 2 ** 30, size=E)
    s1 = np.empty(E, dtype=np.int64)
    s2 = np.empty(E, dtype=np.int64)
    for e0 in range(0, E, 50):
        uu = u[e0:e0 + 50].astype(np.int64)
        s1[e0:e0 + 50] = uu @ wi
        s2[e0:e0 + 50] = (uu * uu) @ wi
    w = np.ldexp(wi.astype(float), -30)
    off = np.zeros(P, dtype=bool)
    if zero_weights:
        off = rng.uniform(size=P) < zero_weights
        w[off] = np.where(rng.uniform(size=off.sum()) < 0.5, 0.0, -0.0)
    v = (torch.as_tensor(u).cuda().to(torch.float64) + torch.as_tensor(c.astype(float)).cuda()[:, None]) * 2.0 ** -40
    if off.any():
        bad = torch.as_tensor(np.flatnonzero(off)).cuda()
        v[:, bad] = torch.as_tensor(rng.choice([np.nan, np.inf, -np.inf], size=(E, off.sum()))).cuda()
        s1 = s1 - np.asarray(u[:, off].astype(np.int64) @ wi[off])
        s2 = s2 - np.asarray((u[:, off].astype(np.int64) ** 2) @ wi[off])
    ref = np.stack((np.ldexp(s1.astype(float), -70), np.ldexp(s2.astype(float), -110)), axis=1)
    assert np.all(np.abs(s2) < 2 ** 52)
    return v, torch.as_tensor(w).cuda(), torch.as_tensor(np.ldexp(c.astype(float), -40)).cuda(), ref


@pytest.mark.gpu
def test_c2_weighted_moments_exact(gb, orc):
    """gb_weighted_moments with explicit shifts on dyadic data, both sums exact: 240 x 259 200 and 500 x 1 036 800;
    1 and 1000 points (most CTAs of the 64-partial stage without points) and 0 points (zeros); 65 535 epochs of 3
    points; 65 536 epochs refused; points with weight +0 or -0 ignored although their values are NaN or +-Inf."""
    import torch
    checks = _Checks("C2")
    rng = np.random.default_rng(41)
    where = lambda i: "epoch %d, %s" % (i[0], ("sum w (v - c)", "sum w (v - c)^2")[i[1]])
    for E, P, z in ((240, 259200, 0.1), (500, 1036800, 0.0), (7, 1000, 0.1), (7, 1, 0.0), (65535, 3, 0.0)):
        v, w, c, ref = _moment_case(rng, E, P, z)
        rc, got = _moments(gb, v, w, c, E, P)
        checks.state("return code, %d epochs x %d points" % (E, P), rc, 0)
        _same(checks, "%d epochs x %d points%s" % (E, P, ", 10 %% zero weights at NaN / Inf" if z else ""), got, ref, where)
        del v, w, c
    v = torch.zeros((7, 1), dtype=torch.float64, device="cuda")
    rc, got = _moments(gb, v, torch.zeros(1, dtype=torch.float64, device="cuda"),
                       torch.zeros(7, dtype=torch.float64, device="cuda"), 7, 0)
    checks.state("return code, 0 points", rc, 0)
    _same(checks, "7 epochs x 0 points: zeros", got, np.zeros((7, 2)), where)
    rc, _ = _moments(gb, v, v[0], None, 65536, 1)
    checks.state("gb_weighted_moments with 65 536 epochs", rc, gb._lib.GB_ERR_ARGUMENT)
    checks.done()


@pytest.mark.gpu
def test_c3_grid_statistics_with_mask(gb):
    """grid_statistics at 240 epochs on the 0.5 degree grid with a mask and NaN outside it, against mean, RMS and
    standard deviation in extended precision."""
    import torch
    checks = _Checks("C3")
    grid = gb.GeographicGrid(0.5, 0.5)
    rng = np.random.default_rng(42)
    mask = rng.uniform(size=grid.point_count) < 0.4
    gen = torch.Generator(device="cuda").manual_seed(43)
    v = torch.randn((240, grid.point_count), generator=gen, dtype=torch.float64, device="cuda") * 0.1 + 0.3
    vh = v.cpu().numpy()
    v[:, torch.as_tensor(~mask).cuda()] = float("nan")
    st = gb.grid_statistics(v, grid, mask)
    w = np.asarray(grid.area, dtype=np.longdouble)[mask]
    x = vh[:, mask].astype(np.longdouble)
    s0 = w.sum()
    mean = (x @ w) / s0
    ref = {"mean": mean, "rms": np.sqrt(((x * x) @ w) / s0), "std": np.sqrt((((x - mean[:, None]) ** 2) @ w) / s0)}
    for key in ("mean", "rms", "std"):
        got = np.asarray(st[key], dtype=np.longdouble)
        err = float(np.max(np.abs(got - ref[key]) / np.abs(ref[key]))) if np.all(np.isfinite(st[key])) else np.inf
        checks.err("240 epochs, masked, " + key, err, TOL_STATS)
    checks.done()


@pytest.mark.gpu
def test_c4_ravel_coefficients(gb, orc):
    """gb_ravel_coefficients of 240 packed sets bit for bit against orc.ravel_coefficients, N = 96, 180, 360 from
    degree 0, 2 and N."""
    import torch
    checks = _Checks("C4")
    rng = np.random.default_rng(44)
    lib = gb._lib.load()
    for nmax in (96, 180, 360):
        X = rng.standard_normal((240, nmax + 1, nmax + 1))
        Xd = _torch(X)
        for nmin in (0, 2, nmax):
            K = (nmax + 1) ** 2 - nmin ** 2
            out = torch.full((240, K), float("nan"), dtype=torch.float64, device="cuda")
            gb._lib.check(lib.gb_ravel_coefficients(_ptr(Xd), 240, nmax, nmin, _ptr(out), torch.cuda.current_device(),
                                                    _stream()))
            _same(checks, "N = %d, from degree %d" % (nmax, nmin), out.cpu().numpy(),
                  orc.ravel_coefficients(X, nmin, nmax), _raveled(nmin, nmax))
        del Xd
    checks.done()


def _quadratic_forms(gb, sigma, vec, K):
    import torch
    n = vec.shape[0]
    out = torch.full((max(n, 1),), float("nan"), dtype=torch.float64, device="cuda")
    gb._lib.check(gb._lib.load().gb_quadratic_forms(_ptr(sigma), K, _ptr(vec), n, _ptr(out), torch.cuda.current_device(),
                                                    _stream()))
    return out.cpu().numpy()[:n]


@pytest.mark.gpu
def test_c5_quadratic_forms(gb, orc):
    """gb_quadratic_forms with a dyadic non-symmetric Sigma (25 bits) and ternary vectors, exact (2^25 K^2 < 2^53):
    K = 9409 and 14 641 (more rows than 8 x 8 x SMs: every CTA loops over rows) with 1, 7, 8, 9, 16 and 17 vectors
    (passes of 8, the last ragged); K = 1, 5, 33; K = 0 gives zeros.  One realistic case at K = 9409 against the
    closed form ||G' a||^2 + (a o a) . d in extended precision."""
    import torch
    checks = _Checks("C5")
    rng = np.random.default_rng(45)
    sm = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    print("C5: %d SMs, row loop above K = %d" % (sm, 64 * sm))
    for K in (9409, 14641, 1, 5, 33):
        S = _dyadic_rows(rng, K, K, 25, -80)
        A = _dyadic(rng, (17, K), 1, -3)
        ref = np.einsum("bk,bk->b", A @ S, A)                         # exact
        Sd, Ad = _torch(S), _torch(A)
        del S
        for nv in ((1, 7, 8, 9, 16, 17) if K > 1000 else (17,)):
            _same(checks, "K = %d, %d vectors" % (K, nv), _quadratic_forms(gb, Sd, Ad[:nv].contiguous(), K), ref[:nv],
                  lambda i: "vector %d" % i[0])
        del Sd, Ad
    dummy = torch.zeros(1, dtype=torch.float64, device="cuda")
    _same(checks, "K = 0, 9 vectors: zeros", _quadratic_forms(gb, dummy, torch.zeros((9, 1), dtype=torch.float64,
                                                                                       device="cuda"), 0), np.zeros(9))
    G, d = _factors(N, 46)
    Sd = _sigma(torch, G, d)
    A = rng.standard_normal((17, G.shape[0])) / (np.repeat(np.arange(N + 1), 2 * np.arange(N + 1) + 1) + 1.0)
    got = _quadratic_forms(gb, Sd, _torch(A), G.shape[0])
    Al = A.astype(np.longdouble)
    y = Al @ G.astype(np.longdouble)
    exact = np.einsum("br,br->b", y, y) + (Al * Al) @ d.astype(np.longdouble)
    checks.err("realistic K = 9409, 17 vectors, per vector",
               float(np.max(np.abs(got - exact) / exact)) if np.all(np.isfinite(got)) else np.inf, TOL_QF)
    checks.done()


# ------------------------------------------------------------------------------ D. basin variances
def _adjoint_sweep(checks, label, plan, U, T, points, width, nmin, tol):
    """A' e_(i,j) for every point (i, j) of ``points`` in batches of ``width`` against U[i] o T[j], per point relative
    to the row maximum; coefficients below min_degree must be zero."""
    import torch
    rows, cols = _degreewise(nmin, plan.max_degree)
    R, C = torch.as_tensor(rows).cuda(), torch.as_tensor(cols).cuda()
    Ud, Td = _torch(U), _torch(T)
    vals = torch.zeros((width, plan.nlat, plan.nlon), dtype=torch.float64, device="cuda")
    worst, where, below = -1.0, "", 0.0
    t0 = time.perf_counter()
    for b0 in range(0, points.shape[0], width):
        pts = points[b0:b0 + width]
        E = pts.shape[0]
        I, J = torch.as_tensor(pts[:, 0]).cuda(), torch.as_tensor(pts[:, 1]).cuda()
        v = vals[:E]
        v.zero_()
        v[torch.arange(E, device="cuda"), I, J] = 1.0
        out = plan.analysis(v)
        if nmin > 0:
            below = max(below, float(out[:, :nmin, :nmin].abs().max()))
        got = out[:, R, C]
        ref = Ud[I] * Td[J]
        d = (got - ref).abs()
        err = d.amax(1) / ref.abs().amax(1)
        err[~torch.isfinite(got).all(1)] = float("inf")
        e = int(err.argmax())
        if not float(err[e]) <= worst:
            k = int(d[e].argmax())
            worst = float(err[e])
            where = "parallel %d, meridian %d, %s" % (pts[e, 0], pts[e, 1], _name(rows[k], cols[k]))
    torch.cuda.synchronize()
    print("%s %s: %.1f s" % (checks.case, label, time.perf_counter() - t0))
    checks.err("%s (worst: %s)" % (label, where), worst, tol)
    if nmin > 0:
        checks.state(label + ", largest coefficient below min_degree", below, 0.0)


@pytest.mark.gpu
def test_d1_every_row_of_the_adjoint(gb, orc):
    """Every point of the 0.5 degree grid at degree 96 (folded production grid, octant Fourier stage): min_degree 0 in
    1080 batches of 240, min_degree 2 in batches of 97 (ragged last batch).  Then every parallel at 3 meridians and
    every meridian at 3 parallels of a grid without four-fold meridian symmetry (721 meridians, 359 parallels: the
    unfolded longitude stage)."""
    from grates_b200 import plan as gplan
    checks = _Checks("D1")
    grid = gb.GeographicGrid(0.5, 0.5)
    plan = gplan.get_plan(grid, N, "ewh", variant="adjoint")
    checks.state("0.5 degree grid: plan.symmetric", plan.symmetric, True)
    allpts = np.stack(np.meshgrid(np.arange(360), np.arange(720), indexing="ij"), axis=-1).reshape(-1, 2)
    for nmin, width in ((0, 240), (2, 97)):
        U, T = _per_order_tables(orc, grid.parallels, grid.meridians, nmin, N)
        plan.set_adjoint(nmin)
        _adjoint_sweep(checks, "0.5 deg, min_degree %d, every point, batches of %d" % (nmin, width), plan, U, T, allpts,
                       width, nmin, TOL_ADJ)
    dlon = 2 * np.pi / 721
    grid = gb.RegularGrid(np.linspace(-np.pi + dlon / 2, np.pi - dlon / 2, 721), gb.GeographicGrid(0.5, 0.5).parallels[:-1])
    plan = gplan.get_plan(grid, N, "ewh", variant="adjoint")
    checks.state("721 x 359 grid: plan.symmetric", plan.symmetric, False)
    nlat, nlon = grid.parallels.size, grid.meridians.size
    pts = np.concatenate([np.stack((np.arange(nlat), np.full(nlat, j)), axis=1) for j in (0, 360, nlon - 1)] +
                         [np.stack((np.full(nlon, i), np.arange(nlon)), axis=1) for i in (0, 179, nlat - 1)])
    for nmin in (0, 2):
        U, T = _per_order_tables(orc, grid.parallels, grid.meridians, nmin, N)
        plan.set_adjoint(nmin)
        _adjoint_sweep(checks, "721 x 359, min_degree %d, partial sweep" % nmin, plan, U, T, pts, 240, nmin, TOL_ADJ)
    checks.done()


@pytest.mark.gpu
def test_d2_basin_variances_end_to_end(gb, orc):
    """basin_variances at the benchmark size: degree 96, the 0.5 degree grid, ewh, 17 basins (three passes of 8 in the
    quadratic forms, the last ragged) with one single-point basin, one global basin and one non-boolean weight mask;
    min_degree 0 and 2; Sigma = G G' + diag(d) as a CUDA tensor; basin by basin against the separable reference."""
    import torch
    checks = _Checks("D2")
    grid = gb.GeographicGrid(0.5, 0.5)
    nlat, nlon = 360, 720
    rng = np.random.default_rng(51)
    masks = np.zeros((17, nlat, nlon))
    for b in range(14):
        i0, j0 = rng.integers(0, nlat - 10), rng.integers(0, nlon - 10)
        masks[b, i0:i0 + rng.integers(1, 60), j0:j0 + rng.integers(1, 120)] = 1.0
    masks[14, 123, 456] = 1.0                                                   # single point
    masks[15] = 1.0                                                             # global
    masks[16, 40:200, 100:400] = rng.uniform(0.1, 2.0, (160, 300))              # weights, not a boolean mask
    masks = masks.reshape(17, -1)
    w = _basin_weights(masks, grid.area).reshape(17, nlat, nlon)
    G, d = _factors(N, 52)
    t0 = time.perf_counter()
    U, T = _per_order_tables(orc, grid.parallels, grid.meridians, 0, N)
    a = _functionals(U, T, w)
    checks.err("functionals vs extended precision", _functional_guard(U, T, w, a, 53), EXACT_TOL)
    print("D2 reference functionals: %.1f s" % (time.perf_counter() - t0))
    for nmin in (0, 2):
        o = nmin * nmin
        ab, Gn, dn = a[:, o:], G[o:], d[o:]
        y = ab @ Gn
        ref = np.einsum("br,br->b", y, y) + (ab * ab) @ dn
        s = _sigma(torch, Gn, dn)
        got = gb.basin_variances(s, grid, masks, nmin, N, "ewh", take_sqrt=False)
        rel = np.abs(got - ref) / ref if np.all(np.isfinite(got)) else np.full(17, np.inf)
        checks.err("17 basins, min_degree %d (worst: basin %d)" % (nmin, int(np.argmax(rel))), float(np.max(rel)), TOL_BASIN)
        del s
    checks.done()
