// Dense FP64 building blocks for the covariance PRODUCERS of the path (SURVEY 8 f4): the block Cholesky factorisation,
// sparse inverse and inverse of reference lstsq.py:698-717, 823-882 are loops over blocks that call
// scipy.linalg.cholesky, solve_triangular, inv and numpy's `@`.  These three entry points replace those four calls on
// device-resident blocks (row-major, arbitrary leading dimension, no alignment requirement beyond 8 bytes):
//
//   gb_dgemm         C = alpha op(A) op(B) + beta C      FP64 tensor cores (DMMA.8x8x4), 64 x 64 tiles, 16-deep chunks
//                                                       double-buffered through shared memory
//   gb_dpotrf_upper  A = W' W in place (upper W)         right-looking over 64-wide panels: one-CTA factorisation of
//                                                       the diagonal block, panel solve, trailing update with gb_dgemm
//   gb_dtrsm_upper   op(W) X = B in place                forward / backward substitution over 64-row blocks + gb_dgemm
//
// The Python mirror (grates_b200/lstsq.py: BlockMatrix, NormalEquations) keeps the reference's block loops and its
// sparsity bookkeeping and calls these per block.
#include "gb_common.cuh"

namespace {

constexpr int LG_T = 64;          // tile edge
constexpr int LG_KC = 16;         // contraction chunk
constexpr int LG_LD = LG_T + 4;   // shared pitch (= 4 mod 16: conflict-free DMMA fragments)

// tile[k][x] <- op(M)[x0 + x][k0 + k]  (zero outside the matrix); kcontig: memory runs along k (M[x][k]), else along x (M[k][x])
__device__ __forceinline__ void lg_fetch(double (&r)[8], const double* __restrict__ M, long long ld, bool kcontig,
                                         long long x0, long long k0, long long xn, long long kn) {
    const int t = threadIdx.x;
    if (kcontig) {
        const long long x = x0 + (t >> 1), kb = k0 + (t & 1) * 8;
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] = (x < xn && kb + j < kn) ? M[x * ld + kb + j] : 0.0;
    } else {
        const long long k = k0 + (t >> 3), xb = x0 + (t & 7) * 8;
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] = (k < kn && xb + j < xn) ? M[k * ld + xb + j] : 0.0;
    }
}
__device__ __forceinline__ void lg_stash(const double (&r)[8], double* tile, bool kcontig) {
    const int t = threadIdx.x;
    if (kcontig) {
        const int x = t >> 1, kb = (t & 1) * 8;
#pragma unroll
        for (int j = 0; j < 8; ++j) tile[(kb + j) * LG_LD + x] = r[j];
    } else {
        const int k = t >> 3, xb = (t & 7) * 8;
#pragma unroll
        for (int j = 0; j < 8; ++j) tile[k * LG_LD + xb + j] = r[j];
    }
}

// C[m][n] = alpha sum_k opA[m][k] opB[k][n] + beta C[m][n];  ta: A is stored [k][m], tb: B is stored [n][k].
// upper: tiles strictly below the diagonal are skipped (symmetric updates of an upper-triangular operand).
__global__ void __launch_bounds__(128)
gb_dgemm_kernel(int ta, int tb, long long m, long long n, long long k, double alpha, const double* __restrict__ A,
                long long lda, const double* __restrict__ B, long long ldb, double beta, double* __restrict__ C,
                long long ldc, int upper) {
    __shared__ double sA[2][LG_KC * LG_LD], sB[2][LG_KC * LG_LD];
    const long long m0 = (long long)blockIdx.y * LG_T, n0 = (long long)blockIdx.x * LG_T;
    if (upper && m0 >= n0 + LG_T) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wm = warp >> 1, wn = warp & 1, g = lane >> 2, q = lane & 3;
    const bool a_kc = !ta, b_kc = tb != 0;      // A[m][k] runs along k when not transposed; B[n][k] when transposed
    double acc[4][4][2];
#pragma unroll
    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
    double ra[8], rb[8];
    lg_fetch(ra, A, lda, a_kc, m0, 0, m, k);
    lg_fetch(rb, B, ldb, b_kc, n0, 0, n, k);
    lg_stash(ra, sA[0], a_kc);
    lg_stash(rb, sB[0], b_kc);
    __syncthreads();
    const long long chunks = (k + LG_KC - 1) / LG_KC;
    for (long long c = 0; c < chunks; ++c) {
        const int cur = (int)(c & 1);
        if (c + 1 < chunks) {
            lg_fetch(ra, A, lda, a_kc, m0, (c + 1) * LG_KC, m, k);
            lg_fetch(rb, B, ldb, b_kc, n0, (c + 1) * LG_KC, n, k);
        }
        const double* pa = sA[cur] + wm * 32 + g;
        const double* pb = sB[cur] + wn * 32 + g;
#pragma unroll
        for (int kk = 0; kk < LG_KC; kk += 4) {
            double a[4], b[4];
#pragma unroll
            for (int mi = 0; mi < 4; ++mi) a[mi] = pa[(kk + q) * LG_LD + mi * 8];
#pragma unroll
            for (int ni = 0; ni < 4; ++ni) b[ni] = pb[(kk + q) * LG_LD + ni * 8];
#pragma unroll
            for (int mi = 0; mi < 4; ++mi)
#pragma unroll
                for (int ni = 0; ni < 4; ++ni) gb::dmma_884(acc[mi][ni][0], acc[mi][ni][1], a[mi], b[ni]);
        }
        if (c + 1 < chunks) {
            lg_stash(ra, sA[cur ^ 1], a_kc);
            lg_stash(rb, sB[cur ^ 1], b_kc);
        }
        __syncthreads();
    }
#pragma unroll
    for (int mi = 0; mi < 4; ++mi) {
        const long long row = m0 + wm * 32 + mi * 8 + g;
        if (row >= m) continue;
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) {
            const long long col = n0 + wn * 32 + ni * 8 + 2 * q;
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                if (col + r >= n) continue;
                double* c = C + row * ldc + col + r;
                *c = (beta == 0.0) ? alpha * acc[mi][ni][r] : fma(alpha, acc[mi][ni][r], beta * *c);
            }
        }
    }
}

// Cholesky factor (upper, A = W' W) of one diagonal block of at most 64 x 64, in place; the strict lower triangle is
// zeroed (scipy.linalg.cholesky(lower=False) returns a clean upper factor).  info: first failing pivot (1-based, absolute).
__global__ void __launch_bounds__(256) gb_potrf64_kernel(double* __restrict__ A, long long lda, int nb, long long j0, int* info) {
    __shared__ double s[LG_T][LG_T + 1];
    __shared__ int bad;
    const int t = threadIdx.x;
    if (t == 0) bad = 0;
    for (int idx = t; idx < nb * nb; idx += blockDim.x) {
        const int i = idx / nb, j = idx % nb;
        s[i][j] = (j >= i) ? A[(size_t)i * lda + j] : 0.0;
    }
    __syncthreads();
    for (int kk = 0; kk < nb; ++kk) {
        if (t == 0) {
            const double d = s[kk][kk];
            if (!(d > 0.0)) {
                if (!bad) bad = kk + 1;
                s[kk][kk] = 1.0;         // keep going with finite numbers; the caller raises
            } else {
                s[kk][kk] = sqrt(d);
            }
        }
        __syncthreads();
        const double piv = s[kk][kk];
        for (int j = kk + 1 + t; j < nb; j += blockDim.x) s[kk][j] /= piv;
        __syncthreads();
        const int rem = nb - kk - 1;
        for (int idx = t; idx < rem * rem; idx += blockDim.x) {
            const int i = kk + 1 + idx / rem, j = kk + 1 + idx % rem;
            if (j >= i) s[i][j] = fma(-s[kk][i], s[kk][j], s[i][j]);
        }
        __syncthreads();
    }
    for (int idx = t; idx < nb * nb; idx += blockDim.x) {
        const int i = idx / nb, j = idx % nb;
        A[(size_t)i * lda + j] = s[i][j];
    }
    if (t == 0 && bad) atomicCAS(info, 0, (int)(j0 + bad));
}

// op(W) X = B for one diagonal block W (upper, nb <= 64) and 64 columns of B per CTA, in place.
// trans = 1: W' X = B (forward substitution), trans = 0: W X = B (backward substitution).
__global__ void __launch_bounds__(64) gb_trsm64_kernel(int trans, const double* __restrict__ W, long long ldw, int nb,
                                                      double* __restrict__ B, long long ldb, long long ncols) {
    extern __shared__ double s_dyn[];                  // 2 x 64 x 65 doubles (66.5 KB: opt-in dynamic shared memory)
    double (*sw)[LG_T + 1] = reinterpret_cast<double (*)[LG_T + 1]>(s_dyn);
    double (*sb)[LG_T + 1] = reinterpret_cast<double (*)[LG_T + 1]>(s_dyn + LG_T * (LG_T + 1));
    const int t = threadIdx.x;
    const long long c0 = (long long)blockIdx.x * LG_T;
    for (int idx = t; idx < nb * nb; idx += 64) sw[idx / nb][idx % nb] = W[(size_t)(idx / nb) * ldw + idx % nb];
    for (int i = 0; i < nb; ++i) sb[i][t] = (c0 + t < ncols) ? B[(size_t)i * ldb + c0 + t] : 0.0;
    __syncthreads();
    if (trans) {
        for (int r = 0; r < nb; ++r) {
            double v = sb[r][t];
            for (int s = 0; s < r; ++s) v = fma(-sw[s][r], sb[s][t], v);
            sb[r][t] = v / sw[r][r];
        }
    } else {
        for (int r = nb - 1; r >= 0; --r) {
            double v = sb[r][t];
            for (int s = r + 1; s < nb; ++s) v = fma(-sw[r][s], sb[s][t], v);
            sb[r][t] = v / sw[r][r];
        }
    }
    if (c0 + t < ncols)
        for (int i = 0; i < nb; ++i) B[(size_t)i * ldb + c0 + t] = sb[i][t];
}

__global__ void gb_zero_lower_kernel(double* __restrict__ A, long long n, long long lda) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
    if (j < i && i < n) A[i * lda + j] = 0.0;
}

constexpr size_t TRSM_SMEM = 2 * LG_T * (LG_T + 1) * sizeof(double);
int launch_trsm64(int trans, const double* W, long long ldw, int nb, double* B, long long ldb, long long ncols, cudaStream_t st) {
    GB_CUDA(cudaFuncSetAttribute(gb_trsm64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TRSM_SMEM));
    gb_trsm64_kernel<<<(unsigned)((ncols + LG_T - 1) / LG_T), 64, TRSM_SMEM, st>>>(trans, W, ldw, nb, B, ldb, ncols);
    GB_LAUNCH_CHECK();
    return GB_OK;
}

int launch_gemm(int ta, int tb, long long m, long long n, long long k, double alpha, const double* A, long long lda,
                const double* B, long long ldb, double beta, double* C, long long ldc, int upper, cudaStream_t st) {
    if (m <= 0 || n <= 0) return GB_OK;
    dim3 grid((unsigned)((n + LG_T - 1) / LG_T), (unsigned)((m + LG_T - 1) / LG_T));
    gb_dgemm_kernel<<<grid, 128, 0, st>>>(ta, tb, m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, upper);
    GB_LAUNCH_CHECK();
    return GB_OK;
}

}  // namespace

extern "C" int gb_dgemm(int trans_a, int trans_b, int64_t m, int64_t n, int64_t k, double alpha, const double* d_a,
                        int64_t lda, const double* d_b, int64_t ldb, double beta, double* d_c, int64_t ldc, int upper_only,
                        int device, void* stream) {
    GB_REQUIRE(m >= 0 && n >= 0 && k >= 0, "gb_dgemm: negative size");
    if (m == 0 || n == 0) return GB_OK;
    GB_REQUIRE(d_c && (k == 0 || (d_a && d_b)), "gb_dgemm: NULL pointer");
    GB_REQUIRE(ldc >= n && (k == 0 || (lda >= (trans_a ? m : k) && ldb >= (trans_b ? k : n))), "gb_dgemm: leading dimension too small");
    GB_REQUIRE((m + LG_T - 1) / LG_T <= 65535, "gb_dgemm: more than 65535 row tiles");
    GB_CUDA(cudaSetDevice(device));
    return launch_gemm(trans_a, trans_b, m, n, k, alpha, d_a, lda, d_b, ldb, beta, d_c, ldc, upper_only,
                       static_cast<cudaStream_t>(stream));
}

extern "C" int gb_dpotrf_upper(double* d_a, int64_t n, int64_t lda, int* d_info, int device, void* stream) {
    GB_REQUIRE(n >= 0 && lda >= n, "gb_dpotrf_upper: bad size");
    GB_REQUIRE(d_info != nullptr, "gb_dpotrf_upper: d_info is NULL");
    // the lower-triangle clear at the end takes one grid row per matrix row (at most 65535): refuse before any write
    GB_REQUIRE(n <= 65535, "gb_dpotrf_upper: blocks of more than 65535 rows are not supported");
    GB_CUDA(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    GB_CUDA(cudaMemsetAsync(d_info, 0, sizeof(int), st));
    if (n == 0) return GB_OK;
    GB_REQUIRE(d_a != nullptr, "gb_dpotrf_upper: NULL pointer");
    for (long long j0 = 0; j0 < n; j0 += LG_T) {
        const int nb = (int)((n - j0 < LG_T) ? (n - j0) : LG_T);
        double* diag = d_a + j0 * lda + j0;
        gb_potrf64_kernel<<<1, 256, 0, st>>>(diag, lda, nb, j0, d_info);
        GB_LAUNCH_CHECK();
        const long long rest = n - j0 - nb;
        if (rest > 0) {
            double* panel = diag + nb;                       // A[j0 .. j0+nb, j0+nb ..]
            {
                int rct = launch_trsm64(1, diag, lda, nb, panel, lda, rest, st);
                if (rct) return rct;
            }
            // trailing update of the upper triangle: A22 -= panel' panel
            int rc = launch_gemm(1, 0, rest, rest, nb, -1.0, panel, lda, panel, lda, 1.0, d_a + (j0 + nb) * lda + j0 + nb, lda,
                                 1, st);
            if (rc) return rc;
        }
    }
    // the strict lower triangle is not referenced above: clear it, scipy.linalg.cholesky(lower=False) returns a clean factor
    gb_zero_lower_kernel<<<dim3((unsigned)((n + 255) / 256), (unsigned)n), 256, 0, st>>>(d_a, n, lda);
    GB_LAUNCH_CHECK();
    return GB_OK;
}

extern "C" int gb_dtrsm_upper(int trans, const double* d_w, int64_t n, int64_t ldw, double* d_b, int64_t m, int64_t ldb,
                              int device, void* stream) {
    GB_REQUIRE(n >= 0 && m >= 0 && ldw >= n && ldb >= m, "gb_dtrsm_upper: bad size");
    if (n == 0 || m == 0) return GB_OK;
    GB_REQUIRE(d_w && d_b, "gb_dtrsm_upper: NULL pointer");
    GB_CUDA(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (trans) {
        for (long long j0 = 0; j0 < n; j0 += LG_T) {
            const int nb = (int)((n - j0 < LG_T) ? (n - j0) : LG_T);
            {
                int rct = launch_trsm64(1, d_w + j0 * ldw + j0, ldw, nb, d_b + j0 * ldb, ldb, m, st);
                if (rct) return rct;
            }
            const long long rest = n - j0 - nb;
            if (rest > 0) {        // B[below] -= W[j-block, below]' X[j-block]
                int rc = launch_gemm(1, 0, rest, m, nb, -1.0, d_w + j0 * ldw + j0 + nb, ldw, d_b + j0 * ldb, ldb, 1.0,
                                     d_b + (j0 + nb) * ldb, ldb, 0, st);
                if (rc) return rc;
            }
        }
    } else {
        for (long long j1 = n; j1 > 0;) {
            const int nb = (int)((j1 % LG_T) ? (j1 % LG_T) : LG_T);
            const long long j0 = j1 - nb;
            {
                int rct = launch_trsm64(0, d_w + j0 * ldw + j0, ldw, nb, d_b + j0 * ldb, ldb, m, st);
                if (rct) return rct;
            }
            if (j0 > 0) {          // B[above] -= W[above, j-block] X[j-block]
                int rc = launch_gemm(0, 0, j0, m, nb, -1.0, d_w + j0, ldw, d_b + j0 * ldb, ldb, 1.0, d_b, ldb, 0, st);
                if (rc) return rc;
            }
            j1 = j0;
        }
    }
    return GB_OK;
}
