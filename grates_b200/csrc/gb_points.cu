// Arbitrary point sets (the reference's IrregularGrid path): synthesis and covariance propagation.
//
//   gb_points_synthesis    replaces the irregular branch of PotentialCoefficients.to_grid
//                          (reference gravityfield.py:370-388): per point the Legendre recursion runs
//                          on the fly (bit-identical values), scaled by kn[p,n], contracted against an
//                          epoch tile of coefficients held in shared memory.
//   gb_points_covariance   replaces IrregularGrid.covariance_propagation (reference grid.py:1096-1120):
//                          var[p] = sum_ab F[p,a] Sigma[a,b] F[p,b] -- the direct, blocked
//                          diag(F Sigma F') of the north star: F tiles generated on the fly
//                          (gb_points_design), (F Sigma)' = Sigma' F' on the shared FP64 tensor-core
//                          GEMM (gb_gemm.cuh) with Sigma as the A operand and F' as the B operand, and
//                          the product with F folded into the epilogue with warp shuffles.
//                          2 P K^2 flops, nothing assumed about the point geometry.
//   gb_points_gradient_covariance
//                          the 3 x 3 covariance of grad V per point, J_p sym(Sigma) J_p' with the Jacobian
//                          J_p = F'_p T of the gradient (Cunningham's transform T, gb_gradient.cuh, followed by the
//                          degree-(N+1) synthesis row F'_p of a gradient point set): the same blocked GEMM with the
//                          three components of 40 points in a 120-column tile, the doubled lower triangle of the
//                          symmetric part of Sigma, and the three cross products of a point folded in the epilogue.
//   gb_points_gradient_normals
//                          the normal equations sum_p J~_p' W_p J~_p of acceleration observations (J~_p = Q_p J_p): the
//                          weighted, rotated Jacobian rows as both GEMM operands, contracted over observations on the
//                          tiles of the upper triangle only, added into N and mirrored.
//   gb_points_gravity_gradient_normals
//                          the same for the six observations of the gravity gradient tensor per point, on a
//                          gravity-gradient point set: one body templated on the order of the derivative, a row writer
//                          per order.
#include <vector>
#include <cmath>
#include "gb_common.cuh"
#include "gb_gemm.cuh"
#include "gb_gradient.cuh"

struct gb_points {
    int device = 0, nmax = 0, L = 0, npts = 0, sm_count = 0;
    double *d_ct = nullptr, *d_kn = nullptr, *d_pmm = nullptr, *d_cml = nullptr, *d_sml = nullptr;
    double *d_ra = nullptr, *d_rb = nullptr, *d_rc = nullptr;
};

namespace {

using gb::legendre_column;

// ---------------------------------------------------------------------------------------------
// synthesis at points: thread = point, CTA = 128 points x 8 epochs, loop over orders
// ---------------------------------------------------------------------------------------------
constexpr int PE = 8;

__global__ void __launch_bounds__(128)
gb_points_synthesis_kernel(const double* __restrict__ anm, double* __restrict__ out, const double* __restrict__ ct,
                           const double* __restrict__ kn, const double* __restrict__ pmm,
                           const double* __restrict__ cml, const double* __restrict__ sml,
                           const double* __restrict__ ra, const double* __restrict__ rb, const double* __restrict__ rc,
                           int L, int npts, int E) {
    extern __shared__ double s_coef[];   // [2][PE][L]
    double* sC = s_coef;
    double* sS = s_coef + PE * L;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    const int e0 = blockIdx.y * PE;
    const int ne = min(PE, E - e0);
    const bool live = p < npts;
    const double ctp = live ? ct[p] : 0.0;
    const double* kn_p = kn + (size_t)(live ? p : 0) * L;
    double v[PE];
#pragma unroll
    for (int e = 0; e < PE; ++e) v[e] = 0.0;
    for (int m = 0; m < L; ++m) {
        __syncthreads();
        const int cnt = L - m;
        for (int idx = threadIdx.x; idx < PE * cnt; idx += blockDim.x) {
            const int e = idx / cnt, nn = idx % cnt;
            const int n = m + nn;
            double c = 0.0, s = 0.0;
            if (e < ne) {
                const double* a = anm + (size_t)(e0 + e) * L * L;
                c = a[(size_t)n * L + m];
                if (m > 0) s = a[(size_t)(m - 1) * L + n];
            }
            sC[e * L + nn] = c;
            sS[e * L + nn] = s;
        }
        __syncthreads();
        if (!live) continue;
        double ac[PE], as[PE];
#pragma unroll
        for (int e = 0; e < PE; ++e) ac[e] = as[e] = 0.0;
        legendre_column(m, L, ctp, pmm[(size_t)p * L + m], ra, rb, rc, [&](int n, double pn) {
            const double pk = __dmul_rn(pn, kn_p[n]);
            const int nn = n - m;
#pragma unroll
            for (int e = 0; e < PE; ++e) {
                ac[e] = fma(pk, sC[e * L + nn], ac[e]);
                as[e] = fma(pk, sS[e * L + nn], as[e]);
            }
        });
        const double cm = cml[(size_t)p * L + m], sm = sml[(size_t)p * L + m];
#pragma unroll
        for (int e = 0; e < PE; ++e) v[e] = fma(cm, ac[e], fma(sm, as[e], v[e]));
    }
    if (live)
        for (int e = 0; e < ne; ++e) out[(size_t)(e0 + e) * npts + p] = v[e];
}

// ---------------------------------------------------------------------------------------------
// design matrix F^T as GEMM tiles [point tile of tn][a][ld], a = degree-wise index - nmin^2: the A operand
// (tn = GB_TM, ld = GB_LDA) of the point synthesis, the B operand (GB_S2_TN, GB_S2_LDB) of the point covariance
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
gb_points_design(double* __restrict__ FT, const double* __restrict__ ct, const double* __restrict__ kn,
                 const double* __restrict__ pmm, const double* __restrict__ cml, const double* __restrict__ sml,
                 const double* __restrict__ ra, const double* __restrict__ rb, const double* __restrict__ rc, int L,
                 int nmin, int npts, int rows, int p0, int tn, int ld) {
    const int p = p0 + blockIdx.x * blockDim.x + threadIdx.x;      // tiles are numbered from point p0
    const int m = blockIdx.y;
    if (p >= npts) return;
    const double* kn_p = kn + (size_t)p * L;
    const double cm = cml[(size_t)p * L + m], sm = sml[(size_t)p * L + m];
    const int off = nmin * nmin;
    double* col = FT + (size_t)((p - p0) / tn) * rows * ld + (p - p0) % tn;
    legendre_column(m, L, ct[p], pmm[(size_t)p * L + m], ra, rb, rc, [&](int n, double pn) {
        if (n < nmin) return;
        const double pk = __dmul_rn(pn, kn_p[n]);
        const int a = n * n + (m == 0 ? 0 : 2 * m - 1) - off;
        col[(size_t)a * ld] = __dmul_rn(pk, cm);
        if (m > 0) col[(size_t)(a + 1) * ld] = __dmul_rn(pk, sm);
    });
}

// ---------------------------------------------------------------------------------------------
// adjoint: design matrix as the GEMM A operand, F[a][p] in tiles [coefficient tile][p][GB_LDA] (K loop over points),
// and the point values as B tiles [epoch tile][p][GB_S2_LDB]
// ---------------------------------------------------------------------------------------------
// CTA = one point, thread = order m, all threads walk the degrees n together: for a fixed n the entries
// a = n^2 .. (n+1)^2 - 1 of the point's row are contiguous, so the stores coalesce.  The recursion is
// gb::legendre_column's, step for step (bit-identical values).  Where the row goes is the layout's business:
struct AdjointTiles {      // GEMM A operand [coefficient tile][point][GB_LDA]; rows beyond the last point are zeroed
    double* at;
    int rows;
    static constexpr bool pad_rows = true;
    __device__ __forceinline__ double* operator()(long long a, int pp) const { return at + gb_ab_offset(a, pp, rows); }
};
struct DenseRows {         // row-major [point][K'], K' = L^2 - nmin^2 (Grid.synthesis_matrix, reference grid.py:412-443)
    double* out;
    long long kc, off;
    static constexpr bool pad_rows = false;
    __device__ __forceinline__ double* operator()(long long a, int pp) const { return out + (size_t)pp * kc + (a - off); }
};

template <class Layout>
__global__ void __launch_bounds__(1024)
gb_points_design_rows(Layout row, const double* __restrict__ ct, const double* __restrict__ kn,
                      const double* __restrict__ pmm, const double* __restrict__ cml, const double* __restrict__ sml,
                      const double* __restrict__ ra, const double* __restrict__ rb, const double* __restrict__ rc, int L,
                      int nmin, int npts, int p0) {
    const int pp = blockIdx.x;
    const int p = p0 + pp;
    if (p >= npts) {
        if (Layout::pad_rows)
            for (long long a = threadIdx.x; a < (long long)L * L; a += blockDim.x) *row(a, pp) = 0.0;
        return;
    }
    const double ctp = ct[p];
    const double* kn_p = kn + (size_t)p * L;
    for (int m0 = threadIdx.x & ~31; m0 < L; m0 += blockDim.x) {        // the warp's orders m0 .. m0 + 31
        const int m = m0 + (threadIdx.x & 31);
        if (m >= L) continue;
        const double cm = cml[(size_t)p * L + m], sm = sml[(size_t)p * L + m];
        double p1 = 0.0, p2 = 0.0;
        for (int n = m0; n < L; ++n) {                                  // same n across the warp at every step
            if (n < m) continue;
            double v;
            if (n == m) v = pmm[(size_t)p * L + m];
            else if (n == m + 1) v = __dmul_rn(__dmul_rn(rc[n], ctp), p1);
            else v = __dsub_rn(__dmul_rn(__dmul_rn(ra[(size_t)n * L + m], ctp), p1), __dmul_rn(rb[(size_t)n * L + m], p2));
            p2 = p1;
            p1 = v;
            if (n < nmin) continue;
            const double pk = __dmul_rn(v, kn_p[n]);
            const long long a = (long long)n * n + (m == 0 ? 0 : 2 * m - 1);
            *row(a, pp) = __dmul_rn(pk, cm);
            if (m > 0) *row(a + 1, pp) = __dmul_rn(pk, sm);
        }
    }
}

__global__ void __launch_bounds__(256)
gb_points_value_tiles(const double* __restrict__ values, double* __restrict__ Bt, int npts, int p0, int count, int rows, int E,
                      int tn, int ldb) {
    const int pp = blockIdx.x * blockDim.x + threadIdx.x;
    const int e = blockIdx.y;
    if (pp >= count) return;
    Bt[((size_t)(e / tn) * rows + pp) * ldb + e % tn] = values[(size_t)e * npts + p0 + pp];
}

// out[p] = (sqrt of) the sum of the point's partial sums, in slot order: bit-identical from run to run
__global__ void gb_points_finish(const double* __restrict__ part, double* __restrict__ out, int nslots, int n, int take_sqrt) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double v = 0.0;
    for (int s = 0; s < nslots; ++s) v += part[(size_t)i * nslots + s];
    out[i] = take_sqrt ? sqrt(v) : v;
}

template <typename T>
int upload(T** d, const std::vector<T>& h) {
    GB_CUDA(cudaMalloc(reinterpret_cast<void**>(d), (h.size() ? h.size() : 1) * sizeof(T)));
    GB_CUDA(cudaMemcpy(*d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
    return GB_OK;
}

}  // namespace

extern "C" int gb_points_create(gb_points** out, int nmax, int npts, const double* cos_theta, const double* sin_theta,
                                const double* kn, const double* cos_mlon, const double* sin_mlon, int device) {
    GB_REQUIRE(out != nullptr, "gb_points_create: out is NULL");
    *out = nullptr;
    GB_REQUIRE(nmax >= 0 && nmax <= 2047, "gb_points_create: nmax=%d out of range [0, 2047]", nmax);
    GB_REQUIRE(npts >= 1, "gb_points_create: empty point set");
    GB_REQUIRE(cos_theta && sin_theta && kn && cos_mlon && sin_mlon, "gb_points_create: NULL table pointer");
    int ndev = 0;
    GB_CUDA(cudaGetDeviceCount(&ndev));
    GB_REQUIRE(device >= 0 && device < ndev, "gb_points_create: device %d not available (%d visible)", device, ndev);
    GB_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    GB_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return gb_set_error(GB_ERR_UNSUPPORTED, "gb_points_create: device %d is sm_%d%d; built for sm_100a", device,
                            prop.major, prop.minor);
    gb_points* p = new gb_points();
    p->device = device;
    p->nmax = nmax;
    p->L = nmax + 1;
    p->npts = npts;
    p->sm_count = prop.multiProcessorCount;
    const int L = p->L;
    std::vector<double> ra, rb, rc, pmm;
    gb_recursion_tables(nmax, npts, sin_theta, ra, rb, rc, pmm);
    const size_t tl = (size_t)npts * L;
    int rc_ = GB_OK;
    if ((rc_ = upload(&p->d_ct, std::vector<double>(cos_theta, cos_theta + npts))) ||
        (rc_ = upload(&p->d_kn, std::vector<double>(kn, kn + tl))) || (rc_ = upload(&p->d_pmm, pmm)) ||
        (rc_ = upload(&p->d_cml, std::vector<double>(cos_mlon, cos_mlon + tl))) ||
        (rc_ = upload(&p->d_sml, std::vector<double>(sin_mlon, sin_mlon + tl))) || (rc_ = upload(&p->d_ra, ra)) ||
        (rc_ = upload(&p->d_rb, rb)) || (rc_ = upload(&p->d_rc, rc))) {
        gb_points_destroy(p);
        return rc_;
    }
    *out = p;
    return GB_OK;
}

extern "C" int gb_points_destroy(gb_points* p) {
    if (!p) return GB_OK;
    cudaSetDevice(p->device);
    cudaFree(p->d_ct); cudaFree(p->d_kn); cudaFree(p->d_pmm); cudaFree(p->d_cml); cudaFree(p->d_sml);
    cudaFree(p->d_ra); cudaFree(p->d_rb); cudaFree(p->d_rc);
    delete p;
    return GB_OK;
}

// epilogue of the batched point synthesis: out[e][p0 + row]
struct PointStore {
    double* out;
    long long npts;
    int p0, count, E;
    __device__ __forceinline__ void operator()(long long row, int col, double v0, double v1) const {
        if (row >= count) return;
        double* o = out + (size_t)col * npts + p0 + row;
        if (col < E) *o = v0;
        if (col + 1 < E) o[npts] = v1;
    }
};

// epilogue of the point covariance: the GEMM rows are the columns b of Sigma, its columns the points of a block, so that
// C[b][p] = (F Sigma)[p][b].  part[p][slot] = sum_b C[b][p] F[p][b] over the warp's 32 rows b, with F[p][b] read back from
// the design tiles (the B operand); slot = (row tile, warp row), one writer per slot.  gb_points_finish adds the slots in
// order.
struct PointQuadForm {
    static constexpr bool whole_tile = true;
    const double* ft;    // design tiles [point tile][rows][GB_S2_LDB]
    double* part;        // [count][nslots]
    long long K;         // coefficients (rows b >= K are padding)
    int rows, count, nslots;
    __device__ __forceinline__ const double* prepare(long long, int nt, int col_base) const {
        return ft + (size_t)nt * rows * GB_S2_LDB + (col_base - nt * GB_S2_TN);
    }
    __device__ __forceinline__ void tile(const double* f, long long row_base, int col_base, double (&acc)[4][5][2]) const {
        // the thread's four rows first, then over g; the sums go to acc[0] (a second set of 10 sums spills at 128 registers)
#pragma unroll
        for (int mi = 0; mi < 4; ++mi) {
            const long long b = row_base + mi * 8;
#pragma unroll
            for (int ni = 0; ni < 5; ++ni) {
                const double2 fb = b < K ? __ldg(reinterpret_cast<const double2*>(f + (size_t)b * GB_S2_LDB + ni * 8))
                                         : make_double2(0.0, 0.0);
                acc[0][ni][0] = mi ? fma(acc[mi][ni][0], fb.x, acc[0][ni][0]) : acc[0][ni][0] * fb.x;
                acc[0][ni][1] = mi ? fma(acc[mi][ni][1], fb.y, acc[0][ni][1]) : acc[0][ni][1] * fb.y;
            }
        }
#pragma unroll
        for (int ni = 0; ni < 5; ++ni)
#pragma unroll
            for (int r = 0; r < 2; ++r)
#pragma unroll
                for (int o = 4; o < 32; o <<= 1) acc[0][ni][r] += __shfl_xor_sync(0xffffffffu, acc[0][ni][r], o);
        if ((threadIdx.x & 31) < 4) {      // g = 0
            const int slot = (int)(row_base >> 5);
#pragma unroll
            for (int ni = 0; ni < 5; ++ni)
#pragma unroll
                for (int r = 0; r < 2; ++r) {
                    const int pp = col_base + ni * 8 + r;
                    if (pp < count) part[(size_t)pp * nslots + slot] = acc[0][ni][r];
                }
        }
    }
};

// Epoch batches at arbitrary points as a GEMM: the design tiles F^T of a block of points are generated once (on-the-fly
// recursion, gb_points_design) and multiplied with ALL epochs on the DMMA GEMM, instead of re-running the recursion for
// every eight epochs.  2 P K E flops; the design matrix only ever exists for one block of points.
static int points_synthesis_gemm(gb_points* p, const double* d_anm, int E, double* d_out, cudaStream_t st) {
    const int L = p->L;
    const long long K = (long long)L * L;
    const int Kp = (int)((K + 3) / 4 * 4);
    const int n_ct = (E + GB_S2_TN - 1) / GB_S2_TN;
    int tiles_per_block = 2 * p->sm_count / n_ct;                 // about two waves of GEMM tiles per block
    if (tiles_per_block < 8) tiles_per_block = 8;
    const int n_mtiles_all = (p->npts + GB_TM - 1) / GB_TM;
    if (tiles_per_block > n_mtiles_all) tiles_per_block = n_mtiles_all;
    gb_scratch scratch(st);
    double *d_ft = nullptr, *d_bt = nullptr;
    const size_t ft_elems = (size_t)tiles_per_block * Kp * GB_LDA;
    const size_t bt_elems = (size_t)n_ct * Kp * GB_S2_LDB;
    GB_CUDA(scratch.alloc(&d_ft, ft_elems));
    GB_CUDA(scratch.alloc(&d_bt, bt_elems));
    GB_CUDA(cudaMemsetAsync(d_bt, 0, bt_elems * sizeof(double), st));
    int rc = gb_launch_ravel_tiles(d_anm, d_bt, L, 0, K, Kp, E, st);
    if (rc) return rc;
    for (int t0 = 0; t0 < n_mtiles_all; t0 += tiles_per_block) {
        const int nt = (n_mtiles_all - t0 < tiles_per_block) ? (n_mtiles_all - t0) : tiles_per_block;
        const int p0 = t0 * GB_TM;
        const int count = (p->npts - p0 < nt * GB_TM) ? (p->npts - p0) : nt * GB_TM;
        GB_CUDA(cudaMemsetAsync(d_ft, 0, (size_t)nt * Kp * GB_LDA * sizeof(double), st));   // padding rows / points
        dim3 grid((count + 127) / 128, L);
        gb_points_design<<<grid, 128, 0, st>>>(d_ft, p->d_ct, p->d_kn, p->d_pmm, p->d_cml, p->d_sml, p->d_ra, p->d_rb,
                                              p->d_rc, L, 0, p0 + count, Kp, p0, GB_TM, GB_LDA);
        GB_LAUNCH_CHECK();
        gbgemm::Shape sh;
        sh.A_t = d_ft;
        sh.a_rows = Kp;
        sh.a_koff_mul = 0;
        sh.tiles_per_group = 1;
        sh.B_t = d_bt;
        sh.b_rows = Kp;
        sh.klen = Kp;
        sh.n_mtiles = nt;
        sh.n_ntiles = n_ct;
        if ((rc = gbgemm::launch(sh, PointStore{d_out, p->npts, p0, count, E}, p->sm_count, st))) return rc;
    }
    return GB_OK;
}

extern "C" int gb_points_synthesis(gb_points* p, const double* d_anm, int n_epochs, double* d_out, void* stream) {
    GB_REQUIRE(p != nullptr, "gb_points_synthesis: point set is NULL");
    GB_REQUIRE(n_epochs >= 0, "gb_points_synthesis: n_epochs=%d is negative", n_epochs);
    if (n_epochs == 0) return GB_OK;
    GB_REQUIRE(d_anm && d_out, "gb_points_synthesis: NULL device pointer");
    GB_CUDA(cudaSetDevice(p->device));
    if (n_epochs >= 16 && !gb_env_flag("GB_POINTS_SIMPLE")) {
        gb_retain_pool_memory(p->device);
        return points_synthesis_gemm(p, d_anm, n_epochs, d_out, static_cast<cudaStream_t>(stream));
    }
    dim3 grid((p->npts + 127) / 128, (n_epochs + PE - 1) / PE);
    const size_t smem = (size_t)2 * PE * p->L * sizeof(double);
    if (smem > 48 * 1024)
        GB_CUDA(cudaFuncSetAttribute(gb_points_synthesis_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    gb_points_synthesis_kernel<<<grid, 128, smem, static_cast<cudaStream_t>(stream)>>>(
        d_anm, d_out, p->d_ct, p->d_kn, p->d_pmm, p->d_cml, p->d_sml, p->d_ra, p->d_rb, p->d_rc, p->L, p->npts,
        n_epochs);
    GB_LAUNCH_CHECK();
    return GB_OK;
}

// Adjoint of the point synthesis: anm_e[n, m] = sum_p F[p, (n, m)] v_e[p]  (the sum over nodal points of
// RadialBasisFunctions.to_potential_coefficients, reference gravityfield.py:707-724, with the plan's per-point
// degree factors as the upward continuation).  One GEMM per block of points on the DMMA kernel, K loop over the
// points of the block; blocks accumulate in launch order, so the result is deterministic.  NI: column fragments per
// warp (epoch tile of 24 NI columns) -- a single value set does not pay for a 120-column tile.
template <int NI>
static int points_adjoint_blocks(gb_points* p, const double* d_values, int E, double* d_anm, cudaStream_t st) {
    constexpr int TN = gbgemm::tile_n(NI), LDB = gbgemm::tile_ldb(NI);
    const int L = p->L;
    const long long K = (long long)L * L;
    const int n_mtiles = (int)((K + GB_TM - 1) / GB_TM);
    const int n_ct = (E + TN - 1) / TN;
    // points per block: A operand of about 512 MB, at least one k chunk
    long long pb = (512LL << 20) / ((long long)n_mtiles * GB_LDA * sizeof(double));
    pb = pb / 128 * 128;
    if (pb < 128) pb = 128;
    if (pb > 16384) pb = 16384;
    if (pb > (p->npts + 3) / 4 * 4) pb = (p->npts + 3) / 4 * 4;
    gb_scratch scratch(st);
    double *d_at = nullptr, *d_bt = nullptr;
    GB_CUDA(scratch.alloc(&d_at, (size_t)n_mtiles * pb * GB_LDA));
    GB_CUDA(scratch.alloc(&d_bt, (size_t)n_ct * pb * LDB));
    GB_CUDA(cudaMemsetAsync(d_anm, 0, (size_t)E * K * sizeof(double), st));
    for (int p0 = 0; p0 < p->npts; p0 += (int)pb) {
        const int count = (p->npts - p0 < pb) ? (p->npts - p0) : (int)pb;
        const int rows = (count + 3) / 4 * 4;
        GB_CUDA(cudaMemsetAsync(d_bt, 0, (size_t)n_ct * rows * LDB * sizeof(double), st));
        const int threads = L >= 1024 ? 1024 : (L + 31) / 32 * 32;
        gb_points_design_rows<<<rows, threads, 0, st>>>(AdjointTiles{d_at, rows}, p->d_ct, p->d_kn, p->d_pmm, p->d_cml,
                                                       p->d_sml, p->d_ra, p->d_rb, p->d_rc, L, 0, p0 + count, p0);
        GB_LAUNCH_CHECK();
        dim3 vgrid((count + 255) / 256, E);
        gb_points_value_tiles<<<vgrid, 256, 0, st>>>(d_values, d_bt, p->npts, p0, count, rows, E, TN, LDB);
        GB_LAUNCH_CHECK();
        gbgemm::Shape sh;
        sh.A_t = d_at;
        sh.a_rows = rows;
        sh.a_koff_mul = 0;
        sh.tiles_per_group = 1;
        sh.B_t = d_bt;
        sh.b_rows = rows;
        sh.klen = rows;
        sh.n_mtiles = n_mtiles;
        sh.n_ntiles = n_ct;
        int rc = gbgemm::launch<gbgemm::UnravelStore<true>, NI>(sh, gbgemm::UnravelStore<true>{d_anm, K, 0, L, E},
                                                               p->sm_count, st);
        if (rc) return rc;
    }
    return GB_OK;
}

extern "C" int gb_points_adjoint(gb_points* p, const double* d_values, int n_epochs, double* d_anm, void* stream) {
    GB_REQUIRE(p != nullptr, "gb_points_adjoint: point set is NULL");
    GB_REQUIRE(n_epochs >= 0, "gb_points_adjoint: n_epochs=%d is negative", n_epochs);
    if (n_epochs == 0) return GB_OK;
    GB_REQUIRE(d_values && d_anm, "gb_points_adjoint: NULL device pointer");
    GB_CUDA(cudaSetDevice(p->device));
    gb_retain_pool_memory(p->device);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (n_epochs <= gbgemm::tile_n(1)) return points_adjoint_blocks<1>(p, d_values, n_epochs, d_anm, st);
    if (n_epochs <= gbgemm::tile_n(2)) return points_adjoint_blocks<2>(p, d_values, n_epochs, d_anm, st);
    return points_adjoint_blocks<5>(p, d_values, n_epochs, d_anm, st);
}

// Dense synthesis operator of the point set, [npts][K'] row-major in degree-wise order (reference grid.py:412-443 with
// IrregularGrid.synthesis_matrix_per_order, grid.py:957-991).
extern "C" int gb_points_synthesis_matrix(gb_points* p, int nmin, double* d_out, void* stream) {
    GB_REQUIRE(p != nullptr, "gb_points_synthesis_matrix: point set is NULL");
    GB_REQUIRE(nmin >= 0 && nmin <= p->nmax, "gb_points_synthesis_matrix: nmin=%d out of range [0, %d]", nmin, p->nmax);
    GB_REQUIRE(d_out != nullptr, "gb_points_synthesis_matrix: NULL device pointer");
    GB_CUDA(cudaSetDevice(p->device));
    const int L = p->L;
    const long long off = (long long)nmin * nmin;
    const int threads = L >= 1024 ? 1024 : (L + 31) / 32 * 32;
    gb_points_design_rows<<<p->npts, threads, 0, static_cast<cudaStream_t>(stream)>>>(
        DenseRows{d_out, (long long)L * L - off, off}, p->d_ct, p->d_kn, p->d_pmm, p->d_cml, p->d_sml, p->d_ra, p->d_rb,
        p->d_rc, L, nmin, p->npts, 0);
    GB_LAUNCH_CHECK();
    return GB_OK;
}

// Sigma as the GEMM A operand, tiles [b tile][a][GB_LDA] with A[k = a][row = b] = Sigma[a][b] (a row tile holds runs of 128
// consecutive entries of the rows of Sigma), zero beyond K' in a and b.  For a symmetric Sigma only its lower triangle is
// kept, the off-diagonal entries doubled:  x' S x = sum_b S_bb x_b^2 + 2 sum_{a>b} S_ab x_a x_b, so that row tile j only
// needs k = a >= 128 j.
enum SigmaTiles { SIGMA_FULL = 0, SIGMA_LOWER = 1, SIGMA_SYMMETRISED_LOWER = 2 };
// SIGMA_LOWER: Sigma is stated symmetric, below the diagonal 2 Sigma_ab.  SIGMA_SYMMETRISED_LOWER: the same for the
// symmetric part (Sigma + Sigma') / 2 of any Sigma, Sigma_ab + Sigma_ba below the diagonal; bit-identical to SIGMA_LOWER
// for an exactly symmetric Sigma.
__global__ void __launch_bounds__(GB_TM)
gb_points_sigma_tiles(const double* __restrict__ sigma, double* __restrict__ St, long long Kc, int Kp, int mode) {
    const long long a = blockIdx.x;
    const long long b = (long long)blockIdx.y * GB_TM + threadIdx.x;
    double v = 0.0;
    if (a < Kc && b < Kc) {
        v = sigma[(size_t)a * Kc + b];
        if (mode != SIGMA_FULL)
            v = (a > b) ? v + (mode == SIGMA_LOWER ? v : sigma[(size_t)b * Kc + a]) : (a == b ? v : 0.0);
    }
    St[gb_ab_offset(b, (int)a, Kp)] = v;
}

extern "C" int gb_points_covariance(gb_points* p, const double* d_sigma, int nmin, double* d_out, int flags,
                                    void* stream) {
    const int take_sqrt = flags & GB_COV_SQRT;
    const int lower = (flags & GB_COV_SYMMETRIC) ? SIGMA_LOWER : SIGMA_FULL;
    GB_REQUIRE(p != nullptr, "gb_points_covariance: point set is NULL");
    GB_REQUIRE(nmin >= 0 && nmin <= p->nmax, "gb_points_covariance: min_degree=%d outside [0, %d]", nmin, p->nmax);
    GB_REQUIRE(d_sigma && d_out, "gb_points_covariance: NULL device pointer");
    GB_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int L = p->L;
    const long long Kc = (long long)L * L - (long long)nmin * nmin;   // coefficients
    const int Kp = (int)((Kc + 3) / 4 * 4);                            // padded to whole k4 steps
    const int n_btiles = (int)((Kc + GB_TM - 1) / GB_TM);              // GEMM row tiles: columns b of Sigma
    const int n_ptiles_all = (p->npts + GB_S2_TN - 1) / GB_S2_TN;       // GEMM column tiles: points
    // the design matrix only ever exists for one block of points (several waves of GEMM tiles): 75 KB per point at
    // degree 96 would otherwise be 12 GB for a 0.5-degree Reuter grid
    int tiles_per_block = 4 * p->sm_count / n_btiles;
    if (tiles_per_block < 16) tiles_per_block = 16;
    if (tiles_per_block > n_ptiles_all) tiles_per_block = n_ptiles_all;
    const int nslots = n_btiles * gbgemm::WM;
    double *d_st = nullptr, *d_ft = nullptr, *d_part = nullptr;
    gb_retain_pool_memory(p->device);
    gb_scratch scratch(st);
    GB_CUDA(scratch.alloc(&d_st, (size_t)n_btiles * Kp * GB_LDA));
    GB_CUDA(scratch.alloc(&d_ft, (size_t)tiles_per_block * Kp * GB_S2_LDB));
    GB_CUDA(scratch.alloc(&d_part, (size_t)tiles_per_block * GB_S2_TN * nslots));
    gb_points_sigma_tiles<<<dim3((unsigned)Kp, (unsigned)n_btiles), GB_TM, 0, st>>>(d_sigma, d_st, Kc, Kp, lower);
    GB_LAUNCH_CHECK();
    gbgemm::Shape sh;
    sh.A_t = d_st;
    sh.a_rows = Kp;
    sh.a_koff_mul = 0;
    sh.tiles_per_group = 1;
    sh.B_t = d_ft;
    sh.b_rows = Kp;
    sh.klen = Kp;
    sh.n_mtiles = n_btiles;
    if (lower) {                // row tile j starts its contraction at k = 128 j (the rows above are zeros)
        sh.mt_kstart_mod = n_btiles;
        sh.mt_kstart_mul = GB_TM;
    }
    for (int t0 = 0; t0 < n_ptiles_all; t0 += tiles_per_block) {
        const int n_ptiles = (n_ptiles_all - t0 < tiles_per_block) ? (n_ptiles_all - t0) : tiles_per_block;
        const int p0 = t0 * GB_S2_TN;
        const int count = (p->npts - p0 < n_ptiles * GB_S2_TN) ? (p->npts - p0) : n_ptiles * GB_S2_TN;
        GB_CUDA(cudaMemsetAsync(d_ft, 0, (size_t)n_ptiles * Kp * GB_S2_LDB * sizeof(double), st));   // padding rows / points
        dim3 grid((count + 127) / 128, L);
        gb_points_design<<<grid, 128, 0, st>>>(d_ft, p->d_ct, p->d_kn, p->d_pmm, p->d_cml, p->d_sml, p->d_ra, p->d_rb,
                                              p->d_rc, L, nmin, p0 + count, Kp, p0, GB_S2_TN, GB_S2_LDB);
        GB_LAUNCH_CHECK();
        sh.n_ntiles = n_ptiles;
        int rc = gbgemm::launch(sh, PointQuadForm{d_ft, d_part, Kc, Kp, count, nslots}, p->sm_count, st);
        if (rc) return rc;
        gb_points_finish<<<(count + 255) / 256, 256, 0, st>>>(d_part, d_out + p0, nslots, count, take_sqrt ? 1 : 0);
        GB_LAUNCH_CHECK();
    }
    return GB_OK;
}

// ---------------------------------------------------------------------------------------------
// covariance of grad V at the points of a gradient point set (degree N + 1, factors GM/R^2 (R/r)^(n'+1))
// ---------------------------------------------------------------------------------------------
namespace {

constexpr int GP_TP = GB_S2_TN / gbgemm::WN;     // 40 points per 120-column tile, one warp column per component

// Jacobian J_c[p][a] = sum_a' F'_p[a'] T_c[a'][a] of a block of points as GEMM B tiles [point tile][Kp][GB_S2_LDB]: tile
// column 40 c + j holds component c of point j of the tile; padding rows (a >= K'), padding points and the four pad
// columns are written as zeros.  fr: the dense degree-(N+1) rows F' of the block, [count][kf] from degree nmin + 1 on.
// An input (n, m, cs) reaches degree n + 1 through the gather of gb_gradient.cu read backwards (gbgrad::grad_terms).
__global__ void __launch_bounds__(256)
gb_points_gradient_design(double* __restrict__ Jt, const double* __restrict__ fr, long long kf, int nmin, long long Kc,
                          int Kp, int count, long long total) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;      // = ((tile * Kp) + a) * LDB + col
    if (idx >= total) return;
    const int col = (int)(idx % GB_S2_LDB);
    const long long ta = idx / GB_S2_LDB;
    const int a = (int)(ta % Kp);
    const int c = col / GP_TP;
    const int pp = (int)(ta / Kp) * GP_TP + (col - c * GP_TP);
    double v = 0.0;
    if (col < GB_S2_TN && a < Kc && pp < count) {
        const long long ad = a + (long long)nmin * nmin;                          // degree-wise index from degree 0
        int n = (int)sqrt((double)ad);
        if ((long long)n * n > ad) --n;
        if ((long long)(n + 1) * (n + 1) <= ad) ++n;
        const int j = (int)(ad - (long long)n * n);                               // 0: C_n0, 2m-1: C_nm, 2m: S_nm
        const int m = (j + 1) >> 1;
        const int s = (j > 0 && (j & 1) == 0) ? 1 : 0;
        const double* f = fr + (size_t)pp * kf + ((long long)(n + 1) * (n + 1) - (long long)(nmin + 1) * (nmin + 1));
        auto at = [&](int mp, int sp) { return f[mp == 0 ? 0 : 2 * mp - 1 + sp]; };    // F' of (n + 1, mp, sp)
        v = gbgrad::apply(gbgrad::grad_terms(c, n, m, s, gbgrad::grad_q(n)), at);
    }
    Jt[idx] = v;
}

// Epilogue of the gradient covariance: the GEMM rows are the columns b of S2 (the doubled lower triangle of sym(Sigma)),
// its columns (component c, point) of a block, so that C[b][(c, p)] = (J_c S2)[p][b].  The warp of component c folds its
// 32 rows with J_0, J_1 and J_2 of the same points, read back from the Jacobian tiles, one c' and one column pair at a
// time (the 40 accumulators stay live beside two sums; ten sums per c' spill at 128 registers), and writes part[p][c][c'][slot] = sum_b (J_c S2)[p][b] J_c'[p][b] over its rows;
// slot = (row tile, warp row), one writer per slot.  gb_points_gradient_finish adds the slots in order.
struct PointGradientQuadForm {
    static constexpr bool whole_tile = true;
    const double* jt;    // Jacobian tiles [point tile][rows][GB_S2_LDB]
    double* part;        // [count][3][3][nslots]
    long long K;         // coefficients (rows b >= K are padding)
    int rows, count, nslots;
    // the tile's row 0 at the thread's first column of component 0 (the component and the point follow from col_base
    // after the K loop: nothing else stays live across it)
    __device__ __forceinline__ const double* prepare(long long, int nt, int col_base) const {
        return jt + (size_t)nt * rows * GB_S2_LDB + (col_base - nt * GB_S2_TN) % GP_TP;
    }
    __device__ __forceinline__ void tile(const double* f, long long row_base, int col_base, double (&acc)[4][5][2]) const {
        const int nt = col_base / GB_S2_TN;
        const int c = (col_base - nt * GB_S2_TN) / GP_TP;                 // the warp's component
        const int pp0 = col_base - nt * GB_S2_TN - c * GP_TP + nt * GP_TP;  // the thread's first point in the block
        const int slot = (int)(row_base >> 5);
#pragma unroll
        for (int c2 = 0; c2 < 3; ++c2) {
#pragma unroll
            for (int ni = 0; ni < 5; ++ni) {        // one column pair at a time: two sums live beside the accumulators
                double s0 = 0.0, s1 = 0.0;
#pragma unroll
                for (int mi = 0; mi < 4; ++mi) {
                    const long long b = row_base + mi * 8;
                    const double2 jb = b < K ? __ldg(reinterpret_cast<const double2*>(f + (size_t)b * GB_S2_LDB +
                                                                                       c2 * GP_TP + ni * 8))
                                             : make_double2(0.0, 0.0);
                    s0 = mi ? fma(acc[mi][ni][0], jb.x, s0) : acc[mi][ni][0] * jb.x;
                    s1 = mi ? fma(acc[mi][ni][1], jb.y, s1) : acc[mi][ni][1] * jb.y;
                }
#pragma unroll
                for (int o = 4; o < 32; o <<= 1) {
                    s0 += __shfl_xor_sync(0xffffffffu, s0, o);
                    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
                }
                const int pp = pp0 + ni * 8;
                if ((threadIdx.x & 31) < 4) {      // g = 0
                    if (pp < count) part[((size_t)(pp * 3 + c) * 3 + c2) * nslots + slot] = s0;
                    if (pp + 1 < count) part[((size_t)((pp + 1) * 3 + c) * 3 + c2) * nslots + slot] = s1;
                }
            }
        }
    }
};

// Per point of the block: M[c][c'] = sum of the slots in order (bit-identical from run to run), the symmetric covariance
// C_cc = M_cc, C_cc' = (M_cc' + M_c'c) / 2, optionally Q C Q' in (east, north, up) (gbgrad::rotate on the columns, then
// on the rows, then made symmetric again); out [npts][3][3], or with take_sqrt [3][npts] square roots of the diagonal.
__global__ void __launch_bounds__(256)
gb_points_gradient_finish(const double* __restrict__ part, const double* __restrict__ frame, double* __restrict__ out,
                          int nslots, int count, int p0, long long npts, int take_sqrt) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    double M[3][3];
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int c2 = 0; c2 < 3; ++c2) {
            const double* pt = part + ((size_t)(i * 3 + c) * 3 + c2) * nslots;
            double v = 0.0;
            for (int s = 0; s < nslots; ++s) v += pt[s];
            M[c][c2] = v;
        }
    double C[3][3];
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int c2 = 0; c2 < 3; ++c2) C[c][c2] = c == c2 ? M[c][c] : __dmul_rn(0.5, __dadd_rn(M[c][c2], M[c2][c]));
    const long long p = p0 + (long long)i;
    if (frame) {
        const gbgrad::Frame f{frame[p], frame[npts + p], frame[2 * npts + p], frame[3 * npts + p]};
        gbgrad::rotate_matrix(f, C);
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int c2 = c + 1; c2 < 3; ++c2) C[c][c2] = C[c2][c] = __dmul_rn(0.5, __dadd_rn(C[c][c2], C[c2][c]));
    }
    if (take_sqrt) {
#pragma unroll
        for (int c = 0; c < 3; ++c) out[c * npts + p] = sqrt(C[c][c]);
    } else {
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int c2 = 0; c2 < 3; ++c2) out[(size_t)p * 9 + 3 * c + c2] = C[c][c2];
    }
}

}  // namespace

extern "C" int gb_points_gradient_covariance(gb_points* p, const double* d_sigma, int nmin, const double* d_frame,
                                             double* d_out, int flags, void* stream) {
    GB_REQUIRE(p != nullptr, "gb_points_gradient_covariance: point set is NULL");
    GB_REQUIRE((flags & ~GB_COV_SQRT) == 0, "gb_points_gradient_covariance: flags=%d; only GB_COV_SQRT is accepted",
               flags);
    GB_REQUIRE(p->nmax >= 1, "gb_points_gradient_covariance: a gradient point set has degree nmax + 1 >= 1 (got %d)",
               p->nmax);
    const int nmax = p->nmax - 1;                                      // degree of the field
    GB_REQUIRE(nmin >= 0 && nmin <= nmax, "gb_points_gradient_covariance: min_degree=%d outside [0, %d]", nmin, nmax);
    GB_REQUIRE(d_sigma && d_out, "gb_points_gradient_covariance: NULL device pointer");
    GB_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const long long Kc = (long long)(nmax + 1) * (nmax + 1) - (long long)nmin * nmin;   // coefficients of the field
    const int Kp = (int)((Kc + 3) / 4 * 4);
    const long long kf = (long long)p->L * p->L - (long long)(nmin + 1) * (nmin + 1);     // F' from degree nmin + 1
    const int n_btiles = (int)((Kc + GB_TM - 1) / GB_TM);
    const int n_ptiles_all = (p->npts + GP_TP - 1) / GP_TP;
    // point blocks as for gb_points_covariance: several waves of GEMM tiles, the Jacobian only ever for one block
    int tiles_per_block = 4 * p->sm_count / n_btiles;
    if (tiles_per_block < 16) tiles_per_block = 16;
    if (tiles_per_block > n_ptiles_all) tiles_per_block = n_ptiles_all;
    const int nslots = n_btiles * gbgemm::WM;
    const int max_count = tiles_per_block * GP_TP;
    double *d_st = nullptr, *d_fr = nullptr, *d_jt = nullptr, *d_part = nullptr;
    gb_retain_pool_memory(p->device);
    gb_scratch scratch(st);
    GB_CUDA(scratch.alloc(&d_st, (size_t)n_btiles * Kp * GB_LDA));
    GB_CUDA(scratch.alloc(&d_fr, (size_t)max_count * kf));
    GB_CUDA(scratch.alloc(&d_jt, (size_t)tiles_per_block * Kp * GB_S2_LDB));
    GB_CUDA(scratch.alloc(&d_part, (size_t)max_count * 9 * nslots));
    gb_points_sigma_tiles<<<dim3((unsigned)Kp, (unsigned)n_btiles), GB_TM, 0, st>>>(d_sigma, d_st, Kc, Kp,
                                                                                    SIGMA_SYMMETRISED_LOWER);
    GB_LAUNCH_CHECK();
    gbgemm::Shape sh;
    sh.A_t = d_st;
    sh.a_rows = Kp;
    sh.a_koff_mul = 0;
    sh.tiles_per_group = 1;
    sh.B_t = d_jt;
    sh.b_rows = Kp;
    sh.klen = Kp;
    sh.n_mtiles = n_btiles;
    sh.mt_kstart_mod = n_btiles;        // row tile j starts its contraction at k = 128 j (the rows above are zeros)
    sh.mt_kstart_mul = GB_TM;
    const int L = p->L;
    const int threads = L >= 1024 ? 1024 : (L + 31) / 32 * 32;
    for (int t0 = 0; t0 < n_ptiles_all; t0 += tiles_per_block) {
        const int n_ptiles = (n_ptiles_all - t0 < tiles_per_block) ? (n_ptiles_all - t0) : tiles_per_block;
        const int p0 = t0 * GP_TP;
        const int count = (p->npts - p0 < n_ptiles * GP_TP) ? (p->npts - p0) : n_ptiles * GP_TP;
        gb_points_design_rows<<<count, threads, 0, st>>>(DenseRows{d_fr, kf, (long long)(nmin + 1) * (nmin + 1)},
                                                         p->d_ct, p->d_kn, p->d_pmm, p->d_cml, p->d_sml, p->d_ra,
                                                         p->d_rb, p->d_rc, L, nmin + 1, p0 + count, p0);
        GB_LAUNCH_CHECK();
        const long long total = (long long)n_ptiles * Kp * GB_S2_LDB;
        gb_points_gradient_design<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(d_jt, d_fr, kf, nmin, Kc, Kp, count,
                                                                                   total);
        GB_LAUNCH_CHECK();
        sh.n_ntiles = n_ptiles;
        int rc = gbgemm::launch(sh, PointGradientQuadForm{d_jt, d_part, Kc, Kp, count, nslots}, p->sm_count, st);
        if (rc) return rc;
        gb_points_gradient_finish<<<(count + 255) / 256, 256, 0, st>>>(d_part, d_frame, d_out, nslots, count, p0,
                                                                       p->npts, (flags & GB_COV_SQRT) ? 1 : 0);
        GB_LAUNCH_CHECK();
    }
    return GB_OK;
}

// ---------------------------------------------------------------------------------------------
// normal equations of acceleration observations at the points of a gradient point set: N += J~' W J~ (upper triangle,
// then mirrored), J~_p = Q_p J_p the rotated Jacobian rows of gb_points_gradient_covariance
// ---------------------------------------------------------------------------------------------
namespace {

// The rows sqrt(w_pc) J~_p[c] of a block of points, observation o = 3 pp + c, straight into the two GEMM operands: A
// tiles [coefficient tile of 128][o][GB_LDA] and B tiles [coefficient tile of 120][o][GB_S2_LDB] (k = observation, like
// the point adjoint).  Thread = (coefficient a, point pp) with a fastest, so the stores of both layouts coalesce; the
// three Cartesian entries of the point come from the same gbgrad::grad_terms as gb_points_gradient_design, then
// gbgrad::rotate for the local frame, then the weights.  Coefficients a >= K' (up to am / bm) and observation rows
// 3 count .. rows - 1 are written as zeros; the pad columns of the tiles are never read by the GEMM.
__global__ void __launch_bounds__(256)
gb_points_gradient_normal_rows(double* __restrict__ At, double* __restrict__ Bt, const double* __restrict__ fr, long long kf,
                               int nmin, long long Kc, int am, int bm, int rows, int count,
                               const double* __restrict__ weights, const double* __restrict__ frame, long long npts, int p0) {
    const int a = blockIdx.x * blockDim.x + threadIdx.x;
    const int pp = blockIdx.y;
    if (a >= am && a >= bm) return;
    double v[3] = {0.0, 0.0, 0.0};
    if (a < Kc && pp < count) {
        const long long ad = a + (long long)nmin * nmin;                          // degree-wise index from degree 0
        int n = (int)sqrt((double)ad);
        if ((long long)n * n > ad) --n;
        if ((long long)(n + 1) * (n + 1) <= ad) ++n;
        const int j = (int)(ad - (long long)n * n);                               // 0: C_n0, 2m-1: C_nm, 2m: S_nm
        const int m = (j + 1) >> 1;
        const int s = (j > 0 && (j & 1) == 0) ? 1 : 0;
        const double* f = fr + (size_t)pp * kf + ((long long)(n + 1) * (n + 1) - (long long)(nmin + 1) * (nmin + 1));
        auto at = [&](int mp, int sp) { return f[mp == 0 ? 0 : 2 * mp - 1 + sp]; };    // F' of (n + 1, mp, sp)
        const double q = gbgrad::grad_q(n);
#pragma unroll
        for (int c = 0; c < 3; ++c) v[c] = gbgrad::apply(gbgrad::grad_terms(c, n, m, s, q), at);
        const long long p = p0 + (long long)pp;
        if (frame) {
            const gbgrad::Frame fq{frame[p], frame[npts + p], frame[2 * npts + p], frame[3 * npts + p]};
            gbgrad::rotate(fq, v[0], v[1], v[2]);
        }
        if (weights) {
#pragma unroll
            for (int c = 0; c < 3; ++c) v[c] = __dmul_rn(__dsqrt_rn(weights[c * npts + p]), v[c]);
        }
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const int o = 3 * pp + c;
        if (o >= rows) break;
        if (a < am) At[gb_ab_offset(a, o, rows)] = v[c];
        if (a < bm) Bt[((size_t)(a / GB_S2_TN) * rows + o) * GB_S2_LDB + a % GB_S2_TN] = v[c];
    }
}

// The rows sqrt(w_pc) J~_p[c] of gravity-gradient observations, observation o = 6 pp + c with the pairs c = xx, xy, xz, yy,
// yz, zz, in the layouts of gb_points_gradient_normal_rows.  fr: the dense degree-(N+2) rows F'' of the block from degree
// nmin + 2 on.  Entry (a, b) of the point is the composed F''_p T_a T_b of gbgrad::apply_pair (the expression of the
// transposed transform), then gbgrad::rotate_tensor for the local frame (the upper triangle of Q V Q', as
// gb_rotate_tensor_to_local), then the weights.
__global__ void __launch_bounds__(256)
gb_points_gravity_gradient_normal_rows(double* __restrict__ At, double* __restrict__ Bt, const double* __restrict__ fr,
                                       long long kf, int nmin, long long Kc, int am, int bm, int rows, int count,
                                       const double* __restrict__ weights, const double* __restrict__ frame,
                                       long long npts, int p0) {
    const int a = blockIdx.x * blockDim.x + threadIdx.x;
    const int pp = blockIdx.y;
    if (a >= am && a >= bm) return;
    double v[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    if (a < Kc && pp < count) {
        const long long ad = a + (long long)nmin * nmin;                          // degree-wise index from degree 0
        int n = (int)sqrt((double)ad);
        if ((long long)n * n > ad) --n;
        if ((long long)(n + 1) * (n + 1) <= ad) ++n;
        const int j = (int)(ad - (long long)n * n);                               // 0: C_n0, 2m-1: C_nm, 2m: S_nm
        const int m = (j + 1) >> 1;
        const int s = (j > 0 && (j & 1) == 0) ? 1 : 0;
        const double* f = fr + (size_t)pp * kf + ((long long)(n + 2) * (n + 2) - (long long)(nmin + 2) * (nmin + 2));
        auto at = [&](int mp, int sp) { return f[mp == 0 ? 0 : 2 * mp - 1 + sp]; };    // F'' of (n + 2, mp, sp)
        const double q0 = gbgrad::grad_q(n), q1 = gbgrad::grad_q(n + 1);
#pragma unroll
        for (int c = 0; c < 6; ++c) v[c] = gbgrad::apply_pair(gbgrad::pair_a(c), gbgrad::pair_b(c), n, m, s, q0, q1, at);
        const long long p = p0 + (long long)pp;
        if (frame) gbgrad::rotate_tensor({frame[p], frame[npts + p], frame[2 * npts + p], frame[3 * npts + p]}, v);
        if (weights) {
#pragma unroll
            for (int c = 0; c < 6; ++c) v[c] = __dmul_rn(__dsqrt_rn(weights[c * npts + p]), v[c]);
        }
    }
#pragma unroll
    for (int c = 0; c < 6; ++c) {
        const int o = 6 * pp + c;
        if (o >= rows) break;
        if (a < am) At[gb_ab_offset(a, o, rows)] = v[c];
        if (a < bm) Bt[((size_t)(a / GB_S2_TN) * rows + o) * GB_S2_LDB + a % GB_S2_TN] = v[c];
    }
}

// Epilogue of the normals: C[a][b] = sum_o J~[o][a] J~[o][b] over the block's observations, added to N[a][b] for b >= a
// (upper triangle).  One thread per entry per launch and the launches in stream order: bit-reproducible.
struct NormalsAddUpper {
    double* out;
    long long K;
    __device__ __forceinline__ void operator()(long long row, int col, double v0, double v1) const {
        if (row >= K) return;
        double* o = out + (size_t)row * K + col;
        if (col >= row && col < K) *o += v0;
        if (col + 1 >= row && col + 1 < K) o[1] += v1;
    }
};

// N[r][c] = N[c][r] for r > c, through 32 x 32 tiles in shared memory (both accesses coalesce).  The block of the lower
// tile (bi, bj), bi >= bj, reads the upper tile (bj, bi), which no block writes.
__global__ void __launch_bounds__(256)
gb_mirror_upper(double* __restrict__ N, long long K) {
    __shared__ double t[32][33];
    const int bi = blockIdx.y, bj = blockIdx.x;
    if (bi < bj) return;
    for (int y = threadIdx.y; y < 32; y += 8) {
        const long long r = (long long)bj * 32 + y, c = (long long)bi * 32 + threadIdx.x;
        if (r < K && c < K) t[y][threadIdx.x] = N[(size_t)r * K + c];
    }
    __syncthreads();
    for (int y = threadIdx.y; y < 32; y += 8) {
        const long long r = (long long)bi * 32 + y, c = (long long)bj * 32 + threadIdx.x;
        if (r < K && c < K && r > c) N[(size_t)r * K + c] = t[threadIdx.x][y];
    }
}

// The normal equations of observations of the derivatives of order ORDER (1: the three components of grad V on a gradient
// point set, 2: the six of the gravity gradient tensor on a gravity-gradient point set, degree nmax + ORDER): NC = 3 or 6
// observation rows per point, written by the row writer of the order.
template <int ORDER>
int points_derivative_normals(const char* name, const char* kind, gb_points* p, int nmin, const double* d_weights,
                              const double* d_frame, double* d_normals, void* stream) {
    constexpr int NC = ORDER == 1 ? 3 : 6;
    GB_REQUIRE(p != nullptr, "%s: point set is NULL", name);
    GB_REQUIRE(p->nmax >= ORDER, "%s: a %s point set has degree nmax + %d >= %d (got %d)", name, kind, ORDER, ORDER,
               p->nmax);
    const int nmax = p->nmax - ORDER;                                  // degree of the field
    GB_REQUIRE(nmin >= 0 && nmin <= nmax, "%s: min_degree=%d outside [0, %d]", name, nmin, nmax);
    GB_REQUIRE(d_normals != nullptr, "%s: NULL device pointer", name);
    GB_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const long long Kc = (long long)(nmax + 1) * (nmax + 1) - (long long)nmin * nmin;   // coefficients of the field
    const long long f0 = (long long)(nmin + ORDER) * (nmin + ORDER);
    const long long kf = (long long)p->L * p->L - f0;                  // the synthesis rows from degree nmin + ORDER
    const int n_mtiles = (int)((Kc + GB_TM - 1) / GB_TM);
    const int n_ntiles = (int)((Kc + GB_S2_TN - 1) / GB_S2_TN);
    const int am = n_mtiles * GB_TM, bm = n_ntiles * GB_S2_TN;
    // points per block: an A operand of about 512 MB (the B operand is as large), a multiple of 4 points so that the NC pb
    // observation rows of a full block are whole k4 steps, and at most 49152 observation rows
    long long pb = (512LL << 20) / ((long long)n_mtiles * GB_LDA * sizeof(double)) / NC;
    pb = pb / 4 * 4;
    if (pb < 4) pb = 4;
    if (pb > 49152 / NC) pb = 49152 / NC;
    if (pb > (p->npts + 3) / 4 * 4) pb = (p->npts + 3) / 4 * 4;
    const int max_rows = (int)(NC * pb);
    double *d_at = nullptr, *d_bt = nullptr, *d_fr = nullptr;
    gb_retain_pool_memory(p->device);
    gb_scratch scratch(st);
    GB_CUDA(scratch.alloc(&d_at, (size_t)n_mtiles * max_rows * GB_LDA));
    GB_CUDA(scratch.alloc(&d_bt, (size_t)n_ntiles * max_rows * GB_S2_LDB));
    GB_CUDA(scratch.alloc(&d_fr, (size_t)pb * kf));
    gbgemm::Shape sh;
    sh.A_t = d_at;
    sh.a_koff_mul = 0;
    sh.tiles_per_group = 1;
    sh.B_t = d_bt;
    sh.n_mtiles = n_mtiles;
    sh.n_ntiles = n_ntiles;
    sh.upper_only = true;                // N is symmetric: the tiles below the diagonal are never contracted
    const int L = p->L;
    const int threads = L >= 1024 ? 1024 : (L + 31) / 32 * 32;
    for (int p0 = 0; p0 < p->npts; p0 += (int)pb) {
        const int count = (p->npts - p0 < pb) ? (p->npts - p0) : (int)pb;
        const int rows = (NC * count + 3) / 4 * 4;
        gb_points_design_rows<<<count, threads, 0, st>>>(DenseRows{d_fr, kf, f0}, p->d_ct, p->d_kn, p->d_pmm, p->d_cml,
                                                         p->d_sml, p->d_ra, p->d_rb, p->d_rc, L, nmin + ORDER,
                                                         p0 + count, p0);
        GB_LAUNCH_CHECK();
        dim3 grid((unsigned)(((am > bm ? am : bm) + 255) / 256), (unsigned)((rows + NC - 1) / NC));
        if constexpr (ORDER == 1)
            gb_points_gradient_normal_rows<<<grid, 256, 0, st>>>(d_at, d_bt, d_fr, kf, nmin, Kc, am, bm, rows, count,
                                                                 d_weights, d_frame, p->npts, p0);
        else
            gb_points_gravity_gradient_normal_rows<<<grid, 256, 0, st>>>(d_at, d_bt, d_fr, kf, nmin, Kc, am, bm, rows,
                                                                         count, d_weights, d_frame, p->npts, p0);
        GB_LAUNCH_CHECK();
        sh.a_rows = rows;
        sh.b_rows = rows;
        sh.klen = rows;
        int rc = gbgemm::launch(sh, NormalsAddUpper{d_normals, Kc}, p->sm_count, st);
        if (rc) return rc;
    }
    const unsigned nt32 = (unsigned)((Kc + 31) / 32);
    gb_mirror_upper<<<dim3(nt32, nt32), dim3(32, 8), 0, st>>>(d_normals, Kc);
    GB_LAUNCH_CHECK();
    return GB_OK;
}

}  // namespace

extern "C" int gb_points_gradient_normals(gb_points* p, int nmin, const double* d_weights, const double* d_frame,
                                          double* d_normals, void* stream) {
    return points_derivative_normals<1>("gb_points_gradient_normals", "gradient", p, nmin, d_weights, d_frame, d_normals,
                                        stream);
}

extern "C" int gb_points_gravity_gradient_normals(gb_points* p, int nmin, const double* d_weights, const double* d_frame,
                                                  double* d_normals, void* stream) {
    return points_derivative_normals<2>("gb_points_gravity_gradient_normals", "gravity gradient", p, nmin, d_weights,
                                        d_frame, d_normals, stream);
}
