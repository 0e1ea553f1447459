// Arbitrary point sets (the reference's IrregularGrid path): synthesis and covariance propagation.
//
//   gb_points_synthesis    replaces the irregular branch of PotentialCoefficients.to_grid
//                          (reference gravityfield.py:370-388): per point the Legendre recursion runs
//                          on the fly (bit-identical values), scaled by kn[p,n], contracted against an
//                          epoch tile of coefficients held in shared memory.
//   gb_points_covariance   replaces IrregularGrid.covariance_propagation (reference grid.py:1096-1120):
//                          var[p] = sum_ab F[p,a] Sigma[a,b] F[p,b] -- the direct, blocked
//                          diag(F Sigma F') of the north star: F tiles generated on the fly
//                          (gb_points_design), T = F Sigma on the FP64 tensor cores with Sigma rows
//                          staged by the TMA unit (cp.async.bulk + mbarrier pipeline), and the
//                          row-wise product with F folded into the epilogue with warp shuffles.
//                          2 P K^2 flops, nothing assumed about the point geometry.
#include <vector>
#include <cmath>
#include "gb_common.cuh"
#include "gb_gemm.cuh"

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
// design matrix F^T in the tiled layout [point tile][a][GB_LDA], a = degree-wise index - nmin^2
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
gb_points_design(double* __restrict__ FT, const double* __restrict__ ct, const double* __restrict__ kn,
                 const double* __restrict__ pmm, const double* __restrict__ cml, const double* __restrict__ sml,
                 const double* __restrict__ ra, const double* __restrict__ rb, const double* __restrict__ rc, int L,
                 int nmin, int npts, int rows, int p0) {
    const int p = p0 + blockIdx.x * blockDim.x + threadIdx.x;      // tiles are numbered from point p0
    const int m = blockIdx.y;
    if (p >= npts) return;
    const double* kn_p = kn + (size_t)p * L;
    const double cm = cml[(size_t)p * L + m], sm = sml[(size_t)p * L + m];
    const int off = nmin * nmin;
    legendre_column(m, L, ct[p], pmm[(size_t)p * L + m], ra, rb, rc, [&](int n, double pn) {
        if (n < nmin) return;
        const double pk = __dmul_rn(pn, kn_p[n]);
        const int a = n * n + (m == 0 ? 0 : 2 * m - 1) - off;
        FT[gb_ab_offset(p - p0, a, rows)] = __dmul_rn(pk, cm);
        if (m > 0) FT[gb_ab_offset(p - p0, a + 1, rows)] = __dmul_rn(pk, sm);
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

// ---------------------------------------------------------------------------------------------
// blocked diag(F Sigma F'): tile = 128 points x 120 columns b; K loop over a in chunks of 28
// ---------------------------------------------------------------------------------------------
constexpr int C_WM = 4, C_WN = 3, C_TM = 128, C_TN = 120, C_KC = 28, C_STAGES = 3;
constexpr int C_LDA = GB_LDA, C_LDB = C_TN + 4;
constexpr int C_CONSUMER_WARPS = C_WM * C_WN;
constexpr int C_THREADS = 32 * (C_CONSUMER_WARPS + 1);
constexpr int C_STAGE_DOUBLES = C_KC * (C_LDA + C_LDB);
constexpr size_t C_SMEM = (size_t)C_STAGES * C_STAGE_DOUBLES * sizeof(double) + 2 * C_STAGES * sizeof(uint64_t);

__global__ void __launch_bounds__(C_THREADS, 1)
gb_points_quadform(const double* __restrict__ FT, int rows, const double* __restrict__ sig, long long lds, int Kp,
                   long long Kc, double* __restrict__ var, int npts, int n_mtiles, int n_ntiles, int upper) {
    extern __shared__ __align__(128) unsigned char s_raw[];
    double* s_tiles = reinterpret_cast<double*>(s_raw);
    uint64_t* full = reinterpret_cast<uint64_t*>(s_raw + (size_t)C_STAGES * C_STAGE_DOUBLES * sizeof(double));
    uint64_t* empty = full + C_STAGES;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < C_STAGES; ++s) {
            gb::mbar_init(&full[s], 1);
            gb::mbar_init(&empty[s], C_CONSUMER_WARPS);
        }
        gb::fence_mbar_init();
    }
    __syncthreads();
    const long long n_tiles = (long long)n_mtiles * n_ntiles;
    int stage = 0;
    uint32_t phase = 0;
    if (warp == C_CONSUMER_WARPS) {
        // producer: one bulk copy for the F^T chunk, one per covariance row
        for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x) {
            // upper-triangular operand: the work of a tile grows with its column tile, so the heaviest column tiles
            // go first (and the CTAs of one wave share the same covariance columns in L2)
            const long long mt = upper ? t % n_mtiles : t / n_ntiles;
            const int n0 = (int)(upper ? n_ntiles - 1 - t / n_mtiles : t % n_ntiles) * C_TN;
            long long w = Kc - n0;
            if (w > C_TN) w = C_TN;
            const int width = (int)((w + 1) & ~1LL);     // even number of doubles (16-byte granules)
            // upper-triangular operand (symmetric Sigma, off-diagonal entries doubled): rows a beyond the tile's last
            // column are zero
            const int kend = upper ? min(Kp, (n0 + C_TN + 3) & ~3) : Kp;
            for (int k0 = 0; k0 < kend; k0 += C_KC) {
                const int kc = min(C_KC, kend - k0);
                gb::mbar_wait(&empty[stage], phase ^ 1u);
                double* sA = s_tiles + (size_t)stage * C_STAGE_DOUBLES;
                double* sB = sA + C_KC * C_LDA;
                if (lane == 0) {
                    const uint32_t bytes_a = (uint32_t)(kc * C_LDA * sizeof(double));
                    gb::mbar_arrive_expect_tx(&full[stage], bytes_a + (uint32_t)(kc * width * sizeof(double)));
                    gb::bulk_g2s(sA, FT + ((size_t)mt * rows + k0) * C_LDA, bytes_a, &full[stage]);
                }
                __syncwarp();
                if (lane < kc)
                    gb::bulk_g2s(sB + lane * C_LDB, sig + (size_t)(k0 + lane) * lds + n0,
                                 (uint32_t)(width * sizeof(double)), &full[stage]);
                if (++stage == C_STAGES) { stage = 0; phase ^= 1u; }
            }
        }
    } else {
        const int wm = warp / C_WN, wn = warp % C_WN;
        const int g = lane >> 2, q = lane & 3;
        for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x) {
            const long long mt = upper ? t % n_mtiles : t / n_ntiles;
            const int n0 = (int)(upper ? n_ntiles - 1 - t / n_mtiles : t % n_ntiles) * C_TN;
            double acc[4][5][2];
#pragma unroll
            for (int mi = 0; mi < 4; ++mi)
#pragma unroll
                for (int ni = 0; ni < 5; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
            const int kend = upper ? min(Kp, (n0 + C_TN + 3) & ~3) : Kp;
            for (int k0 = 0; k0 < kend; k0 += C_KC) {
                const int kc = min(C_KC, kend - k0);
                gb::mbar_wait(&full[stage], phase);
                const double* sA = s_tiles + (size_t)stage * C_STAGE_DOUBLES + wm * 32 + g;
                const double* sB = s_tiles + (size_t)stage * C_STAGE_DOUBLES + C_KC * C_LDA + wn * 40 + g;
#pragma unroll
                for (int kk = 0; kk < C_KC; kk += 4) {
                    if (kk >= kc) break;
                    double a[4], b[5];
#pragma unroll
                    for (int mi = 0; mi < 4; ++mi) a[mi] = sA[(kk + q) * C_LDA + mi * 8];
#pragma unroll
                    for (int ni = 0; ni < 5; ++ni) b[ni] = sB[(kk + q) * C_LDB + ni * 8];
#pragma unroll
                    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
                        for (int ni = 0; ni < 5; ++ni) gb::dmma_884(acc[mi][ni][0], acc[mi][ni][1], a[mi], b[ni]);
                }
                __syncwarp();
                if (lane == 0) gb::mbar_arrive(&empty[stage]);
                if (++stage == C_STAGES) { stage = 0; phase ^= 1u; }
            }
            // epilogue: var[p] += sum_b T[p,b] F[p,b] over this tile's columns
            const double* ft = FT + (size_t)mt * rows * C_LDA;
#pragma unroll
            for (int mi = 0; mi < 4; ++mi) {
                const int r = wm * 32 + mi * 8 + g;
                double part = 0.0;
#pragma unroll
                for (int ni = 0; ni < 5; ++ni) {
                    const long long b = (long long)n0 + wn * 40 + ni * 8 + 2 * q;
                    if (b < Kc) part = fma(acc[mi][ni][0], ft[(size_t)b * C_LDA + r], part);
                    if (b + 1 < Kc) part = fma(acc[mi][ni][1], ft[(size_t)(b + 1) * C_LDA + r], part);
                }
                part += __shfl_xor_sync(0xffffffffu, part, 1);
                part += __shfl_xor_sync(0xffffffffu, part, 2);
                const long long p = mt * C_TM + r;
                // one writer per (point, column tile, warp column): gb_points_finish adds the slots in order
                if (q == 0 && p < npts) var[(size_t)p * (n_ntiles * C_WN) + (n0 / C_TN) * C_WN + wn] = part;
            }
        }
    }
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
    {   // keep stream-ordered workspace allocations in the pool between calls (default threshold 0
        // returns them to the driver at every synchronisation: milliseconds per GB on the next call)
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            unsigned long long keep = ~0ULL;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
    }
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
                                              p->d_rc, L, 0, p0 + count, Kp, p0);
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

// Sigma re-pitched to an even leading dimension; for a symmetric Sigma only its upper triangle is kept, the
// off-diagonal entries doubled:  x' S x = sum_a S_aa x_a^2 + 2 sum_{a<b} S_ab x_a x_b
__global__ void __launch_bounds__(256)
gb_points_sigma_operand(const double* __restrict__ sigma, double* __restrict__ sig, long long Kc, long long lds, int upper) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long a = blockIdx.y;
    if (b >= Kc) return;
    double v = sigma[(size_t)a * Kc + b];
    if (upper) v = (a < b) ? v + v : (a == b ? v : 0.0);
    sig[(size_t)a * lds + b] = v;
}

extern "C" int gb_points_covariance(gb_points* p, const double* d_sigma, int nmin, double* d_out, int flags,
                                    void* stream) {
    const int take_sqrt = flags & GB_COV_SQRT;
    const int upper = (flags & GB_COV_SYMMETRIC) ? 1 : 0;
    GB_REQUIRE(p != nullptr, "gb_points_covariance: point set is NULL");
    GB_REQUIRE(nmin >= 0 && nmin <= p->nmax, "gb_points_covariance: min_degree=%d outside [0, %d]", nmin, p->nmax);
    GB_REQUIRE(d_sigma && d_out, "gb_points_covariance: NULL device pointer");
    GB_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int L = p->L;
    const long long Kc = (long long)L * L - (long long)nmin * nmin;   // coefficients
    const int Kp = (int)((Kc + 3) / 4 * 4);                            // padded to whole k4 steps
    const long long lds = (Kc + 1) / 2 * 2 + 2;                        // even leading dimension, room for the tail
    const int n_mtiles_all = (p->npts + C_TM - 1) / C_TM;
    const int n_ntiles = (int)((Kc + C_TN - 1) / C_TN);
    // the design matrix only ever exists for one block of points (about four waves of GEMM tiles): 75 KB per point at
    // degree 96 would otherwise be 12 GB for a 0.5-degree Reuter grid
    int tiles_per_block = 4 * p->sm_count / (n_ntiles > 0 ? n_ntiles : 1);
    if (tiles_per_block < 16) tiles_per_block = 16;
    if (tiles_per_block > n_mtiles_all) tiles_per_block = n_mtiles_all;
    double *d_ft = nullptr, *d_sig = nullptr, *d_part = nullptr;
    const size_t ft_elems = (size_t)tiles_per_block * Kp * C_LDA;
    const int nslots = n_ntiles * C_WN;
    gb_retain_pool_memory(p->device);
    gb_scratch scratch(st);
    GB_CUDA(scratch.alloc(&d_ft, ft_elems));
    GB_CUDA(scratch.alloc(&d_sig, (size_t)Kp * lds));
    GB_CUDA(scratch.alloc(&d_part, (size_t)tiles_per_block * C_TM * nslots));
    GB_CUDA(cudaMemsetAsync(d_sig, 0, (size_t)Kp * lds * sizeof(double), st));
    {   // covariance rows re-pitched to an even leading dimension (16-byte aligned rows for the bulk copies)
        dim3 grid((unsigned)((Kc + 255) / 256), (unsigned)Kc);
        gb_points_sigma_operand<<<grid, 256, 0, st>>>(d_sigma, d_sig, Kc, lds, upper);
        GB_LAUNCH_CHECK();
    }
    GB_CUDA(cudaFuncSetAttribute(gb_points_quadform, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C_SMEM));
    for (int t0 = 0; t0 < n_mtiles_all; t0 += tiles_per_block) {
        const int n_mtiles = (n_mtiles_all - t0 < tiles_per_block) ? (n_mtiles_all - t0) : tiles_per_block;
        const int p0 = t0 * C_TM;
        const int count = (p->npts - p0 < n_mtiles * C_TM) ? (p->npts - p0) : n_mtiles * C_TM;
        GB_CUDA(cudaMemsetAsync(d_ft, 0, (size_t)n_mtiles * Kp * C_LDA * sizeof(double), st));
        dim3 grid((count + 127) / 128, L);
        gb_points_design<<<grid, 128, 0, st>>>(d_ft, p->d_ct, p->d_kn, p->d_pmm, p->d_cml, p->d_sml, p->d_ra, p->d_rb,
                                              p->d_rc, L, nmin, p0 + count, Kp, p0);
        GB_LAUNCH_CHECK();
        const long long n_tiles = (long long)n_mtiles * n_ntiles;
        const int gridq = (int)(n_tiles < p->sm_count ? n_tiles : p->sm_count);
        gb_points_quadform<<<gridq, C_THREADS, C_SMEM, st>>>(d_ft, Kp, d_sig, lds, Kp, Kc, d_part, count, n_mtiles,
                                                             n_ntiles, upper);
        GB_LAUNCH_CHECK();
        gb_points_finish<<<(count + 255) / 256, 256, 0, st>>>(d_part, d_out + p0, nslots, count, take_sqrt ? 1 : 0);
        GB_LAUNCH_CHECK();
    }
    return GB_OK;
}
