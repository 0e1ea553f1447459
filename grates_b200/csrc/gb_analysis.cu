// Spherical-harmonic analysis on B200, epoch-batched.
//
// Replaces RegularGrid.to_potential_coefficients (reference grid.py:776-785), whose per-order
// operator solve(A'WA, A'W) (grid.py:690-696) factors on a regular grid with rank-one area
// weights W_ij = w_i u_j into
//
//   G[e,i,(m,cs)] = sum_j V[e,i,j] * lon_op[(m,cs)][j]                         (longitude stage)
//   x[e,n,(m,cs)] = sum_i lat_op_m[n - n0(m)][i] * G[e,i,(m,cs)]              (latitude stage)
//
// with lon_op = u_j trig(m lon_j) / sum_j u_j trig^2 and lat_op_m = solve(P'WP, P'W), built once
// per plan on the host (grates_b200/plan.py: analysis_operators).
//
// Both stages run on the persistent DMMA GEMM of gb_gemm.cuh.  The rows of the longitude stage are
// ordered (parallel i, epoch e) with the epochs fastest, so that its epilogue writes the B operand of
// the latitude stage, Gt[order m][column tile][parallel i][column (cs, e)], in contiguous 64-byte runs
// (eight epochs of one fragment slab); the latitude stage then is one GEMM per order (row tiles of the
// per-order operators, contraction over the parallels) batched into a single launch.
//
// HBM layout:  V [E][nlat][nlon] (input), VF folded input tiles [row tile][j'][132],
//              Gt [L][n_ct][nlat_p4][124], lat operator tiles [row tile][nlat_p4][132],
//              anm [E][L][L] packed (output).  GB_SIMPLE_ANALYSIS=1 runs plain FMA kernels with
//              G [kpad][mpad] and lat_ops concatenated [cnt_m][nlat] blocks as a cross-check.
#include <vector>
#include <cmath>
#include "gb_common.cuh"
#include "gb_gemm.cuh"

namespace {

// ---- longitude stage on the tensor cores ---------------------------------------------------------
// gb_analysis_fold transposes V into the tiled k-major operand layout of gb_gemm.cuh.  With four-fold
// symmetric meridians / weights it also folds the four mirrored meridians of every first-quadrant
// longitude mu = lon[h+j'] (v1 = V(mu), v2 = V(pi-mu), v3 = V(-mu), v4 = V(mu-pi)):
//   set 0 (even m, cos) (v1+v3)+(v2+v4)      set 1 (odd m, cos) (v1+v3)-(v2+v4)
//   set 2 (even m, sin) (v1-v3)+(v4-v2)      set 3 (odd m, sin) (v1-v3)-(v4-v2)
// so that the contraction runs over one quadrant only (a quarter of the multiply-adds).
// GEMM row rho = i * E + e  (epochs fastest, see above)
__global__ void __launch_bounds__(256)
gb_analysis_fold(const double* __restrict__ V, double* __restrict__ VF, long long M, int nlon, int nsets, int kp,
                 int kvalid, int E, int nlat) {
    __shared__ double s_f[4][32][33];
    const int j0 = blockIdx.x * 32;                 // first k (j or j') of this block
    const long long r0 = (long long)blockIdx.y * 32;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;   // 8 warps, 4 rows each
    const int h = nlon >> 1;
    for (int rr = w; rr < 32; rr += 8) {
        const long long row = r0 + rr;
        const int j = j0 + lane;
        double f0 = 0.0, f1 = 0.0, f2 = 0.0, f3 = 0.0;
        if (row < M && j < kvalid) {
            const long long i = row / E, e = row - i * E;
            const double* v = V + (size_t)(e * nlat + i) * nlon;
            if (nsets == 4) {
                const double v1 = v[h + j], v2 = v[nlon - 1 - j], v3 = v[h - 1 - j], v4 = v[j];
                const double p13 = v1 + v3, p24 = v2 + v4, m13 = v1 - v3, m42 = v4 - v2;
                f0 = p13 + p24; f1 = p13 - p24; f2 = m13 + m42; f3 = m13 - m42;
            } else {
                f0 = v[j];
            }
        }
        s_f[0][lane][rr] = f0;
        if (nsets == 4) { s_f[1][lane][rr] = f1; s_f[2][lane][rr] = f2; s_f[3][lane][rr] = f3; }
    }
    __syncthreads();
    const int a_rows = nsets * kp;
    for (int idx = threadIdx.x; idx < nsets * 32 * 32; idx += 256) {
        const int set = idx >> 10, jj = (idx >> 5) & 31, rr = idx & 31;
        const int k = j0 + jj;
        if (k >= kp) continue;
        VF[gb_ab_offset(r0 + rr, set * kp + k, a_rows)] = s_f[set][jj][rr];
    }
}

// epilogue of the longitude stage: row rho = i * E + e, column -> spectral row k = 2m + cs;
// Gt[((m * n_ct + c / 120) * nlat_p4 + i) * 124 + c % 120] with c = cs * E + e
struct LatOperandStore {
    static constexpr bool whole_tile = true;
    double* Gt;
    long long M;
    const int* kmap;
    int E, n_ct, nlat_p4;
    struct Pre { int i[4], e[4]; };
    __device__ __forceinline__ Pre prepare(long long row_base, int, int) const {
        Pre pr;
#pragma unroll
        for (int mi = 0; mi < 4; ++mi) {
            const long long row = row_base + mi * 8;
            pr.i[mi] = row < M ? (int)(row / E) : -1;
            pr.e[mi] = (int)(row - (long long)pr.i[mi] * E);
        }
        return pr;
    }
    template <int NI>
    __device__ __forceinline__ void tile(const Pre& pr, long long, int col_base, double (&acc)[4][NI][2]) const {
#pragma unroll
        for (int ni = 0; ni < NI; ++ni) {
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const int k = kmap[col_base + ni * 8 + r];
                if (k < 0) continue;
                const int m = k >> 1, cs = k & 1;
#pragma unroll
                for (int mi = 0; mi < 4; ++mi) {
                    if (pr.i[mi] < 0) continue;
                    const int c = cs * E + pr.e[mi];
                    const int ct = c / GB_S2_TN, cc = c - ct * GB_S2_TN;
                    Gt[(((size_t)m * n_ct + ct) * nlat_p4 + pr.i[mi]) * GB_S2_LDB + cc] = acc[mi][ni][r];
                }
            }
        }
    }
};

// epilogue of the latitude stage: row tile -> (order m, first degree), column c = cs * E + e
struct CoefficientStore {
    static constexpr bool whole_tile = true;
    double* anm;
    const int* tile_m;
    const int* tile_n;
    int L, E;
    struct Pre { int m, n; };
    __device__ __forceinline__ Pre prepare(long long row_base, int, int) const {
        const int t = (int)(row_base >> 7);
        return Pre{tile_m[t], tile_n[t] + (int)(row_base & 127)};
    }
    __device__ __forceinline__ void tile(const Pre& pr, long long, int col_base, double (&acc)[4][5][2]) const {
        // columns are local to the order's column tiles: col_base = ct * 120 + ...
#pragma unroll
        for (int ni = 0; ni < 5; ++ni) {
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const int c = col_base + ni * 8 + r;
                if (c >= 2 * E) continue;
                const int cs = c >= E, e = c - cs * E;
                if (cs && pr.m == 0) continue;
                double* a = anm + (size_t)e * L * L;
#pragma unroll
                for (int mi = 0; mi < 4; ++mi) {
                    const int n = pr.n + mi * 8;
                    if (n >= L) continue;
                    if (cs) a[(size_t)(pr.m - 1) * L + n] = acc[mi][ni][r];
                    else a[(size_t)n * L + pr.m] = acc[mi][ni][r];
                }
            }
        }
    }
};

// ---- longitude stage: G[k][row] = sum_j V[row][j] * lonT[j][k] ;  64 x 64 tile, 4 x 4 per thread
constexpr int LT = 64, LK = 16;

__global__ void __launch_bounds__(256)
gb_analysis_lon_kernel(const double* __restrict__ V, const double* __restrict__ lonT, double* __restrict__ G,
                       long long M, int nlon, int kpad, long long mpad) {
    __shared__ double sV[LK][LT + 1];   // [j][row]
    __shared__ double sT[LK][LT];       // [j][k]
    const long long row0 = (long long)blockIdx.x * LT;
    const int k0 = blockIdx.y * LT;
    const int tx = threadIdx.x & 15;    // k direction
    const int ty = threadIdx.x >> 4;    // row direction
    double acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;

    for (int j0 = 0; j0 < nlon; j0 += LK) {
        // V tile: 64 rows x 16 j, read with j fastest
        for (int idx = threadIdx.x; idx < LT * LK; idx += 256) {
            const int r = idx / LK, jj = idx % LK;
            const long long row = row0 + r;
            const int j = j0 + jj;
            sV[jj][r] = (row < M && j < nlon) ? V[(size_t)row * nlon + j] : 0.0;
        }
        for (int idx = threadIdx.x; idx < LK * LT; idx += 256) {
            const int jj = idx / LT, kk = idx % LT;
            const int j = j0 + jj, k = k0 + kk;
            sT[jj][kk] = (j < nlon && k < kpad) ? lonT[(size_t)j * kpad + k] : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int jj = 0; jj < LK; ++jj) {
            double v[4], t[4];
#pragma unroll
            for (int a = 0; a < 4; ++a) v[a] = sV[jj][ty * 4 + a];
#pragma unroll
            for (int b = 0; b < 4; ++b) t[b] = sT[jj][tx * 4 + b];
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) acc[a][b] = fma(v[a], t[b], acc[a][b]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        const int k = k0 + tx * 4 + b;
        if (k >= kpad) continue;
#pragma unroll
        for (int a = 0; a < 4; ++a) {
            const long long row = row0 + ty * 4 + a;
            if (row < M) G[(size_t)k * mpad + row] = acc[a][b];
        }
    }
}

// ---- latitude stage: one CTA per (order m, epoch tile); a warp owns an output degree, lanes stride
//      over the parallels, sums are combined with warp shuffles.
constexpr int AE = 4;  // epochs per CTA

__global__ void __launch_bounds__(256)
gb_analysis_lat_kernel(const double* __restrict__ G, const double* __restrict__ lat_ops,
                       const long long* __restrict__ lat_off, double* __restrict__ anm, int L, int nlat, int E,
                       int nmin, long long mpad) {
    extern __shared__ double s_g[];  // [2][AE][nlat]
    const int m = blockIdx.x;
    const int e0 = blockIdx.y * AE;
    const int ne = min(AE, E - e0);
    const int n0 = max(m, nmin);
    const int cnt = L - n0;
    if (cnt <= 0) return;
    const double* op = lat_ops + lat_off[m];
    for (int idx = threadIdx.x; idx < 2 * AE * nlat; idx += blockDim.x) {
        const int cs = idx / (AE * nlat);
        const int rem = idx % (AE * nlat);
        const int e = rem / nlat, i = rem % nlat;
        s_g[idx] = (e < ne) ? G[(size_t)(2 * m + cs) * mpad + (size_t)(e0 + e) * nlat + i] : 0.0;
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    for (int r = warp; r < cnt; r += nwarps) {
        double acc[2][AE];
#pragma unroll
        for (int cs = 0; cs < 2; ++cs)
#pragma unroll
            for (int e = 0; e < AE; ++e) acc[cs][e] = 0.0;
        const double* row = op + (size_t)r * nlat;
        for (int i = lane; i < nlat; i += 32) {
            const double w = __ldg(row + i);
#pragma unroll
            for (int cs = 0; cs < 2; ++cs)
#pragma unroll
                for (int e = 0; e < AE; ++e) acc[cs][e] = fma(w, s_g[(cs * AE + e) * nlat + i], acc[cs][e]);
        }
#pragma unroll
        for (int cs = 0; cs < 2; ++cs)
#pragma unroll
            for (int e = 0; e < AE; ++e)
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) acc[cs][e] += __shfl_xor_sync(0xffffffffu, acc[cs][e], off);
        if (lane == 0) {
            const int n = n0 + r;
#pragma unroll
            for (int e = 0; e < AE; ++e) {
                if (e >= ne) break;
                double* a = anm + (size_t)(e0 + e) * L * L;
                a[(size_t)n * L + m] = acc[0][e];
                if (m > 0) a[(size_t)(m - 1) * L + n] = acc[1][e];
            }
        }
    }
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// The latitude-side least-squares operators on the device (reference grid.py:690-696 per order:
// op_m = solve(P' W P, P' W), P[i][n] = kn[i,n] P_nm(theta_i), W = diag(w_lat)): P and (W P)' by the bit-exact recursion,
// then per order the normal matrix (gb_dgemm, FP64 tensor cores), its Cholesky factor (gb_dpotrf_upper) and two
// triangular solves (gb_dtrsm_upper) in place of (W P)'.  The host variant (plan.py: analysis_operators, numpy LU) costs
// 0.5-0.8 s at degree 180; the normal matrices of a quadrature-like grid are well conditioned, the two agree to 1e-14.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32)
gb_ana_design_kernel(double* __restrict__ P, double* __restrict__ PW, const long long* __restrict__ off,
                     const double* __restrict__ ct, const double* __restrict__ kn, const double* __restrict__ pmm,
                     const double* __restrict__ ra, const double* __restrict__ rb, const double* __restrict__ rc, int L,
                     int nlat, int nmin, const double* __restrict__ w) {
    const int i = blockIdx.x * 32 + threadIdx.x, m = blockIdx.y;
    if (i >= nlat) return;
    const int n0 = max(m, nmin), cnt = L - n0;
    if (cnt <= 0) return;
    double* Pm = P + off[m] + (size_t)i * cnt;           // [nlat][cnt]
    double* PWm = PW + off[m] + i;                       // [cnt][nlat]
    const double* kn_i = kn + (size_t)i * L;
    const double wi = w[i];
    gb::legendre_column(m, L, ct[i], pmm[(size_t)i * L + m], ra, rb, rc, [&](int n, double p) {
        if (n < n0) return;
        const double v = __dmul_rn(p, kn_i[n]);
        Pm[n - n0] = v;
        PWm[(size_t)(n - n0) * nlat] = v * wi;
    });
}

// lt[(tile * nlat_p4 + i) * GB_LDA + r] = op_m[r0 + r][i]   (the A operand of the latitude GEMM)
__global__ void __launch_bounds__(GB_TM)
gb_ana_tile_lat_kernel(const double* __restrict__ lat_ops, const long long* __restrict__ off, double* __restrict__ lt,
                       const int* __restrict__ tile_m, const int* __restrict__ tile_n, int nlat, int nlat_p4, int L, int nmin) {
    __shared__ double s_t[32][GB_TM + 1];
    const int t = blockIdx.x, m = tile_m[t];
    const int n0 = max(m, nmin), r0 = tile_n[t] - n0;
    const int rows = min(GB_TM, L - tile_n[t]);
    const int i0 = blockIdx.y * 32;
    const double* op = lat_ops + off[m] + (size_t)r0 * nlat;
    // coalesced along the parallels on the way in, along the rows on the way out
    for (int idx = threadIdx.x; idx < rows * 32; idx += GB_TM) {
        const int r = idx >> 5, ii = idx & 31;
        s_t[ii][r] = (i0 + ii < nlat) ? op[(size_t)r * nlat + i0 + ii] : 0.0;
    }
    __syncthreads();
    const int r = threadIdx.x;
    if (r < rows)
        for (int ii = 0; ii < 32 && i0 + ii < nlat; ++ii) lt[((size_t)t * nlat_p4 + i0 + ii) * GB_LDA + r] = s_t[ii][r];
}

static int build_lat_operators(gb_plan* p, int nmin, const double* w_lat) {
    const int L = p->L, nlat = p->nlat, dev = p->device;
    const size_t total = (size_t)p->h_lat_off[L];
    if (total == 0) return GB_OK;
    double *d_p = nullptr, *d_n = nullptr, *d_w = nullptr;
    int* d_info = nullptr;
    auto cleanup = [&] { cudaFree(d_p); cudaFree(d_n); cudaFree(d_w); cudaFree(d_info); };
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&d_p), total * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&d_n), (size_t)L * L * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&d_w), (size_t)nlat * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&d_info), (size_t)L * sizeof(int));
    if (e == cudaSuccess) e = cudaMemcpy(d_w, w_lat, (size_t)nlat * sizeof(double), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        cleanup();
        return gb_set_error(GB_ERR_CUDA, "gb_plan_set_analysis_weights: %s", cudaGetErrorString(e));
    }
    gb_ana_design_kernel<<<dim3((nlat + 31) / 32, L), 32>>>(d_p, p->d_lat_ops, p->d_lat_off, p->d_ct, p->d_kn, p->d_pmm, p->d_ra,
                                                          p->d_rb, p->d_rc, L, nlat, nmin, d_w);
    gb_count_launch();
    int rc = GB_OK;
    for (int m = 0; m < L && !rc; ++m) {
        const long long cnt = L - (m > nmin ? m : nmin);
        if (cnt <= 0) continue;
        double* pw = p->d_lat_ops + p->h_lat_off[m];      // (W P)' [cnt][nlat] -> the operator, in place
        const double* pm = d_p + p->h_lat_off[m];         // P [nlat][cnt]
        rc = gb_dgemm(0, 0, cnt, cnt, nlat, 1.0, pw, nlat, pm, cnt, 0.0, d_n, cnt, 1, dev, nullptr);
        if (!rc) rc = gb_dpotrf_upper(d_n, cnt, cnt, d_info + m, dev, nullptr);
        if (!rc) rc = gb_dtrsm_upper(1, d_n, cnt, cnt, pw, nlat, nlat, dev, nullptr);
        if (!rc) rc = gb_dtrsm_upper(0, d_n, cnt, cnt, pw, nlat, nlat, dev, nullptr);
    }
    if (!rc) {
        std::vector<int> info(L, 0);
        e = cudaMemcpy(info.data(), d_info, (size_t)L * sizeof(int), cudaMemcpyDeviceToHost);   // also waits for the stream
        if (e != cudaSuccess) rc = gb_set_error(GB_ERR_CUDA, "gb_plan_set_analysis_weights: %s", cudaGetErrorString(e));
        for (int m = 0; m < L && !rc; ++m)
            if (L - (m > nmin ? m : nmin) > 0 && info[m] != 0)
                rc = gb_set_error(GB_ERR_ARGUMENT, "gb_plan_set_analysis_weights: the normal matrix of order %d is not positive "
                                  "definite (pivot %d): the grid does not resolve degree %d", m, info[m], p->nmax);
    }
    cleanup();
    return rc;
}

// lat_ops != nullptr: host operators (gb_plan_set_analysis); else they are built on the device from the latitude
// weights w_lat (gb_plan_set_analysis_weights)
static int set_analysis(gb_plan* plan, int nmin, const double* lon_ops, const double* lat_ops, const int64_t* lat_op_offsets,
                        const double* w_lat) {
    GB_REQUIRE(plan != nullptr, "gb_plan_set_analysis: plan is NULL");
    GB_REQUIRE(nmin >= 0 && nmin <= plan->nmax, "gb_plan_set_analysis: min_degree=%d outside [0, %d]", nmin, plan->nmax);
    GB_REQUIRE(lon_ops && ((lat_ops && lat_op_offsets) || w_lat), "gb_plan_set_analysis: NULL pointer");
    gb_plan* p = plan;
    GB_CUDA(cudaSetDevice(p->device));
    GB_CUDA(cudaDeviceSynchronize());
    cudaFree(p->d_lon_ops); p->d_lon_ops = nullptr;
    cudaFree(p->d_lat_ops); p->d_lat_ops = nullptr;
    cudaFree(p->d_lat_off); p->d_lat_off = nullptr;
    delete[] p->h_lat_off; p->h_lat_off = nullptr;
    p->ana_nmin = -1;
    const int L = p->L;
    // transposed + zero padded longitude operator: lonT[j][k], k = 2m + cs
    std::vector<double> lonT((size_t)p->nlp * p->kpad, 0.0);
    for (int k = 0; k < 2 * L; ++k)
        for (int j = 0; j < p->nlon; ++j) lonT[(size_t)j * p->kpad + k] = lon_ops[(size_t)k * p->nlon + j];
    GB_CUDA(cudaMalloc(reinterpret_cast<void**>(&p->d_lon_ops), lonT.size() * sizeof(double)));
    GB_CUDA(cudaMemcpy(p->d_lon_ops, lonT.data(), lonT.size() * sizeof(double), cudaMemcpyHostToDevice));
    p->h_lat_off = new long long[L + 1];
    p->h_lat_off[0] = 0;
    for (int m = 0; m < L; ++m) {
        const long long expect = (long long)(L - (m > nmin ? m : nmin)) * p->nlat;
        if (lat_ops) {
            GB_REQUIRE(lat_op_offsets[m + 1] - lat_op_offsets[m] == (expect > 0 ? expect : 0),
                       "gb_plan_set_analysis: operator of order %d has %lld elements, expected %lld", m,
                       (long long)(lat_op_offsets[m + 1] - lat_op_offsets[m]), expect);
        }
        p->h_lat_off[m + 1] = p->h_lat_off[m] + (expect > 0 ? expect : 0);
    }
    const size_t total = (size_t)p->h_lat_off[L];
    GB_CUDA(cudaMalloc(reinterpret_cast<void**>(&p->d_lat_ops), (total ? total : 1) * sizeof(double)));
    GB_CUDA(cudaMalloc(reinterpret_cast<void**>(&p->d_lat_off), (L + 1) * sizeof(long long)));
    GB_CUDA(cudaMemcpy(p->d_lat_off, p->h_lat_off, (L + 1) * sizeof(long long), cudaMemcpyHostToDevice));
    if (lat_ops) {
        GB_CUDA(cudaMemcpy(p->d_lat_ops, lat_ops, total * sizeof(double), cudaMemcpyHostToDevice));
    } else {
        int rcb = build_lat_operators(p, nmin, w_lat);
        if (rcb) return rcb;
    }

    // ---- operator tiles for the tensor-core longitude stage ----
    cudaFree(p->d_ana_w_t); p->d_ana_w_t = nullptr;
    cudaFree(p->d_ana_kmap); p->d_ana_kmap = nullptr;
    const int nlon = p->nlon, h = nlon / 2, q = nlon / 4;
    bool sym = (nlon % 8 == 0);
    for (int k = 0; k < 2 * L && sym; ++k) {
        const int m = k >> 1;
        const bool sine = (k & 1) != 0;
        if (sine && m == 0) continue;
        const double* row = lon_ops + (size_t)k * nlon;
        double amax = 0.0;
        for (int j = 0; j < nlon; ++j) amax = std::fmax(amax, std::fabs(row[j]));
        const double tol = 4.0 * (m + 1) * 2.220446049250313e-16 * 3.141592653589793 * amax;
        const double sg = (m & 1) ? -1.0 : 1.0;
        for (int j = 0; j < q; ++j) {
            const double c = row[h + j];
            const double e2 = sine ? -sg * c : sg * c;   // at pi - mu
            const double e3 = sine ? -c : c;             // at -mu
            const double e4 = sg * c;                    // at mu - pi
            if (std::fabs(row[nlon - 1 - j] - e2) > tol || std::fabs(row[h - 1 - j] - e3) > tol ||
                std::fabs(row[j] - e4) > tol) {
                sym = false;
                break;
            }
        }
    }
    if (gb_env_flag("GB_NO_SYMMETRY")) sym = false;
    std::vector<std::vector<int>> cols;   // spectral rows (2m+cs) per set
    if (sym) {
        cols.resize(4);
        for (int m = 0; m < L; ++m) {
            cols[m & 1].push_back(2 * m);
            if (m > 0) cols[2 + (m & 1)].push_back(2 * m + 1);
        }
        p->ana_nsets = 4;
        p->ana_kp = (q + 3) / 4 * 4;
    } else {
        cols.resize(1);
        for (int k = 0; k < 2 * L; ++k) cols[0].push_back(k);
        p->ana_nsets = 1;
        p->ana_kp = (nlon + 3) / 4 * 4;
    }
    size_t widest = 1;
    for (auto& c : cols) widest = c.size() > widest ? c.size() : widest;
    // column tile width of the longitude GEMM: 24 NI columns with NI = 2..5 fragments per warp; every set gets whole
    // tiles, so the width that wastes the fewest padded columns wins (91 columns per set at degree 180: 96, not 120)
    int best_ni = 5;
    size_t best_cols = ~(size_t)0;
    for (int ni = 2; ni <= 5; ++ni) {
        const size_t tn = (size_t)gbgemm::tile_n(ni);
        const size_t padded = (widest + tn - 1) / tn * tn;
        if (padded < best_cols) { best_cols = padded; best_ni = ni; }
    }
    p->ana_ni = best_ni;
    const int tn = gbgemm::tile_n(best_ni), ldb = gbgemm::tile_ldb(best_ni);
    p->ana_tps = (int)((widest + tn - 1) / tn);
    const int ntiles = p->ana_nsets * p->ana_tps;
    std::vector<double> wt((size_t)ntiles * p->ana_kp * ldb, 0.0);
    std::vector<int> kmap((size_t)ntiles * tn, -1);
    const int kvalid = sym ? q : nlon;
    for (int s = 0; s < p->ana_nsets; ++s)
        for (size_t c = 0; c < cols[s].size(); ++c) {
            const int tile = s * p->ana_tps + (int)(c / tn), cc = (int)(c % tn);
            const int k = cols[s][c];
            kmap[(size_t)tile * tn + cc] = k;
            const double* row = lon_ops + (size_t)k * nlon;
            for (int j = 0; j < kvalid; ++j)
                wt[((size_t)tile * p->ana_kp + j) * ldb + cc] = sym ? row[h + j] : row[j];
        }
    GB_CUDA(cudaMalloc(reinterpret_cast<void**>(&p->d_ana_w_t), wt.size() * sizeof(double)));
    GB_CUDA(cudaMemcpy(p->d_ana_w_t, wt.data(), wt.size() * sizeof(double), cudaMemcpyHostToDevice));
    GB_CUDA(cudaMalloc(reinterpret_cast<void**>(&p->d_ana_kmap), kmap.size() * sizeof(int)));
    GB_CUDA(cudaMemcpy(p->d_ana_kmap, kmap.data(), kmap.size() * sizeof(int), cudaMemcpyHostToDevice));
    // ---- operator tiles for the tensor-core latitude stage: A[i][r] = lat_op_m[r][i] ----
    cudaFree(p->d_ana_lat_t); p->d_ana_lat_t = nullptr;
    cudaFree(p->d_ana_lat_m); p->d_ana_lat_m = nullptr;
    cudaFree(p->d_ana_lat_n); p->d_ana_lat_n = nullptr;
    {
        const int nlat = p->nlat;
        p->ana_nlat_p4 = (nlat + 3) / 4 * 4;
        std::vector<int> tile_m, tile_n;
        for (int m = 0; m < L; ++m) {
            const int n0 = m > nmin ? m : nmin;
            for (int r0 = 0; r0 < L - n0; r0 += GB_TM) {
                tile_m.push_back(m);
                tile_n.push_back(n0 + r0);
            }
        }
        p->ana_lat_tiles = (int)tile_m.size();
        const size_t lt_elems = (size_t)p->ana_lat_tiles * p->ana_nlat_p4 * GB_LDA;
        GB_CUDA(cudaMalloc(reinterpret_cast<void**>(&p->d_ana_lat_t), (lt_elems ? lt_elems : 1) * sizeof(double)));
        GB_CUDA(cudaMemset(p->d_ana_lat_t, 0, (lt_elems ? lt_elems : 1) * sizeof(double)));
        GB_CUDA(cudaMalloc(reinterpret_cast<void**>(&p->d_ana_lat_m), (tile_m.size() + 1) * sizeof(int)));
        GB_CUDA(cudaMemcpy(p->d_ana_lat_m, tile_m.data(), tile_m.size() * sizeof(int), cudaMemcpyHostToDevice));
        GB_CUDA(cudaMalloc(reinterpret_cast<void**>(&p->d_ana_lat_n), (tile_n.size() + 1) * sizeof(int)));
        GB_CUDA(cudaMemcpy(p->d_ana_lat_n, tile_n.data(), tile_n.size() * sizeof(int), cudaMemcpyHostToDevice));
        if (p->ana_lat_tiles > 0) {
            // A[i][r] = lat_op_m[r][i]: the operators (host-built and uploaded, or built on the device) re-tiled on the device
            gb_ana_tile_lat_kernel<<<dim3(p->ana_lat_tiles, (nlat + 31) / 32), GB_TM>>>(
                p->d_lat_ops, p->d_lat_off, p->d_ana_lat_t, p->d_ana_lat_m, p->d_ana_lat_n, nlat, p->ana_nlat_p4, L, nmin);
            GB_LAUNCH_CHECK();
            GB_CUDA(cudaDeviceSynchronize());
        }
    }
    p->ana_nmin = nmin;
    return GB_OK;
}

extern "C" int gb_plan_set_analysis(gb_plan* plan, int nmin, const double* lon_ops, const double* lat_ops,
                                    const int64_t* lat_op_offsets) {
    GB_REQUIRE(lat_ops && lat_op_offsets, "gb_plan_set_analysis: NULL pointer");
    return set_analysis(plan, nmin, lon_ops, lat_ops, lat_op_offsets, nullptr);
}

extern "C" int gb_plan_set_analysis_weights(gb_plan* plan, int nmin, const double* lon_ops, const double* w_lat) {
    GB_REQUIRE(w_lat, "gb_plan_set_analysis_weights: NULL pointer");
    return set_analysis(plan, nmin, lon_ops, nullptr, nullptr, w_lat);
}

static int launch_analysis(gb_plan* p, const double* d_grid, int E, double* d_anm, cudaStream_t st) {
    {
        int rca = gb_plan_acquire(p, st);   // one workspace per plan: order this call behind the previous one
        if (rca) return rca;
    }
    const int L = p->L;
    const long long M = (long long)E * p->nlat;
    const long long mpad = p->ws_mpad;
    GB_CUDA(cudaMemsetAsync(d_anm, 0, (size_t)E * L * L * sizeof(double), st));
    if (gb_env_flag("GB_SIMPLE_ANALYSIS")) {
        // plain FMA longitude stage (cross-check of the tensor-core path)
        dim3 grid((unsigned)((M + LT - 1) / LT), (p->kpad + LT - 1) / LT);
        gb_analysis_lon_kernel<<<grid, 256, 0, st>>>(d_grid, p->d_lon_ops, p->d_ab, M, p->nlon, p->kpad, mpad);
        GB_LAUNCH_CHECK();
        dim3 grid2(L, (E + AE - 1) / AE);
        const size_t smem = (size_t)2 * AE * p->nlat * sizeof(double);
        if (smem > 48 * 1024)
            GB_CUDA(cudaFuncSetAttribute(gb_analysis_lat_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        gb_analysis_lat_kernel<<<grid2, 256, smem, st>>>(p->d_ab, p->d_lat_ops, p->d_lat_off, d_anm, L, p->nlat, E,
                                                         p->ana_nmin, mpad);
        GB_LAUNCH_CHECK();
        return GB_OK;
    }
    // fold / transpose V into the tiled operand layout (rows (i, e), epochs fastest), then one persistent
    // DMMA GEMM over all sets whose epilogue writes the B tiles of the latitude stage
    const int n_mtiles = (int)((M + GB_TM - 1) / GB_TM);
    const int a_rows = p->ana_nsets * p->ana_kp;
    const size_t vf_elems = (size_t)n_mtiles * a_rows * GB_LDA;
    const int n_ct = (2 * E + GB_S2_TN - 1) / GB_S2_TN;
    const size_t gt_elems = (size_t)L * n_ct * p->ana_nlat_p4 * GB_S2_LDB;
    if (vf_elems > p->ana_vf_elems || gt_elems > p->ana_gt_elems) {   // grow-only workspaces (a fresh 1 GB allocation per call costs milliseconds)
        GB_CUDA(cudaStreamSynchronize(st));
        if (vf_elems > p->ana_vf_elems) {
            cudaFree(p->d_ana_vf);
            p->d_ana_vf = nullptr;
            p->ana_vf_elems = 0;
            GB_CUDA(cudaMalloc(reinterpret_cast<void**>(&p->d_ana_vf), vf_elems * sizeof(double)));
            p->ana_vf_elems = vf_elems;
        }
        if (gt_elems > p->ana_gt_elems) {
            cudaFree(p->d_ana_gt);
            p->d_ana_gt = nullptr;
            p->ana_gt_elems = 0;
            GB_CUDA(cudaMalloc(reinterpret_cast<void**>(&p->d_ana_gt), gt_elems * sizeof(double)));
            p->ana_gt_elems = gt_elems;
            p->ana_gt_epochs = -1;
        }
    }
    // padding parallels / columns and the sine columns of order 0 are never written: they must be finite (zero).
    // Everything else is overwritten by every call, so the buffer is cleared only when its layout changes.
    if (p->ana_gt_epochs != E) {
        GB_CUDA(cudaMemsetAsync(p->d_ana_gt, 0, p->ana_gt_elems * sizeof(double), st));
        p->ana_gt_epochs = E;
    }
    {
        dim3 grid((p->ana_kp + 31) / 32, n_mtiles * 4);
        gb_analysis_fold<<<grid, 256, 0, st>>>(d_grid, p->d_ana_vf, M, p->nlon, p->ana_nsets, p->ana_kp,
                                               p->ana_nsets == 4 ? p->nlon / 4 : p->nlon, E, p->nlat);
        GB_LAUNCH_CHECK();
    }
    {
        gbgemm::Shape sh;
        sh.A_t = p->d_ana_vf;
        sh.a_rows = a_rows;
        sh.a_koff_mul = p->ana_kp;
        sh.tiles_per_group = p->ana_tps;
        sh.B_t = p->d_ana_w_t;
        sh.b_rows = p->ana_kp;
        sh.klen = p->ana_kp;
        sh.n_mtiles = n_mtiles;
        sh.n_ntiles = p->ana_nsets * p->ana_tps;
        const LatOperandStore epi{p->d_ana_gt, M, p->d_ana_kmap, E, n_ct, p->ana_nlat_p4};
        int rc;
        switch (p->ana_ni) {
            case 2: rc = gbgemm::launch<LatOperandStore, 2>(sh, epi, p->sm_count, st); break;
            case 3: rc = gbgemm::launch<LatOperandStore, 3>(sh, epi, p->sm_count, st); break;
            case 4: rc = gbgemm::launch<LatOperandStore, 4>(sh, epi, p->sm_count, st); break;
            default: rc = gbgemm::launch<LatOperandStore, 5>(sh, epi, p->sm_count, st); break;
        }
        if (rc) return rc;
    }
    {
        gbgemm::Shape sh;
        sh.A_t = p->d_ana_lat_t;
        sh.a_rows = p->ana_nlat_p4;
        sh.a_koff_mul = 0;
        sh.tiles_per_group = 1;
        sh.B_t = p->d_ana_gt;
        sh.b_rows = p->ana_nlat_p4;
        sh.klen = p->ana_nlat_p4;
        sh.n_mtiles = p->ana_lat_tiles;
        sh.n_ntiles = n_ct;
        sh.mt_bgroup = p->d_ana_lat_m;
        int rc = gbgemm::launch(sh, CoefficientStore{d_anm, p->d_ana_lat_m, p->d_ana_lat_n, L, E}, p->sm_count, st);
        if (rc) return rc;
    }
    return GB_OK;
}

extern "C" int gb_analysis(gb_plan* plan, const double* d_grid, int n_epochs, double* d_anm, void* stream) {
    GB_REQUIRE(plan != nullptr, "gb_analysis: plan is NULL");
    GB_REQUIRE(plan->ana_nmin >= 0, "gb_analysis: gb_plan_set_analysis has not been called for this plan");
    GB_REQUIRE(n_epochs >= 0, "gb_analysis: n_epochs=%d is negative", n_epochs);
    if (n_epochs == 0) return GB_OK;
    GB_REQUIRE(d_grid && d_anm, "gb_analysis: NULL device pointer");
    GB_CUDA(cudaSetDevice(plan->device));
    int rc = gb_plan_ensure_workspace(plan, n_epochs);
    if (rc) return rc;
    return launch_analysis(plan, d_grid, n_epochs, d_anm, static_cast<cudaStream_t>(stream));
}

extern "C" int gb_analysis_host(gb_plan* plan, const double* h_grid, int n_epochs, double* h_anm) {
    GB_REQUIRE(plan != nullptr, "gb_analysis_host: plan is NULL");
    GB_REQUIRE(plan->ana_nmin >= 0, "gb_analysis_host: gb_plan_set_analysis has not been called for this plan");
    GB_REQUIRE(n_epochs >= 0, "gb_analysis_host: n_epochs=%d is negative", n_epochs);
    if (n_epochs == 0) return GB_OK;
    GB_REQUIRE(h_grid && h_anm, "gb_analysis_host: NULL host pointer");
    gb_plan* p = plan;
    GB_CUDA(cudaSetDevice(p->device));
    const size_t pts = (size_t)p->nlat * p->nlon, coef = (size_t)p->L * p->L;
    // epoch chunks: the upload of chunk c+1 overlaps the kernels of chunk c
    int chunk = (n_epochs + 7) / 8;
    if (chunk < 1) chunk = 1;
    int rc = gb_plan_ensure_workspace(p, chunk);
    if (rc) return rc;
    if (!p->s_compute) GB_CUDA(cudaStreamCreateWithFlags(&p->s_compute, cudaStreamNonBlocking));
    if (!p->s_copy) GB_CUDA(cudaStreamCreateWithFlags(&p->s_copy, cudaStreamNonBlocking));
    for (auto& e : p->ev)
        if (!e) GB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    double* d_in[2] = {nullptr, nullptr};
    double* d_out = nullptr;
    for (int b = 0; b < 2; ++b) GB_CUDA(cudaMalloc(reinterpret_cast<void**>(&d_in[b]), (size_t)chunk * pts * sizeof(double)));
    GB_CUDA(cudaMalloc(reinterpret_cast<void**>(&d_out), (size_t)n_epochs * coef * sizeof(double)));
    int c = 0;
    for (int e0 = 0; e0 < n_epochs; e0 += chunk, ++c) {
        const int ne = (n_epochs - e0 < chunk) ? (n_epochs - e0) : chunk;
        const int b = c & 1;
        if (c >= 2) GB_CUDA(cudaStreamWaitEvent(p->s_copy, p->ev[2 + b], 0));  // kernels done with buffer b
        GB_CUDA(cudaMemcpyAsync(d_in[b], h_grid + (size_t)e0 * pts, (size_t)ne * pts * sizeof(double),
                                cudaMemcpyHostToDevice, p->s_copy));
        GB_CUDA(cudaEventRecord(p->ev[b], p->s_copy));
        GB_CUDA(cudaStreamWaitEvent(p->s_compute, p->ev[b], 0));
        if ((rc = launch_analysis(p, d_in[b], ne, d_out + (size_t)e0 * coef, p->s_compute))) break;
        GB_CUDA(cudaEventRecord(p->ev[2 + b], p->s_compute));
    }
    if (rc == GB_OK) {
        cudaError_t e = cudaMemcpyAsync(h_anm, d_out, (size_t)n_epochs * coef * sizeof(double), cudaMemcpyDeviceToHost,
                                        p->s_compute);
        if (e != cudaSuccess) rc = gb_set_error(GB_ERR_CUDA, "gb_analysis_host: result copy failed: %s", cudaGetErrorString(e));
    }
    cudaStreamSynchronize(p->s_compute);
    cudaStreamSynchronize(p->s_copy);
    cudaFree(d_in[0]); cudaFree(d_in[1]); cudaFree(d_out);
    return rc;
}
