// Covariance propagation to grid-point variances on B200: diag(F Sigma F') for a regular grid.
//
// Replaces the per-parallel products of RegularGrid.covariance_propagation (reference
// grid.py:833-835), F[(i,j), a] = U_i[a] * t_a(j) with U_i[a] = kn[i,n] P_nm(theta_i) and
// t_a(j) = cos/sin(m lon_j).  The reference forms F Sigma F' (nlon x nlon) per parallel and keeps
// its diagonal: 2 P K^2 flops.  On a regular grid F factors, so the same numbers follow from
//
//   H_i[k,k'] = sum_{a in k} sum_{b in k'} U_i[a] Sigma[a,b] U_i[b]        (k = (m, cos|sin) group)
//   var[i,j]  = sum_k T[k,j] * ( sum_k' H_i[k,k'] T[k',j] )
//
// i.e. 2 nlat K^2 + 2 P (2L)^2 flops (config 4: 83.6 GF instead of 45.9 TF).  This restructuring is
// DECLARED in DESIGN.md; bench_configs.py reports contract and executed flops separately, and the
// direct kernel without any structure assumption is gb_points_covariance (gb_points.cu).
//
// Second declared shortcut, the equator fold (same gate as the folded Legendre stage of the synthesis,
// gb_plan::fold_ns / fold_cap): U_{i'}[a] = (-1)^(n-m) U_i[a] for the mirror image i' of parallel i, so with the
// coefficients of every group split into the parity classes of n - m
//   S_i = same-class pairs (a, b),  D_i = cross-class pairs:   H_i = S_i + D_i,   H_i' = S_i - D_i
// and the first contraction runs for the northern parallels only, class by class: half its flops.  The split
// itself is exact for any parallel (it is a partition of the index pairs), so ONE kernel serves folded and
// unfolded calls: a parallel without usable mirror image simply is its own "representative" with sign +.
//
// Every partial sum has ONE writer and the partials are added in a fixed order by small reduction kernels: the
// result is bit-identical from run to run.
//
//   1. gb_cov_permute_degree   Sigma (degree-wise order) -> tiled operand St[row tile a'][b][132]: order-wise order;
//                        rows a': groups padded to 8; columns b: every group as [class 0 | class 1], each padded to 4;
//                        zeros in the padding.  For a symmetric Sigma only the blocks k <= k' are read and written.
//   2. gb_cov_legendre   on-the-fly Legendre recursion * kn for the representative parallels -> U as GEMM
//                        B tiles [group k' * nti + parallel tile][b][tn + 4] (same class order of the rows b)
//   3. gb_cov_quad_kernel   C[a', i] = sum_{b in k', class c'} St[a'][b] U[b][i] on the FP64 tensor cores, then
//                        Hpart[i][k'][piece(a')][c'][row parity] = sum over the rows of the piece of U[a'][i] C[a'][i].
//                        A CTA walks "segments" = (row tile, parallel tile, range of k'), so the row-side factor
//                        U[a'][i] of its tile is fetched once per segment and parked in TENSOR MEMORY (thread-private
//                        columns) instead of 20 L2 loads per thread and tile.
//      gb_cov_reduce_h   S, D = ordered sums of the pieces; H = S + D -> northern row, S - D -> mirrored row,
//                        written in the A-tile layout of stage 4
//   4. GEMM + LonEpilogue    W_i[k, j] = sum_k' H_i[k][k'] T[k'][j];          varpart[i][slot][j] = sum T[k][j] W
//   5. gb_cov_finish     var = sum of the slots in order, optional sqrt
#include <vector>
#include <cmath>
#include <algorithm>
#include "gb_common.cuh"
#include "gb_gemm.cuh"

namespace {

using gb::legendre_column;

// row of degree offset r (n = n0 + r) inside its group: class (r + po) & 1, po = (n0 - m) & 1; class 1 starts at ne4
__host__ __device__ __forceinline__ int cov_cls_pos(int r, int po, int ne4) { return (((r + po) & 1) ? ne4 : 0) + (r >> 1); }

// St[gb_ab_offset(a', b, Kp4)] = Sigma[perm8[a']][perm4[b]] (0 where either index is padding), one CTA per (32 rows a',
// 64 columns of degree n): the 2n+1 columns of a degree are contiguous in the degree-wise order, so Sigma is read in
// row segments of up to 512 bytes and St written in 256-byte runs (an element-wise gather fetches a 32-byte sector per
// double); 16 KB of shared memory per CTA keeps a dozen CTAs resident per SM.
// Symmetric Sigma (first_group != nullptr): a row tile only meets column groups k' >= its own first group kmin,
// i.e. the columns j >= jmin of every degree: the rest of the row block is neither read nor written (the quadratic-form
// kernel never touches it).
constexpr int CP_ROWS = 32, CP_COLS = 64, CP_PITCH = CP_COLS + 1;     // odd pitch: conflict-free column reads
__global__ void __launch_bounds__(256)
gb_cov_permute_degree(const double* __restrict__ sigma, double* __restrict__ St, const int* __restrict__ perm8,
                      const int* __restrict__ goff4, const int* __restrict__ ne4, int Kp4, long long K, int nmin,
                      const int* __restrict__ first_group) {
    __shared__ double s_p[CP_ROWS * CP_PITCH];
    __shared__ int s_b[CP_COLS];                                      // row of St of every column of this CTA
    const int a0 = blockIdx.x * CP_ROWS;
    const int n = nmin + blockIdx.y;
    const int width = 2 * n + 1;
    int jmin = 0;
    if (first_group) {
        const int kmin = first_group[a0 >> 7];                        // first group of the 128-row tile
        jmin = kmin <= 1 ? 0 : kmin - 1;                              // group 2m (cos) is column 2m-1, group 2m+1 (sin) column 2m
    }
    const int j0 = blockIdx.z * CP_COLS;                              // this CTA: columns [j0, j1) of the degree
    const int j1 = min(width, j0 + CP_COLS);
    const int jlo = max(jmin, j0);
    if (jlo >= j1) return;
    const long long col0 = (long long)n * n - (long long)nmin * nmin;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // the two dependent table look-ups per column run here, beside the loads of Sigma, not in front of every store
    if (threadIdx.x < CP_COLS && jlo + (int)threadIdx.x < j1) {
        const int j = jlo + threadIdx.x;
        const int m = (j + 1) >> 1;
        const int k = (j == 0) ? 0 : 2 * m + ((j & 1) ? 0 : 1);          // j = 2m-1: cos, j = 2m: sin
        const int n0 = max(m, nmin);
        s_b[j - j0] = goff4[k] + cov_cls_pos(n - n0, (n0 - m) & 1, ne4[k]);
    }
    for (int r = warp; r < CP_ROWS; r += 8) {
        const int pa = perm8[a0 + r];
        const double* src = sigma + (size_t)(pa < 0 ? 0 : pa) * K + col0;
        // Sigma is read once: streaming loads keep the re-tiled operand (and U) in L2 instead
        for (int j = jlo + lane; j < j1; j += 32) s_p[r * CP_PITCH + j - j0] = pa < 0 ? 0.0 : __ldcs(src + j);
    }
    __syncthreads();
    for (int j = jlo + warp; j < j1; j += 8) {
        const int b = s_b[j - j0];
        double* dst = St + ((size_t)(a0 >> 7) * Kp4 + b) * GB_LDA + (a0 & (GB_TM - 1));
#pragma unroll
        for (int r = lane; r < CP_ROWS; r += 32) dst[r] = s_p[r * CP_PITCH + j - j0];
    }
}

// rows b of St that pad a class to a multiple of four
__global__ void __launch_bounds__(128)
gb_cov_zero_rows(double* __restrict__ St, const int* __restrict__ padrows, int n_padrows, int Kp4) {
    for (int r = blockIdx.y * 16; r < min(n_padrows, blockIdx.y * 16 + 16); ++r)
        St[((size_t)blockIdx.x * Kp4 + padrows[r]) * GB_LDA + threadIdx.x] = 0.0;
}

// U as B tiles: Ut[((k * nti + r / tn) * Kg + row(n)) * ldb + r % tn] = kn[i][n] * P_nm(theta_i), i = rep[r]
__global__ void __launch_bounds__(128)
gb_cov_legendre(double* __restrict__ Ut, const double* __restrict__ ct, const double* __restrict__ kn,
                const double* __restrict__ pmm, const double* __restrict__ ra, const double* __restrict__ rb,
                const double* __restrict__ rc, int L, int nmin, const int* __restrict__ rep, int nrep, int nti, int Kg,
                int tn, int ldb, const double* __restrict__ wn, const int* __restrict__ ne4) {
    const int il = blockIdx.x * blockDim.x + threadIdx.x;
    const int m = blockIdx.y;
    if (il >= nrep) return;
    const int i = rep[il];
    const int n0 = max(m, nmin);
    const int po = (n0 - m) & 1, e4 = ne4[2 * m];
    const double* kn_i = kn + (size_t)i * L;
    const int it = il / tn, ic = il % tn;
    double* uc = Ut + ((size_t)(2 * m) * nti + it) * Kg * ldb + ic;
    double* us = Ut + ((size_t)(2 * m + 1) * nti + it) * Kg * ldb + ic;
    legendre_column(m, L, ct[i], pmm[(size_t)i * L + m], ra, rb, rc, [&](int n, double p) {
        if (n < n0) return;
        double v = __dmul_rn(p, kn_i[n]);
        if (wn) v *= wn[n];                       // isotropic filter: F = diag(w_n)
        const size_t row = (size_t)cov_cls_pos(n - n0, po, e4) * ldb;
        uc[row] = v;
        if (m > 0) us[row] = v;
    });
}

// Filtered covariances: diag(A F Sigma F' A') = diag((A F) Sigma (A F)').  An order-wise filter F only mixes
// coefficients of one (order, cos|sin) group, so A F keeps the product structure of A with
//   U'[b][i] = sum_{a in group} W_g[a][b] U[a][i]          (W_g: the group's block of F, reference filter.py:193-222)
// One thread per parallel, eight output degrees per CTA; the U tile of the group is re-read from L2.  (F mixes the
// parity classes, so filtered calls never fold; the class order of the rows is only a layout here.)
constexpr int CF_B = 8;
__global__ void __launch_bounds__(128)
gb_cov_apply_blocks(const double* __restrict__ Ut, double* __restrict__ Ut2, const double* __restrict__ blocks,
                    const long long* __restrict__ offsets, int nf, int L, int nmin, int nti, int Kg, int ldb,
                    const int* __restrict__ ne4) {
    const int k = blockIdx.x;                 // group 2m + cs
    const int it = blockIdx.y;
    const int b0 = blockIdx.z * CF_B;
    const int m = k >> 1, cs = k & 1;
    if (m >= L || (m == 0 && cs == 1)) return;
    const int n0 = max(m, nmin);
    const int cnt = L - n0;
    if (b0 >= cnt) return;
    const int po = (n0 - m) & 1, e4 = ne4[k];
    const int g = (m == 0) ? 0 : 2 * m - 1 + cs;          // block index of the filter (filter.py:180-187)
    const int kf = nf + 1 - m;
    const double* W = blocks + offsets[g] + (size_t)(n0 - m) * kf + (n0 - m);   // rows / columns of degree >= n0
    const size_t tile = ((size_t)k * nti + it) * Kg * ldb;
    const double* u = Ut + tile + threadIdx.x;
    double acc[CF_B];
#pragma unroll
    for (int j = 0; j < CF_B; ++j) acc[j] = 0.0;
    if (threadIdx.x < ldb) {
        for (int a = 0; a < cnt; ++a) {
            const double ua = u[(size_t)cov_cls_pos(a, po, e4) * ldb];
            const double* wrow = W + (size_t)a * kf + b0;
#pragma unroll
            for (int j = 0; j < CF_B; ++j)
                if (b0 + j < cnt) acc[j] = fma(__ldg(wrow + j), ua, acc[j]);
        }
#pragma unroll
        for (int j = 0; j < CF_B; ++j)
            if (b0 + j < cnt) Ut2[tile + (size_t)cov_cls_pos(b0 + j, po, e4) * ldb + threadIdx.x] = acc[j];
    }
}

// ---------------------------------------------------------------------------------------------
// The quadratic-form contraction.  Persistent, 12 consumer warps (4 x 3, 32 x 8 NI register tiles) + a producer warp
// with a 3-stage bulk-copy ring (as gbgemm::kernel).  Work = segments (row tile mt, parallel tile it, groups [k0, k1)):
// at the head of a segment every consumer thread fetches the 8 NI row-side factors U[a'][i] of its fragments and parks
// them in tensor memory; then per (k', class c') one short K loop (the class holds at most (L + 1) / 2 rows) and the
// epilogue: multiply by the parked factors, add the slabs of one group inside the thread, reduce over the rows of equal
// parity inside the slab (two shuffles) and store the piece.
// ---------------------------------------------------------------------------------------------
struct QuadArgs {
    const double* St;        // [n_atiles][Kp4][GB_LDA]
    const double* Ut;        // [kpad * nti][Kg][ldb]
    double* Hpart;           // [nrep][kpad][n_pieces][2 classes of b][2 row parities]
    const int4* segs;        // (mt, it, k0, k1)
    const int* rowgroup;     // [rows_a / 8] group k of each 8-row slab, -1: padding
    const int* goff8;        // [kpad] first a' of each group
    const int* gcnt;         // [kpad] coefficients in each group
    const int* piece_of;     // [rows_a / 8] piece of the run of slabs that starts here (valid at run heads)
    const int* goff4;        // [kpad] first b of each group
    const int* ne4;          // [kpad] rows of class 0 (padded to 4) = offset of class 1
    const int* no4;          // [kpad] rows of class 1 (padded to 4)
    int n_segs, Kp4, Kg, nti, kpad, n_pieces, nrep, nmin, symmetric;
};

constexpr int CQ_KC = 28, CQ_STAGES = 3, CQ_WM = 4;
// WN warps along the parallels, NI 8-column fragments each: 3 x 5 (120 parallels per tile), 3 x 3 (72) or 4 x 3 (96: sixteen
// consumer warps, four per scheduler -- a warp that is busy with its epilogue leaves three, not two, to feed the DMMA pipe)
__host__ __device__ constexpr int cq_threads(int wn) { return 32 * (CQ_WM * wn + 1); }
__host__ __device__ constexpr int cq_tn(int ni, int wn) { return 8 * ni * wn; }
__host__ __device__ constexpr size_t cq_smem(int ni, int wn) {
    return (size_t)CQ_STAGES * CQ_KC * (GB_LDA + cq_tn(ni, wn) + 4) * sizeof(double) + 2 * CQ_STAGES * sizeof(uint64_t) + 16;
}

template <int NI, int CQ_WN>
__global__ void __launch_bounds__(cq_threads(CQ_WN), 1) gb_cov_quad_kernel(QuadArgs qa) {
    constexpr int CQ_CONSUMER_WARPS = CQ_WM * CQ_WN;
    constexpr int TN = cq_tn(NI, CQ_WN), LDB = TN + 4, STAGE_DOUBLES = CQ_KC * (GB_LDA + LDB);
    extern __shared__ __align__(128) unsigned char s_raw[];
    double* s_tiles = reinterpret_cast<double*>(s_raw);
    uint64_t* full = reinterpret_cast<uint64_t*>(s_raw + (size_t)CQ_STAGES * STAGE_DOUBLES * sizeof(double));
    uint64_t* empty = full + CQ_STAGES;
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(empty + CQ_STAGES);
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < CQ_STAGES; ++s) {
            gb::mbar_init(&full[s], 1);
            gb::mbar_init(&empty[s], CQ_CONSUMER_WARPS);
        }
        gb::fence_mbar_init();
    }
    if (warp == 0) gb::tmem_alloc(s_tmem, 512);
    gb::tmem_fence_before_sync();
    __syncthreads();
    gb::tmem_fence_after_sync();
    int stage = 0;
    uint32_t phase = 0;

    if (warp == CQ_CONSUMER_WARPS) {
        if (lane == 0) {
            for (int s = blockIdx.x; s < qa.n_segs; s += gridDim.x) {
                const int4 sg = qa.segs[s];
                for (int kp = sg.z; kp < sg.w; ++kp) {
                    const int e4 = qa.ne4[kp], o4 = qa.no4[kp];
                    const double* a_g = qa.St + ((size_t)sg.x * qa.Kp4 + qa.goff4[kp]) * GB_LDA;
                    const double* b_g = qa.Ut + ((size_t)kp * qa.nti + sg.y) * qa.Kg * LDB;
                    for (int c = 0; c < 2; ++c) {
                        const int klen = c ? o4 : e4, koff = c ? e4 : 0;
                        for (int k0 = 0; k0 < klen; k0 += CQ_KC) {
                            const int kc = min(CQ_KC, klen - k0);
                            gb::mbar_wait(&empty[stage], phase ^ 1u);
                            double* sA = s_tiles + (size_t)stage * STAGE_DOUBLES;
                            double* sB = sA + CQ_KC * GB_LDA;
                            const uint32_t bytes_a = (uint32_t)(kc * GB_LDA * sizeof(double));
                            const uint32_t bytes_b = (uint32_t)(kc * LDB * sizeof(double));
                            gb::mbar_arrive_expect_tx(&full[stage], bytes_a + bytes_b);
                            gb::bulk_g2s(sA, a_g + (size_t)(koff + k0) * GB_LDA, bytes_a, &full[stage]);
                            gb::bulk_g2s(sB, b_g + (size_t)(koff + k0) * LDB, bytes_b, &full[stage]);
                            if (++stage == CQ_STAGES) { stage = 0; phase ^= 1u; }
                        }
                    }
                }
            }
        }
    } else {
        const int wm = warp / CQ_WN;
        const int wn = warp % CQ_WN;
        const int g = lane >> 2, q = lane & 3;
        // this thread's tensor-memory columns: lanes 32 (warp % 4) .., the three warps of a lane quarter side by side
        const uint32_t tbase = *s_tmem + ((uint32_t)(32 * (warp & 3)) << 16) + (uint32_t)((warp >> 2) * (16 * NI));
        const size_t hstep = (size_t)qa.kpad * qa.n_pieces * 4;             // doubles per representative parallel
        for (int s = blockIdx.x; s < qa.n_segs; s += gridDim.x) {
            const int4 sg = qa.segs[s];
            const int mt = sg.x, it = sg.y;
            const int cc = wn * (8 * NI) + 2 * q;                       // first column of the thread inside the tile (even)
            const int i0 = it * TN + cc;                                // its first representative parallel
            int kslab[4];
            // runs of slabs with one group (warp-uniform): bit mi of head_mask = slab mi starts a run, of valid_mask = it
            // belongs to a group; hb[mi] = where this lane stores the piece of the run starting at slab mi (see below)
            int head_mask = 0, valid_mask = 0;
            double* hb[4];
            // ---- segment head: row-side factors -> tensor memory ----
#pragma unroll
            for (int mi = 0; mi < 4; ++mi) {
                const int row = mt * GB_TM + wm * 32 + mi * 8 + g;
                const int k = qa.rowgroup[row >> 3];
                kslab[mi] = k;
                if (k >= 0) {
                    valid_mask |= 1 << mi;
                    if (mi == 0 || k != kslab[mi > 0 ? mi - 1 : 0]) head_mask |= 1 << mi;
                }
                // lanes 0..15 store: value r = bit 3 of the lane (parallel i0 + r), row parity = bit 2
                hb[mi] = qa.Hpart + ((size_t)(i0 + ((lane >> 3) & 1)) * qa.kpad * qa.n_pieces + qa.piece_of[row >> 3]) * 4 + (g & 1);
                double u[2 * NI];
#pragma unroll
                for (int j = 0; j < 2 * NI; ++j) u[j] = 0.0;
                if (k >= 0) {
                    const int r = row - qa.goff8[k];
                    if (r < qa.gcnt[k]) {
                        const int m = k >> 1, n0 = max(m, qa.nmin);
                        const double* up = qa.Ut + (((size_t)k * qa.nti + it) * qa.Kg + cov_cls_pos(r, (n0 - m) & 1, qa.ne4[k])) * LDB + cc;
#pragma unroll
                        for (int ni = 0; ni < NI; ++ni) {
                            const double2 v = __ldg(reinterpret_cast<const double2*>(up + ni * 8));   // 16-byte aligned
                            u[2 * ni] = v.x;
                            u[2 * ni + 1] = v.y;
                        }
                    }
                }
                gb::tmem_st_n<2 * NI>(tbase + mi * (4 * NI), u);
            }
            gb::tmem_wait_st();
            for (int kp = sg.z; kp < sg.w; ++kp) {
                const int e4 = qa.ne4[kp], o4 = qa.no4[kp];
#pragma unroll 1
                for (int c = 0; c < 2; ++c) {
                    const int klen = c ? o4 : e4;
                    if (klen == 0) continue;
                    double acc[4][NI][2];
#pragma unroll
                    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
                        for (int ni = 0; ni < NI; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
                    for (int k0 = 0; k0 < klen; k0 += CQ_KC) {
                        const int kc = min(CQ_KC, klen - k0);
                        gb::mbar_wait(&full[stage], phase);
                        const double* sA = s_tiles + (size_t)stage * STAGE_DOUBLES + wm * 32 + g;
                        const double* sB = s_tiles + (size_t)stage * STAGE_DOUBLES + CQ_KC * GB_LDA + wn * (8 * NI) + g;
#pragma unroll
                        for (int kk = 0; kk < CQ_KC; kk += 4) {
                            if (kk >= kc) break;
                            double a[4], b[NI];
#pragma unroll
                            for (int mi = 0; mi < 4; ++mi) a[mi] = sA[(kk + q) * GB_LDA + mi * 8];
#pragma unroll
                            for (int ni = 0; ni < NI; ++ni) b[ni] = sB[(kk + q) * LDB + ni * 8];
#pragma unroll
                            for (int mi = 0; mi < 4; ++mi)
#pragma unroll
                                for (int ni = 0; ni < NI; ++ni) gb::dmma_884(acc[mi][ni][0], acc[mi][ni][1], a[mi], b[ni]);
                        }
                        __syncwarp();
                        if (lane == 0) gb::mbar_arrive(&empty[stage]);
                        if (++stage == CQ_STAGES) { stage = 0; phase ^= 1u; }
                    }
                    // ---- epilogue ----
#pragma unroll
                    for (int mi = 0; mi < 4; ++mi) {
                        if (kslab[mi] < 0) continue;                     // warp-uniform
                        double u[2 * NI];
                        gb::tmem_ld_n<2 * NI>(tbase + mi * (4 * NI), u);
#pragma unroll
                        for (int ni = 0; ni < NI; ++ni) {
                            acc[mi][ni][0] *= u[2 * ni];
                            acc[mi][ni][1] *= u[2 * ni + 1];
                        }
                    }
                    const size_t toff = ((size_t)kp * qa.n_pieces) * 4 + c * 2;
#pragma unroll
                    for (int head = 0; head < 4; ++head) {
                        if (!((head_mask >> head) & 1)) continue;                       // warp-uniform
                        if (qa.symmetric && kslab[head] > kp) continue;
                        double s0[NI], s1[NI];
#pragma unroll
                        for (int ni = 0; ni < NI; ++ni) {
                            s0[ni] = acc[head][ni][0];
                            s1[ni] = acc[head][ni][1];
                        }
#pragma unroll
                        for (int mi = head + 1; mi < 4; ++mi) {
                            if (((head_mask >> mi) & 1) || !((valid_mask >> mi) & 1)) break;
#pragma unroll
                            for (int ni = 0; ni < NI; ++ni) {
                                s0[ni] += acc[mi][ni][0];
                                s1[ni] += acc[mi][ni][1];
                            }
                        }
                        // rows g, g + 2, g + 4, g + 6 of the slab are the degrees of one parity.  Two shuffles per pair of
                        // values: the lanes with bit 3 clear collect the first value, those with bit 3 set the second
                        double* h = hb[head] + toff;
#pragma unroll
                        for (int ni = 0; ni < NI; ++ni) {
                            const bool second = (lane & 8) != 0;
                            double mine = second ? s1[ni] : s0[ni];
                            const double theirs = second ? s0[ni] : s1[ni];
                            mine += __shfl_xor_sync(0xffffffffu, theirs, 8);
                            mine += __shfl_xor_sync(0xffffffffu, mine, 16);
                            if (lane < 16 && i0 + ((lane >> 3) & 1) + ni * 8 < qa.nrep) h[(size_t)(ni * 8) * hstep] = mine;
                        }
                    }
                }
            }
        }
    }
    gb::tmem_fence_before_sync();
    __syncthreads();
    if (warp == 0) gb::tmem_dealloc(*s_tmem, 512);
}

// S[k][k'] / D[k][k'] = ordered sums of the pieces of group k whose rows have the class of the column class c' / the
// other class; H = scale (S + D) goes to output row out_n[r], scale (S - D) to the mirrored row out_s[r] (-1: none), in
// the A-tile layout of stage 4: Ht[((row * hmt + k / 128) * kpad + k') * 132 + k % 128] (every element is written,
// padding with zero).  Symmetric: pairs k > k' are zero, pairs k < k' count twice.  CTA = (representative r, column
// group k'), thread = row group k.
// krow != nullptr: H goes out in the AB layout of the synthesis' Fourier stage instead (rows (output row, k), spectral
// index k' at row krow[k'] of the symmetric order): the plain values S +- D, both triangles when Sigma is symmetric; the
// buffer was cleared (padding rows of the spectral groups stay zero).
__global__ void __launch_bounds__(256)
gb_cov_reduce_h(const double* __restrict__ Hpart, double* __restrict__ Ht, const int* __restrict__ pstart,
                const int* __restrict__ ne4, const int* __restrict__ no4, const int* __restrict__ out_n,
                const int* __restrict__ out_s, int kpad, int n_pieces, int hmt, int symmetric, int nmin,
                const int* __restrict__ krow, int ab_rows, int L) {
    const int r = blockIdx.x, kp = blockIdx.y;
    const double* src = Hpart + ((size_t)r * kpad + kp) * n_pieces * 4;
    const bool has0 = ne4[kp] > 0, has1 = no4[kp] > 0;
    const int on = out_n[r], os = out_s[r];
    if (krow) {
        if ((kp >> 1) >= L || kp == 1) return;                    // not a spectral row
        const int colp = krow[kp];
        for (int kg = threadIdx.x; kg < kpad; kg += blockDim.x) {
            if ((kg >> 1) >= L || kg == 1 || (symmetric && kg > kp)) continue;
            const int m = kg >> 1;
            const int po = (max(m, nmin) - m) & 1;
            double S = 0.0, D = 0.0;
            for (int pc = pstart[kg]; pc < pstart[kg + 1]; ++pc) {
                const double* v = src + (size_t)pc * 4;
                if (has0) { S += po ? v[1] : v[0]; D += po ? v[0] : v[1]; }
                if (has1) { S += po ? v[2] : v[3]; D += po ? v[3] : v[2]; }
            }
            const int colk = krow[kg];
            if (on >= 0) {
                Ht[gb_ab_offset((long long)on * kpad + kg, colp, ab_rows)] = S + D;
                if (symmetric && kg != kp) Ht[gb_ab_offset((long long)on * kpad + kp, colk, ab_rows)] = S + D;
            }
            if (os >= 0) {
                Ht[gb_ab_offset((long long)os * kpad + kg, colp, ab_rows)] = S - D;
                if (symmetric && kg != kp) Ht[gb_ab_offset((long long)os * kpad + kp, colk, ab_rows)] = S - D;
            }
        }
        return;
    }
    for (int k = threadIdx.x; k < hmt * GB_LDA; k += blockDim.x) {
        const int kt = k / GB_LDA, kk = k - kt * GB_LDA;
        const int kg = kt * GB_TM + kk;
        double S = 0.0, D = 0.0;
        if (kk < GB_TM && kg < kpad && !(symmetric && kg > kp)) {
            const int m = kg >> 1;
            const int po = (max(m, nmin) - m) & 1;                 // class of the group's first row
            for (int pc = pstart[kg]; pc < pstart[kg + 1]; ++pc) {
                const double* v = src + (size_t)pc * 4;            // [class of b][row parity]
                if (has0) {
                    const double same = po ? v[1] : v[0], cross = po ? v[0] : v[1];
                    S += same;
                    D += cross;
                }
                if (has1) {
                    const double same = po ? v[2] : v[3], cross = po ? v[3] : v[2];
                    S += same;
                    D += cross;
                }
            }
            if (symmetric && kg < kp) {
                S *= 2.0;
                D *= 2.0;
            }
        }
        if (on >= 0) Ht[(((size_t)on * hmt + kt) * kpad + kp) * GB_LDA + kk] = S + D;
        if (os >= 0) Ht[(((size_t)os * hmt + kt) * kpad + kp) * GB_LDA + kk] = S - D;
    }
}

// sum over the 8 rows of a fragment slab (lanes with equal lane % 4)
__device__ __forceinline__ double slab_sum(double v) {
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    v += __shfl_xor_sync(0xffffffffu, v, 8);
    v += __shfl_xor_sync(0xffffffffu, v, 16);
    return v;
}

// varpart[(i * 4 hmt + slot) * nlon + j] = sum_k T[k][j] * W_i[k][j] over the 32 spectral rows of one warp row of one
// row tile (slot = 4 * (row tile of the parallel) + warp row: one writer); rows of the GEMM = (i, k), all 128 rows of a
// tile belong to one parallel, so the thread sums its four rows before the slab reduction.  gb_cov_finish adds the slots.
struct LonEpilogue {
    static constexpr bool whole_tile = true;
    const double* trig;      // [kpad][nlp]
    double* var;             // [nrows][4 hmt][nlon]
    int hmt, kpad, nlp, nlon;
    __device__ __forceinline__ int prepare(long long, int, int) const { return 0; }
    __device__ __forceinline__ void tile(int, long long row_base, int col_base, double (&acc)[4][5][2]) const {
        const int mt = (int)(row_base >> 7);
        const int i = mt / hmt;
        const int kb = (mt % hmt) * 128 + (int)(row_base & 127);
#pragma unroll
        for (int ni = 0; ni < 5; ++ni) {
            const int col = col_base + ni * 8;
            double p0 = 0.0, p1 = 0.0;
#pragma unroll
            for (int mi = 0; mi < 4; ++mi) {
                const int k = kb + mi * 8;
                if (k < kpad) {
                    const double* t = trig + (size_t)k * nlp + col;
                    if (col < nlp) p0 = fma(acc[mi][ni][0], t[0], p0);
                    if (col + 1 < nlp) p1 = fma(acc[mi][ni][1], t[1], p1);
                }
            }
            p0 = slab_sum(p0);
            p1 = slab_sum(p1);
            if ((threadIdx.x & 31) < 4) {
                const int slot = (mt % hmt) * 4 + (int)((row_base & 127) >> 5);
                double* o = var + ((size_t)i * (4 * hmt) + slot) * nlon + col;
                if (col < nlon) o[0] = p0;
                if (col + 1 < nlon) o[1] = p1;
            }
        }
    }
};

// var[i][j] = sum_k T[k][j] W[(i, k)][j]: the second half of the longitude quadratic form when W = H T came from the
// synthesis' Fourier stage; four partial sums in a fixed order (deterministic), optional sqrt.
__global__ void __launch_bounds__(256)
gb_cov_lon_reduce(const double* __restrict__ W, const double* __restrict__ trig, double* __restrict__ out, int kpad, int nlp,
                  int nlon, long long n, int take_sqrt) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n) return;
    const long long i = idx / nlon;
    const int j = (int)(idx - i * nlon);
    const double* w = W + (size_t)i * kpad * nlon + j;
    const double* t = trig + j;
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    int k = 0;
    for (; k + 3 < kpad; k += 4) {
        a0 = fma(t[(size_t)k * nlp], __ldcs(w + (size_t)k * nlon), a0);
        a1 = fma(t[(size_t)(k + 1) * nlp], __ldcs(w + (size_t)(k + 1) * nlon), a1);
        a2 = fma(t[(size_t)(k + 2) * nlp], __ldcs(w + (size_t)(k + 2) * nlon), a2);
        a3 = fma(t[(size_t)(k + 3) * nlp], __ldcs(w + (size_t)(k + 3) * nlon), a3);
    }
    for (; k < kpad; ++k) a0 = fma(t[(size_t)k * nlp], __ldcs(w + (size_t)k * nlon), a0);
    const double v = (a0 + a1) + (a2 + a3);
    out[idx] = take_sqrt ? sqrt(v) : v;
}

__global__ void gb_cov_finish(const double* __restrict__ part, double* __restrict__ out, int nslots, int nlon, long long n,
                              int take_sqrt) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n) return;
    const long long i = idx / nlon;
    const int j = (int)(idx - i * nlon);
    double v = 0.0;
    for (int s = 0; s < nslots; ++s) v += part[((size_t)i * nslots + s) * nlon + j];
    out[idx] = take_sqrt ? sqrt(v) : v;
}

// Index tables of one call shape (min_degree, row block, flags): order-wise layouts, permutations, pieces, the
// representative parallels and the segment list.  Built on the host and uploaded once, kept with the plan: a repeated
// propagation launches its kernels without host work or copies.
struct CovLayout {
    int nmin = -1, row0 = -1, nrows = -1, key_flags = -1;
    int Kp8 = 0, Kp4 = 0, Kg = 8, n_atiles = 0, rows_a = 0, nti = 0, hmt = 0, n_padrows = 0, n_pieces = 0;
    int nrep = 0, nout = 0, ni = 5, n_segs = 0, folded = 0;
    int* d_all = nullptr;     // one allocation; the pointers below point into it
    int *d_perm8 = nullptr, *d_rowgroup = nullptr, *d_goff8 = nullptr, *d_gcnt = nullptr,
        *d_goff4 = nullptr, *d_ne4 = nullptr, *d_no4 = nullptr, *d_padrows = nullptr, *d_piece_of = nullptr,
        *d_pstart = nullptr, *d_first_group = nullptr, *d_rep = nullptr, *d_out_n = nullptr, *d_out_s = nullptr,
        *d_segs = nullptr;
};

constexpr int COV_KEY_MIRRORED = 1, COV_KEY_SYMMETRIC = 2, COV_KEY_NOFOLD = 4;

int build_layout(gb_plan* p, int nmin, int row0, int nrows, int key_flags, CovLayout** out) {
    CovLayout* c = static_cast<CovLayout*>(p->cov_layout);
    if (c && c->nmin == nmin && c->row0 == row0 && c->nrows == nrows && c->key_flags == key_flags) {
        *out = c;
        return GB_OK;
    }
    gb_cov_layout_free(p);
    c = new CovLayout();
    const int L = p->L, kpad = p->kpad, nlat = p->nlat;
    const bool mirrored = key_flags & COV_KEY_MIRRORED, symmetric = key_flags & COV_KEY_SYMMETRIC;
    const bool foldable = p->fold_ns && !(key_flags & COV_KEY_NOFOLD);
    // ---- output rows and representative parallels ----
    std::vector<int> out_par;                       // parallel of every output row
    for (int il = 0; il < nrows; ++il) out_par.push_back(row0 + il);
    if (mirrored)
        for (int il = 0; il < nrows; ++il) out_par.push_back(nlat - row0 - nrows + il);
    const int nout = (int)out_par.size();
    std::vector<int> rep, out_n, out_s, taken(nout, 0);
    {
        std::vector<int> row_of(nlat, -1);          // first output row of a parallel
        for (int o = nout - 1; o >= 0; --o) row_of[out_par[o]] = o;
        for (int o = 0; o < nout; ++o) {
            if (taken[o]) continue;
            const int i = out_par[o], im = nlat - 1 - i;
            taken[o] = 1;
            int partner = -1;
            // a parallel of the northern hemisphere outside the polar cap shares its factors with its mirror image
            if (foldable && i < im && i >= p->fold_cap && row_of[im] >= 0 && !taken[row_of[im]]) partner = row_of[im];
            if (partner >= 0) taken[partner] = 1;
            rep.push_back(i);
            out_n.push_back(o);
            out_s.push_back(partner);
            if (partner >= 0) c->folded = 1;
        }
    }
    const int nrep = (int)rep.size();
    // column tile of the quadratic form: 24 NI representatives, the NI with the least padding (ties: the wider tile)
    int ni = 5;
    {
        long long best = -1;
        for (int cand = 5; cand >= 3; --cand) {
            const long long padded = (long long)((nrep + 24 * cand - 1) / (24 * cand)) * 24 * cand;
            if (best < 0 || padded < best) { best = padded; ni = cand; }
        }
    }
    const int tn = 24 * ni;
    const int nti = (nrep + tn - 1) / tn;
    // ---- order-wise layouts: group k = 2m + cs holds degrees n0(m)..nmax; columns b in parity classes ----
    std::vector<int> gcnt(kpad, 0), goff8(kpad, 0), goff4(kpad, 0), ne4(kpad, 0), no4(kpad, 0);
    int Kp8 = 0, Kp4 = 0, Kg = 8;   // Kg: rows per U tile
    for (int k = 0; k < kpad; ++k) {
        const int m = k >> 1, cs = k & 1;
        int cnt = 0;
        if (m < L && !(m == 0 && cs == 1)) cnt = L - (m > nmin ? m : nmin);
        const int n0 = (m > nmin ? m : nmin), po = (n0 - m) & 1;
        const int ne = po ? cnt / 2 : (cnt + 1) / 2, no = cnt - ne;          // class 0: rows with (r + po) even
        gcnt[k] = cnt;
        goff8[k] = Kp8;
        goff4[k] = Kp4;
        ne4[k] = (ne + 3) / 4 * 4;
        no4[k] = (no + 3) / 4 * 4;
        Kp8 += (cnt + 7) / 8 * 8;
        Kp4 += ne4[k] + no4[k];
        if (ne4[k] + no4[k] > Kg) Kg = ne4[k] + no4[k];
    }
    const int n_atiles = (Kp8 + GB_TM - 1) / GB_TM;
    const int rows_a = n_atiles * GB_TM;
    std::vector<int> perm8(rows_a, -1), perm4(Kp4 > 0 ? Kp4 : 1, -1), rowgroup(rows_a / 8, -1);
    for (int k = 0; k < kpad; ++k) {
        const int m = k >> 1, cs = k & 1;
        const int n0 = (m > nmin ? m : nmin), po = (n0 - m) & 1;
        for (int r = 0; r < gcnt[k]; ++r) {
            const int n = n0 + r;
            const long long idx = (long long)n * n + (m == 0 ? 0 : 2 * m - 1 + cs) - (long long)nmin * nmin;
            perm8[goff8[k] + r] = (int)idx;
            perm4[goff4[k] + cov_cls_pos(r, po, ne4[k])] = (int)idx;
        }
        for (int r = 0; r < (gcnt[k] + 7) / 8; ++r) rowgroup[goff8[k] / 8 + r] = k;
    }
    std::vector<int> padrows;
    for (int b = 0; b < Kp4; ++b)
        if (perm4[b] < 0) padrows.push_back(b);
    // first group of every row tile (symmetric Sigma: H_i is symmetric, the tile needs the column groups k' >= it only)
    std::vector<int> first_group(n_atiles, kpad);
    for (int t = 0; t < n_atiles; ++t)
        for (int sl = t * (GB_TM / 8); sl < (t + 1) * (GB_TM / 8); ++sl)
            if (rowgroup[sl] >= 0 && rowgroup[sl] < first_group[t]) first_group[t] = rowgroup[sl];
    // pieces: runs of slabs of one group inside a warp's 32 rows (4 slabs); the pieces of a group are consecutive
    std::vector<int> piece_of(rows_a / 8, -1), pstart(kpad + 1, 0);
    int n_pieces = 0;
    {
        std::vector<int> count(kpad, 0);
        for (int w = 0; w < rows_a / 32; ++w)
            for (int sl = 0; sl < 4; ++sl) {
                const int k = rowgroup[w * 4 + sl];
                if (k < 0 || (sl > 0 && rowgroup[w * 4 + sl - 1] == k)) continue;
                piece_of[w * 4 + sl] = n_pieces++;
                ++count[k];
            }
        for (int k = 0; k < kpad; ++k) pstart[k + 1] = pstart[k] + count[k];   // groups appear in increasing order of a'
    }
    // ---- segments: (row tile, parallel tile, [k0, k1)) of about equal cost; a tile costs its K rows + its epilogue ----
    std::vector<int> segs;
    {
        constexpr int EPI = 12;                    // epilogue of one (tile, class) in units of K rows
        auto cost = [&](int k) { return (ne4[k] ? ne4[k] + EPI : 0) + (no4[k] ? no4[k] + EPI : 0); };
        long long total = 0;
        for (int t = 0; t < n_atiles; ++t)
            for (int k = symmetric ? first_group[t] : 0; k < kpad; ++k) total += (long long)cost(k) * nti;
        const int sms = p->sm_count > 0 ? p->sm_count : 148;
        long long target = total / ((long long)sms * 8) + 1;
        if (target < 400) target = 400;            // a segment pays one fetch of the row factors
        // heaviest row tiles first (static round-robin over the CTAs)
        for (int t = 0; t < n_atiles; ++t)
            for (int it = 0; it < nti; ++it) {
                const int kfirst = symmetric ? first_group[t] : 0;
                if (kfirst >= kpad) continue;
                long long w = 0;
                int k0 = kfirst;
                for (int k = kfirst; k < kpad; ++k) {
                    w += cost(k);
                    if (w >= target || k == kpad - 1) {
                        if (w > 0) { segs.push_back(t); segs.push_back(it); segs.push_back(k0); segs.push_back(k + 1); }
                        k0 = k + 1;
                        w = 0;
                    }
                }
            }
    }
    c->n_segs = (int)(segs.size() / 4);
    c->nmin = nmin; c->row0 = row0; c->nrows = nrows; c->key_flags = key_flags;
    c->Kp8 = Kp8; c->Kp4 = Kp4; c->Kg = Kg; c->n_atiles = n_atiles; c->rows_a = rows_a; c->nti = nti;
    c->hmt = (kpad + GB_TM - 1) / GB_TM;
    c->n_padrows = (int)padrows.size();
    c->n_pieces = n_pieces;
    c->nrep = nrep; c->nout = nout; c->ni = ni;
    constexpr int NT = 15;
    const std::vector<int>* parts[NT] = {&perm8, &rowgroup, &goff8, &gcnt, &goff4, &ne4, &no4, &padrows, &piece_of,
                                         &pstart, &first_group, &rep, &out_n, &out_s, &segs};
    int** slots[NT] = {&c->d_perm8, &c->d_rowgroup, &c->d_goff8, &c->d_gcnt, &c->d_goff4, &c->d_ne4, &c->d_no4,
                       &c->d_padrows, &c->d_piece_of, &c->d_pstart, &c->d_first_group, &c->d_rep, &c->d_out_n, &c->d_out_s,
                       &c->d_segs};
    std::vector<int> all;
    size_t offs[NT];
    for (int i = 0; i < NT; ++i) {
        offs[i] = all.size();
        all.insert(all.end(), parts[i]->begin(), parts[i]->end());
        all.resize((all.size() + 3) / 4 * 4);                   // keep every table 16-byte aligned
    }
    if (cudaMalloc(reinterpret_cast<void**>(&c->d_all), (all.size() ? all.size() : 4) * sizeof(int)) != cudaSuccess) {
        delete c;
        return gb_set_error(GB_ERR_CUDA, "gb_covariance_propagation: cannot allocate the index tables");
    }
    if (cudaMemcpy(c->d_all, all.data(), all.size() * sizeof(int), cudaMemcpyHostToDevice) != cudaSuccess) {
        cudaFree(c->d_all);
        delete c;
        return gb_set_error(GB_ERR_CUDA, "gb_covariance_propagation: cannot upload the index tables");
    }
    for (int i = 0; i < NT; ++i) *slots[i] = c->d_all + offs[i];
    p->cov_layout = c;
    *out = c;
    return GB_OK;
}

template <int NI, int WN>
int launch_quad(const QuadArgs& qa, int sm_count, cudaStream_t st) {
    if (qa.n_segs == 0) return GB_OK;
    const int grid = qa.n_segs < sm_count ? qa.n_segs : sm_count;
    constexpr size_t SMEM = cq_smem(NI, WN);
    GB_CUDA(cudaFuncSetAttribute(gb_cov_quad_kernel<NI, WN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
    gb_cov_quad_kernel<NI, WN><<<grid, cq_threads(WN), SMEM, st>>>(qa);
    GB_LAUNCH_CHECK();
    return GB_OK;
}

}  // namespace

void gb_cov_layout_free(gb_plan* p) {
    CovLayout* c = static_cast<CovLayout*>(p->cov_layout);
    if (!c) return;
    cudaFree(c->d_all);
    delete c;
    p->cov_layout = nullptr;
}

extern "C" int gb_covariance_propagation(gb_plan* plan, const double* d_sigma, int nmin, int row0, int nrows,
                                         double* d_out, int flags, void* stream) {
    return gb_covariance_propagation_filtered(plan, d_sigma, nmin, row0, nrows, d_out, flags, nullptr, nullptr, 0, nullptr,
                                              stream);
}

extern "C" int gb_covariance_propagation_filtered(gb_plan* plan, const double* d_sigma, int nmin, int row0, int nrows,
                                                  double* d_out, int flags, const double* d_blocks,
                                                  const int64_t* block_offsets, int nf, const double* d_wn, void* stream) {
    const int take_sqrt = flags & GB_COV_SQRT;
    const int symmetric = (flags & GB_COV_SYMMETRIC) ? 1 : 0;
    const int mirrored = (flags & GB_COV_MIRRORED) ? 1 : 0;
    GB_REQUIRE(plan != nullptr, "gb_covariance_propagation: plan is NULL");
    gb_plan* p = plan;
    GB_REQUIRE(nmin >= 0 && nmin <= p->nmax, "gb_covariance_propagation: min_degree=%d outside [0, %d]", nmin, p->nmax);
    GB_REQUIRE(row0 >= 0 && nrows >= 0 && row0 + nrows <= p->nlat,
               "gb_covariance_propagation: parallels [%d, %d) outside the grid (%d parallels)", row0, row0 + nrows, p->nlat);
    GB_REQUIRE(!mirrored || 2 * (row0 + nrows) <= p->nlat,
               "gb_covariance_propagation: a mirrored block must lie north of the equator (parallels [%d, %d) of %d)", row0,
               row0 + nrows, p->nlat);
    if (nrows == 0) return GB_OK;
    GB_REQUIRE(d_sigma && d_out, "gb_covariance_propagation: NULL device pointer");
    GB_REQUIRE(!d_blocks || (block_offsets && nf >= p->nmax),
               "gb_covariance_propagation_filtered: the order-wise filter (degree %d) does not reach degree %d", nf, p->nmax);
    GB_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    {
        int rca = gb_plan_acquire(p, st);   // the cached index tables are rebuilt when the shape changes
        if (rca) return rca;
    }
    gb_scratch scratch(st);           // frees every temporary of this call on all return paths
    const int L = p->L, kpad = p->kpad;
    const long long K = (long long)L * L - (long long)nmin * nmin;

    CovLayout* lay = nullptr;
    {
        // an order-wise filter mixes the parity classes of a group: no fold then (GB_COV_NO_FOLD=1: never)
        const bool nofold = d_blocks != nullptr || gb_env_flag("GB_COV_NO_FOLD");
        const int key = (mirrored ? COV_KEY_MIRRORED : 0) | (symmetric ? COV_KEY_SYMMETRIC : 0) | (nofold ? COV_KEY_NOFOLD : 0);
        int rc0 = build_layout(p, nmin, row0, nrows, key, &lay);
        if (rc0) return rc0;
    }
    const int Kp4 = lay->Kp4, Kg = lay->Kg, n_atiles = lay->n_atiles, rows_a = lay->rows_a, nti = lay->nti, hmt = lay->hmt;
    const int nrep = lay->nrep, nout = lay->nout, tn = 24 * lay->ni, ldb = tn + 4;
    const int n_ct = kpad * nti;
    GB_REQUIRE(Kp4 <= 65535, "gb_covariance_propagation: degree %d is too large for this path", p->nmax);
    GB_REQUIRE((long long)n_ct * Kg * ldb < (1LL << 31),
               "gb_covariance_propagation: %d parallels at degree %d exceed the 32-bit tile index; pass row blocks", nrows, p->nmax);
    const int n_pieces = lay->n_pieces, nslots = 4 * hmt;
    double *d_st = nullptr, *d_ut = nullptr, *d_ht = nullptr, *d_hpart = nullptr, *d_vpart = nullptr;
    int rc = GB_OK;
    const size_t st_elems = (size_t)n_atiles * Kp4 * GB_LDA;
    const size_t ut_elems = (size_t)n_ct * Kg * ldb;
    const size_t ht_elems = (size_t)nout * hmt * kpad * GB_LDA;
    const size_t hp_elems = (size_t)nrep * kpad * n_pieces * 4;
    const size_t vp_elems = (size_t)nout * nslots * p->nlon;
    GB_CUDA(scratch.alloc(&d_st, st_elems));
    GB_CUDA(scratch.alloc(&d_ut, ut_elems));
    GB_CUDA(scratch.alloc(&d_hpart, hp_elems));
    GB_CUDA(cudaMemsetAsync(d_ut, 0, ut_elems * sizeof(double), st));
    {
        dim3 grid((nrep + 31) / 32, L);      // thread = (parallel, order): a serial recursion each, so many small CTAs
        gb_cov_legendre<<<grid, 32, 0, st>>>(d_ut, p->d_ct, p->d_kn, p->d_pmm, p->d_ra, p->d_rb, p->d_rc, L, nmin,
                                              lay->d_rep, nrep, nti, Kg, tn, ldb, d_wn, lay->d_ne4);
        GB_LAUNCH_CHECK();
    }
    long long* d_boff = nullptr;
    if (d_blocks) {
        // U <- F' U group by group (see gb_cov_apply_blocks); the contractions below then run on A F
        const int nblocks = 2 * nf + 1;
        GB_CUDA(scratch.alloc(&d_boff, (size_t)nblocks + 1));
        GB_CUDA(cudaMemcpyAsync(d_boff, block_offsets, (nblocks + 1) * sizeof(long long), cudaMemcpyHostToDevice, st));
        double* d_ut2 = nullptr;
        GB_CUDA(scratch.alloc(&d_ut2, ut_elems));
        GB_CUDA(cudaMemsetAsync(d_ut2, 0, ut_elems * sizeof(double), st));
        dim3 grid(kpad, nti, (Kg + CF_B - 1) / CF_B);
        gb_cov_apply_blocks<<<grid, 128, 0, st>>>(d_ut, d_ut2, d_blocks, d_boff, nf, L, nmin, nti, Kg, ldb, lay->d_ne4);
        GB_LAUNCH_CHECK();
        d_ut = d_ut2;
    }
    // the padding rows of the classes are the only part of St the permutation does not write
    if (lay->n_padrows > 0) {
        gb_cov_zero_rows<<<dim3(n_atiles, (lay->n_padrows + 15) / 16), 128, 0, st>>>(d_st, lay->d_padrows, lay->n_padrows, Kp4);
        GB_LAUNCH_CHECK();
    }
    const dim3 pgrid(rows_a / CP_ROWS, L - nmin, (2 * p->nmax + 1 + CP_COLS - 1) / CP_COLS);
    gb_cov_permute_degree<<<pgrid, 256, 0, st>>>(d_sigma, d_st, lay->d_perm8, lay->d_goff4, lay->d_ne4, Kp4, K, nmin,
                                                 symmetric ? lay->d_first_group : nullptr);
    GB_LAUNCH_CHECK();
    {
        QuadArgs qa;
        qa.St = d_st; qa.Ut = d_ut; qa.Hpart = d_hpart;
        qa.segs = reinterpret_cast<const int4*>(lay->d_segs);
        qa.rowgroup = lay->d_rowgroup; qa.goff8 = lay->d_goff8; qa.gcnt = lay->d_gcnt; qa.piece_of = lay->d_piece_of;
        qa.goff4 = lay->d_goff4; qa.ne4 = lay->d_ne4; qa.no4 = lay->d_no4;
        qa.n_segs = lay->n_segs; qa.Kp4 = Kp4; qa.Kg = Kg; qa.nti = nti; qa.kpad = kpad; qa.n_pieces = n_pieces;
        qa.nrep = nrep; qa.nmin = nmin; qa.symmetric = symmetric;
        rc = lay->ni == 5 ? launch_quad<5, 3>(qa, p->sm_count, st) : lay->ni == 4 ? launch_quad<3, 4>(qa, p->sm_count, st)
                                                                                  : launch_quad<3, 3>(qa, p->sm_count, st);
        if (rc) return rc;
    }
    // longitude quadratic form.  Four-fold symmetric meridians (every grid the reference builds): W = H T is exactly the
    // Fourier stage of the synthesis on the rows (parallel, k) -- one quarter of the multiply-adds of a plain GEMM, no padded
    // spectral rows -- followed by a streaming reduction over k.  Otherwise: the GEMM with the fused reduction below.
    if (p->sym) {
        const long long Mrows = (long long)nout * kpad;
        const size_t h2_elems = (size_t)((Mrows + GB_TM - 1) / GB_TM) * p->ab_rows * GB_LDA;
        const size_t w_elems = (size_t)Mrows * p->nlon;
        double *d_h2 = nullptr, *d_w = nullptr;
        GB_CUDA(scratch.alloc(&d_h2, h2_elems));
        GB_CUDA(scratch.alloc(&d_w, w_elems));
        GB_CUDA(cudaMemsetAsync(d_h2, 0, h2_elems * sizeof(double), st));
        gb_cov_reduce_h<<<dim3(nrep, kpad), 256, 0, st>>>(d_hpart, d_h2, lay->d_pstart, lay->d_ne4, lay->d_no4, lay->d_out_n,
                                                          lay->d_out_s, kpad, n_pieces, hmt, symmetric, nmin, gb_stage2_krow(p),
                                                          p->ab_rows, L);
        GB_LAUNCH_CHECK();
        if ((rc = gb_launch_stage2_sym(p, d_h2, Mrows, d_w, st, false))) return rc;
        const long long n = (long long)nout * p->nlon;
        gb_cov_lon_reduce<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_w, p->d_trig, d_out, kpad, p->nlp, p->nlon, n,
                                                                      take_sqrt ? 1 : 0);
        GB_LAUNCH_CHECK();
        return GB_OK;
    }
    GB_CUDA(scratch.alloc(&d_ht, ht_elems));
    GB_CUDA(scratch.alloc(&d_vpart, vp_elems));
    {
        dim3 grid(nrep, kpad);
        gb_cov_reduce_h<<<grid, 256, 0, st>>>(d_hpart, d_ht, lay->d_pstart, lay->d_ne4, lay->d_no4, lay->d_out_n, lay->d_out_s,
                                              kpad, n_pieces, hmt, symmetric, nmin, nullptr, 0, L);
        GB_LAUNCH_CHECK();
    }
    {
        gbgemm::Shape sh;
        sh.A_t = d_ht;
        sh.a_rows = kpad;
        sh.a_koff_mul = 0;
        sh.tiles_per_group = 1;
        sh.B_t = p->d_trig_t;
        sh.b_rows = kpad;
        sh.klen = kpad;
        sh.n_mtiles = nout * hmt;
        sh.n_ntiles = p->n_ntiles;
        if (symmetric) {            // H is upper triangular then: spectral rows k >= 128 j only meet columns k' >= 128 j
            sh.mt_kstart_mod = hmt;
            sh.mt_kstart_mul = GB_TM;
        }
        LonEpilogue epi{p->d_trig, d_vpart, hmt, kpad, p->nlp, p->nlon};
        if ((rc = gbgemm::launch(sh, epi, p->sm_count, st))) return rc;
    }
    {
        const long long n = (long long)nout * p->nlon;
        gb_cov_finish<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_vpart, d_out, nslots, p->nlon, n, take_sqrt ? 1 : 0);
        GB_LAUNCH_CHECK();
    }
    return GB_OK;
}
