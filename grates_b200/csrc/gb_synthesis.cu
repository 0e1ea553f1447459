// Spherical-harmonic synthesis on B200 (sm_100a), epoch-batched.
//
// Replaces the hot loop of PotentialCoefficients.to_grid (reference gravityfield.py:358-368):
//
//   V[e,i,j] = sum_m ( A[e,i,m] cos(m lon_j) + B[e,i,m] sin(m lon_j) )                (stage 2)
//   A[e,i,m] = sum_n kn[i,n] P_nm(theta_i) C_nm^e ,  B likewise with S_nm^e           (stage 1)
//
// HBM layout
//   anm   [E][L][L]          packed coefficients as the reference stores them
//   X     [order][column tile][degree row][tn+4]  X_m[n-m][cs*E+e], degree rows in the Legendre table's order
//                            (tb_fold_row, gb_pack.cu); order-wise X_m[n-m][cs*E+e] for the FMA cross-check
//   AB    [row tile][k][132]  spectral intermediate, tiled by 128 grid rows (e*nlat + i), see gb_common.cuh;
//                            row order k = 2m+cs, or [CE|CO|SE|SO] groups for the symmetric stage 2
//   trig  [col tile][k][124]  row 2m = cos(m lon_j), row 2m+1 = sin(m lon_j) (first quadrant only when symmetric)
//   V     [E][nlat][nlon]    output
//
// Kernels
//   gb_pack_rows_kernel / gb_pack_kernel   transpose anm into X (gb_pack.cu; HBM-bound)
//   gb_stage1            per (order pair, latitude tile, column tile): contracts kn[i,n] P_nm(theta_i) against all
//                        epochs on the FP64 tensor cores (DMMA.8x8x4) and writes AB; the Legendre values (unfused IEEE
//                        ops -> bit-identical to utilities.py:37-54) come from the plan's table (gb_ptab_kernel) or
//                        from the recursion run inside the kernel
//   gb_fourier_stage2_oct / gb_fourier_stage2_sym   stage 2 on meridians with eight- / four-fold symmetry
//   gbgemm::kernel       stage 2 on other meridians: persistent FP64 tensor-core GEMM  V = AB^T * trig (gb_gemm.cuh)
// All stage-1 and stage-2 kernels stage their operands with the TMA unit (cp.async.bulk) through mbarrier rings fed
// by a producer lane.
#include <type_traits>
#include <vector>
#include "gb_common.cuh"
#include "gb_gemm.cuh"

#ifdef GB_TRACE
// development aid (-DGB_TRACE): in-kernel timeline of the stage-1 / stage-2 kernels, read back with gb_debug_trace
__device__ unsigned long long gb_trace_buf[2][160][24][2];      // [kernel][CTA][slot][globaltimer ns, clock64]
#define GB_TRACE_MARK(k, slot)                                                                      \
    do {                                                                                            \
        unsigned long long gt_;                                                                     \
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt_));                                      \
        if (blockIdx.x < 160 && (slot) < 24) {                                                      \
            gb_trace_buf[k][blockIdx.x][slot][0] = gt_;                                             \
            gb_trace_buf[k][blockIdx.x][slot][1] = (unsigned long long)clock64();                   \
        }                                                                                           \
    } while (0)
#else
#define GB_TRACE_MARK(k, slot) ((void)0)
#endif

namespace {

using gb::legendre_column;   // f(n, P_nm), n = m..L-1 (gb_common.cuh)

constexpr int S1_TI = 32;  // latitudes per CTA

__global__ void __launch_bounds__(256)
gb_legendre_stage1_simple(const double* __restrict__ X, double* __restrict__ AB, const double* __restrict__ ct,
                   const double* __restrict__ kn, const double* __restrict__ pmm, const double* __restrict__ ra,
                   const double* __restrict__ rb, const double* __restrict__ rc, const int* __restrict__ krow, int L,
                   int nlat, int E, int ab_rows) {
    extern __shared__ double s_pk[];  // [Kn][S1_TI]
    const int m = blockIdx.y;
    const int i0 = blockIdx.x * S1_TI;
    const int Kn = L - m;
    const int tid = threadIdx.x;
    if (tid < S1_TI) {
        const int i = i0 + tid;
        if (i < nlat) {
            const double* kn_i = kn + (size_t)i * L + m;
            legendre_column(m, L, ct[i], pmm[(size_t)i * L + m], ra, rb, rc,
                            [&](int n, double p) { s_pk[(n - m) * S1_TI + tid] = __dmul_rn(p, kn_i[n - m]); });
        } else {
            for (int nn = 0; nn < Kn; ++nn) s_pk[nn * S1_TI + tid] = 0.0;
        }
    }
    __syncthreads();

    const int cols = 2 * E;
    const int lane = tid & 31;
    const int ig = tid >> 5;  // 8 groups of 4 latitudes
    const long long xo = (long long)cols * ((long long)m * L - (long long)m * (m - 1) / 2);
    const double* Xm = X + xo;
    for (int col0 = 0; col0 < cols; col0 += 32) {
        const int col = col0 + lane;
        if (col >= cols) continue;
        double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
        const double* xp = Xm + col;
        const double* pk = s_pk + ig * 4;
#pragma unroll 4
        for (int nn = 0; nn < Kn; ++nn) {
            const double x = __ldg(xp + (size_t)nn * cols);
            const double2 p01 = *reinterpret_cast<const double2*>(pk + nn * S1_TI);
            const double2 p23 = *reinterpret_cast<const double2*>(pk + nn * S1_TI + 2);
            a0 = fma(p01.x, x, a0);
            a1 = fma(p01.y, x, a1);
            a2 = fma(p23.x, x, a2);
            a3 = fma(p23.y, x, a3);
        }
        const int cs = col >= E, e = col - cs * E;
        const int i = i0 + ig * 4;
        const int k = krow[2 * m + cs];
        const long long row = (long long)e * nlat + i;
        if (i + 0 < nlat) AB[gb_ab_offset(row + 0, k, ab_rows)] = a0;
        if (i + 1 < nlat) AB[gb_ab_offset(row + 1, k, ab_rows)] = a1;
        if (i + 2 < nlat) AB[gb_ab_offset(row + 2, k, ab_rows)] = a2;
        if (i + 3 < nlat) AB[gb_ab_offset(row + 3, k, ab_rows)] = a3;
    }
}


// ---------------------------------------------------------------------------------------------
// stage 1 on the FP64 tensor cores, persistent.  Work item = (order pair (p, nmax-p), 32 or 64 parallels, TN = 8 MI NWN
// columns (e, cos|sin)); every item carries L+1 degrees, so items cost the same:
//   D[i, col] = sum_n Pk[i, n] X_m[n, col],  Pk[i, n] = kn[i,n] * P_nm(theta_i)
// A ring stage holds 16 degrees of both operands: Pk [16][lda] and X_m [16][TN + 4].  A copy lane fills the X half with
// one bulk copy from the tiled X; where the Pk half comes from is the Source:
//   Table      the plan's Legendre table (the default).  Pk does not depend on the epoch, so the plan holds it -- written
//              once by gb_ptab_kernel with the same bit-exact recursion -- in exactly the tile layout a stage needs, and
//              the copy lane fetches it with one more bulk copy.  No FP64 instruction competes with the DMMA stream for
//              the pipe (a recursion warp shares its scheduler with three DMMA-issuing warps: 300 cycles per degree,
//              DMMA pipe 45 % active at config 2).
//   Recursion  Legendre warps (lane = column of the tile, recursion state in registers) run the recursion on the fly and
//              write the stage: the fallback when the table is over its memory budget or cannot be allocated.
// Both sources lay a stage out alike: column li holds parallel s1_parallel(li), degree offset nn sits in row
// tb_fold_row(nn) ([even n-m | odd n-m] per 8 rows, so both parity classes of a folded chunk read consecutive
// shared-memory rows; pitch 36 = 4 mod 16: conflict-free fragments).  The consumers and epilogues are therefore the same,
// and so are the results, bit for bit.
// ---------------------------------------------------------------------------------------------
enum class S1Source { Table, Recursion };
__host__ __device__ constexpr int s1_lda(bool fold) { return fold ? 36 : 68; }
// one Legendre warp per 32 parallels of an item
__host__ __device__ constexpr int s1_legendre_warps(bool fold, S1Source src) {
    return src == S1Source::Recursion ? (fold ? 1 : 2) : 0;
}
// Narrow column tiles run several CTAs per SM.  The recursion keeps at most two (an item there is paced by the Legendre
// warps' dependent recursion, so resident items add throughput, but a third CTA would leave its warps too few registers).
__host__ __device__ constexpr int s1_ctas_per_sm(int nwn, bool fold, S1Source src) {
    return src == S1Source::Recursion ? (nwn <= 3 ? 2 : 1) : nwn <= 2 ? (fold ? 3 : 2) : nwn == 3 ? 2 : 1;
}
__host__ __device__ constexpr int s1_threads(int nwn, bool fold, S1Source src) {
    return 32 * (2 * nwn + 1 + s1_legendre_warps(fold, src));    // consumers + copy warp + Legendre warps
}
__host__ __device__ constexpr size_t s1_stage_bytes(int nwn, bool fold) {
    return (size_t)GB_T1_KC * (s1_lda(fold) + 40 * nwn + 4) * sizeof(double);
}
// as many ring stages (at most 6) as the CTA's share of the 227 KB of shared memory holds
__host__ __device__ constexpr int s1_stages(int nwn, bool fold, S1Source src) {
    const size_t budget = (232448 - 1024 * s1_ctas_per_sm(nwn, fold, src)) / s1_ctas_per_sm(nwn, fold, src) - 128;
    const int s = (int)(budget / s1_stage_bytes(nwn, fold));
    return s > 6 ? 6 : s;
}
__host__ __device__ constexpr size_t s1_smem(int nwn, bool fold, S1Source src) {
    return (size_t)s1_stages(nwn, fold, src) * s1_stage_bytes(nwn, fold) + 2 * s1_stages(nwn, fold, src) * sizeof(uint64_t);
}
// row of degree offset nn inside a Legendre table / ring stage / tiled X: even offsets first
__host__ __device__ __forceinline__ int tb_fold_row(int nn) { return (nn & ~7) + ((nn & 1) << 2) + ((nn & 7) >> 1); }
__host__ __device__ __forceinline__ int tb_fold_degree(int row) {
    const int r = row & 7;
    return (row & ~7) + (r < 4 ? 2 * r : 2 * (r - 4) + 1);
}
// Parallel of column li of a stage-1 tile whose first (northern) parallel is i0, by tile kind (gb_common.cuh):
// 0 folded -- inside every 16-column slab of a warp the columns are interleaved so that a lane's two DMMA fragments (tile
//   columns 2q, 2q+1 and 8+2q, 9+2q) are FOUR CONSECUTIVE parallels 4q .. 4q+3: one 32-byte store per lane (parallels
//   beyond the equator keep their own values: a lane's parallels may straddle it);
// 1 polar cap -- 32 northern parallels, then their 32 mirror images (i_south = nlat - 64 - i0 onwards);
// 2 plain -- 64 consecutive parallels.
__host__ __device__ __forceinline__ int s1_parallel(int kind, int i0, int li, int nlat) {
    if (kind == 0) {
        const int cc = li & 15;
        return i0 + (li & 16) + 4 * ((cc & 7) >> 1) + 2 * (cc >> 3) + (cc & 1);
    }
    return (kind == 1 && li >= 32) ? nlat - 64 - i0 + li : i0 + li;
}

struct S1Args {
    const int* roff;        // [L + 1] first row of every order in the table and in the tiled X
    const int* krow;
    const double* tab;      // Table: [lat tile][rtot][lda]
    long long tile_stride;  // Table: rtot * lda
    // Recursion: the plan's transposed, zero-padded recursion tables (gb_common.cuh)
    const double* ct_pad;   // [nlat_pad]
    const double* kn_t;     // [L + 16][nlat_pad]
    const double* pmm_t;    // [L][nlat_pad]
    const double* rec_a;    // [L][lpad]   rec_a[m][n - m]
    const double* rec_b;    // [L][lpad]
    int nlat_pad, lpad;
};

// PAIRS: nlat even, rows (e, i), (e, i+1) with i even are 16-byte aligned in AB.
// FOLD (declared shortcut, grids that are symmetric about the equator): P_nm(pi - theta) = (-1)^(n-m) P_nm(theta), so an
// item covers 32 northern parallels AND their mirror images: the degrees of a chunk are contracted in two parity
// classes, north = even + odd, south = even - odd.  Half the recursion steps and half the DMMAs for the same output.
// MI: 8-column fragments per consumer warp (5: 40 columns; 4: shards of at most 32 epochs, whose 64 columns then carry
// no padding fragment)
template <S1Source SRC, bool PAIRS, int NWN, bool FOLD, int MI>
__global__ void __launch_bounds__(s1_threads(NWN, FOLD, SRC), s1_ctas_per_sm(NWN, FOLD, SRC))
gb_stage1(const double* __restrict__ X, double* __restrict__ AB, S1Args tb, int L, int nlat, int E, int ab_rows,
          int n_lattiles, int n_coltiles, int n_items, int polar) {
    // polar: FOLD -- number of leading 32-parallel tiles left to the unfolded launch; !FOLD -- nonzero selects the
    // "polar cap" tiling (tile t = northern parallels [32t, 32t+32) and their mirror images), see launch_synthesis
    constexpr bool REC = SRC == S1Source::Recursion;
    constexpr int KC = GB_T1_KC, STAGES = s1_stages(NWN, FOLD, SRC);
    static_assert(STAGES >= 2, "the ring needs at least two stages");
    constexpr int TN = 8 * MI * NWN, LDA = s1_lda(FOLD), LDB = TN + 4, CONSUMER_WARPS = 2 * NWN;
    constexpr int STAGE_DOUBLES = KC * (LDA + LDB);
    extern __shared__ __align__(128) unsigned char s_raw[];
    double* s_tiles = reinterpret_cast<double*>(s_raw);
    uint64_t* full = reinterpret_cast<uint64_t*>(s_raw + (size_t)STAGES * STAGE_DOUBLES * sizeof(double));
    uint64_t* empty = full + STAGES;
    const int cols = 2 * E;
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        GB_TRACE_MARK(0, 0);
        for (int s = 0; s < STAGES; ++s) {
            gb::mbar_init(&full[s], 1 + s1_legendre_warps(FOLD, SRC));    // copy lane (+tx bytes), Legendre warps
            gb::mbar_init(&empty[s], CONSUMER_WARPS);
        }
        gb::fence_mbar_init();
    }
    __syncthreads();
    gb::griddep_launch_dependents();
    // griddepcontrol.wait (X comes from the pack kernel, AB is still being read by the previous call) is executed by the
    // copy lane alone: the Legendre table and the recursion tables are plan constants, so the table halves of the first
    // ring stages are already in flight (a cold DRAM round trip after an L2 flush) when the wait returns, and the
    // Legendre warps start their recursion at once; the consumers touch global memory only after they have seen chunks
    // of X, which the copy lane requests after the wait.
    const int tiles_per_pair = n_lattiles * n_coltiles;
    int n_pre = 0;                      // chunks whose table half (and byte count) went out before the wait
    if (warp == CONSUMER_WARPS && lane == 0) {
        for (int item = blockIdx.x; !REC && item < n_items && n_pre < STAGES; item += gridDim.x) {
            const int m_first = item / tiles_per_pair;
            const int lt = (item - m_first * tiles_per_pair) / n_coltiles;
            const int m_second = L - 1 - m_first;
            const int npass = (m_second == m_first) ? 1 : 2;
            const double* tab_t = tb.tab + (size_t)lt * tb.tile_stride;
            for (int pass = 0; pass < npass && n_pre < STAGES; ++pass) {
                const int m = pass ? m_second : m_first;
                const int r0 = tb.roff[m], kn_pad = tb.roff[m + 1] - r0;
                for (int r = 0; r < kn_pad && n_pre < STAGES; r += KC, ++n_pre) {
                    const int rows = min(KC, kn_pad - r);
                    gb::mbar_arrive_expect_tx(&full[n_pre], (uint32_t)(rows * (LDB + LDA) * sizeof(double)));
                    gb::bulk_g2s(s_tiles + (size_t)n_pre * STAGE_DOUBLES, tab_t + ((size_t)r0 + r) * LDA,
                                 (uint32_t)(rows * LDA * sizeof(double)), &full[n_pre]);
                }
            }
        }
        gb::griddep_wait();
        GB_TRACE_MARK(0, 1);
    }

    int stage = 0;
    uint32_t phase = 0;
    int chunk_idx = 0;                  // copy lane: chunks handed to the ring so far
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        const int m_first = item / tiles_per_pair;
        const int rem = item - m_first * tiles_per_pair;
        const int lt = rem / n_coltiles;
        const int i0 = FOLD ? (polar + lt) * 32 : lt * (polar ? 32 : GB_T1_TM);
        const int i_south = nlat - 64 - i0;
        const int c0 = (rem % n_coltiles) * TN;
        const int m_second = L - 1 - m_first;
        const int npass = (m_second == m_first) ? 1 : 2;
        const int width = min(TN, cols - c0);

        if (warp == CONSUMER_WARPS) {
            // ===== copy warp (one elected lane): one bulk copy for the chunk of X_m (and one for the table chunk) =====
            if (lane == 0) {
                const double* tab_t = tb.tab + (size_t)lt * tb.tile_stride;
                const int ct = rem % n_coltiles;
                for (int pass = 0; pass < npass; ++pass) {
                    const int m = pass ? m_second : m_first;
                    const int r0 = tb.roff[m], kn_pad = tb.roff[m + 1] - r0;       // rows of the order, padded to 8
                    const double* tab_m = tab_t + (size_t)r0 * LDA;
                    const double* x_m = X + ((size_t)r0 * n_coltiles + (size_t)ct * kn_pad) * LDB;
                    for (int r = 0; r < kn_pad; r += KC) {
                        const int rows = min(KC, kn_pad - r);
                        double* sA = s_tiles + (size_t)stage * STAGE_DOUBLES;
                        if (REC || chunk_idx++ >= n_pre) {
                            gb::mbar_wait(&empty[stage], phase ^ 1u);
                            gb::mbar_arrive_expect_tx(&full[stage], (uint32_t)(rows * (REC ? LDB : LDB + LDA) * sizeof(double)));
                            if (!REC)
                                gb::bulk_g2s(sA, tab_m + (size_t)r * LDA, (uint32_t)(rows * LDA * sizeof(double)), &full[stage]);
                        }
                        gb::bulk_g2s(sA + KC * LDA, x_m + (size_t)r * LDB, (uint32_t)(rows * LDB * sizeof(double)), &full[stage]);
                        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
                    }
                }
            }
        } else if (REC && warp > CONSUMER_WARPS) {
            // ===== Legendre warps: lane = column li of the tile, recursion state lives in registers =====
            const int li = (warp - CONSUMER_WARPS - 1) * 32 + lane;
            const int i = s1_parallel(FOLD ? 0 : polar ? 1 : 2, i0, li, nlat);   // < nlat_pad; padded parallels read zeros
            const double cti = tb.ct_pad[i];
            for (int pass = 0; pass < npass; ++pass) {
                const int m = pass ? m_second : m_first;
                const int n_chunks = (L - m + KC - 1) / KC;
                const double* kn_i = tb.kn_t + (size_t)m * tb.nlat_pad + i;
                const double* c_ra = tb.rec_a + (size_t)m * tb.lpad;
                const double* c_rb = tb.rec_b + (size_t)m * tb.lpad;
                const double seed = tb.pmm_t[(size_t)m * tb.nlat_pad + i];
                double p1 = 0.0, p2 = 0.0;
                for (int c = 0; c < n_chunks; ++c) {
                    // factors and recursion coefficients of the chunk first (independent loads in flight
                    // together), then the serial chain: per degree one dependent multiply + subtract
                    double knv[KC], act[KC], rbv[KC];
#pragma unroll
                    for (int kk = 0; kk < KC; ++kk) {
                        const int nn = c * KC + kk;
                        knv[kk] = __ldg(kn_i + (size_t)nn * tb.nlat_pad);     // 0 beyond nmax / nlat
                        act[kk] = __dmul_rn(__ldg(c_ra + nn), cti);
                        rbv[kk] = __ldg(c_rb + nn);
                    }
                    gb::mbar_wait(&empty[stage], phase ^ 1u);
                    double* sA = s_tiles + (size_t)stage * STAGE_DOUBLES + li;
#pragma unroll
                    for (int kk = 0; kk < KC; ++kk) {
                        double pn;
                        if (c == 0 && kk == 0) pn = seed;
                        else pn = __dsub_rn(__dmul_rn(act[kk], p1), __dmul_rn(rbv[kk], p2));
                        p2 = p1;
                        p1 = pn;
                        sA[tb_fold_row(kk) * LDA] = __dmul_rn(pn, knv[kk]);
                    }
                    __syncwarp();
                    if (lane == 0) gb::mbar_arrive(&full[stage]);
                    if (++stage == STAGES) { stage = 0; phase ^= 1u; }
                }
            }
        } else {
            // ===== consumer warps: D[col][i] = sum_n X_m[n][col] Pk[n][i], the columns (e, cos|sin) on the M side of the
            // DMMA tiles and the parallels on the N side =====
            const int wm = warp / NWN;
            const int wn = warp % NWN;
            const int g = lane >> 2, q = lane & 3;
            const bool has_columns = wn * (8 * MI) < width;    // narrow batches: the other warps only keep the ring moving
            if constexpr (FOLD) {
                const int nh = nlat >> 1;
                for (int pass = 0; pass < npass; ++pass) {
                    const int m = pass ? m_second : m_first;
                    const int Kn = L - m;
                    const int n_chunks = (Kn + KC - 1) / KC;
                    const int kc_row = gb::ld_nc_early(tb.krow + 2 * m), ks_row = gb::ld_nc_early(tb.krow + 2 * m + 1);   // latency hides behind the K loop
                    double ev[MI][2][2], od[MI][2][2];
#pragma unroll
                    for (int mi = 0; mi < MI; ++mi)
#pragma unroll
                        for (int ni = 0; ni < 2; ++ni) ev[mi][ni][0] = ev[mi][ni][1] = od[mi][ni][0] = od[mi][ni][1] = 0.0;
                    for (int c = 0; c < n_chunks; ++c) {
                        const int rows = Kn - c * KC;
                        gb::mbar_wait(&full[stage], phase);
#ifdef GB_TRACE
                        if (warp == 0 && lane == 0 && item == (int)blockIdx.x && pass == 0 && c == 0) GB_TRACE_MARK(0, 3);
#endif
                        const double* sP = s_tiles + (size_t)stage * STAGE_DOUBLES + wm * 16 + g;
                        const double* sX = s_tiles + (size_t)stage * STAGE_DOUBLES + KC * LDA + wn * (8 * MI) + g;
#pragma unroll
                        for (int kk = 0; kk < KC; kk += 8) {
                            if (kk >= rows || !has_columns) break;
                            double a[MI], b[2];
#pragma unroll
                            for (int mi = 0; mi < MI; ++mi) a[mi] = sX[(kk + q) * LDB + mi * 8];
#pragma unroll
                            for (int ni = 0; ni < 2; ++ni) b[ni] = sP[(kk + q) * LDA + ni * 8];
#pragma unroll
                            for (int mi = 0; mi < MI; ++mi)
#pragma unroll
                                for (int ni = 0; ni < 2; ++ni) gb::dmma_884(ev[mi][ni][0], ev[mi][ni][1], a[mi], b[ni]);
#pragma unroll
                            for (int mi = 0; mi < MI; ++mi) a[mi] = sX[(kk + 4 + q) * LDB + mi * 8];
#pragma unroll
                            for (int ni = 0; ni < 2; ++ni) b[ni] = sP[(kk + 4 + q) * LDA + ni * 8];
#pragma unroll
                            for (int mi = 0; mi < MI; ++mi)
#pragma unroll
                                for (int ni = 0; ni < 2; ++ni) gb::dmma_884(od[mi][ni][0], od[mi][ni][1], a[mi], b[ni]);
                        }
                        __syncwarp();
                        if (lane == 0) gb::mbar_arrive(&empty[stage]);
                        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
                    }
#ifdef GB_TRACE
                    if (warp == 0 && lane == 0 && item == (int)blockIdx.x) GB_TRACE_MARK(0, 4 + 2 * pass);
#endif
                    // the store addresses are derived here, behind an opaque copy of the item's column offset: hoisted to the
                    // item prologue they would live (spilled) across the whole K loop
                    int c0e = c0;
                    asm volatile("" : "+r"(c0e));
                    // the table interleaves the parallels of a slab: this lane holds the four consecutive parallels
                    // ib .. ib+3 (fragment ni = parallels ib + 2 ni, ib + 2 ni + 1)
                    const int ib = i0 + wm * 16 + 4 * q;
                    const bool quads = (nh & 3) == 0;            // 32-byte stores: whole quads on either side of the equator
#pragma unroll
                    for (int mi = 0; mi < MI; ++mi) {
                        const int col = c0e + wn * (8 * MI) + mi * 8 + g;
                        if (col >= cols) continue;
                        const int cs = col >= E;
                        const int e = col - cs * E;
                        const int k = cs ? ks_row : kc_row;
                        if (quads) {
                            if (ib >= nh) continue;
                            const long long rn = (long long)e * nlat + ib;
                            const long long rs = (long long)e * nlat + (nlat - 4 - ib);
                            gb::st_v4(AB + gb_ab_offset(rn, k, ab_rows), ev[mi][0][0] + od[mi][0][0], ev[mi][0][1] + od[mi][0][1],
                                      ev[mi][1][0] + od[mi][1][0], ev[mi][1][1] + od[mi][1][1]);
                            gb::st_v4(AB + gb_ab_offset(rs, k, ab_rows), ev[mi][1][1] - od[mi][1][1], ev[mi][1][0] - od[mi][1][0],
                                      ev[mi][0][1] - od[mi][0][1], ev[mi][0][0] - od[mi][0][0]);
                            continue;
                        }
#pragma unroll
                        for (int ni = 0; ni < 2; ++ni) {
                            // pairs: the northern store may straddle the equator (the table holds the southern parallel's
                            // own values there), the mirrored store only covers what no northern store wrote
                            const int i = ib + ni * 2;
                            if (i < nh) {
                                const long long rn = (long long)e * nlat + i;
                                gb::st_v2(AB + gb_ab_offset(rn, k, ab_rows), ev[mi][ni][0] + od[mi][ni][0],
                                          ev[mi][ni][1] + od[mi][ni][1]);
                            }
                            if (i + 2 <= nh) {
                                const long long rs = (long long)e * nlat + (nlat - 2 - i);
                                gb::st_v2(AB + gb_ab_offset(rs, k, ab_rows), ev[mi][ni][1] - od[mi][ni][1],
                                          ev[mi][ni][0] - od[mi][ni][0]);
                            }
                        }
                    }
#ifdef GB_TRACE
                    if (warp == 0 && lane == 0 && item == (int)blockIdx.x) GB_TRACE_MARK(0, 5 + 2 * pass);
#endif
                }
                continue;
            }
            for (int pass = 0; pass < npass; ++pass) {
                const int m = pass ? m_second : m_first;
                const int Kn = L - m;
                const int n_chunks = (Kn + KC - 1) / KC;
                const int kc_row = gb::ld_nc_early(tb.krow + 2 * m), ks_row = gb::ld_nc_early(tb.krow + 2 * m + 1);
                double acc[MI][4][2];
#pragma unroll
                for (int mi = 0; mi < MI; ++mi)
#pragma unroll
                    for (int ni = 0; ni < 4; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
                for (int c = 0; c < n_chunks; ++c) {
                    const int rows = (Kn - c * KC + 7) & ~7;      // the degrees of an 8-row group are interleaved
                    gb::mbar_wait(&full[stage], phase);
                    const double* sP = s_tiles + (size_t)stage * STAGE_DOUBLES + wm * 32 + g;
                    const double* sX = s_tiles + (size_t)stage * STAGE_DOUBLES + KC * LDA + wn * (8 * MI) + g;
#pragma unroll
                    for (int kk = 0; kk < KC; kk += 4) {
                        if (kk >= rows || !has_columns) break;
                        double a[MI], b[4];
#pragma unroll
                        for (int mi = 0; mi < MI; ++mi) a[mi] = sX[(kk + q) * LDB + mi * 8];
#pragma unroll
                        for (int ni = 0; ni < 4; ++ni) b[ni] = sP[(kk + q) * LDA + ni * 8];
#pragma unroll
                        for (int mi = 0; mi < MI; ++mi)
#pragma unroll
                            for (int ni = 0; ni < 4; ++ni) gb::dmma_884(acc[mi][ni][0], acc[mi][ni][1], a[mi], b[ni]);
                    }
                    __syncwarp();
                    if (lane == 0) gb::mbar_arrive(&empty[stage]);
                    if (++stage == STAGES) { stage = 0; phase ^= 1u; }
                }
                int c0e = c0;
                asm volatile("" : "+r"(c0e));
                const int ib = ((polar && wm) ? i_south : i0) + wm * 32 + 2 * q;
                const int tile_step = ab_rows * GB_LDA - GB_TM;
#pragma unroll
                for (int mi = 0; mi < MI; ++mi) {
                    const int col = c0e + wn * (8 * MI) + mi * 8 + g;
                    if (col >= cols) continue;
                    const int cs = col >= E;
                    const int e = col - cs * E;
                    const long long row = (long long)e * nlat + ib;
                    const int o0 = (int)(row & (GB_TM - 1));
                    double* base = AB + ((size_t)(row >> 7) * ab_rows + (cs ? ks_row : kc_row)) * GB_LDA + o0;
#pragma unroll
                    for (int ni = 0; ni < 4; ++ni) {
                        const int i = ib + ni * 8;
                        if (PAIRS) {
                            if (i < nlat)
                                gb::st_v2(base + ni * 8 + ((o0 + ni * 8 >= GB_TM) ? tile_step : 0), acc[mi][ni][0],
                                          acc[mi][ni][1]);
                        } else {
                            if (i < nlat) base[ni * 8 + ((o0 + ni * 8 >= GB_TM) ? tile_step : 0)] = acc[mi][ni][0];
                            if (i + 1 < nlat)
                                base[ni * 8 + 1 + ((o0 + ni * 8 + 1 >= GB_TM) ? tile_step : 0)] = acc[mi][ni][1];
                        }
                    }
                }
            }
        }
    }
    if (threadIdx.x == 0) GB_TRACE_MARK(0, 10);
}


// The table itself: thread = (lat tile, order, parallel of the tile) runs the recursion of utilities.py:37-54 once.
__global__ void __launch_bounds__(128)
gb_ptab_kernel(double* __restrict__ tab, const int* __restrict__ roff, long long rtot, int kind, int tile0, int n_tiles,
               int L, int nlat, const double* __restrict__ ct, const double* __restrict__ kn,
               const double* __restrict__ pmm, const double* __restrict__ ra, const double* __restrict__ rb,
               const double* __restrict__ rc) {
    const int per_tile = kind == 0 ? 32 : 64;
    const int lda = kind == 0 ? 36 : 68;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)n_tiles * L * per_tile) return;
    const int li = (int)(idx % per_tile);
    const int m = (int)((idx / per_tile) % L);
    const int t = (int)(idx / ((long long)per_tile * L));
    const int i = s1_parallel(kind, kind == 2 ? t * 64 : (kind == 0 ? tile0 + t : t) * 32, li, nlat);   // i0 as in gb_stage1
    if (i < 0 || i >= nlat) return;
    double* out = tab + ((size_t)t * rtot + roff[m]) * lda + li;
    const double* kn_i = kn + (size_t)i * L;
    legendre_column(m, L, ct[i], pmm[(size_t)i * L + m], ra, rb, rc, [&](int n, double p) {
        const int nn = n - m;
        out[(size_t)tb_fold_row(nn) * lda] = __dmul_rn(p, kn_i[n]);   // same row order in every table kind and in X
    });
}

// ---------------------------------------------------------------------------------------------
// stage 2, direct contraction: V[row][j] = sum_k AB[k][row] * trig[k][j]  (M = E*nlat rows, K = kpad,
// N = nlon) on the shared persistent DMMA GEMM (gb_gemm.cuh) with a streaming row-major epilogue.
// ---------------------------------------------------------------------------------------------
struct RowMajorStore {
    double* out;
    long long M;
    int nlon;
    __device__ __forceinline__ void operator()(long long row, int col, double v0, double v1) const {
        if (row >= M) return;
        double* o = out + (size_t)row * nlon + col;
        if ((nlon & 1) == 0 && col + 1 < nlon) {
            gb::st_cs_v2(o, v0, v1);
        } else {
            if (col < nlon) gb::st_cs(o, v0);
            if (col + 1 < nlon) gb::st_cs(o + 1, v1);
        }
    }
};

// ---------------------------------------------------------------------------------------------
// stage 2 with four-fold longitude symmetry.  For mu = lon[h + j'] in the first quadrant
//   CE = sum_{m even} A_m cos(m mu)   CO = sum_{m odd} A_m cos(m mu)
//   SE = sum_{m even} B_m sin(m mu)   SO = sum_{m odd} B_m sin(m mu)
//   V(mu)      = CE + CO + SE + SO  -> column h + j'        V(pi - mu) = CE - CO - SE + SO -> nlon-1-j'
//   V(-mu)     = CE + CO - SE - SO  -> column h - 1 - j'    V(mu - pi) = CE - CO + SE - SO -> j'
// so one quarter of the multiply-adds of the direct contraction produce all four columns.
// AB rows are grouped [CE | CO | SE | SO] (gb_plan::grp_off); the K loop walks the groups in
// turn, each feeding its own accumulator set.  CTA tile: 128 rows x 32 first-quadrant columns
// (= 128 x 128 outputs), 8 consumer warps (4 x 2) with 32 x 16 x 4-set register tiles.
// ---------------------------------------------------------------------------------------------
constexpr int Q_WM = 4, Q_WN = 2;
constexpr int Q_TM = 32 * Q_WM;               // 128
constexpr int Q_TN = 16 * Q_WN;               // 32 first-quadrant columns
static_assert(Q_TM == GB_TM && Q_TN == GB_Q_TN, "tile shape must match the tiled HBM layouts");
constexpr int Q_KC = 28;
constexpr int Q_STAGES = 4;
constexpr int Q_LDA = Q_TM + 4;               // 132
constexpr int Q_LDB = Q_TN + 4;               // 36
constexpr int Q_CONSUMER_WARPS = Q_WM * Q_WN;
constexpr int Q_STAGE_DOUBLES = Q_KC * (Q_LDA + Q_LDB);
constexpr size_t Q_SMEM = (size_t)Q_STAGES * Q_STAGE_DOUBLES * sizeof(double) + (2 * Q_STAGES + 4) * sizeof(uint64_t) + 16;

struct QGroups { int off[5]; };

// 16 warps.  The eight consumer warps never store to global memory: a finished
// accumulator tile is parked in tensor memory (thread-private columns, gb::tmem_st16; double buffered: 2 x 2 x 128 of
// the 512 columns per sub-partition) and the warp goes straight back to the next tile's K loop.  Four epilogue warps,
// one per sub-partition (a warp reaches the tensor-memory lanes 32 (warp % 4) .. only), read the tile back, apply the
// butterfly and issue the stores, so the store back-pressure of the 128 KB burst per tile (every store waits for the
// LSU to drain its predecessors: 13 % of the consumers' time in the direct kernel) lands on warps that have a whole
// tile period to absorb it.  Registers are rebalanced with setmaxnreg: the kernel starts with 128 per thread
// (512 threads), consumers grow to 168, epilogue warps shrink to 104, the producer's warpgroup to 40.
// Work list of a CTA: whole tiles t = b, b + grid, ... of the full rounds; when the last, partial round holds at most
// grid / 2 tiles they are cut into halves of 64 rows, one per CTA, so that the tail costs half a tile period.
struct QWork {
    long long n_tiles, n_full;
    int n_ntiles, split, grid;
    __device__ QWork(int n_mtiles, int n_nt, int g) : n_tiles((long long)n_mtiles * n_nt), n_ntiles(n_nt), grid(g) {
        n_full = n_tiles / grid * grid;
        const long long rest = n_tiles - n_full;
        split = rest > 0 && 2 * rest <= grid;
    }
    // i-th work item of CTA b: returns false when there is none; half = -1 for a whole tile
    __device__ bool get(int b, long long i, long long& mt, int& nt, int& half) const {
        long long t = b + i * grid;
        half = -1;
        if (split && t >= n_full) {
            if (t >= n_full + grid) return false;
            const long long j = t - n_full;
            if (j >= 2 * (n_tiles - n_full)) return false;
            t = n_full + (j >> 1);
            half = (int)(j & 1);
        } else if (t >= n_tiles) {
            return false;
        }
        mt = t / n_ntiles;
        nt = (int)(t % n_ntiles);
        return true;
    }
};

constexpr int QE_THREADS = 512;
__global__ void __launch_bounds__(QE_THREADS, 1)
gb_fourier_stage2_sym(const double* __restrict__ AB, int ab_rows, const double* __restrict__ trig_q_t, int kpad_s,
                      QGroups grp, double* __restrict__ out, long long M, int nlon, int nq, int n_mtiles,
                      int n_ntiles, int wide) {
    extern __shared__ __align__(128) unsigned char s_raw[];
    double* s_tiles = reinterpret_cast<double*>(s_raw);
    uint64_t* full = reinterpret_cast<uint64_t*>(s_raw + (size_t)Q_STAGES * Q_STAGE_DOUBLES * sizeof(double));
    uint64_t* empty = full + Q_STAGES;
    uint64_t* tfull = empty + Q_STAGES;     // [2] accumulator tile parked in tensor memory
    uint64_t* tempty = tfull + 2;           // [2] tensor-memory buffer read back
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(tempty + 2);
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    constexpr int PRODUCER_WARP = 12;
    if (threadIdx.x == 0) {
        for (int s = 0; s < Q_STAGES; ++s) {
            gb::mbar_init(&full[s], 1);
            gb::mbar_init(&empty[s], Q_CONSUMER_WARPS);
        }
        for (int b = 0; b < 2; ++b) {
            gb::mbar_init(&tfull[b], Q_CONSUMER_WARPS);
            gb::mbar_init(&tempty[b], 4);
        }
        gb::fence_mbar_init();
    }
    if (warp == 0) gb::tmem_alloc(s_tmem, 512);
    gb::tmem_fence_before_sync();
    __syncthreads();
    gb::tmem_fence_after_sync();
    gb::griddep_wait();                 // AB comes from stage 1; `out` may still be read by whatever ran before
    gb::griddep_launch_dependents();

    const QWork work(n_mtiles, n_ntiles, (int)gridDim.x);
    const int h = nlon >> 1;
    // butterfly + stores of one 8-row slab of a warp tile: output row `row`, first-quadrant meridians jq .. jq+3;
    // v[4 s + 2 ni + r] = accumulator set s.  The trig tiles interleave the columns of a warp's slab (gb_plan.cu), so a
    // lane's two fragments are four consecutive meridians: one 32-byte store per lane and quadrant.
    auto emit_row = [&](long long row, int jq, const double (&v)[16]) {
        if (row >= M || jq >= nq) return;
        double* orow = out + (size_t)row * nlon;
        double v1[4], v2[4], v3[4], v4[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const double ce = v[c], co = v[4 + c], se = v[8 + c], so = v[12 + c];
            const double cp = ce + co, cm = ce - co, sp = se + so, sm = se - so;
            v1[c] = cp + sp;   // mu
            v2[c] = cm - sm;   // pi - mu
            v3[c] = cp - sp;   // -mu
            v4[c] = cm + sm;   // mu - pi
        }
        if (wide && jq + 4 <= nq) {
            gb::st_cs_v4(orow + h + jq, v1[0], v1[1], v1[2], v1[3]);
            gb::st_cs_v4(orow + nlon - 4 - jq, v2[3], v2[2], v2[1], v2[0]);
            gb::st_cs_v4(orow + h - 4 - jq, v3[3], v3[2], v3[1], v3[0]);
            gb::st_cs_v4(orow + jq, v4[0], v4[1], v4[2], v4[3]);
        } else {
#pragma unroll
            for (int c = 0; c < 4; c += 2) {          // nq is even: pairs are all in or all out
                const int j = jq + c;
                if (j >= nq) continue;
                gb::st_cs_v2(orow + h + j, v1[c], v1[c + 1]);
                gb::st_cs_v2(orow + nlon - 2 - j, v2[c + 1], v2[c]);
                gb::st_cs_v2(orow + h - 2 - j, v3[c + 1], v3[c]);
                gb::st_cs_v2(orow + j, v4[c], v4[c + 1]);
            }
        }
    };
    // first row (inside the 128-row tile) of consumer warp row wm: whole tiles 32 rows per warp, half tiles 16
    auto warp_row0 = [](int wm, int half) { return half < 0 ? wm * 32 : half * 64 + wm * 16; };

    if (warp >= PRODUCER_WARP) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 40;\n");
        if (warp == PRODUCER_WARP && lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            long long mt;
            int nt, half;
            for (long long i = 0; work.get(blockIdx.x, i, mt, nt, half); ++i) {
                for (int k0 = 0; k0 < grp.off[4];) {
                    // chunks never straddle a group boundary
                    int gend = grp.off[1];
#pragma unroll
                    for (int s = 1; s < 4; ++s)
                        if (k0 >= grp.off[s]) gend = grp.off[s + 1];
                    const int kc = min(Q_KC, gend - k0);
                    gb::mbar_wait(&empty[stage], phase ^ 1u);
                    double* sA = s_tiles + (size_t)stage * Q_STAGE_DOUBLES;
                    double* sB = sA + Q_KC * Q_LDA;
                    const uint32_t bytes_a = (uint32_t)(kc * Q_LDA * sizeof(double));
                    const uint32_t bytes_b = (uint32_t)(kc * Q_LDB * sizeof(double));
                    gb::mbar_arrive_expect_tx(&full[stage], bytes_a + bytes_b);
                    gb::bulk_g2s(sA, AB + ((size_t)mt * ab_rows + k0) * Q_LDA, bytes_a, &full[stage]);
                    gb::bulk_g2s(sB, trig_q_t + ((size_t)nt * kpad_s + k0) * Q_LDB, bytes_b, &full[stage]);
                    if (++stage == Q_STAGES) { stage = 0; phase ^= 1u; }
                    k0 += kc;
                }
            }
        }
    } else if (warp >= Q_CONSUMER_WARPS) {
        // ===== epilogue warp of sub-partition sp: the tiles of consumer warps sp and sp + 4 =====
        asm volatile("setmaxnreg.dec.sync.aligned.u32 104;\n");
        const int sp = warp & 3;
        int tb = 0;
        uint32_t tphase = 0;
        long long mt;
        int nt, half;
        for (long long i = 0; work.get(blockIdx.x, i, mt, nt, half); ++i) {
            gb::mbar_wait(&tfull[tb], tphase);
            gb::tmem_fence_after_sync();
            const int n_slabs = half < 0 ? 4 : 2;
#pragma unroll 1
            for (int cw = 0; cw < 2; ++cw) {
                const int w = sp + 4 * cw;                 // consumer warp whose tile this is
                const uint32_t taddr = *s_tmem + ((uint32_t)(32 * sp) << 16) + (uint32_t)(tb * 256 + cw * 128);
                const long long row0 = mt * Q_TM + warp_row0(w / Q_WN, half) + (lane >> 2);
                const int jq = nt * Q_TN + (w % Q_WN) * 16 + 4 * (lane & 3);
#pragma unroll 1
                for (int mi = 0; mi < n_slabs; ++mi) {
                    double v[16];
                    gb::tmem_ld16(taddr + 32u * mi, v);
                    emit_row(row0 + mi * 8, jq, v);
                }
            }
            gb::tmem_fence_before_sync();
            __syncwarp();
            if (lane == 0) gb::mbar_arrive(&tempty[tb]);
            if (++tb == 2) { tb = 0; tphase ^= 1u; }
        }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 168;\n");
        const int wm = warp / Q_WN;
        const int wn = warp % Q_WN;
        const int g = lane >> 2, q = lane & 3;
        int stage = 0, tb = 0;
        uint32_t phase = 0, tphase = 0;
        // one tile: MI 8-row slabs per warp (4: whole tile, 2: half tile)
        auto run_tile = [&](auto mi_tag, int half) {
            constexpr int MI = decltype(mi_tag)::value;
            const int r0 = warp_row0(wm, half);
            double acc[4][MI][2][2];   // [set][mi][ni][2]
#pragma unroll
            for (int s = 0; s < 4; ++s)
#pragma unroll
                for (int mi = 0; mi < MI; ++mi)
#pragma unroll
                    for (int ni = 0; ni < 2; ++ni) acc[s][mi][ni][0] = acc[s][mi][ni][1] = 0.0;
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                for (int k0 = grp.off[s]; k0 < grp.off[s + 1];) {
                    const int kc = min(Q_KC, grp.off[s + 1] - k0);
                    gb::mbar_wait(&full[stage], phase);
                    const double* sA = s_tiles + (size_t)stage * Q_STAGE_DOUBLES + r0 + g;
                    const double* sB = s_tiles + (size_t)stage * Q_STAGE_DOUBLES + Q_KC * Q_LDA + wn * 16 + g;
                    auto k_step = [&](int kk) {
                        double a[MI], b[2];
#pragma unroll
                        for (int mi = 0; mi < MI; ++mi) a[mi] = sA[(kk + q) * Q_LDA + mi * 8];
#pragma unroll
                        for (int ni = 0; ni < 2; ++ni) b[ni] = sB[(kk + q) * Q_LDB + ni * 8];
#pragma unroll
                        for (int mi = 0; mi < MI; ++mi)
#pragma unroll
                            for (int ni = 0; ni < 2; ++ni)
                                gb::dmma_884(acc[s][mi][ni][0], acc[s][mi][ni][1], a[mi], b[ni]);
                    };
                    if (kc == Q_KC) {                 // whole chunk: no per-step test in the DMMA stream
#pragma unroll
                        for (int kk = 0; kk < Q_KC; kk += 4) k_step(kk);
                    } else {
#pragma unroll
                        for (int kk = 0; kk < Q_KC; kk += 4) {
                            if (kk >= kc) break;
                            k_step(kk);
                        }
                    }
                    __syncwarp();
                    if (lane == 0) gb::mbar_arrive(&empty[stage]);
                    if (++stage == Q_STAGES) { stage = 0; phase ^= 1u; }
                    k0 += kc;
                }
            }
            // park the tile: this warp's 128 columns of buffer tb (lanes 32 (warp % 4) .., columns 256 tb + 128 (warp / 4) ..)
            gb::mbar_wait(&tempty[tb], tphase ^ 1u);
            gb::tmem_fence_after_sync();
            const uint32_t taddr = *s_tmem + ((uint32_t)(32 * (warp & 3)) << 16) + (uint32_t)(tb * 256 + (warp >> 2) * 128);
#pragma unroll
            for (int mi = 0; mi < MI; ++mi) {
                double v[16];
#pragma unroll
                for (int s = 0; s < 4; ++s)
#pragma unroll
                    for (int c = 0; c < 4; ++c) v[4 * s + c] = acc[s][mi][c >> 1][c & 1];
                gb::tmem_st16(taddr + 32u * mi, v);
            }
            gb::tmem_wait_st();
            gb::tmem_fence_before_sync();
            __syncwarp();
            if (lane == 0) gb::mbar_arrive(&tfull[tb]);
            if (++tb == 2) { tb = 0; tphase ^= 1u; }
        };
        long long mt;
        int nt, half;
        for (long long i = 0; work.get(blockIdx.x, i, mt, nt, half); ++i) {
            if (half < 0) run_tile(std::integral_constant<int, 4>{}, half);
            else run_tile(std::integral_constant<int, 2>{}, half);
        }
    }
    gb::tmem_fence_before_sync();
    __syncthreads();
    if (warp == 0) gb::tmem_dealloc(*s_tmem, 512);
}

// ---------------------------------------------------------------------------------------------
// stage 2 with EIGHT-fold longitude symmetry -- third declared shortcut of the synthesis (gb_plan::oct, gated on the
// trig tables like the four-fold one).  The first-quadrant meridians mirror about pi/4: with nu = lon[h + j] in the first
// octant and mu' = pi/2 - nu, the orders m = 0, 2 (mod 4) only change the SIGN of their cosine / sine rows, the odd
// orders swap them (gb_plan.cu).  Per octant meridian eight sums
//   E0, E2 = sum_{m = 0, 2 (4)} A_m cos(m nu)     F0, F2 = sum_{m = 0, 2 (4)} B_m sin(m nu)         (even orders: K / 2 each)
//   CO = sum_odd A_m cos(m nu),  AS = sum_odd A_m (+-) sin(m nu)      SO = sum_odd B_m sin(m nu),  BC = sum_odd B_m (+-) cos(m nu)
// give the quadrant sums at nu (CE = E0 + E2, SE = F0 + F2, CO, SO) and at pi/2 - nu (CE = E0 - E2, SE = F2 - F0,
// CO = AS, SO = BC), hence eight meridians: the even orders cost half the multiply-adds of the quadrant kernel, the odd
// ones the same -- 3/4 in total -- and an odd k-step feeds two accumulator sets from ONE coefficient fragment (8 LDS per
// 16 DMMA instead of 6 per 8).
// Same structure as gb_fourier_stage2_sym: persistent, 8 consumer warps (4 x 2, 32 rows x 16 octant columns), 4
// epilogue warps, 1 producer lane, 4-stage ring (coefficient chunk + one or two table chunks).  CTA tile 128 rows x 32 octant
// columns = 128 x 256 outputs.  A tile is parked in tensor memory in two halves (the four even sets after the even groups,
// the four odd sets at the end: 2 x 128 columns per consumer warp, single buffered -- the epilogue warp of the lane quarter
// hands each consumer's buffers back as soon as it has read them).
// ---------------------------------------------------------------------------------------------
constexpr int O_KC = 28, O_STAGES = 4;
constexpr int O_STAGE_DOUBLES = O_KC * (Q_LDA + 2 * Q_LDB);
constexpr size_t O_SMEM = (size_t)O_STAGES * O_STAGE_DOUBLES * sizeof(double) + (2 * O_STAGES + 4 * Q_CONSUMER_WARPS) * sizeof(uint64_t) + 16;

struct OGroups { int off[7]; };

__global__ void __launch_bounds__(QE_THREADS, 1)
gb_fourier_stage2_oct(const double* __restrict__ AB, int ab_rows, const double* __restrict__ trig_o_t, int kpad_o, OGroups grp,
                      double* __restrict__ out, long long M, int nlon, int no, int n_mtiles, int n_ntiles, int wide) {
    extern __shared__ __align__(128) unsigned char s_raw[];
    double* s_tiles = reinterpret_cast<double*>(s_raw);
    uint64_t* full = reinterpret_cast<uint64_t*>(s_raw + (size_t)O_STAGES * O_STAGE_DOUBLES * sizeof(double));
    uint64_t* empty = full + O_STAGES;
    uint64_t* tfull = empty + O_STAGES;                 // [2 halves][8 consumer warps]
    uint64_t* tempty = tfull + 2 * Q_CONSUMER_WARPS;    // [2 halves][8 consumer warps]
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(tempty + 2 * Q_CONSUMER_WARPS);
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    constexpr int PRODUCER_WARP = 12;
    if (threadIdx.x == 0) {
        GB_TRACE_MARK(1, 0);
        for (int s = 0; s < O_STAGES; ++s) {
            gb::mbar_init(&full[s], 1);
            gb::mbar_init(&empty[s], Q_CONSUMER_WARPS);
        }
        for (int b = 0; b < 2 * Q_CONSUMER_WARPS; ++b) {
            gb::mbar_init(&tfull[b], 1);
            gb::mbar_init(&tempty[b], 1);
        }
        gb::fence_mbar_init();
    }
    if (warp == 0) gb::tmem_alloc(s_tmem, 512);
    gb::tmem_fence_before_sync();
    __syncthreads();
    gb::tmem_fence_after_sync();
    gb::griddep_launch_dependents();
    // griddepcontrol.wait (AB comes from stage 1; `out` may still be read by whatever ran before) is executed by the
    // producer lane alone, right before its first copy: everything else -- the work list, the register hand-over, the
    // first fetch of the kernel parameters (a DRAM round trip after an L2 flush) -- overlaps the predecessor's tail.
    // No other thread touches global memory before it has seen data those copies delivered.

    const QWork work(n_mtiles, n_ntiles, (int)gridDim.x);
    const int h = nlon >> 1, nq = nlon >> 2;
    auto warp_row0 = [](int wm, int half) { return half < 0 ? wm * 32 : half * 64 + wm * 16; };
    // butterfly + stores of one 8-row slab of a warp tile (output row `row`, octant meridians jo .. jo+3):
    // ve = [E0 | E2 | F0 | F2] x 4 meridians, vo = [CO | AS | SO | BC] x 4 meridians
    auto emit_slab = [&](long long row, int jo, const double (&ve)[16], const double (&vo)[16]) {
        if (row >= M || jo >= no) return;
        double* orow = out + (size_t)row * nlon;
        // the quadrant sums at nu (p = 0) and at pi/2 - nu (p = 1), then the four mirrored meridians of each
#pragma unroll
        for (int p = 0; p < 2; ++p) {
            double v1[4], v2[4], v3[4], v4[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const double ce = p ? ve[c] - ve[4 + c] : ve[c] + ve[4 + c];
                const double se = p ? ve[12 + c] - ve[8 + c] : ve[8 + c] + ve[12 + c];
                const double co = p ? vo[4 + c] : vo[c];
                const double so = p ? vo[12 + c] : vo[8 + c];
                const double cp = ce + co, cm = ce - co, sp_ = se + so, sm = se - so;
                v1[c] = cp + sp_;   // mu
                v2[c] = cm - sm;    // pi - mu
                v3[c] = cp - sp_;   // -mu
                v4[c] = cm + sm;    // mu - pi
            }
            // quadrant index of meridian c: jo + c (p = 0, ascending) or nq - 1 - jo - c (p = 1, descending)
            if (wide && jo + 4 <= no) {
                if (p == 0) {
                    gb::st_cs_v4(orow + h + jo, v1[0], v1[1], v1[2], v1[3]);
                    gb::st_cs_v4(orow + nlon - 4 - jo, v2[3], v2[2], v2[1], v2[0]);
                    gb::st_cs_v4(orow + h - 4 - jo, v3[3], v3[2], v3[1], v3[0]);
                    gb::st_cs_v4(orow + jo, v4[0], v4[1], v4[2], v4[3]);
                } else {
                    const int jb = nq - 4 - jo;       // quadrant index of c = 3
                    gb::st_cs_v4(orow + h + jb, v1[3], v1[2], v1[1], v1[0]);
                    gb::st_cs_v4(orow + nlon - 4 - jb, v2[0], v2[1], v2[2], v2[3]);
                    gb::st_cs_v4(orow + h - 4 - jb, v3[0], v3[1], v3[2], v3[3]);
                    gb::st_cs_v4(orow + jb, v4[3], v4[2], v4[1], v4[0]);
                }
            } else {
#pragma unroll
                for (int c = 0; c < 4; c += 2) {          // no is even: pairs are all in or all out
                    if (jo + c >= no) continue;
                    if (p == 0) {
                        const int j = jo + c;
                        gb::st_cs_v2(orow + h + j, v1[c], v1[c + 1]);
                        gb::st_cs_v2(orow + nlon - 2 - j, v2[c + 1], v2[c]);
                        gb::st_cs_v2(orow + h - 2 - j, v3[c + 1], v3[c]);
                        gb::st_cs_v2(orow + j, v4[c], v4[c + 1]);
                    } else {
                        const int j = nq - 2 - jo - c;    // quadrant index of c + 1
                        gb::st_cs_v2(orow + h + j, v1[c + 1], v1[c]);
                        gb::st_cs_v2(orow + nlon - 2 - j, v2[c], v2[c + 1]);
                        gb::st_cs_v2(orow + h - 2 - j, v3[c], v3[c + 1]);
                        gb::st_cs_v2(orow + j, v4[c + 1], v4[c]);
                    }
                }
            }
        }
    };
    // The LAST tile of a CTA has no K loop behind it to hide its epilogue: the epilogue warps take only the first
    // S_TAIL_EPI slab(s) of every consumer's tile, each consumer warp reads the rest of its own tile back and stores it.
    constexpr int S_TAIL_EPI = 1;

    if (warp >= PRODUCER_WARP) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 40;\n");
        if (warp == PRODUCER_WARP && lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            long long mt;
            int nt, half;
            {
                // the parameters and the first work item are in registers before the wait
                const bool any = work.get(blockIdx.x, 0, mt, nt, half);
                const double* a0 = AB + ((size_t)mt * ab_rows + grp.off[4]) * Q_LDA;
                const double* b0 = trig_o_t + ((size_t)nt * 2 * kpad_o + grp.off[4]) * Q_LDB;
                asm volatile("" ::"r"((int)any), "l"(a0), "l"(b0), "r"(grp.off[5]), "r"(grp.off[6]), "r"(grp.off[0]), "r"(grp.off[1]),
                             "r"(grp.off[2]), "r"(grp.off[3]));
            }
            gb::griddep_wait();
            GB_TRACE_MARK(1, 1);
            for (long long i = 0; work.get(blockIdx.x, i, mt, nt, half); ++i) {
                const double* t1 = trig_o_t + (size_t)nt * 2 * kpad_o * Q_LDB;
                const double* t2 = t1 + (size_t)kpad_o * Q_LDB;
                for (int go = 0; go < 6; ++go) {
                    const int gi = go < 2 ? 4 + go : go - 2;        // the odd groups first (see the consumers)
                    for (int k0 = grp.off[gi]; k0 < grp.off[gi + 1];) {
                        const int kc = min(O_KC, grp.off[gi + 1] - k0);
                        gb::mbar_wait(&empty[stage], phase ^ 1u);
                        double* sA = s_tiles + (size_t)stage * O_STAGE_DOUBLES;
                        double* sB = sA + O_KC * Q_LDA;
                        const uint32_t bytes_a = (uint32_t)(kc * Q_LDA * sizeof(double));
                        const uint32_t bytes_b = (uint32_t)(kc * Q_LDB * sizeof(double));
                        gb::mbar_arrive_expect_tx(&full[stage], bytes_a + (gi >= 4 ? 2 : 1) * bytes_b);
                        gb::bulk_g2s(sA, AB + ((size_t)mt * ab_rows + k0) * Q_LDA, bytes_a, &full[stage]);
                        gb::bulk_g2s(sB, t1 + (size_t)k0 * Q_LDB, bytes_b, &full[stage]);
                        if (gi >= 4) gb::bulk_g2s(sB + O_KC * Q_LDB, t2 + (size_t)k0 * Q_LDB, bytes_b, &full[stage]);
#ifdef GB_TRACE
                        if (i == 0 && go == 0 && k0 == grp.off[gi]) GB_TRACE_MARK(1, 2);
#endif
                        if (++stage == O_STAGES) { stage = 0; phase ^= 1u; }
                        k0 += kc;
                    }
                }
            }
        }
    } else if (warp >= Q_CONSUMER_WARPS) {
        // ===== epilogue warp of lane quarter sp: the tiles of consumer warps sp and sp + 4 =====
        asm volatile("setmaxnreg.inc.sync.aligned.u32 136;\n");
        const int sp = warp & 3;
        uint32_t tphase = 0;
        long long mt, mt_next = 0;
        int nt, half, nt_next = 0, half_next = 0;
        bool more = work.get(blockIdx.x, 0, mt, nt, half);
        for (long long i = 0; more; ++i) {
            more = work.get(blockIdx.x, i + 1, mt_next, nt_next, half_next);
            const int n_slabs = half < 0 ? 4 : 2;
            const int n_mine = more ? n_slabs : S_TAIL_EPI;      // last tile: the consumers store the other slabs themselves
#pragma unroll 1
            for (int cw = 0; cw < 2; ++cw) {
                const int w = sp + 4 * cw;                 // consumer warp whose tile this is
                const uint32_t taddr = *s_tmem + ((uint32_t)(32 * sp) << 16) + (uint32_t)(cw * 256);
                const long long row0 = mt * Q_TM + warp_row0(w / Q_WN, half) + (lane >> 2);
                const int jo = nt * Q_TN + (w % Q_WN) * 16 + 4 * (lane & 3);      // first of this lane's four octant meridians
                gb::mbar_wait(&tfull[w], tphase);
                gb::mbar_wait(&tfull[Q_CONSUMER_WARPS + w], tphase);
                gb::tmem_fence_after_sync();
#ifdef GB_TRACE
                if (warp == 8 && lane == 0 && cw == 0 && i < 3) GB_TRACE_MARK(1, 16 + 2 * (int)i);
#endif
#pragma unroll 1
                for (int mi = 0; mi < n_mine; ++mi) {
                    double ve[16], vo[16];
                    gb::tmem_ld16(taddr + 32u * mi, ve);             // [E0 | E2 | F0 | F2] x 4 meridians
                    gb::tmem_ld16(taddr + 128u + 32u * mi, vo);      // [CO | AS | SO | BC] x 4 meridians
                    if (mi == n_mine - 1 && more) {
                        // both halves of this consumer's tile have been read: hand its buffers back
                        gb::tmem_fence_before_sync();
                        __syncwarp();
                        if (lane == 0) {
                            gb::mbar_arrive(&tempty[w]);
                            gb::mbar_arrive(&tempty[Q_CONSUMER_WARPS + w]);
                        }
                    }
                    emit_slab(row0 + mi * 8, jo, ve, vo);
                }
            }
#ifdef GB_TRACE
            if (warp == 8 && lane == 0 && i < 3) GB_TRACE_MARK(1, 17 + 2 * (int)i);
#endif
            tphase ^= 1u;
            mt = mt_next; nt = nt_next; half = half_next;
        }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 168;\n");
        const int wm = warp / Q_WN;
        const int wn = warp % Q_WN;
        const int g = lane >> 2, q = lane & 3;
        int stage = 0;
        uint32_t phase = 0, tphase = 0;
        const uint32_t taddr = *s_tmem + ((uint32_t)(32 * (warp & 3)) << 16) + (uint32_t)((warp >> 2) * 256);
        long long trace_item = 0;
        auto run_tile = [&](auto mi_tag, long long mt, int nt, int half, bool last) {
            constexpr int MI = decltype(mi_tag)::value;
            const int r0 = warp_row0(wm, half);
            // the odd part (two thirds of the tile's DMMAs) first: its half is parked two thirds into the tile period, by
            // when the epilogue warp has long read the previous tile (the tensor-memory buffers are single)
#pragma unroll 1
            for (int part = 1; part >= 0; --part) {
                double acc[4][MI][2][2];   // [set][mi][ni][2]: even part E0 E2 F0 F2, odd part CO AS SO BC
#pragma unroll
                for (int s = 0; s < 4; ++s)
#pragma unroll
                    for (int mi = 0; mi < MI; ++mi)
#pragma unroll
                        for (int ni = 0; ni < 2; ++ni) acc[s][mi][ni][0] = acc[s][mi][ni][1] = 0.0;
                auto chunks = [&](int gi, auto&& k_step) {
                    for (int k0 = grp.off[gi]; k0 < grp.off[gi + 1];) {
                        const int kc = min(O_KC, grp.off[gi + 1] - k0);
                        gb::mbar_wait(&full[stage], phase);
#ifdef GB_TRACE
                        if (warp == 0 && lane == 0 && trace_item == 0 && part == 1 && gi == 4 && k0 == grp.off[4]) GB_TRACE_MARK(1, 3);
#endif
                        const double* sA = s_tiles + (size_t)stage * O_STAGE_DOUBLES + r0 + g;
                        const double* sB = s_tiles + (size_t)stage * O_STAGE_DOUBLES + O_KC * Q_LDA + wn * 16 + g;
                        if (kc == O_KC) {
#pragma unroll
                            for (int kk = 0; kk < O_KC; kk += 4) k_step(sA, sB, kk);
                        } else {
#pragma unroll
                            for (int kk = 0; kk < O_KC; kk += 4) {
                                if (kk >= kc) break;
                                k_step(sA, sB, kk);
                            }
                        }
                        __syncwarp();
                        if (lane == 0) gb::mbar_arrive(&empty[stage]);
                        if (++stage == O_STAGES) { stage = 0; phase ^= 1u; }
                        k0 += kc;
                    }
                };
                if (part == 0) {
#pragma unroll
                    for (int s = 0; s < 4; ++s)
                        chunks(s, [&](const double* sA, const double* sB, int kk) {
                            double a[MI], b[2];
#pragma unroll
                            for (int mi = 0; mi < MI; ++mi) a[mi] = sA[(kk + q) * Q_LDA + mi * 8];
#pragma unroll
                            for (int ni = 0; ni < 2; ++ni) b[ni] = sB[(kk + q) * Q_LDB + ni * 8];
#pragma unroll
                            for (int mi = 0; mi < MI; ++mi)
#pragma unroll
                                for (int ni = 0; ni < 2; ++ni) gb::dmma_884(acc[s][mi][ni][0], acc[s][mi][ni][1], a[mi], b[ni]);
                        });
                } else {
#pragma unroll
                    for (int s = 0; s < 2; ++s)
                        chunks(4 + s, [&](const double* sA, const double* sB, int kk) {
                            // one coefficient fragment, two table rows: cos and (+-) sin of the octant meridian
                            double a[MI], b1[2], b2[2];
#pragma unroll
                            for (int mi = 0; mi < MI; ++mi) a[mi] = sA[(kk + q) * Q_LDA + mi * 8];
#pragma unroll
                            for (int ni = 0; ni < 2; ++ni) {
                                b1[ni] = sB[(kk + q) * Q_LDB + ni * 8];
                                b2[ni] = sB[(O_KC + kk + q) * Q_LDB + ni * 8];
                            }
#pragma unroll
                            for (int mi = 0; mi < MI; ++mi)
#pragma unroll
                                for (int ni = 0; ni < 2; ++ni) {
                                    gb::dmma_884(acc[2 * s][mi][ni][0], acc[2 * s][mi][ni][1], a[mi], b1[ni]);
                                    gb::dmma_884(acc[2 * s + 1][mi][ni][0], acc[2 * s + 1][mi][ni][1], a[mi], b2[ni]);
                                }
                        });
                }
#ifdef GB_TRACE
                if (warp == 0 && lane == 0 && trace_item < 3) GB_TRACE_MARK(1, 4 + 4 * (int)trace_item + 2 * (1 - part));
#endif
                // park this half of the tile: columns 256 (warp / 4) + 128 part + 32 mi of this warp's lanes
                gb::mbar_wait(&tempty[part * Q_CONSUMER_WARPS + warp], tphase ^ 1u);
                gb::tmem_fence_after_sync();
#pragma unroll
                for (int mi = 0; mi < MI; ++mi) {
                    double v[16];
#pragma unroll
                    for (int s = 0; s < 4; ++s)
#pragma unroll
                        for (int c = 0; c < 4; ++c) v[4 * s + c] = acc[s][mi][c >> 1][c & 1];
                    gb::tmem_st16(taddr + 128u * part + 32u * mi, v);
                }
                gb::tmem_wait_st();
                gb::tmem_fence_before_sync();
                __syncwarp();
                if (lane == 0) gb::mbar_arrive(&tfull[part * Q_CONSUMER_WARPS + warp]);
#ifdef GB_TRACE
                if (warp == 0 && lane == 0 && trace_item < 3) GB_TRACE_MARK(1, 5 + 4 * (int)trace_item + 2 * (1 - part));
#endif
            }
            if (last) {
                // no K loop follows: this warp stores the slabs the epilogue warp leaves to it (its own parked values)
                const long long row0 = mt * Q_TM + r0 + g;
                const int jo = nt * Q_TN + wn * 16 + 4 * q;
#pragma unroll 1
                for (int mi = S_TAIL_EPI; mi < MI; ++mi) {
                    double ve[16], vo[16];
                    gb::tmem_ld16(taddr + 32u * mi, ve);
                    gb::tmem_ld16(taddr + 128u + 32u * mi, vo);
                    emit_slab(row0 + mi * 8, jo, ve, vo);
                }
            }
            tphase ^= 1u;
            ++trace_item;
        };
        long long mt, mt_next = 0;
        int nt, half, nt_next = 0, half_next = 0;
        bool more = work.get(blockIdx.x, 0, mt, nt, half);
        for (long long i = 0; more; ++i) {
            more = work.get(blockIdx.x, i + 1, mt_next, nt_next, half_next);
            if (half < 0) run_tile(std::integral_constant<int, 4>{}, mt, nt, half, !more);
            else run_tile(std::integral_constant<int, 2>{}, mt, nt, half, !more);
            mt = mt_next; nt = nt_next; half = half_next;
        }
    }
    if (threadIdx.x == 0) GB_TRACE_MARK(1, 22);
    gb::tmem_fence_before_sync();
    __syncthreads();
    if (threadIdx.x == 0) GB_TRACE_MARK(1, 23);
    if (warp == 0) gb::tmem_dealloc(*s_tmem, 512);
}

// Plain one-thread-per-output stage 2 (debug cross-check of the tensor-core kernel, GB_NAIVE_STAGE2=1).
__global__ void __launch_bounds__(256)
gb_fourier_stage2_naive(const double* __restrict__ AB, int ab_rows, const double* __restrict__ trig, int nlp,
                        int kpad, double* __restrict__ out, long long M, int nlon) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= M * nlon) return;
    const long long row = idx / nlon;
    const int j = (int)(idx % nlon);
    double s = 0.0;
    for (int k = 0; k < kpad; ++k) s = fma(AB[gb_ab_offset(row, k, ab_rows)], trig[(size_t)k * nlp + j], s);
    out[idx] = s;
}

// Legendre table in the reference's packed layout (bit-exactness hook).
__global__ void __launch_bounds__(128)
gb_legendre_table_kernel(double* __restrict__ out, const double* __restrict__ ct, const double* __restrict__ kn,
                         const double* __restrict__ pmm, const double* __restrict__ ra, const double* __restrict__ rb,
                         const double* __restrict__ rc, int L, int nlat, int scaled) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= nlat * L) return;
    const int i = idx / L, m = idx % L;
    double* o = out + (size_t)i * L * L;
    const double* kn_i = kn + (size_t)i * L;
    legendre_column(m, L, ct[i], pmm[(size_t)i * L + m], ra, rb, rc, [&](int n, double p) {
        const double v = scaled ? __dmul_rn(p, kn_i[n]) : p;
        o[(size_t)n * L + m] = v;
        if (m > 0) o[(size_t)(m - 1) * L + n] = v;
    });
}

}  // namespace

constexpr size_t PTAB_MAX_BYTES = (size_t)2048 << 20;     // memory budget of one Legendre table

// Build (once) the Legendre table of `kind` (gb_common.cuh: 0 folded tiles, 1 polar-cap tiles, 2 plain tiles).
// Returns 1 if the table exists, 0 if it is over PTAB_MAX_BYTES or cannot be allocated (the caller then runs stage 1
// in its Recursion mode), < 0 on error (-code).
static int ensure_ptab(gb_plan* p, int kind, int n_tiles, int tile0, cudaStream_t st) {
    if (p->ptab_state[kind] != 0) return p->ptab_state[kind] > 0 ? 1 : 0;
    const int L = p->L;
    const int lda = kind == 0 ? 36 : 68, per_tile = kind == 0 ? 32 : 64;
    const size_t elems = (size_t)n_tiles * p->ptab_rtot * lda;
    if (elems * sizeof(double) > PTAB_MAX_BYTES) {
        p->ptab_state[kind] = -1;
        return 0;
    }
    if (cudaMalloc(reinterpret_cast<void**>(&p->d_ptab[kind]), elems * sizeof(double)) != cudaSuccess) {
        cudaGetLastError();
        p->ptab_state[kind] = -1;          // no room: the Recursion mode needs none
        return 0;
    }
    cudaError_t e = cudaMemsetAsync(p->d_ptab[kind], 0, elems * sizeof(double), st);
    if (e == cudaSuccess) {
        const long long total = (long long)n_tiles * L * per_tile;
        gb_ptab_kernel<<<(unsigned)((total + 127) / 128), 128, 0, st>>>(p->d_ptab[kind], p->d_ptab_roff, p->ptab_rtot, kind,
                                                                      tile0, n_tiles, L, p->nlat, p->d_ct, p->d_kn, p->d_pmm,
                                                                      p->d_ra, p->d_rb, p->d_rc);
        gb_count_launch();
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) return -gb_set_error(GB_ERR_CUDA, "Legendre table build failed: %s", cudaGetErrorString(e));
    p->ptab_state[kind] = 1;
    return 1;
}

// order-wise block filter applied between the pack and the Legendre stage (gb_synthesis_orderwise_filtered)
struct SynthesisFilter {
    const double* d_blocks;
    const int64_t* block_offsets;
    int nf;
};

// Column tiling of the stage-1 items: NWN column warps of MI 8-column fragments, tn = 8 MI NWN columns (e, cos|sin).
struct S1Tiling {
    int nwn, mi;
    int tn() const { return 8 * mi * nwn; }
};

// Narrow batches (at most 80 epochs) run 80-column items, several CTAs per SM; wider batches 240-column items.  Folded
// grids without polar caps (fold_only: nothing runs the unfolded instances there) have two more tilings.
static S1Tiling stage1_tiling(int E, bool fold_only) {
    const int cols = 2 * E;
    if (fold_only && cols <= 64) return {2, 4};      // shards of at most 32 epochs: 64-column items (no padding fragment)
    // 41 .. 60 epochs: ONE 120-column tile per order pair and latitude tile, two CTAs per SM (80-column tiles would leave
    // a second, mostly empty round of items)
    if (fold_only && cols > 80 && cols <= 120) return {3, 5};
    return cols <= 160 ? S1Tiling{2, 5} : S1Tiling{6, 5};
}

// what the stage-1 launches of one synthesis share
struct S1Launch {
    gb_plan* p;
    const int* krow;
    S1Tiling tiling;
    int E, n_coltiles;
    cudaStream_t st;
};

// Stage 1 over `lattiles` latitude tiles of `kind` (gb_common.cuh).  Threads and shared memory follow from the template
// arguments.
template <S1Source SRC, bool PAIRS, int NWN, bool FOLD, int MI>
static int launch_stage1(const S1Launch& a, int kind, int lattiles, int items, int polar) {
    const gb_plan* p = a.p;
    auto kernel = gb_stage1<SRC, PAIRS, NWN, FOLD, MI>;
    constexpr int ctas_per_sm = s1_ctas_per_sm(NWN, FOLD, SRC);
    const int max_ctas = ctas_per_sm * p->sm_count;
    const int grid = items < max_ctas ? items : max_ctas;
    size_t smem = s1_smem(NWN, FOLD, SRC);
    // Fewer items than CTA slots (a narrow shard): the CTAs are launched while the pack kernel still holds part of every
    // SM (programmatic dependent launch) and the block scheduler fills whatever is free first -- three CTAs on some SMs,
    // one on others, and the crowded SMs finish last.  Asking for more shared memory than a CTA needs caps the CTAs per
    // SM at the even share.
    const int per_sm = (grid + p->sm_count - 1) / p->sm_count;
    if (per_sm < ctas_per_sm) {
        const size_t forbid = 233472 / (size_t)(per_sm + 1) - 1024 + 256;      // per_sm + 1 CTAs no longer fit
        const size_t allow = 233472 / (size_t)per_sm - 1024;                    // per_sm CTAs still do
        if (forbid > smem && forbid <= allow && forbid <= 232448) smem = forbid;
    }
    const S1Args args{p->d_ptab_roff, a.krow,     p->d_ptab[kind], p->ptab_rtot * s1_lda(FOLD), p->d_ct_pad, p->d_kn_t,
                      p->d_pmm_t,     p->d_rec_a, p->d_rec_b,      p->nlat_pad,                 p->lpad};
    GB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    GB_CUDA(gb_launch_pdl(kernel, dim3(grid), dim3(s1_threads(NWN, FOLD, SRC)), smem, a.st, p->d_x, p->d_ab, args, p->L,
                          p->nlat, a.E, p->ab_rows, lattiles, a.n_coltiles, items, polar));
    GB_LAUNCH_CHECK();
    return GB_OK;
}

// The stage-1 instance for the tiling, the fold and the parity of the parallel count (folded grids have an even one).
template <S1Source SRC>
static int dispatch_stage1(const S1Launch& a, bool fold, bool pairs, int kind, int lattiles, int items, int polar) {
    const S1Tiling t = a.tiling;
    if (fold) {
        if (t.mi == 4) return launch_stage1<SRC, true, 2, true, 4>(a, kind, lattiles, items, polar);
        if (t.nwn == 2) return launch_stage1<SRC, true, 2, true, 5>(a, kind, lattiles, items, polar);
        if (t.nwn == 3) return launch_stage1<SRC, true, 3, true, 5>(a, kind, lattiles, items, polar);
        return launch_stage1<SRC, true, 6, true, 5>(a, kind, lattiles, items, polar);
    }
    if (t.nwn == 2)
        return pairs ? launch_stage1<SRC, true, 2, false, 5>(a, kind, lattiles, items, polar)
                     : launch_stage1<SRC, false, 2, false, 5>(a, kind, lattiles, items, polar);
    return pairs ? launch_stage1<SRC, true, 6, false, 5>(a, kind, lattiles, items, polar)
                 : launch_stage1<SRC, false, 6, false, 5>(a, kind, lattiles, items, polar);
}

// the eight-fold symmetric stage 2: plan gate + override
static bool stage2_octant(const gb_plan* p) { return p->sym && p->oct && !gb_env_flag("GB_S2_QUADRANT"); }

// spectral row k = 2m + cs -> row of the AB layout the symmetric Fourier stage of this plan reads (octant or quadrant order)
const int* gb_stage2_krow(const gb_plan* p) { return stage2_octant(p) ? p->d_krow_oct : p->d_krow_sym; }

template <typename... KArgs, typename... Args>
static cudaError_t launch_maybe_pdl(bool pdl, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                    Args... args) {
    if (pdl) return gb_launch_pdl(kernel, grid, block, smem, st, args...);
    kernel<<<grid, block, smem, st>>>(args...);
    return cudaSuccess;      // launch errors: GB_LAUNCH_CHECK
}

// The symmetric Fourier stage on any row set in the AB layout: d_out[row][j] = sum_k d_ab[row][k] trig[k][j], rows
// [0, M).  The synthesis launches it behind its stage 1 with programmatic dependent launch (pdl); the covariance
// propagation, whose longitude quadratic form starts with the same contraction, launches it plainly.
int gb_launch_stage2_sym(gb_plan* p, const double* d_ab, long long M, double* d_out, cudaStream_t st, bool pdl) {
    GB_REQUIRE(p->sym, "gb_launch_stage2_sym: the plan's meridians are not four-fold symmetric");
    const bool oct = stage2_octant(p);
    const int n_mtiles = (int)((M + Q_TM - 1) / Q_TM);
    const int n_ntiles = oct ? p->n_otiles : p->n_qtiles;
    const long long n_tiles = (long long)n_mtiles * n_ntiles;
    if (n_tiles == 0) return GB_OK;
    const int grid = (int)((n_tiles < p->sm_count) ? n_tiles : p->sm_count);
    // 32-byte stores need 32-byte aligned rows: the base pointer, and a meridian count that keeps every row aligned
    const bool out32 = reinterpret_cast<uintptr_t>(d_out) % 32 == 0;
    if (oct) {
        OGroups grp;
        for (int g = 0; g < 7; ++g) grp.off[g] = p->ogrp_off[g];
        const int wide = out32 && p->nlon % 16 == 0;
        GB_CUDA(cudaFuncSetAttribute(gb_fourier_stage2_oct, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)O_SMEM));
        GB_CUDA(launch_maybe_pdl(pdl, gb_fourier_stage2_oct, dim3(grid), dim3(QE_THREADS), O_SMEM, st, d_ab, p->ab_rows,
                                 p->d_trig_o_t, p->kpad_o, grp, d_out, M, p->nlon, p->no, n_mtiles, n_ntiles, wide));
    } else {
        QGroups grp;
        for (int g = 0; g < 5; ++g) grp.off[g] = p->grp_off[g];
        const int wide = out32 && p->nlon % 8 == 0;
        GB_CUDA(cudaFuncSetAttribute(gb_fourier_stage2_sym, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Q_SMEM));
        GB_CUDA(launch_maybe_pdl(pdl, gb_fourier_stage2_sym, dim3(grid), dim3(QE_THREADS), Q_SMEM, st, d_ab, p->ab_rows,
                                 p->d_trig_q_t, p->kpad_s, grp, d_out, M, p->nlon, p->nq, n_mtiles, n_ntiles, wide));
    }
    GB_LAUNCH_CHECK();
    return GB_OK;
}

static int launch_synthesis(gb_plan* p, const double* d_anm, int E, double* d_out, cudaStream_t st,
                            const double* d_wn = nullptr, const SynthesisFilter* flt = nullptr) {
    const int L = p->L;
    const long long M = (long long)E * p->nlat;
    {
        int rca = gb_plan_acquire(p, st);   // one workspace (X, AB) per plan: order this call behind the previous one
        if (rca) return rca;
    }
    cudaEvent_t* prof = (p->prof_ev && p->prof_count < p->prof_capacity) ? p->prof_ev + (size_t)p->prof_count * 4 : nullptr;
    const bool naive2 = gb_env_flag("GB_NAIVE_STAGE2");
    const bool use_sym = p->sym && !naive2 && !gb_env_flag("GB_NO_SYMMETRY");
    const int* d_krow = use_sym ? gb_stage2_krow(p) : p->d_krow_id;
    const bool simple1 = gb_env_flag("GB_SIMPLE_STAGE1");           // FMA cross-check on the order-wise X
    const bool fold = p->fold_ns && !gb_env_flag("GB_NO_FOLD");     // equatorial symmetry: 32 northern parallels per item
    const int cap_tiles = fold ? p->fold_cap / 32 : 0;              // polar tiles that stay unfolded
    const int n_lattiles = fold ? (p->nlat / 2 + 31) / 32 - cap_tiles : (p->nlat + GB_T1_TM - 1) / GB_T1_TM;
    // the Legendre table(s) of these latitude tiles; 0 = over budget -> recursion on the fly
    int have_tab = (simple1 || gb_env_flag("GB_S1_ONTHEFLY")) ? 0 : ensure_ptab(p, fold ? 0 : 2, n_lattiles, cap_tiles, st);
    if (have_tab > 0 && cap_tiles > 0) have_tab = ensure_ptab(p, 1, cap_tiles, 0, st);
    if (have_tab < 0) return -have_tab;
    const S1Tiling tiling = stage1_tiling(E, fold && cap_tiles == 0);
    const int tn = tiling.tn();
    const int n_coltiles = (2 * E + tn - 1) / tn;
    const int n_items = (L + 1) / 2 * n_lattiles * n_coltiles;     // order pairs (p, nmax - p) x tiles
    const int cap_items = (L + 1) / 2 * cap_tiles * n_coltiles;
    if (!simple1) {
        // tiled X: pad rows, pad columns and the (non-existent) sine plane of order 0 are never written by the pack
        const long long key = ((long long)E << 16) | tn;
        if (p->x_layout_key != key) {
            GB_CUDA(cudaMemsetAsync(p->d_x, 0, p->x_elems * sizeof(double), st));
            p->x_layout_key = key;
        }
    } else {
        p->x_layout_key = 0;
    }
    if (prof) GB_CUDA(cudaEventRecord(prof[0], st));
    if (flt) {
        // pack -> filter, whose epilogue writes X in the layout the Legendre stage reads (no unpack / second pack)
        int rc = gb_filter_into_x(flt->d_blocks, flt->block_offsets, flt->nf, d_anm, E, p->nmax, p->d_x,
                                  simple1 ? nullptr : p->d_ptab_roff, tn, n_coltiles, st);
        if (rc) return rc;
    } else {
        int rc = simple1 ? gb_launch_pack(d_anm, p->d_x, L, E, st, d_wn)
                         : gb_launch_pack_tiled(d_anm, p->d_x, L, E, p->d_ptab_roff, tn, n_coltiles, st, d_wn);
        if (rc) return rc;
    }
    if (prof) GB_CUDA(cudaEventRecord(prof[1], st));
    if (simple1) {
        dim3 grid((p->nlat + S1_TI - 1) / S1_TI, L);
        const size_t smem = (size_t)L * S1_TI * sizeof(double);
        if (smem > 48 * 1024)
            GB_CUDA(cudaFuncSetAttribute(gb_legendre_stage1_simple, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        gb_legendre_stage1_simple<<<grid, 256, smem, st>>>(p->d_x, p->d_ab, p->d_ct, p->d_kn, p->d_pmm, p->d_ra,
                                                           p->d_rb, p->d_rc, d_krow, L, p->nlat, E, p->ab_rows);
        GB_LAUNCH_CHECK();
    } else {
        // the polar caps (parallels whose mirror image is not close enough in the reference's tables) run the unfolded
        // kernel on tiles of 32 northern parallels + their 32 mirror images (kind 1, polar = 1)
        const S1Launch a{p, d_krow, tiling, E, n_coltiles, st};
        const bool pairs = p->nlat % 2 == 0;
        auto stage1 = [&](bool f, int kind, int lattiles, int items, int polar) {
            return have_tab ? dispatch_stage1<S1Source::Table>(a, f, pairs, kind, lattiles, items, polar)
                            : dispatch_stage1<S1Source::Recursion>(a, f, pairs, kind, lattiles, items, polar);
        };
        int rc = stage1(fold, fold ? 0 : 2, n_lattiles, n_items, cap_tiles);
        if (!rc && cap_tiles > 0) rc = stage1(false, 1, cap_tiles, cap_items, 1);
        if (rc) return rc;
    }
    if (prof) GB_CUDA(cudaEventRecord(prof[2], st));
    if (naive2) {
        const long long total = M * p->nlon;
        gb_fourier_stage2_naive<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(p->d_ab, p->ab_rows, p->d_trig, p->nlp,
                                                                                p->kpad, d_out, M, p->nlon);
        GB_LAUNCH_CHECK();
    } else if (use_sym) {
        int rc = gb_launch_stage2_sym(p, p->d_ab, M, d_out, st, true);
        if (rc) return rc;
    } else {
        gbgemm::Shape sh;
        sh.A_t = p->d_ab;
        sh.a_rows = p->ab_rows;
        sh.a_koff_mul = 0;
        sh.tiles_per_group = 1;
        sh.B_t = p->d_trig_t;
        sh.b_rows = p->kpad;
        sh.klen = p->kpad;
        sh.n_mtiles = (int)((M + gbgemm::TM - 1) / gbgemm::TM);
        sh.n_ntiles = p->n_ntiles;
        int rc = gbgemm::launch(sh, RowMajorStore{d_out, M, p->nlon}, p->sm_count, st);
        if (rc) return rc;
    }
    if (prof) {
        GB_CUDA(cudaEventRecord(prof[3], st));
        p->prof_count++;
    }
    return GB_OK;
}

extern "C" int gb_synthesis(gb_plan* plan, const double* d_anm, int n_epochs, double* d_out, void* stream) {
    GB_REQUIRE(plan != nullptr, "gb_synthesis: plan is NULL");
    GB_REQUIRE(n_epochs >= 0, "gb_synthesis: n_epochs=%d is negative", n_epochs);
    if (n_epochs == 0) return GB_OK;
    GB_REQUIRE(d_anm && d_out, "gb_synthesis: NULL device pointer");
    GB_REQUIRE(reinterpret_cast<uintptr_t>(d_out) % 16 == 0, "gb_synthesis: d_out is not 16-byte aligned");
    GB_CUDA(cudaSetDevice(plan->device));
    int rc = gb_plan_ensure_workspace(plan, n_epochs);
    if (rc) return rc;
    return launch_synthesis(plan, d_anm, n_epochs, d_out, static_cast<cudaStream_t>(stream));
}

extern "C" int gb_synthesis_weighted(gb_plan* plan, const double* d_anm, const double* d_wn, int n_epochs, double* d_out,
                                     void* stream) {
    GB_REQUIRE(plan != nullptr, "gb_synthesis_weighted: plan is NULL");
    GB_REQUIRE(n_epochs >= 0, "gb_synthesis_weighted: n_epochs=%d is negative", n_epochs);
    if (n_epochs == 0) return GB_OK;
    GB_REQUIRE(d_anm && d_out && d_wn, "gb_synthesis_weighted: NULL device pointer");
    GB_REQUIRE(reinterpret_cast<uintptr_t>(d_out) % 16 == 0, "gb_synthesis_weighted: d_out is not 16-byte aligned");
    GB_CUDA(cudaSetDevice(plan->device));
    int rc = gb_plan_ensure_workspace(plan, n_epochs);
    if (rc) return rc;
    return launch_synthesis(plan, d_anm, n_epochs, d_out, static_cast<cudaStream_t>(stream), d_wn);
}

extern "C" int gb_synthesis_orderwise_filtered(gb_plan* plan, const double* d_blocks, const int64_t* block_offsets, int nf,
                                               const double* d_anm, int n_epochs, double* d_out, void* stream) {
    GB_REQUIRE(plan != nullptr, "gb_synthesis_orderwise_filtered: plan is NULL");
    GB_REQUIRE(n_epochs >= 0, "gb_synthesis_orderwise_filtered: n_epochs=%d is negative", n_epochs);
    GB_REQUIRE(nf >= plan->nmax, "gb_synthesis_orderwise_filtered: the filter (degree %d) does not reach degree %d", nf,
               plan->nmax);
    if (n_epochs == 0) return GB_OK;
    GB_REQUIRE(d_anm && d_out && d_blocks && block_offsets, "gb_synthesis_orderwise_filtered: NULL pointer");
    GB_REQUIRE(reinterpret_cast<uintptr_t>(d_out) % 16 == 0, "gb_synthesis_orderwise_filtered: d_out is not 16-byte aligned");
    GB_CUDA(cudaSetDevice(plan->device));
    int rc = gb_plan_ensure_workspace(plan, n_epochs);
    if (rc) return rc;
    const SynthesisFilter flt{d_blocks, block_offsets, nf};
    return launch_synthesis(plan, d_anm, n_epochs, d_out, static_cast<cudaStream_t>(stream), nullptr, &flt);
}

static int ensure_pipeline(gb_plan* p) {
    if (!p->s_compute) GB_CUDA(cudaStreamCreateWithFlags(&p->s_compute, cudaStreamNonBlocking));
    if (!p->s_copy) GB_CUDA(cudaStreamCreateWithFlags(&p->s_copy, cudaStreamNonBlocking));
    for (auto& e : p->ev)
        if (!e) GB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    return GB_OK;
}

static int ensure_io(gb_plan* p, size_t in_bytes, size_t out_bytes) {
    if (in_bytes > p->io_in_bytes) {
        GB_CUDA(cudaDeviceSynchronize());
        cudaFree(p->d_io_in);
        p->d_io_in = nullptr; p->io_in_bytes = 0;
        GB_CUDA(cudaMalloc(reinterpret_cast<void**>(&p->d_io_in), in_bytes));
        p->io_in_bytes = in_bytes;
    }
    if (out_bytes > p->io_out_bytes) {
        GB_CUDA(cudaDeviceSynchronize());
        for (int b = 0; b < 2; ++b) {
            cudaFree(p->d_io_out[b]);
            p->d_io_out[b] = nullptr;
        }
        p->io_out_bytes = 0;
        for (int b = 0; b < 2; ++b) GB_CUDA(cudaMalloc(reinterpret_cast<void**>(&p->d_io_out[b]), out_bytes));
        p->io_out_bytes = out_bytes;
    }
    return GB_OK;
}

extern "C" int gb_synthesis_host(gb_plan* plan, const double* h_anm, int n_epochs, double* h_out) {
    GB_REQUIRE(plan != nullptr, "gb_synthesis_host: plan is NULL");
    GB_REQUIRE(n_epochs >= 0, "gb_synthesis_host: n_epochs=%d is negative", n_epochs);
    if (n_epochs == 0) return GB_OK;
    GB_REQUIRE(h_anm && h_out, "gb_synthesis_host: NULL host pointer");
    gb_plan* p = plan;
    GB_CUDA(cudaSetDevice(p->device));
    int rc = ensure_pipeline(p);
    if (rc) return rc;
    const size_t coef = (size_t)p->L * p->L;
    const size_t pts = (size_t)p->nlat * p->nlon;
    // chunk the epochs so that the device->host copy of chunk c overlaps the kernels of chunk c+1
    int chunk = (n_epochs + 15) / 16;
    if (chunk < 1) chunk = 1;
    if ((rc = ensure_io(p, (size_t)n_epochs * coef * sizeof(double), (size_t)chunk * pts * sizeof(double)))) return rc;
    if ((rc = gb_plan_ensure_workspace(p, chunk))) return rc;
    // the coefficients go up chunk by chunk in front of their kernels (1 MB each at config 2): only the first
    // chunk's upload is exposed, the rest hides behind the result copies of the previous chunks
    int c = 0;
    for (int e0 = 0; e0 < n_epochs; e0 += chunk, ++c) {
        const int ne = (n_epochs - e0 < chunk) ? (n_epochs - e0) : chunk;
        const int b = c & 1;
        GB_CUDA(cudaMemcpyAsync(p->d_io_in + (size_t)e0 * coef, h_anm + (size_t)e0 * coef, (size_t)ne * coef * sizeof(double),
                                cudaMemcpyHostToDevice, p->s_compute));
        if (c >= 2) GB_CUDA(cudaStreamWaitEvent(p->s_compute, p->ev[2 + b], 0));  // buffer b drained
        if ((rc = launch_synthesis(p, p->d_io_in + (size_t)e0 * coef, ne, p->d_io_out[b], p->s_compute))) return rc;
        GB_CUDA(cudaEventRecord(p->ev[b], p->s_compute));
        GB_CUDA(cudaStreamWaitEvent(p->s_copy, p->ev[b], 0));
        GB_CUDA(cudaMemcpyAsync(h_out + (size_t)e0 * pts, p->d_io_out[b], (size_t)ne * pts * sizeof(double),
                                cudaMemcpyDeviceToHost, p->s_copy));
        GB_CUDA(cudaEventRecord(p->ev[2 + b], p->s_copy));
    }
    GB_CUDA(cudaStreamSynchronize(p->s_copy));
    GB_CUDA(cudaStreamSynchronize(p->s_compute));
    return GB_OK;
}

#ifdef GB_TRACE
extern "C" int gb_debug_trace(unsigned long long* h_out, int reset) {
    if (reset) {
        void* sym = nullptr;
        GB_CUDA(cudaGetSymbolAddress(&sym, gb_trace_buf));
        GB_CUDA(cudaMemset(sym, 0, sizeof(gb_trace_buf)));
        return GB_OK;
    }
    GB_CUDA(cudaDeviceSynchronize());
    GB_CUDA(cudaMemcpyFromSymbol(h_out, gb_trace_buf, sizeof(gb_trace_buf)));
    return GB_OK;
}
#endif

extern "C" int gb_legendre_table(gb_plan* plan, double* d_out, int scaled, void* stream) {
    GB_REQUIRE(plan != nullptr && d_out != nullptr, "gb_legendre_table: NULL argument");
    GB_CUDA(cudaSetDevice(plan->device));
    const int total = plan->nlat * plan->L;
    GB_CUDA(cudaMemsetAsync(d_out, 0, (size_t)plan->nlat * plan->L * plan->L * sizeof(double),
                            static_cast<cudaStream_t>(stream)));
    gb_legendre_table_kernel<<<(total + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(
        d_out, plan->d_ct, plan->d_kn, plan->d_pmm, plan->d_ra, plan->d_rb, plan->d_rc, plan->L, plan->nlat, scaled);
    GB_LAUNCH_CHECK();
    return GB_OK;
}
