// Persistent FP64 tensor-core GEMM building block (sm_100a).  Users: synthesis stage 2 (direct path), both analysis
// stages (longitude and latitude), the dense filter, the covariance longitude form of grids without four-fold symmetric
// meridians, and at arbitrary points the synthesis, the adjoint, the covariance diag(F Sigma F') and the normal
// equations J'WJ of the acceleration (upper_only: the tiles of the upper triangle only).
//
//   C[row, col] = sum_k A[k, row] * B[k, col]
//
// Operands live in HBM in the tiled + padded layouts of gb_common.cuh:
//   A_t [row tile][k][GB_LDA]        (128 rows + 4 pad doubles per k)
//   B_t [col tile][k][GB_S2_LDB]     (120 cols + 4 pad doubles per k)
// so that every pipeline chunk (28 consecutive k) is ONE contiguous cp.async.bulk per operand and
// lands in shared memory with k-rows 4 doubles apart modulo 16 (conflict-free DMMA.8x8x4 fragments).
//
// CTA: 12 consumer warps (4 x 3, 32 x 40 register tiles, 20 DMMA per k4 step) + 1 producer warp
// (one elected lane), 3-stage mbarrier pipeline, static round-robin tile schedule over <= #SM CTAs.
// The column tiles may be partitioned into groups that read different k ranges of A
// (a_koff = (col tile / tiles_per_group) * a_koff_mul): the analysis uses this for its four folded
// inputs.  The epilogue functor receives accumulator pairs (row, col, col+1); an epilogue that
// declares `static constexpr bool whole_tile = true` gets the warp's 32 x 40 register tile at once
// (`tile(row_base, col_base, acc)`, rows row_base + 8 mi, columns col_base + 8 ni + {0, 1}) so that it
// can reduce inside the thread before it touches shuffles or atomics; its `prepare(row_base, nt, col_base)`
// runs before the K loop (index look-ups and prefetches whose latency then hides behind the tile's DMMAs)
// and its result is handed back to `tile`.
#pragma once
#include <type_traits>
#include "gb_common.cuh"

namespace gbgemm {

constexpr int WM = 4, WN = 3;
constexpr int TM = 32 * WM;   // 128
constexpr int TN = 40 * WN;   // 120 (default column tile; narrower tiles: NI < 5 fragments per warp, TN = 24 NI)
constexpr int KC = 28;
constexpr int STAGES = 3;
constexpr int LDA = GB_LDA;
constexpr int LDB = GB_S2_LDB;
constexpr int CONSUMER_WARPS = WM * WN;
constexpr int THREADS = 32 * (CONSUMER_WARPS + 1);
static_assert(TM == GB_TM && TN == GB_S2_TN, "tile shape must match the tiled HBM layouts");
// column tile of NI 8-column fragments per warp: width, pitch (= 4 mod 16 for every NI), stage size
__host__ __device__ constexpr int tile_n(int ni) { return 8 * ni * WN; }
__host__ __device__ constexpr int tile_ldb(int ni) { return tile_n(ni) + 4; }
__host__ __device__ constexpr size_t smem_bytes(int ni) {
    return (size_t)STAGES * KC * (LDA + tile_ldb(ni)) * sizeof(double) + 2 * STAGES * sizeof(uint64_t);
}

struct Shape {
    const double* A_t;      // [n_mtiles][a_rows][LDA]
    int a_rows;             // k rows allocated per A tile
    int a_koff_mul;         // see above
    int tiles_per_group;    // column tiles per group (>= 1)
    const double* B_t;      // [n_ntiles][b_rows][LDB]
    int b_rows;             // k rows per B tile
    int klen;               // contraction length (multiple of 4), k = 0..klen-1 of B, a_koff.. of A
    int n_mtiles, n_ntiles;
    int mt_kstart_mod = 0, mt_kstart_mul = 0;   // optional: row tile mt starts its contraction at k = (mt % mod) * mul
                                        // (operand rows below are known zeros: triangular A blocks)
    const int* mt_bgroup = nullptr;     // optional: row tile mt multiplies B tile mt_bgroup[mt] * n_ntiles + nt
                                        // (block-diagonal batches: the analysis latitude stage, one group per order)
    bool upper_only = false;            // optional: tiles whose columns all lie below their first row (col < row
                                        // everywhere) are skipped -- the upper triangle of a symmetric product
};

// the tile (mt, nt) of a column tile width tn holds no entry with col >= row
__host__ __device__ __forceinline__ bool below_diagonal(const Shape& sh, int mt, int nt, int tn) {
    return sh.upper_only && (long long)(nt + 1) * tn <= (long long)mt * TM;
}

template <class E, class = void>
struct wants_whole_tile { static constexpr bool value = false; };
template <class E>
struct wants_whole_tile<E, std::enable_if_t<E::whole_tile>> { static constexpr bool value = true; };

template <class Epilogue, int NI = 5>
__global__ void __launch_bounds__(THREADS, 1) kernel(Shape sh, Epilogue epi) {
    constexpr int TN = tile_n(NI), LDB = tile_ldb(NI), STAGE_DOUBLES = KC * (LDA + LDB);
    extern __shared__ __align__(128) unsigned char s_raw[];
    double* s_tiles = reinterpret_cast<double*>(s_raw);
    uint64_t* full = reinterpret_cast<uint64_t*>(s_raw + (size_t)STAGES * STAGE_DOUBLES * sizeof(double));
    uint64_t* empty = full + STAGES;
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            gb::mbar_init(&full[s], 1);
            gb::mbar_init(&empty[s], CONSUMER_WARPS);
        }
        gb::fence_mbar_init();
    }
    __syncthreads();

    // tiles t = mt * n_ntiles + nt are walked with stride gridDim.x; (mt, nt) advance incrementally (a 64-bit
    // division per tile costs the single producer thread, and every consumer warp, hundreds of dependent cycles)
    const int step_m = (int)(gridDim.x / sh.n_ntiles), step_n = (int)(gridDim.x % sh.n_ntiles);
    int mt = (int)(blockIdx.x / sh.n_ntiles), nt = (int)(blockIdx.x % sh.n_ntiles);
    int stage = 0;
    uint32_t phase = 0;

    if (warp == CONSUMER_WARPS) {
        if (lane == 0) {
            for (; mt < sh.n_mtiles; mt += step_m, nt += step_n) {
                if (nt >= sh.n_ntiles) { nt -= sh.n_ntiles; ++mt; if (mt >= sh.n_mtiles) break; }
                if (below_diagonal(sh, mt, nt, TN)) continue;
                const int a_koff = (nt / sh.tiles_per_group) * sh.a_koff_mul;
                const int kstart = sh.mt_kstart_mod ? (mt % sh.mt_kstart_mod) * sh.mt_kstart_mul : 0;
                for (int k0 = kstart; k0 < sh.klen; k0 += KC) {
                    const int kc = min(KC, sh.klen - k0);
                    gb::mbar_wait(&empty[stage], phase ^ 1u);
                    double* sA = s_tiles + (size_t)stage * STAGE_DOUBLES;
                    double* sB = sA + KC * LDA;
                    const uint32_t bytes_a = (uint32_t)(kc * LDA * sizeof(double));
                    const uint32_t bytes_b = (uint32_t)(kc * LDB * sizeof(double));
                    gb::mbar_arrive_expect_tx(&full[stage], bytes_a + bytes_b);
                    gb::bulk_g2s(sA, sh.A_t + ((size_t)mt * sh.a_rows + a_koff + k0) * LDA, bytes_a, &full[stage]);
                    const size_t bt = sh.mt_bgroup ? (size_t)sh.mt_bgroup[mt] * sh.n_ntiles + nt : (size_t)nt;
                    gb::bulk_g2s(sB, sh.B_t + (bt * sh.b_rows + k0) * LDB, bytes_b, &full[stage]);
                    if (++stage == STAGES) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else {
        const int wm = warp / WN;
        const int wn = warp % WN;
        const int g = lane >> 2;
        const int q = lane & 3;
        for (; mt < sh.n_mtiles; mt += step_m, nt += step_n) {
            if (nt >= sh.n_ntiles) { nt -= sh.n_ntiles; ++mt; if (mt >= sh.n_mtiles) break; }
            if (below_diagonal(sh, mt, nt, TN)) continue;
            double acc[4][NI][2];
#pragma unroll
            for (int mi = 0; mi < 4; ++mi)
#pragma unroll
                for (int ni = 0; ni < NI; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
            const long long row_base = (long long)mt * TM + wm * 32 + g;
            const int col_base = nt * TN + wn * (8 * NI) + 2 * q;
            auto pre = [&] {
                if constexpr (wants_whole_tile<Epilogue>::value) return epi.prepare(row_base, nt, col_base);
                else return 0;
            }();
            const int kstart = sh.mt_kstart_mod ? (mt % sh.mt_kstart_mod) * sh.mt_kstart_mul : 0;
            for (int k0 = kstart; k0 < sh.klen; k0 += KC) {
                const int kc = min(KC, sh.klen - k0);
                gb::mbar_wait(&full[stage], phase);
                const double* sA = s_tiles + (size_t)stage * STAGE_DOUBLES + wm * 32 + g;
                const double* sB = s_tiles + (size_t)stage * STAGE_DOUBLES + KC * LDA + wn * (8 * NI) + g;
#pragma unroll
                for (int kk = 0; kk < KC; kk += 4) {
                    if (kk >= kc) break;
                    double a[4], b[NI];
#pragma unroll
                    for (int mi = 0; mi < 4; ++mi) a[mi] = sA[(kk + q) * LDA + mi * 8];
#pragma unroll
                    for (int ni = 0; ni < NI; ++ni) b[ni] = sB[(kk + q) * LDB + ni * 8];
#pragma unroll
                    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
                        for (int ni = 0; ni < NI; ++ni) gb::dmma_884(acc[mi][ni][0], acc[mi][ni][1], a[mi], b[ni]);
                }
                __syncwarp();
                if (lane == 0) gb::mbar_arrive(&empty[stage]);
                if (++stage == STAGES) { stage = 0; phase ^= 1u; }
            }
            if constexpr (wants_whole_tile<Epilogue>::value) {
                epi.tile(pre, row_base, col_base, acc);
            } else {
                (void)pre;
#pragma unroll
                for (int mi = 0; mi < 4; ++mi)
#pragma unroll
                    for (int ni = 0; ni < NI; ++ni)
                        epi(row_base + mi * 8, col_base + ni * 8, acc[mi][ni][0], acc[mi][ni][1]);
            }
        }
    }
}

template <class Epilogue, int NI = 5>
inline int launch(const Shape& sh, const Epilogue& epi, int sm_count, cudaStream_t st) {
    const long long n_tiles = (long long)sh.n_mtiles * sh.n_ntiles;
    if (n_tiles == 0) return GB_OK;
    const int grid = (int)(n_tiles < sm_count ? n_tiles : sm_count);
    constexpr size_t SMEM = smem_bytes(NI);
    GB_CUDA(cudaFuncSetAttribute(kernel<Epilogue, NI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
    kernel<Epilogue, NI><<<grid, THREADS, SMEM, st>>>(sh, epi);
    GB_LAUNCH_CHECK();
    return GB_OK;
}

// degree-wise index c (counted from degree 0; reference utilities.py:310-360) -> position in the packed [L][L] array
__device__ __forceinline__ void degreewise_position(long long c, int& row, int& col, int& degree) {
    int n = (int)floor(sqrt((double)c));
    if ((long long)n * n > c) --n;
    if ((long long)(n + 1) * (n + 1) <= c) ++n;
    const int j = (int)(c - (long long)n * n);             // 0: C_n0, 2m-1: C_nm, 2m: S_nm
    const int m = (j + 1) >> 1;
    const bool sine = j > 0 && (j & 1) == 0;
    row = sine ? m - 1 : n;
    col = sine ? n : m;
    degree = n;
}

// Epilogue: GEMM rows are degree-wise coefficient indices (from nmin^2), columns epochs; scatter into packed
// out[e][Lout][Lout].  ACCUMULATE adds to what is there (K loop split over several launches on one stream).
template <bool ACCUMULATE>
struct UnravelStore {
    static constexpr bool whole_tile = true;
    double* out;
    long long K;
    int nmin, Lout, E;
    struct Pre { int pos[4]; };          // packed position of the thread's four rows, -1: not stored
    __device__ __forceinline__ Pre prepare(long long row_base, int, int) const {
        Pre pr;
#pragma unroll
        for (int mi = 0; mi < 4; ++mi) {
            const long long r = row_base + mi * 8;
            pr.pos[mi] = -1;
            if (r < K) {
                int row, col, n;
                degreewise_position(r + (long long)nmin * nmin, row, col, n);
                if (n < Lout) pr.pos[mi] = row * Lout + col;
            }
        }
        return pr;
    }
    template <int NI>
    __device__ __forceinline__ void tile(const Pre& pr, long long, int col_base, double (&acc)[4][NI][2]) const {
#pragma unroll
        for (int ni = 0; ni < NI; ++ni)
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const int e = col_base + ni * 8 + r;
                if (e >= E) continue;
                double* o = out + (size_t)e * Lout * Lout;
#pragma unroll
                for (int mi = 0; mi < 4; ++mi)
                    if (pr.pos[mi] >= 0) {
                        if (ACCUMULATE) o[pr.pos[mi]] += acc[mi][ni][r];
                        else o[pr.pos[mi]] = acc[mi][ni][r];
                    }
            }
    }
};

}  // namespace gbgemm

