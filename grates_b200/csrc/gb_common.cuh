// Shared declarations of the grates_b200 CUDA library (sm_100a only).
#pragma once
#include <cstdint>
#include <cstdio>
#include <cstdarg>
#include <cstdlib>
#include <cuda_runtime.h>
#include "../../include/grates_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "grates_b200 targets sm_100a (B200) only"
#endif

// ---------------------------------------------------------------------------------------------
// error handling: thread-local message + error code returns (no exceptions cross the C ABI)
// ---------------------------------------------------------------------------------------------
int gb_set_error(int code, const char* fmt, ...);
void gb_count_launch(int n = 1);

#define GB_CUDA(expr)                                                                           \
    do {                                                                                        \
        cudaError_t gb_e_ = (expr);                                                             \
        if (gb_e_ != cudaSuccess)                                                               \
            return gb_set_error(GB_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,                    \
                                cudaGetErrorString(gb_e_), __FILE__, __LINE__);                 \
    } while (0)

#define GB_REQUIRE(cond, ...)                                                                   \
    do {                                                                                        \
        if (!(cond)) return gb_set_error(GB_ERR_ARGUMENT, __VA_ARGS__);                         \
    } while (0)

#define GB_LAUNCH_CHECK()                                                                       \
    do {                                                                                        \
        gb_count_launch();                                                                      \
        GB_CUDA(cudaGetLastError());                                                            \
    } while (0)

// Environment switch `name`: set, non-empty and not starting with '0'.  Read on every call, so that a process (a test)
// can change it between calls.
inline bool gb_env_flag(const char* name) {
    const char* v = getenv(name);
    return v && v[0] && v[0] != '0';
}

// ---------------------------------------------------------------------------------------------
// tiled HBM layouts shared by the synthesis kernels
//   AB   [row tile][spectral row k][GB_LDA]   128 grid rows (e, i) per tile, 4 pad doubles so that a
//        chunk of consecutive k lands in shared memory with one bulk copy AND with the k-rows 4
//        doubles apart modulo 16 (conflict-free DMMA fragment loads)
//   trig [column tile][k][tile width + 4]     same idea for the longitude tables
// ---------------------------------------------------------------------------------------------
constexpr int GB_TM = 128;          // grid rows per AB tile
constexpr int GB_LDA = GB_TM + 4;   // 132
constexpr int GB_S2_TN = 120;       // meridians per tile, general stage 2
constexpr int GB_S2_LDB = GB_S2_TN + 4;
constexpr int GB_Q_TN = 32;         // first-quadrant meridians per tile, symmetric stage 2
constexpr int GB_Q_LDB = GB_Q_TN + 4;
constexpr int GB_T1_TM = 64;        // parallels per stage-1 work item
constexpr int GB_T1_KC = 16;        // degrees per stage-1 pipeline chunk

__host__ __device__ __forceinline__ size_t gb_ab_offset(long long row, int k, int ab_rows) {
    return ((size_t)(row >> 7) * ab_rows + k) * GB_LDA + (size_t)(row & 127);
}

// ---------------------------------------------------------------------------------------------
// plan
// ---------------------------------------------------------------------------------------------
struct gb_plan {
    int device = 0;
    int nmax = 0, L = 0, nlat = 0, nlon = 0;
    int kpad = 0;   // spectral rows of one grid row: k = 2m + {0: cos, 1: sin}, padded to a multiple of 4
    int nlp = 0;    // nlon padded to a multiple of 8
    // tables on the device
    double* d_ct = nullptr;     // [nlat]      cos(theta_i)
    double* d_kn = nullptr;     // [nlat][L]   per-latitude degree factors
    double* d_pmm = nullptr;    // [nlat][L]   sectorial seeds P_mm(theta_i)
    double* d_ra = nullptr;     // [L][L]      recursion coefficient a_nm (utilities.py:52)
    double* d_rb = nullptr;     // [L][L]      recursion coefficient b_nm (utilities.py:54)
    double* d_rc = nullptr;     // [L]         sqrt(2n+1), first off-diagonal (utilities.py:46)
    double* d_trig = nullptr;   // [kpad][nlp] row 2m: cos(m lon_j), row 2m+1: sin(m lon_j)
    // recursion tables of stage 1 (Source Recursion), transposed and zero padded so that the Legendre warps read them
    // coalesced and unguarded: parallels padded to GB_T1_TM, degrees of one order padded to whole GB_T1_KC chunks
    int nlat_pad = 0, lpad = 0;
    double* d_ct_pad = nullptr; // [nlat_pad]
    double* d_kn_t = nullptr;   // [L + GB_T1_KC][nlat_pad]   kn_t[n][i]
    double* d_pmm_t = nullptr;  // [L][nlat_pad]              pmm_t[m][i]
    double* d_rec_a = nullptr;  // [L][lpad]  rec_a[m][n-m]: sqrt(2n+1) at n = m+1 (utilities.py:46), a_nm beyond
    double* d_rec_b = nullptr;  // [L][lpad]  rec_b[m][n-m]: 0 at n = m+1, b_nm beyond
    // four-fold longitude symmetry (meridians symmetric about 0 and invariant under a half turn):
    // spectral rows regrouped as [even-m cos | odd-m cos | even-m sin | odd-m sin], each padded to 4
    int sym = 0;                // 1 if the meridians allow the symmetric stage 2
    int fold_ns = 0;            // 1 if the parallels are symmetric about the equator (folded stage 1)
    int fold_cap = 0;           // leading parallels per hemisphere (0, 32 or 64) that stay with the unfolded stage
    int kpad_s = 0;             // rows of AB in the symmetric layout (incl. 4 dummy rows at the end)
    int grp_off[5] = {0, 0, 0, 0, 0};
    int nq = 0, nqp = 0;        // first-quadrant meridians, padded to a multiple of 8
    int* d_krow_id = nullptr;   // [kpad] k = 2m+cs -> AB row, general layout (identity)
    int* d_krow_sym = nullptr;  // [kpad] k = 2m+cs -> AB row, symmetric layout
    double* d_trig_q = nullptr; // [kpad_s][nqp] first-quadrant trig table in the symmetric row order
    double* d_trig_t = nullptr;   // tiled copy of d_trig:   [n_ntiles][kpad][GB_S2_LDB]
    double* d_trig_q_t = nullptr; // tiled copy of d_trig_q: [n_qtiles][kpad_s][GB_Q_LDB]
    int n_ntiles = 0, n_qtiles = 0;
    // eight-fold longitude symmetry (the first-quadrant meridians are also symmetric about pi/4): spectral rows grouped by
    // order mod 4 as [CE0 | CE2 | SE0 | SE2 | CO | SO], each padded to 4; two first-OCTANT tables (gb_synthesis.cu)
    int oct = 0;                // 1 if the octant stage 2 is usable
    int no = 0;                 // first-octant meridians (nlon / 8)
    int kpad_o = 0;             // rows of AB in the octant layout (incl. 4 dummy rows at the end)
    int ogrp_off[7] = {0, 0, 0, 0, 0, 0, 0};
    int* d_krow_oct = nullptr;  // [kpad] k = 2m+cs -> AB row, octant layout
    double* d_trig_o_t = nullptr; // [n_otiles][2 tables][kpad_o][GB_Q_LDB]
    int n_otiles = 0;
    int ab_rows = 0;            // spectral rows allocated per AB tile = max(kpad, kpad_s, kpad_o)
    // synthesis workspace, grown on demand (epochs)
    int ws_epochs = 0;
    long long ws_mpad = 0;
    double* d_x = nullptr;      // packed coefficients: tiled for stage 1 (gb_launch_pack_tiled), order-wise for the FMA
                                // cross-check (gb_launch_pack), see gb_synthesis.cu
    double* d_ab = nullptr;     // [mpad/128][ab_rows][GB_LDA] spectral intermediate (see above)
    // host-buffer pipeline
    cudaStream_t s_compute = nullptr, s_copy = nullptr;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    double* d_io_in = nullptr;  size_t io_in_bytes = 0;
    double* d_io_out[2] = {nullptr, nullptr}; size_t io_out_bytes = 0;
    // analysis
    int ana_nmin = -1;
    double* d_lon_ops = nullptr;     // [kpad][nlp]
    double* d_lat_ops = nullptr;
    long long* d_lat_off = nullptr;  // [L+1]
    long long* h_lat_off = nullptr;
    // longitude stage on the tensor cores: nsets = 4 folded inputs (four-fold symmetric meridians and
    // weights) or 1 (plain transpose); operator tiles [nsets*tiles_per_set][ana_kp][GB_S2_LDB]
    int ana_nsets = 0, ana_kp = 0, ana_tps = 0;
    int ana_ni = 5;                  // 8-column fragments per warp in the longitude GEMM (column tile = 24 * ana_ni)
    double* d_ana_w_t = nullptr;
    int* d_ana_kmap = nullptr;       // [nsets*tiles_per_set*GB_S2_TN] output column -> spectral row 2m+cs, or -1
    double* d_ana_vf = nullptr;      // folded / transposed input tiles (grow-only workspace)
    size_t ana_vf_elems = 0;
    // latitude stage on the tensor cores: per-order operators as A tiles [row tile][parallel][GB_LDA]
    int ana_lat_tiles = 0, ana_nlat_p4 = 0;
    double* d_ana_lat_t = nullptr;
    int* d_ana_lat_m = nullptr;      // [ana_lat_tiles] order of each row tile
    int* d_ana_lat_n = nullptr;      // [ana_lat_tiles] degree of the tile's first row
    void* cov_layout = nullptr;      // index tables of the last covariance propagation (owned by gb_covprop.cu)
    double* d_ana_gt = nullptr;      // longitude-stage output as B tiles [order][column tile][parallel][GB_S2_LDB]
    size_t ana_gt_elems = 0;
    int ana_gt_epochs = -1;          // epoch count the buffer was last cleared for (its tiling depends on it)
    // optional per-kernel event timing (gb_plan_set_profiling)
    cudaEvent_t* prof_ev = nullptr;  // [capacity][4]
    int prof_capacity = 0, prof_count = 0;
    // Legendre tables of stage 1: kn[i,n] * P_nm(theta_i), written once per plan by the bit-exact device recursion
    // (gb_synthesis.cu) in the tile layout the stage-1 kernel bulk-copies: [lat tile][order m: rows roff[m]..][pitch].
    // kind 0: folded tiles (32 northern parallels, pitch 36, even/odd degrees grouped), 1: polar-cap tiles
    // (32 northern + 32 mirrored parallels, pitch 68), 2: plain tiles of 64 parallels (pitch 68)
    double* d_ptab[3] = {nullptr, nullptr, nullptr};
    int* d_ptab_roff = nullptr;      // [L + 1] first table row of every order (orders padded to 8 rows)
    long long ptab_rtot = 0;         // rows per lat tile
    int ptab_state[3] = {0, 0, 0};   // 0: not built yet, 1: built, -1: over the budget or no memory (recursion instead)
    long long x_layout_key = 0;      // (epochs, tile width) d_x was last cleared for; 0: order-wise layout / unknown
    size_t x_elems = 0;              // doubles allocated in d_x
    // stream ordering of the shared workspace (d_x, d_ab, analysis / covariance scratch, cached index tables): a call
    // on another stream than the previous call's first waits for everything that stream holds (gb_plan_acquire)
    cudaEvent_t ws_free = nullptr;
    cudaStream_t ws_stream = nullptr;
    int ws_used = 0;
    // device facts
    int sm_count = 0;
};

// The plan's workspace is one buffer set: make `st` wait until the previous call that used it (on whatever stream) is
// done.  Free when consecutive calls share a stream.  Host threads must not call into one plan concurrently.
int gb_plan_acquire(gb_plan* p, cudaStream_t st);

int gb_plan_ensure_workspace(gb_plan* p, int n_epochs);
void gb_cov_layout_free(gb_plan* p);
// the library's own stream-ordered memory pool of `device` (gb_plan.cu); nullptr if it cannot be created
cudaMemPool_t gb_scratch_pool(int device);
void gb_retain_pool_memory(int device);   // makes sure the pool exists

// anm [E][L][L] <-> order-wise packed X (gb_pack.cu): block of order m at 2E (m L - m(m-1)/2),
// X_m[n - m][cs * E + e]
int gb_launch_pack(const double* d_anm, double* d_x, int L, int E, cudaStream_t st, const double* d_wn = nullptr);
int gb_launch_unpack(const double* d_x, double* d_anm, int L, int E, cudaStream_t st);
// anm -> X in the tiled layout of the table-fed stage 1: [order][column tile of tn][degree row][tn + 4] (gb_pack.cu);
// d_roff [L + 1] = first row of every order (gb_plan::d_ptab_roff).  The buffer must have been cleared for this layout.
int gb_launch_pack_tiled(const double* d_anm, double* d_x, int L, int E, const int* d_roff, int tn, int n_ct,
                         cudaStream_t st, const double* d_wn = nullptr);
// symmetric Fourier stage of the synthesis on rows [0, M) of an AB-layout operand (gb_synthesis.cu); needs p->sym.
// pdl: launched with programmatic dependent launch (the kernel may start while its predecessor drains)
int gb_launch_stage2_sym(gb_plan* p, const double* d_ab, long long M, double* d_out, cudaStream_t st, bool pdl);
const int* gb_stage2_krow(const gb_plan* p);    // spectral row 2m + cs -> row of that stage's AB layout
// order-wise block filter of a batch, written straight into a synthesis workspace X (gb_filter.cu): order-wise packed
// (d_roff == nullptr) or the tiled layout of gb_launch_pack_tiled (the buffer must have been cleared for it)
int gb_filter_into_x(const double* d_blocks, const int64_t* block_offsets, int nf, const double* d_anm, int E, int nmax,
                     double* d_x, const int* d_roff, int tn, int n_ct, cudaStream_t st);
// packed batch -> degree-wise vectors as GEMM B tiles [epoch tile of 120][c][124] (gb_densefilter.cu); K = number of
// coefficients from degree nmin on, kp4 = K padded to 4, degrees above Lin - 1 read as zero
int gb_launch_ravel_tiles(const double* d_anm, double* d_bt, int Lin, int nmin, long long K, int kp4, int E, cudaStream_t st);

// Stream-ordered scratch memory of one C-ABI call: everything allocated through it is returned to the pool
// (cudaFreeAsync on the same stream) when the call leaves, on every path including the error returns.
struct gb_scratch {
    cudaStream_t st;
    void* ptrs[24];
    int n = 0;
    explicit gb_scratch(cudaStream_t s) : st(s) {}
    gb_scratch(const gb_scratch&) = delete;
    gb_scratch& operator=(const gb_scratch&) = delete;
    ~gb_scratch() {
        for (int i = n - 1; i >= 0; --i) cudaFreeAsync(ptrs[i], st);
    }
    template <typename T>
    cudaError_t alloc(T** out, size_t count) {
        *out = nullptr;
        if (n >= 24) return cudaErrorMemoryAllocation;
        void* p = nullptr;
        int dev = 0;
        cudaGetDevice(&dev);
        cudaMemPool_t pool = gb_scratch_pool(dev);
        cudaError_t e = pool ? cudaMallocFromPoolAsync(&p, (count ? count : 1) * sizeof(T), pool, st)
                             : cudaMallocAsync(&p, (count ? count : 1) * sizeof(T), st);
        if (e == cudaSuccess) {
            ptrs[n++] = p;
            *out = static_cast<T*>(p);
        }
        return e;
    }
};

// Kernel launch with the programmatic-stream-serialization attribute (PDL).
#ifdef __CUDACC__
#include <utility>
template <typename... KArgs, typename... Args>
inline cudaError_t gb_launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                 Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(std::forward<Args>(args))...);
}
#endif

// Recursion coefficients a_nm, b_nm [L][L], sqrt(2n+1) [L] and sectorial seeds P_mm [npts][L],
// evaluated in IEEE double in the operation order of reference utilities.py:37-54.
#include <vector>
void gb_recursion_tables(int nmax, int npts, const double* sin_theta, std::vector<double>& ra,
                         std::vector<double>& rb, std::vector<double>& rc, std::vector<double>& pmm);

// ---------------------------------------------------------------------------------------------
// PTX helpers (device)
// ---------------------------------------------------------------------------------------------
#ifdef __CUDACC__
namespace gb {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// D(8x8) += A(8x4, row) * B(4x8, col); FP64 tensor op, SASS DMMA.8x8x4
__device__ __forceinline__ void dmma_884(double& d0, double& d1, double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(d0), "+d"(d1)
                 : "d"(a), "d"(b));
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// 1-D bulk copy global -> shared through the TMA unit (SASS UBLKCP); completes on an mbarrier.
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// Fully normalised Legendre functions of one (point, order): calls f(n, P_nm) for n = m..L-1.
// Forward column recursion of reference utilities.py:37-54 with unfused multiplies / subtract in numpy's evaluation
// order, so that the values are bit-identical to the reference table (seed P_mm from the plan, a/b/sqrt(2n+1) tables).
template <typename F>
__device__ __forceinline__ void legendre_column(int m, int L, double ct, double pmm, const double* __restrict__ ra,
                                                const double* __restrict__ rb, const double* __restrict__ rc, F&& f) {
    double p2 = pmm;  // P_mm
    f(m, p2);
    if (m + 1 >= L) return;
    double p1 = __dmul_rn(__dmul_rn(rc[m + 1], ct), p2);  // P_{m+1,m} = sqrt(2n+1) * cos * P_mm
    f(m + 1, p1);
    for (int n = m + 2; n < L; ++n) {
        const double p = __dsub_rn(__dmul_rn(__dmul_rn(ra[(size_t)n * L + m], ct), p1),
                                   __dmul_rn(rb[(size_t)n * L + m], p2));
        f(n, p);
        p2 = p1;
        p1 = p;
    }
}

// Tensor memory (256 KB per SM, otherwise unused by FP64 kernels) as a thread-private spill area for accumulators:
// the 32x32b shape gives lane l of warp w its own TMEM lane 32 (w % 4) + l, `x32` = 32 consecutive 32-bit columns
// = 16 doubles (SASS STTM.x32 / LDTM.x32).  Used to take finished accumulator tiles out of the registers so that
// their epilogue can be spread over the next tile's K loop.
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {   // one whole warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(smem_result)), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {        // the warp that allocated
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tmem_fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory"); }
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const double (&v)[16]) {
    asm volatile(
        "{\n.reg .b32 l<16>, h<16>;\n"
        "mov.b64 {l0,h0}, %1; mov.b64 {l1,h1}, %2; mov.b64 {l2,h2}, %3; mov.b64 {l3,h3}, %4;\n"
        "mov.b64 {l4,h4}, %5; mov.b64 {l5,h5}, %6; mov.b64 {l6,h6}, %7; mov.b64 {l7,h7}, %8;\n"
        "mov.b64 {l8,h8}, %9; mov.b64 {l9,h9}, %10; mov.b64 {l10,h10}, %11; mov.b64 {l11,h11}, %12;\n"
        "mov.b64 {l12,h12}, %13; mov.b64 {l13,h13}, %14; mov.b64 {l14,h14}, %15; mov.b64 {l15,h15}, %16;\n"
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {l0,h0,l1,h1,l2,h2,l3,h3,l4,h4,l5,h5,l6,h6,l7,h7,"
        "l8,h8,l9,h9,l10,h10,l11,h11,l12,h12,l13,h13,l14,h14,l15,h15};\n}\n" ::"r"(taddr),
        "d"(v[0]), "d"(v[1]), "d"(v[2]), "d"(v[3]), "d"(v[4]), "d"(v[5]), "d"(v[6]), "d"(v[7]), "d"(v[8]), "d"(v[9]),
        "d"(v[10]), "d"(v[11]), "d"(v[12]), "d"(v[13]), "d"(v[14]), "d"(v[15])
        : "memory");
}
// load + wait: the values are valid when this returns
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, double (&v)[16]) {
    asm volatile(
        "{\n.reg .b32 l<16>, h<16>;\n"
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {l0,h0,l1,h1,l2,h2,l3,h3,l4,h4,l5,h5,l6,h6,l7,h7,"
        "l8,h8,l9,h9,l10,h10,l11,h11,l12,h12,l13,h13,l14,h14,l15,h15}, [%16];\n"
        "tcgen05.wait::ld.sync.aligned;\n"
        "mov.b64 %0, {l0,h0}; mov.b64 %1, {l1,h1}; mov.b64 %2, {l2,h2}; mov.b64 %3, {l3,h3};\n"
        "mov.b64 %4, {l4,h4}; mov.b64 %5, {l5,h5}; mov.b64 %6, {l6,h6}; mov.b64 %7, {l7,h7};\n"
        "mov.b64 %8, {l8,h8}; mov.b64 %9, {l9,h9}; mov.b64 %10, {l10,h10}; mov.b64 %11, {l11,h11};\n"
        "mov.b64 %12, {l12,h12}; mov.b64 %13, {l13,h13}; mov.b64 %14, {l14,h14}; mov.b64 %15, {l15,h15};\n}\n"
        : "=d"(v[0]), "=d"(v[1]), "=d"(v[2]), "=d"(v[3]), "=d"(v[4]), "=d"(v[5]), "=d"(v[6]), "=d"(v[7]), "=d"(v[8]),
          "=d"(v[9]), "=d"(v[10]), "=d"(v[11]), "=d"(v[12]), "=d"(v[13]), "=d"(v[14]), "=d"(v[15])
        : "r"(taddr)
        : "memory");
}

// The same thread-private tensor-memory access for 2 / 4 / 8 doubles (.x4 / .x8 / .x16); loads wait.
__device__ __forceinline__ void tmem_st2(uint32_t taddr, double a, double b) {
    asm volatile(
        "{\n.reg .b32 l<2>, h<2>;\nmov.b64 {l0,h0}, %1; mov.b64 {l1,h1}, %2;\n"
        "tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {l0,h0,l1,h1};\n}\n" ::"r"(taddr), "d"(a), "d"(b)
        : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const double* v) {
    asm volatile(
        "{\n.reg .b32 l<4>, h<4>;\nmov.b64 {l0,h0}, %1; mov.b64 {l1,h1}, %2; mov.b64 {l2,h2}, %3; mov.b64 {l3,h3}, %4;\n"
        "tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {l0,h0,l1,h1,l2,h2,l3,h3};\n}\n" ::"r"(taddr), "d"(v[0]), "d"(v[1]),
        "d"(v[2]), "d"(v[3])
        : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const double* v) {
    asm volatile(
        "{\n.reg .b32 l<8>, h<8>;\n"
        "mov.b64 {l0,h0}, %1; mov.b64 {l1,h1}, %2; mov.b64 {l2,h2}, %3; mov.b64 {l3,h3}, %4;\n"
        "mov.b64 {l4,h4}, %5; mov.b64 {l5,h5}, %6; mov.b64 {l6,h6}, %7; mov.b64 {l7,h7}, %8;\n"
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {l0,h0,l1,h1,l2,h2,l3,h3,l4,h4,l5,h5,l6,h6,l7,h7};\n}\n" ::"r"(taddr),
        "d"(v[0]), "d"(v[1]), "d"(v[2]), "d"(v[3]), "d"(v[4]), "d"(v[5]), "d"(v[6]), "d"(v[7])
        : "memory");
}
__device__ __forceinline__ void tmem_ld2(uint32_t taddr, double* v) {
    asm volatile(
        "{\n.reg .b32 l<2>, h<2>;\n"
        "tcgen05.ld.sync.aligned.32x32b.x4.b32 {l0,h0,l1,h1}, [%2];\n"
        "tcgen05.wait::ld.sync.aligned;\n"
        "mov.b64 %0, {l0,h0}; mov.b64 %1, {l1,h1};\n}\n"
        : "=d"(v[0]), "=d"(v[1])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, double* v) {
    asm volatile(
        "{\n.reg .b32 l<4>, h<4>;\n"
        "tcgen05.ld.sync.aligned.32x32b.x8.b32 {l0,h0,l1,h1,l2,h2,l3,h3}, [%4];\n"
        "tcgen05.wait::ld.sync.aligned;\n"
        "mov.b64 %0, {l0,h0}; mov.b64 %1, {l1,h1}; mov.b64 %2, {l2,h2}; mov.b64 %3, {l3,h3};\n}\n"
        : "=d"(v[0]), "=d"(v[1]), "=d"(v[2]), "=d"(v[3])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, double* v) {
    asm volatile(
        "{\n.reg .b32 l<8>, h<8>;\n"
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {l0,h0,l1,h1,l2,h2,l3,h3,l4,h4,l5,h5,l6,h6,l7,h7}, [%8];\n"
        "tcgen05.wait::ld.sync.aligned;\n"
        "mov.b64 %0, {l0,h0}; mov.b64 %1, {l1,h1}; mov.b64 %2, {l2,h2}; mov.b64 %3, {l3,h3};\n"
        "mov.b64 %4, {l4,h4}; mov.b64 %5, {l5,h5}; mov.b64 %6, {l6,h6}; mov.b64 %7, {l7,h7};\n}\n"
        : "=d"(v[0]), "=d"(v[1]), "=d"(v[2]), "=d"(v[3]), "=d"(v[4]), "=d"(v[5]), "=d"(v[6]), "=d"(v[7])
        : "r"(taddr)
        : "memory");
}
// N doubles (N even, <= 10) at 32-bit column `taddr`
template <int N>
__device__ __forceinline__ void tmem_st_n(uint32_t taddr, const double* v) {
    static_assert(N == 6 || N == 8 || N == 10, "unsupported row-factor width");
    if constexpr (N == 6) { tmem_st4(taddr, v); tmem_st2(taddr + 8, v[4], v[5]); }
    if constexpr (N == 8) tmem_st8(taddr, v);
    if constexpr (N == 10) { tmem_st8(taddr, v); tmem_st2(taddr + 16, v[8], v[9]); }
}
template <int N>
__device__ __forceinline__ void tmem_ld_n(uint32_t taddr, double* v) {
    static_assert(N == 6 || N == 8 || N == 10, "unsupported row-factor width");
    if constexpr (N == 6) { tmem_ld4(taddr, v); tmem_ld2(taddr + 8, v + 4); }
    if constexpr (N == 8) tmem_ld8(taddr, v);
    if constexpr (N == 10) { tmem_ld8(taddr, v); tmem_ld2(taddr + 16, v + 8); }
}

// Programmatic dependent launch: a kernel launched with gb_launch_pdl may start while its predecessor in the stream
// drains; everything it reads or writes that the predecessor (or anything before it) touches comes after griddep_wait().
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;\n" ::: "memory"); }
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory"); }

// Read-only load that stays where it is written (volatile asm keeps its place among the barrier waits): issued at the top
// of a K loop, its latency is over by the epilogue.  A plain __ldg is sunk by the compiler to its first use.
__device__ __forceinline__ int ld_nc_early(const int* p) {
    int v;
    asm volatile("ld.global.nc.s32 %0, [%1];\n" : "=r"(v) : "l"(p));
    return v;
}

__device__ __forceinline__ void st_cs_v2(double* p, double a, double b) {
    asm volatile("st.global.cs.v2.f64 [%0], {%1, %2};\n" ::"l"(p), "d"(a), "d"(b) : "memory");
}
__device__ __forceinline__ void st_v2(double* p, double a, double b) {
    asm volatile("st.global.v2.f64 [%0], {%1, %2};\n" ::"l"(p), "d"(a), "d"(b) : "memory");
}
// 32-byte store; p must be 32-byte aligned
__device__ __forceinline__ void st_v4(double* p, double a, double b, double c, double d) {
    asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};\n" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
}
// 32-byte streaming store (SASS STG.E.EF.256, sm_100); p must be 32-byte aligned
__device__ __forceinline__ void st_cs_v4(double* p, double a, double b, double c, double d) {
    asm volatile("st.global.cs.v4.f64 [%0], {%1, %2, %3, %4};\n" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
}
__device__ __forceinline__ void st_cs(double* p, double a) {
    asm volatile("st.global.cs.f64 [%0], %1;\n" ::"l"(p), "d"(a) : "memory");
}

}  // namespace gb
#endif
