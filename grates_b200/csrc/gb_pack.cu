// Order-wise packing of epoch batches of potential coefficients (HBM-bound transposes).
//
//   anm [E][L][L]   reference layout (gravityfield.py:149-159): C_nm = anm[n][m], S_nm = anm[m-1][n]
//   X               order-wise: the block of order m starts at 2E (m L - m(m-1)/2) and is
//                   X_m[n - m][cs * E + e], cs = 0 (cos) / 1 (sin), epochs contiguous
//
// Row r of anm[e] holds C_{r,0..r} followed by S_{r+1, r+1..nmax}; one CTA moves that row for 32 (8 for small
// shards) epochs through shared memory, so both sides are touched in full contiguous lines: reads are
// rows of L doubles, writes are 32 consecutive epochs (256 B).  The sine plane of order 0 does not
// exist in anm and is kept at zero (stage 1 contracts it like any other column).  Optional per-degree
// weights w[n] (Gaussian / Butterworth filters, reference filter.py:31-130) are multiplied in while
// packing: element (r, c) of anm has degree max(r, c).
#include "gb_common.cuh"

#ifdef GB_TRACE
// development aid (-DGB_TRACE): timeline of the pack kernel, read back with gb_debug_trace_pack
__device__ unsigned long long gb_trace_pack[512][4];
#define GB_PACK_MARK(slot)                                                                          \
    do {                                                                                            \
        const unsigned cta_ = blockIdx.x + gridDim.x * blockIdx.y;                                  \
        if (threadIdx.x == 0 && cta_ < 512) {                                                       \
            unsigned long long gt_;                                                                 \
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt_));                                  \
            gb_trace_pack[cta_][slot] = gt_;                                                        \
        }                                                                                           \
    } while (0)
#else
#define GB_PACK_MARK(slot) ((void)0)
#endif

namespace {

constexpr int PK_C = 512;         // columns of anm per CTA (bounds shared memory at high degree)

__device__ __forceinline__ long long x_block_offset(int m, int L, int E) {
    return 2LL * E * ((long long)m * L - (long long)m * (m - 1) / 2);
}

// X position of element (row r, column c) of anm: (order, degree offset, cos|sin)
__device__ __forceinline__ long long x_position(int r, int c, int L, int E) {
    const int m = (c <= r) ? c : r + 1;
    const int nn = (c <= r) ? r - c : c - r - 1;
    const int cs = (c <= r) ? 0 : 1;
    return x_block_offset(m, L, E) + (long long)nn * 2 * E + (long long)cs * E;
}

// Tiled layout for the table-fed stage 1 (gb_synthesis.cu): [order m][column tile][degree row][tn + 4], the rows of an
// order padded to a multiple of 8 and, inside every 8, ordered [even n-m | odd n-m] like the Legendre table, so that a
// pipeline chunk of stage 1 is ONE contiguous bulk copy.  roff[m] = first row of order m, columns (cs * E + e).
struct XTiling {
    const int* roff;
    int tn, n_ct;
};
__device__ __forceinline__ long long x_tiled_position(int r, int c, int e, int E, const XTiling& xt, const int* roff) {
    const int m = (c <= r) ? c : r + 1;
    const int nn = (c <= r) ? r - c : c - r - 1;
    const int col = ((c <= r) ? 0 : E) + e;
    const int ct = col / xt.tn, cc = col - ct * xt.tn;
    const int r0 = roff[m], kn_pad = roff[m + 1] - r0;
    const int row = (nn & ~7) + ((nn & 1) << 2) + ((nn & 7) >> 1);
    return ((long long)r0 * xt.n_ct + (long long)ct * kn_pad + row) * (xt.tn + 4) + cc;
}

// PKE epochs per CTA: 32 for epoch batches (256-byte runs on the X side), 8 for small shards (four times as many
// CTAs: a 30-epoch shard is latency-, not bandwidth-bound)
template <bool PACK, int PKE, bool TILED = false>
__global__ void __launch_bounds__(256) gb_pack_kernel(const double* __restrict__ src, double* __restrict__ dst, int L,
                                                      int E, const double* __restrict__ wn, XTiling xt) {
    constexpr int PK_LD = PKE + 1;    // shared-memory pitch
    extern __shared__ double s_t[];   // [min(L, PK_C)][PK_LD] (+ the row offsets of the tiled layout)
    int* s_roff = reinterpret_cast<int*>(s_t + (size_t)min(L, PK_C) * PK_LD);
    const int r = blockIdx.x;
    const int cb = blockIdx.z * PK_C;                 // first column of this CTA
    const int nc = min(PK_C, L - cb);
    const int e0 = blockIdx.y * PKE;
    const int ne = min(PKE, E - e0);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    GB_PACK_MARK(0);
    if (TILED)
        for (int i = threadIdx.x; i <= L; i += blockDim.x) s_roff[i] = xt.roff[i];    // plan constant: before the wait
    gb::griddep_wait();
    gb::griddep_launch_dependents();
    GB_PACK_MARK(1);
    if (PACK) {
        for (int e = warp; e < ne; e += nwarps) {
            const double* row = src + ((size_t)(e0 + e) * L + r) * L;
            if (wn) {
                for (int c = lane; c < nc; c += 32) s_t[c * PK_LD + e] = __dmul_rn(row[cb + c], wn[max(r, cb + c)]);
            } else {
                for (int c = lane; c < nc; c += 32) s_t[c * PK_LD + e] = row[cb + c];
            }
        }
        __syncthreads();
        GB_PACK_MARK(2);
        if (TILED) {
            // PKE lanes share one column c of anm: its order / degree / plane and the row of the tiled layout are
            // computed once per column, the epoch only moves the position inside (at most two) column tiles
            constexpr int CPW = 32 / PKE;                      // columns per warp pass
            const int sub = lane / PKE, e = lane % PKE;
            for (int c = warp * CPW + sub; c < nc; c += nwarps * CPW) {
                const int cc_anm = cb + c;
                const int m = (cc_anm <= r) ? cc_anm : r + 1;
                const int nn = (cc_anm <= r) ? r - cc_anm : cc_anm - r - 1;
                const int r0 = s_roff[m], kn_pad = s_roff[m + 1] - r0;
                const int row = (nn & ~7) + ((nn & 1) << 2) + ((nn & 7) >> 1);
                const int col = ((cc_anm <= r) ? 0 : E) + e0 + e;
                const int ct = col / xt.tn;
                if (e < ne)
                    dst[((long long)r0 * xt.n_ct + (long long)ct * kn_pad + row) * (xt.tn + 4) + (col - ct * xt.tn)] =
                        s_t[c * PK_LD + e];
            }
        } else {
            for (int idx = threadIdx.x; idx < nc * PKE; idx += blockDim.x) {
                const int c = idx / PKE, e = idx % PKE;
                if (e < ne) dst[x_position(r, cb + c, L, E) + e0 + e] = s_t[c * PK_LD + e];
            }
        }
        // sine plane of order 0, degree r (the tiled buffer is cleared when its layout changes: nothing to write)
        if (!TILED && blockIdx.z == 0 && threadIdx.x < ne) dst[(long long)r * 2 * E + E + e0 + threadIdx.x] = 0.0;
        GB_PACK_MARK(3);
    } else {
        for (int idx = threadIdx.x; idx < nc * PKE; idx += blockDim.x) {
            const int c = idx / PKE, e = idx % PKE;
            if (e < ne) s_t[c * PK_LD + e] = src[x_position(r, cb + c, L, E) + e0 + e];
        }
        __syncthreads();
        for (int e = warp; e < ne; e += nwarps) {
            double* row = dst + ((size_t)(e0 + e) * L + r) * L;
            for (int c = lane; c < nc; c += 32) row[cb + c] = s_t[c * PK_LD + e];
        }
    }
}

// The tiled pack with its rows fetched by the TMA unit.  One CTA = row r of anm for PKE epochs, as above, but every row is
// ONE bulk copy (cp.async.bulk) issued by its own lane, so all of the CTA's bytes are in flight at once instead of a few
// 8-byte loads per lane (the scalar-load kernel needed 7 us to read the 18 MB of a 240-epoch batch).  Bulk copies move
// whole 16-byte units: a row that starts on an odd double is fetched from the double before it (`off` = 1) and rows are
// an even number of doubles long in shared memory; a row whose widened range would leave the array (the very first or
// last one) is read with plain loads by its lane.  The write side is the one of gb_pack_kernel<true, PKE, true>.
template <int PKE>
__global__ void __launch_bounds__(256) gb_pack_rows_kernel(const double* __restrict__ src, double* __restrict__ dst, int L,
                                                            int E, const double* __restrict__ wn, XTiling xt) {
    extern __shared__ __align__(16) double s_rows[];       // [PKE][lp], lp = L + 3 rounded up to even + 2 (bank spread)
    const int lp = ((L + 3) & ~1) + 2;
    int* s_roff = reinterpret_cast<int*>(s_rows + (size_t)PKE * lp);
    uint64_t* bar = reinterpret_cast<uint64_t*>(s_roff + ((L + 2 + 1) & ~1));
    const int r = blockIdx.x;
    const int e0 = blockIdx.y * PKE;
    const int ne = min(PKE, E - e0);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    GB_PACK_MARK(0);
    for (int i = threadIdx.x; i <= L; i += blockDim.x) s_roff[i] = xt.roff[i];    // plan constant: before the wait
    if (threadIdx.x == 0) {
        gb::mbar_init(bar, (uint32_t)ne);
        gb::fence_mbar_init();
    }
    __syncthreads();
    gb::griddep_wait();
    gb::griddep_launch_dependents();
    GB_PACK_MARK(1);
    const long long a0 = (long long)((reinterpret_cast<uintptr_t>(src) >> 3) & 1);
    const long long total = (long long)E * L * L;
    if (threadIdx.x < ne) {
        const int e = threadIdx.x;
        const long long start = ((long long)(e0 + e) * L + r) * L;
        const int off = (int)((a0 + start) & 1);
        const int cnt = (L + off + 1) & ~1;
        double* row = s_rows + (size_t)e * lp;
        if (start - off >= 0 && start - off + cnt <= total) {
            gb::mbar_arrive_expect_tx(bar, (uint32_t)(cnt * sizeof(double)));
            gb::bulk_g2s(row, src + (start - off), (uint32_t)(cnt * sizeof(double)), bar);
        } else {
            for (int c = 0; c < L; ++c) row[off + c] = src[start + c];
            gb::mbar_arrive(bar);
        }
    }
    gb::mbar_wait(bar, 0);
    GB_PACK_MARK(2);
    // PKE lanes share one column c of anm: its order / degree / plane and the row of the tiled layout are computed once
    // per column, the epoch only moves the position inside (at most two) column tiles
    constexpr int CPW = 32 / PKE;                      // columns per warp pass
    const int sub = lane / PKE, e = lane % PKE;
    const int off_e = (int)((a0 + ((long long)(e0 + e) * L + r) * L) & 1);
    const double* my_row = s_rows + (size_t)e * lp + off_e;
    for (int c = warp * CPW + sub; c < L; c += nwarps * CPW) {
        const int m = (c <= r) ? c : r + 1;
        const int nn = (c <= r) ? r - c : c - r - 1;
        const int r0 = s_roff[m], kn_pad = s_roff[m + 1] - r0;
        const int row = (nn & ~7) + ((nn & 1) << 2) + ((nn & 7) >> 1);
        const int col = ((c <= r) ? 0 : E) + e0 + e;
        const int ct = col / xt.tn;
        if (e < ne) {
            double v = my_row[c];
            if (wn) v = __dmul_rn(v, wn[max(r, c)]);
            dst[((long long)r0 * xt.n_ct + (long long)ct * kn_pad + row) * (xt.tn + 4) + (col - ct * xt.tn)] = v;
        }
    }
    GB_PACK_MARK(3);
}

// out[e][r][c] = in[e][r][c] * w[max(r, c)]
__global__ void __launch_bounds__(256) gb_scale_degree_kernel(const double* __restrict__ in, double* __restrict__ out,
                                                              const double* __restrict__ wn, int L, long long total) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int rc = (int)(idx % ((long long)L * L));
    const int r = rc / L, c = rc - r * L;
    out[idx] = __dmul_rn(in[idx], wn[max(r, c)]);
}

template <bool PACK, int PKE, bool TILED>
int launch_pke(const double* src, double* dst, int L, int E, const double* wn, XTiling xt, cudaStream_t st) {
    const size_t smem = (size_t)(L < PK_C ? L : PK_C) * (PKE + 1) * sizeof(double) + (TILED ? (L + 2) * sizeof(int) : 0);
    if (smem > 48 * 1024)
        GB_CUDA(cudaFuncSetAttribute(gb_pack_kernel<PACK, PKE, TILED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid(L, (E + PKE - 1) / PKE, (L + PK_C - 1) / PK_C);
    GB_CUDA(gb_launch_pdl(gb_pack_kernel<PACK, PKE, TILED>, grid, dim3(256), smem, st, src, dst, L, E, wn, xt));
    GB_LAUNCH_CHECK();
    return GB_OK;
}

template <bool PACK>
int launch(const double* src, double* dst, int L, int E, const double* wn, cudaStream_t st) {
    const XTiling none{nullptr, 0, 0};
    return E <= 64 ? launch_pke<PACK, 8, false>(src, dst, L, E, wn, none, st)
                   : launch_pke<PACK, 32, false>(src, dst, L, E, wn, none, st);
}

}  // namespace

int gb_launch_pack(const double* d_anm, double* d_x, int L, int E, cudaStream_t st, const double* d_wn) {
    return launch<true>(d_anm, d_x, L, E, d_wn, st);
}
template <int PKE>
static int launch_rows(const double* src, double* dst, int L, int E, const double* wn, XTiling xt, cudaStream_t st) {
    const int lp = ((L + 3) & ~1) + 2;
    const size_t smem = (size_t)PKE * lp * sizeof(double) + (size_t)((L + 3) & ~1) * sizeof(int) + sizeof(uint64_t);
    if (smem > 48 * 1024)
        GB_CUDA(cudaFuncSetAttribute(gb_pack_rows_kernel<PKE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid(L, (E + PKE - 1) / PKE, 1);
    GB_CUDA(gb_launch_pdl(gb_pack_rows_kernel<PKE>, grid, dim3(256), smem, st, src, dst, L, E, wn, xt));
    GB_LAUNCH_CHECK();
    return GB_OK;
}

int gb_launch_pack_tiled(const double* d_anm, double* d_x, int L, int E, const int* d_roff, int tn, int n_ct,
                         cudaStream_t st, const double* d_wn) {
    const XTiling xt{d_roff, tn, n_ct};
    if (L <= PK_C)      // rows fetched by the TMA unit
        return E <= 64 ? launch_rows<8>(d_anm, d_x, L, E, d_wn, xt, st) : launch_rows<32>(d_anm, d_x, L, E, d_wn, xt, st);
    return E <= 64 ? launch_pke<true, 8, true>(d_anm, d_x, L, E, d_wn, xt, st)
                   : launch_pke<true, 32, true>(d_anm, d_x, L, E, d_wn, xt, st);
}
int gb_launch_unpack(const double* d_x, double* d_anm, int L, int E, cudaStream_t st) {
    return launch<false>(d_x, d_anm, L, E, nullptr, st);
}

#ifdef GB_TRACE
extern "C" int gb_debug_trace_pack(unsigned long long* h_out, int reset) {
    if (reset) {
        void* sym = nullptr;
        GB_CUDA(cudaGetSymbolAddress(&sym, gb_trace_pack));
        GB_CUDA(cudaMemset(sym, 0, sizeof(gb_trace_pack)));
        return GB_OK;
    }
    GB_CUDA(cudaDeviceSynchronize());
    GB_CUDA(cudaMemcpyFromSymbol(h_out, gb_trace_pack, sizeof(gb_trace_pack)));
    return GB_OK;
}
#endif

extern "C" int gb_scale_by_degree(const double* d_anm_in, const double* d_wn, int n_epochs, int nmax, double* d_anm_out,
                                  int device, void* stream) {
    GB_REQUIRE(n_epochs >= 0 && nmax >= 0, "gb_scale_by_degree: negative size");
    if (n_epochs == 0) return GB_OK;
    GB_REQUIRE(d_anm_in && d_wn && d_anm_out, "gb_scale_by_degree: NULL pointer");
    GB_CUDA(cudaSetDevice(device));
    const int L = nmax + 1;
    const long long total = (long long)n_epochs * L * L;
    gb_scale_degree_kernel<<<(unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        d_anm_in, d_anm_out, d_wn, L, total);
    GB_LAUNCH_CHECK();
    return GB_OK;
}
