// Gravitational acceleration (gradient of the potential) as scalar syntheses: two HBM-bound passes around gb_synthesis /
// gb_points_synthesis.
//
//   gb_gradient_coefficients   Cunningham's relation for solid harmonics: each Cartesian component of grad V of a
//                              degree-N field is a synthesis at degree N + 1 of linearly transformed coefficients
//                              (the general form of the zonal code behind GRS80 normal gravity, reference
//                              gravityfield.py:437-454 with the factors f_zero, f_plus).  With q = (2n+1)/(2n+3), the
//                              input (C_nm, S_nm) contributes to degree n' = n + 1:
//                                Z[n+1, m]              -sqrt((n-m+1)(n+m+1) q) (C, S)
//                                X[n+1, m+1]            -fp (C, S)            Y[n+1, m+1]  (+fp S, -fp C)
//                                X[n+1, m-1], m >= 1    +fm (C, S)            Y[n+1, m-1]  (+fm S, -fm C)
//                              fp = sqrt((n+m+1)(n+m+2) q) / 2 (times sqrt 2 for m = 0),
//                              fm = sqrt((n-m+1)(n-m+2) q) / 2 (times sqrt 2 for m = 1); sine terms of order 0 are
//                              dropped.  Written as a GATHER: one thread per output coefficient computes its factors
//                              once and reads at most two inputs in each of eight sets, so there are no atomics and
//                              the result is bit-reproducible.
//   gb_rotate_to_local         (gx, gy, gz) -> (east, north, up) of the geocentric spherical frame, in place.
#include "gb_common.cuh"

namespace {

constexpr double GB_SQRT2 = 1.41421356237309504880;   // == sqrt(2.0) correctly rounded

// Factors in one fixed expression order, every operation rounded on its own (no contraction):
//   q  = (2n+1) / (2n+3)
//   f  = sqrt(p * q) * 0.5 [* sqrt2]   p = the integer product of the table, converted exactly to double
__device__ __forceinline__ double grad_q(int n) { return __ddiv_rn((double)(2 * n + 1), (double)(2 * n + 3)); }

__device__ __forceinline__ double grad_fz(int n, int m, double q) {
    return __dsqrt_rn(__dmul_rn((double)(n - m + 1) * (double)(n + m + 1), q));
}

__device__ __forceinline__ double grad_fp(int n, int m, double q) {
    const double f = __dmul_rn(__dsqrt_rn(__dmul_rn((double)(n + m + 1) * (double)(n + m + 2), q)), 0.5);
    return m == 0 ? __dmul_rn(f, GB_SQRT2) : f;
}

__device__ __forceinline__ double grad_fm(int n, int m, double q) {
    const double f = __dmul_rn(__dsqrt_rn(__dmul_rn((double)(n - m + 1) * (double)(n - m + 2), q)), 0.5);
    return m == 1 ? __dmul_rn(f, GB_SQRT2) : f;
}

constexpr int GC_EB = 8;      // epochs per thread: the factors of an output coefficient are computed once for them

// out [E][3][L+1][L+1] packed (x, y, z); one thread per output coefficient of one set, for GC_EB sets.  An output
// coefficient (n', m', sine) of a component is at most two products f1 a[i1] + f2 a[i2]: its fp term (source order
// m' - 1) first, then its fm term (source order m' + 1); a source index of -1 is a missing term (out of range, or the
// sine of order 0).
__global__ void __launch_bounds__(256)
gb_gradient_coefficients_kernel(const double* __restrict__ anm, double* __restrict__ out, int L, int E) {
    const int Lo = L + 1;
    const int per_set = 3 * Lo * Lo;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= per_set) return;
    const int comp = idx / (Lo * Lo);
    const int rc = idx - comp * Lo * Lo;
    const int r = rc / Lo, c = rc - r * Lo;
    const bool sine = r < c;                                  // S_{n', m'} = out[m' - 1][n'], C_{n', m'} = out[n'][m']
    const int np = sine ? c : r, mp = sine ? r + 1 : c;
    int i1 = -1, i2 = -1;
    double f1 = 0.0, f2 = 0.0;
    if (np > 0) {
        const int n = np - 1;
        const double q = grad_q(n);
        // packed index of the cosine / sine of input order m <= n; the sine of order 0 does not exist
        auto Ci = [&](int m) { return n * L + m; };
        auto Si = [&](int m) { return m > 0 ? (m - 1) * L + n : -1; };
        if (comp == 2) {
            if (mp <= n) { i1 = sine ? Si(mp) : Ci(mp); f1 = -grad_fz(n, mp, q); }
        } else if (comp == 0) {
            if (mp >= 1) { i1 = sine ? Si(mp - 1) : Ci(mp - 1); f1 = -grad_fp(n, mp - 1, q); }
            if (mp + 1 <= n) { i2 = sine ? Si(mp + 1) : Ci(mp + 1); f2 = grad_fm(n, mp + 1, q); }
        } else {
            if (mp >= 1) {
                const double f = grad_fp(n, mp - 1, q);
                i1 = sine ? Ci(mp - 1) : Si(mp - 1);
                f1 = sine ? -f : f;
            }
            if (mp + 1 <= n) {
                const double f = grad_fm(n, mp + 1, q);
                i2 = sine ? Ci(mp + 1) : Si(mp + 1);
                f2 = sine ? -f : f;
            }
        }
    }
    const int e0 = blockIdx.y * GC_EB;
    const int e1 = e0 + GC_EB < E ? e0 + GC_EB : E;
    for (int e = e0; e < e1; ++e) {
        const double* a = anm + (size_t)e * L * L;
        double v = 0.0;
        if (i1 >= 0) v = __dmul_rn(f1, a[i1]);
        if (i2 >= 0) v = __dadd_rn(v, __dmul_rn(f2, a[i2]));
        out[(size_t)e * per_set + idx] = v;
    }
}

constexpr int ROT_EB = 8;     // epochs per thread: the frame of a point is read once for them

struct Frame { double ct, st, cl, sl; };

// east  = -sl gx + cl gy
// north = -ct cl gx - ct sl gy + st gz
// up    =  st cl gx + st sl gy + ct gz       each product and sum rounded on its own, left to right
__device__ __forceinline__ void rotate(const Frame& f, double& gx, double& gy, double& gz) {
    const double east = __dadd_rn(__dmul_rn(-f.sl, gx), __dmul_rn(f.cl, gy));
    const double north = __dadd_rn(__dadd_rn(__dmul_rn(__dmul_rn(-f.ct, f.cl), gx), __dmul_rn(__dmul_rn(-f.ct, f.sl), gy)),
                                   __dmul_rn(f.st, gz));
    const double up = __dadd_rn(__dadd_rn(__dmul_rn(__dmul_rn(f.st, f.cl), gx), __dmul_rn(__dmul_rn(f.st, f.sl), gy)),
                                __dmul_rn(f.ct, gz));
    gx = east;
    gy = north;
    gz = up;
}

// Two points per thread with 16-byte accesses (n_points even, xyz and frame 16-byte aligned), ROT_EB epochs per thread.
__global__ void __launch_bounds__(256)
gb_rotate_local_vec2(double* __restrict__ xyz, const double* __restrict__ frame, int E, long long P) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;      // point pair
    if (2 * j >= P) return;
    const double2 ct = reinterpret_cast<const double2*>(frame)[j];
    const double2 st = reinterpret_cast<const double2*>(frame + P)[j];
    const double2 cl = reinterpret_cast<const double2*>(frame + 2 * P)[j];
    const double2 sl = reinterpret_cast<const double2*>(frame + 3 * P)[j];
    const Frame f0{ct.x, st.x, cl.x, sl.x}, f1{ct.y, st.y, cl.y, sl.y};
    const int e0 = blockIdx.y * ROT_EB;
    const int e1 = e0 + ROT_EB < E ? e0 + ROT_EB : E;
    for (int e = e0; e < e1; ++e) {
        double2* gx = reinterpret_cast<double2*>(xyz + (size_t)e * 3 * P);
        double2* gy = reinterpret_cast<double2*>(xyz + (size_t)e * 3 * P + P);
        double2* gz = reinterpret_cast<double2*>(xyz + (size_t)e * 3 * P + 2 * P);
        double2 x = gx[j], y = gy[j], z = gz[j];
        rotate(f0, x.x, y.x, z.x);
        rotate(f1, x.y, y.y, z.y);
        gx[j] = x;
        gy[j] = y;
        gz[j] = z;
    }
}

// Any point count or alignment: one point per thread, the same arithmetic.
__global__ void __launch_bounds__(256)
gb_rotate_local_scalar(double* __restrict__ xyz, const double* __restrict__ frame, int E, long long P) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const Frame f{frame[p], frame[P + p], frame[2 * P + p], frame[3 * P + p]};
    const int e0 = blockIdx.y * ROT_EB;
    const int e1 = e0 + ROT_EB < E ? e0 + ROT_EB : E;
    for (int e = e0; e < e1; ++e) {
        double* g = xyz + (size_t)e * 3 * P;
        double x = g[p], y = g[P + p], z = g[2 * P + p];
        rotate(f, x, y, z);
        g[p] = x;
        g[P + p] = y;
        g[2 * P + p] = z;
    }
}

}  // namespace

extern "C" int gb_gradient_coefficients(const double* d_anm, int n_sets, int nmax, double* d_out, int device,
                                        void* stream) {
    GB_REQUIRE(n_sets >= 0 && nmax >= 0, "gb_gradient_coefficients: negative size (n_sets=%d, nmax=%d)", n_sets, nmax);
    if (n_sets == 0) return GB_OK;
    GB_REQUIRE(d_anm && d_out, "gb_gradient_coefficients: NULL device pointer");
    GB_REQUIRE(nmax < 8192, "gb_gradient_coefficients: nmax=%d too large (at most 8191)", nmax);
    const int eb = (n_sets + GC_EB - 1) / GC_EB;
    GB_REQUIRE(eb <= 65535, "gb_gradient_coefficients: at most %d sets per call", 65535 * GC_EB);
    GB_CUDA(cudaSetDevice(device));
    const int L = nmax + 1;
    const int per_set = 3 * (L + 1) * (L + 1);
    dim3 grid((per_set + 255) / 256, eb);
    gb_gradient_coefficients_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(d_anm, d_out, L, n_sets);
    GB_LAUNCH_CHECK();
    return GB_OK;
}

extern "C" int gb_rotate_to_local(double* d_xyz, const double* d_frame, int n_sets, int64_t n_points, int device,
                                  void* stream) {
    GB_REQUIRE(n_sets >= 0 && n_points >= 0, "gb_rotate_to_local: negative size (n_sets=%d, n_points=%lld)", n_sets,
               (long long)n_points);
    if (n_sets == 0 || n_points == 0) return GB_OK;
    GB_REQUIRE(d_xyz && d_frame, "gb_rotate_to_local: NULL device pointer");
    const int eb = (n_sets + ROT_EB - 1) / ROT_EB;
    GB_REQUIRE(eb <= 65535, "gb_rotate_to_local: at most %d sets per call", 65535 * ROT_EB);
    GB_CUDA(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool vec = n_points % 2 == 0 && reinterpret_cast<uintptr_t>(d_xyz) % 16 == 0 &&
                     reinterpret_cast<uintptr_t>(d_frame) % 16 == 0;
    if (vec) {
        dim3 grid((unsigned)((n_points / 2 + 255) / 256), eb);
        gb_rotate_local_vec2<<<grid, 256, 0, st>>>(d_xyz, d_frame, n_sets, n_points);
    } else {
        dim3 grid((unsigned)((n_points + 255) / 256), eb);
        gb_rotate_local_scalar<<<grid, 256, 0, st>>>(d_xyz, d_frame, n_sets, n_points);
    }
    GB_LAUNCH_CHECK();
    return GB_OK;
}
