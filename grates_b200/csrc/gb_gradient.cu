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
//   gb_gradient_coefficients_adjoint, gb_rotate_from_local
//                              the transposes T' (summed over the three components) and Q', for the adjoint of the
//                              acceleration at points (PointsPlan.gradient_adjoint): the same factors (gbgrad::grad_terms)
//                              and the same rotation kernels, templated on the direction.
//   gb_gravity_gradient_coefficients, gb_rotate_tensor_to_local
//                              the gravity gradient tensor: applying the transform twice gives every second derivative
//                              V_ab as a synthesis at degree N + 2 (T_a T_b, in one gather), and the same rotation kernels
//                              turn its six components into (east, north, up).
//   gb_gravity_gradient_coefficients_adjoint, gb_rotate_tensor_from_local
//                              their transposes, for the adjoint of the gravity gradient at points
//                              (PointsPlan.gravity_gradient_adjoint): the composed terms of gbgrad::apply_pair and
//                              gbgrad::rotate_tensor_transpose.
#include "gb_gradient.cuh"

namespace {

using gbgrad::grad_q;
using gbgrad::grad_fz;
using gbgrad::grad_fp;
using gbgrad::grad_fm;
using gbgrad::Frame;
using gbgrad::rotate_dir;

constexpr int GC_EB = 8;      // epochs per thread: the factors of an output coefficient are computed once for them

// An output coefficient (n', m', sine) of component comp of the transform of a packed [L][L] set is at most two products
// f1 a[i1] + f2 a[i2]: its fp term (source order m' - 1) first, then its fm term (source order m' + 1); a source index of
// -1 is a missing term (out of range, or the sine of order 0).
struct Gather {
    int i1, i2;
    double f1, f2;
};

__device__ __forceinline__ Gather gather_terms(int comp, int np, int mp, bool sine, int L) {
    Gather g{-1, -1, 0.0, 0.0};
    if (np > 0) {
        const int n = np - 1;
        const double q = grad_q(n);
        // packed index of the cosine / sine of input order m <= n; the sine of order 0 does not exist
        auto Ci = [&](int m) { return n * L + m; };
        auto Si = [&](int m) { return m > 0 ? (m - 1) * L + n : -1; };
        if (comp == 2) {
            if (mp <= n) { g.i1 = sine ? Si(mp) : Ci(mp); g.f1 = -grad_fz(n, mp, q); }
        } else if (comp == 0) {
            if (mp >= 1) { g.i1 = sine ? Si(mp - 1) : Ci(mp - 1); g.f1 = -grad_fp(n, mp - 1, q); }
            if (mp + 1 <= n) { g.i2 = sine ? Si(mp + 1) : Ci(mp + 1); g.f2 = grad_fm(n, mp + 1, q); }
        } else {
            if (mp >= 1) {
                const double f = grad_fp(n, mp - 1, q);
                g.i1 = sine ? Ci(mp - 1) : Si(mp - 1);
                g.f1 = sine ? -f : f;
            }
            if (mp + 1 <= n) {
                const double f = grad_fm(n, mp + 1, q);
                g.i2 = sine ? Ci(mp + 1) : Si(mp + 1);
                g.f2 = sine ? -f : f;
            }
        }
    }
    return g;
}

// The terms of the output coefficient at packed position idx of a [Lo][Lo] component (Lo = L + 1)
__device__ __forceinline__ Gather gather_at(int comp, int idx, int L) {
    const int Lo = L + 1;
    const int r = idx / Lo, c = idx - r * Lo;
    const bool sine = r < c;                                  // S_{n', m'} = out[m' - 1][n'], C_{n', m'} = out[n'][m']
    return gather_terms(comp, sine ? c : r, sine ? r + 1 : c, sine, L);
}

// f1 x(i1) [+ f2 x(i2)] in the order of the transform, each product and sum rounded on its own; x is called for present
// terms only.
template <class Read>
__device__ __forceinline__ double gather(const Gather& g, Read x) {
    double v = 0.0;
    if (g.i1 >= 0) v = __dmul_rn(g.f1, x(g.i1));
    if (g.i2 >= 0) v = __dadd_rn(v, __dmul_rn(g.f2, x(g.i2)));
    return v;
}

// out [E][3][L+1][L+1] packed (x, y, z); one thread per output coefficient of one set, for GC_EB sets.
__global__ void __launch_bounds__(256)
gb_gradient_coefficients_kernel(const double* __restrict__ anm, double* __restrict__ out, int L, int E) {
    const int Lo = L + 1;
    const int per_set = 3 * Lo * Lo;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= per_set) return;
    const int comp = idx / (Lo * Lo);
    const Gather g = gather_at(comp, idx - comp * Lo * Lo, L);
    const int e0 = blockIdx.y * GC_EB;
    const int e1 = e0 + GC_EB < E ? e0 + GC_EB : E;
    for (int e = e0; e < e1; ++e) {
        const double* a = anm + (size_t)e * L * L;
        out[(size_t)e * per_set + idx] = gather(g, [&](int i) { return a[i]; });
    }
}

// out [E][6][L+2][L+2] packed, pairs (a, b) = xx, xy, xz, yy, yz, zz: T_a applied to component b of T(anm), with the
// arithmetic of two gb_gradient_coefficients calls.  One thread per output coefficient of one set, for GC_EB sets: the
// outer terms (T_a at degree L) name at most two intermediate coefficients of component b, each of them the inner terms
// (T_b at degree L - 1) of at most two inputs, so an output reads at most four inputs and nothing is stored in between.
__global__ void __launch_bounds__(256)
gb_gravity_gradient_coefficients_kernel(const double* __restrict__ anm, double* __restrict__ out, int L, int E) {
    const int Lo = L + 2;
    const int per_set = 6 * Lo * Lo;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= per_set) return;
    const int pair = idx / (Lo * Lo);
    const int ca = pair < 3 ? 0 : pair < 5 ? 1 : 2;
    const int cb = pair < 3 ? pair : pair < 5 ? pair - 2 : 2;
    const Gather outer = gather_at(ca, idx - pair * Lo * Lo, L + 1);
    const Gather inner1 = outer.i1 >= 0 ? gather_at(cb, outer.i1, L) : Gather{-1, -1, 0.0, 0.0};
    const Gather inner2 = outer.i2 >= 0 ? gather_at(cb, outer.i2, L) : Gather{-1, -1, 0.0, 0.0};
    const int e0 = blockIdx.y * GC_EB;
    const int e1 = e0 + GC_EB < E ? e0 + GC_EB : E;
    for (int e = e0; e < e1; ++e) {
        const double* a = anm + (size_t)e * L * L;
        auto read = [&](int i) { return a[i]; };
        const double g1 = gather(inner1, read), g2 = gather(inner2, read);
        out[(size_t)e * per_set + idx] = gather(outer, [&](int i) { return i == outer.i1 ? g1 : g2; });
    }
}

constexpr int ROT_EB = 8;     // epochs per thread: the frame of a point is read once for them

// What the rotation kernels do to the NC values of one point of one set:
//   ToLocal / FromLocal   a vector (x, y, z) <-> (east, north, up): Q (gbgrad::rotate) or Q' (gbgrad::rotate_back)
//   TensorToLocal         a symmetric tensor, upper triangle (xx, xy, xz, yy, yz, zz) -> (ee, en, eu, nn, nu, uu) of
//                         Q V Q' (gbgrad::rotate_matrix: the columns of V, then the rows of the result)
template <bool TO_LOCAL>
struct VectorRotation {
    static constexpr int NC = 3;
    __device__ static void apply(const Frame& f, double (&v)[NC]) { rotate_dir<TO_LOCAL>(f, v[0], v[1], v[2]); }
};
using ToLocal = VectorRotation<true>;
using FromLocal = VectorRotation<false>;

struct TensorToLocal {
    static constexpr int NC = 6;
    __device__ static void apply(const Frame& f, double (&v)[NC]) { gbgrad::rotate_tensor(f, v); }
};

//   TensorFromLocal       the transpose of TensorToLocal on the 6-vectors (gbgrad::rotate_tensor_transpose)
struct TensorFromLocal {
    static constexpr int NC = 6;
    __device__ static void apply(const Frame& f, double (&v)[NC]) { gbgrad::rotate_tensor_transpose(f, v); }
};

// Two points per thread with 16-byte accesses (n_points even, values and frame 16-byte aligned), ROT_EB epochs per
// thread; values [E][Op::NC][P].
template <class Op>
__global__ void __launch_bounds__(256)
gb_rotate_vec2(double* __restrict__ vals, const double* __restrict__ frame, int E, long long P) {
    constexpr int NC = Op::NC;
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
        double2* g = reinterpret_cast<double2*>(vals + (size_t)e * NC * P);
        double v0[NC], v1[NC];
#pragma unroll
        for (int c = 0; c < NC; ++c) {
            const double2 x = g[c * (P / 2) + j];
            v0[c] = x.x;
            v1[c] = x.y;
        }
        Op::apply(f0, v0);
        Op::apply(f1, v1);
#pragma unroll
        for (int c = 0; c < NC; ++c) g[c * (P / 2) + j] = make_double2(v0[c], v1[c]);
    }
}

// Any point count or alignment: one point per thread, the same arithmetic.
template <class Op>
__global__ void __launch_bounds__(256)
gb_rotate_scalar(double* __restrict__ vals, const double* __restrict__ frame, int E, long long P) {
    constexpr int NC = Op::NC;
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const Frame f{frame[p], frame[P + p], frame[2 * P + p], frame[3 * P + p]};
    const int e0 = blockIdx.y * ROT_EB;
    const int e1 = e0 + ROT_EB < E ? e0 + ROT_EB : E;
    for (int e = e0; e < e1; ++e) {
        double* g = vals + (size_t)e * NC * P;
        double v[NC];
#pragma unroll
        for (int c = 0; c < NC; ++c) v[c] = g[c * P + p];
        Op::apply(f, v);
#pragma unroll
        for (int c = 0; c < NC; ++c) g[c * P + p] = v[c];
    }
}

template <class Op>
int rotate_sets(const char* name, double* d_xyz, const double* d_frame, int n_sets, int64_t n_points, int device,
                void* stream) {
    GB_REQUIRE(n_sets >= 0 && n_points >= 0, "%s: negative size (n_sets=%d, n_points=%lld)", name, n_sets,
               (long long)n_points);
    if (n_sets == 0 || n_points == 0) return GB_OK;
    GB_REQUIRE(d_xyz && d_frame, "%s: NULL device pointer", name);
    const int eb = (n_sets + ROT_EB - 1) / ROT_EB;
    GB_REQUIRE(eb <= 65535, "%s: at most %d sets per call", name, 65535 * ROT_EB);
    GB_CUDA(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool vec = n_points % 2 == 0 && reinterpret_cast<uintptr_t>(d_xyz) % 16 == 0 &&
                     reinterpret_cast<uintptr_t>(d_frame) % 16 == 0;
    if (vec) {
        dim3 grid((unsigned)((n_points / 2 + 255) / 256), eb);
        gb_rotate_vec2<Op><<<grid, 256, 0, st>>>(d_xyz, d_frame, n_sets, n_points);
    } else {
        dim3 grid((unsigned)((n_points + 255) / 256), eb);
        gb_rotate_scalar<Op><<<grid, 256, 0, st>>>(d_xyz, d_frame, n_sets, n_points);
    }
    GB_LAUNCH_CHECK();
    return GB_OK;
}

// T' of gb_gradient_coefficients_kernel, summed over the components: in [E][3][L+1][L+1] -> anm [E][L][L] packed.  One
// thread per output coefficient (n, m, s) of one set, for GC_EB sets: the terms of gbgrad::grad_terms read the degree
// n + 1 of the three input components, component by component in the order x, y, z (a gather, no atomics).
__global__ void __launch_bounds__(256)
gb_gradient_coefficients_adjoint_kernel(const double* __restrict__ in, double* __restrict__ anm, int L, int E) {
    const int Lo = L + 1;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= L * L) return;
    const int r = idx / L, c = idx - r * L;
    const int s = r < c ? 1 : 0;                             // S_nm = anm[m - 1][n], C_nm = anm[n][m]
    const int n = s ? c : r, m = s ? r + 1 : c;
    const double q = grad_q(n);
    gbgrad::Terms t[3];
#pragma unroll
    for (int comp = 0; comp < 3; ++comp) t[comp] = gbgrad::grad_terms(comp, n, m, s, q);
    const int e0 = blockIdx.y * GC_EB;
    const int e1 = e0 + GC_EB < E ? e0 + GC_EB : E;
    for (int e = e0; e < e1; ++e) {
        double v = 0.0;
#pragma unroll
        for (int comp = 0; comp < 3; ++comp) {
            const double* g = in + ((size_t)e * 3 + comp) * Lo * Lo;
            // packed position of (n + 1, mp, sp): C at [n + 1][mp], S at [mp - 1][n + 1]
            v = __dadd_rn(v, gbgrad::apply(t[comp], [&](int mp, int sp) {
                return g[sp ? (mp - 1) * Lo + n + 1 : (n + 1) * Lo + mp];
            }));
        }
        anm[(size_t)e * L * L + idx] = v;
    }
}

// The transpose of gb_gravity_gradient_coefficients_kernel, summed over the pairs: in [E][6][L+2][L+2] -> anm [E][L][L]
// packed.  One thread per output coefficient (n, m, s) of one set, for GC_EB sets: the composed terms of
// gbgrad::apply_pair read degree n + 2 of each pair, added in the order xx, xy, xz, yy, yz, zz (a gather, no atomics).
__global__ void __launch_bounds__(256)
gb_gravity_gradient_coefficients_adjoint_kernel(const double* __restrict__ in, double* __restrict__ anm, int L, int E) {
    const int Lo = L + 2;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= L * L) return;
    const int r = idx / L, c = idx - r * L;
    const int s = r < c ? 1 : 0;                             // S_nm = anm[m - 1][n], C_nm = anm[n][m]
    const int n = s ? c : r, m = s ? r + 1 : c;
    const double q0 = grad_q(n), q1 = grad_q(n + 1);
    const int e0 = blockIdx.y * GC_EB;
    const int e1 = e0 + GC_EB < E ? e0 + GC_EB : E;
    for (int e = e0; e < e1; ++e) {
        double v = 0.0;
#pragma unroll
        for (int pair = 0; pair < 6; ++pair) {
            const double* g = in + ((size_t)e * 6 + pair) * Lo * Lo;
            // packed position of (n + 2, mp, sp): C at [n + 2][mp], S at [mp - 1][n + 2]
            v = __dadd_rn(v, gbgrad::apply_pair(gbgrad::pair_a(pair), gbgrad::pair_b(pair), n, m, s, q0, q1,
                                                [&](int mp, int sp) {
                                                    return g[sp ? (mp - 1) * Lo + n + 2 : (n + 2) * Lo + mp];
                                                }));
        }
        anm[(size_t)e * L * L + idx] = v;
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
    return rotate_sets<ToLocal>("gb_rotate_to_local", d_xyz, d_frame, n_sets, n_points, device, stream);
}

extern "C" int gb_rotate_from_local(double* d_xyz, const double* d_frame, int n_sets, int64_t n_points, int device,
                                    void* stream) {
    return rotate_sets<FromLocal>("gb_rotate_from_local", d_xyz, d_frame, n_sets, n_points, device, stream);
}

extern "C" int gb_gradient_coefficients_adjoint(const double* d_in, int n_sets, int nmax, double* d_anm, int device,
                                                void* stream) {
    GB_REQUIRE(n_sets >= 0 && nmax >= 0, "gb_gradient_coefficients_adjoint: negative size (n_sets=%d, nmax=%d)", n_sets,
               nmax);
    if (n_sets == 0) return GB_OK;
    GB_REQUIRE(d_in && d_anm, "gb_gradient_coefficients_adjoint: NULL device pointer");
    GB_REQUIRE(nmax < 8192, "gb_gradient_coefficients_adjoint: nmax=%d too large (at most 8191)", nmax);
    const int eb = (n_sets + GC_EB - 1) / GC_EB;
    GB_REQUIRE(eb <= 65535, "gb_gradient_coefficients_adjoint: at most %d sets per call", 65535 * GC_EB);
    GB_CUDA(cudaSetDevice(device));
    const int L = nmax + 1;
    dim3 grid((L * L + 255) / 256, eb);
    gb_gradient_coefficients_adjoint_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(d_in, d_anm, L, n_sets);
    GB_LAUNCH_CHECK();
    return GB_OK;
}

extern "C" int gb_gravity_gradient_coefficients(const double* d_anm, int n_sets, int nmax, double* d_out, int device,
                                                void* stream) {
    GB_REQUIRE(n_sets >= 0 && nmax >= 0, "gb_gravity_gradient_coefficients: negative size (n_sets=%d, nmax=%d)", n_sets,
               nmax);
    if (n_sets == 0) return GB_OK;
    GB_REQUIRE(d_anm && d_out, "gb_gravity_gradient_coefficients: NULL device pointer");
    GB_REQUIRE(nmax < 8192, "gb_gravity_gradient_coefficients: nmax=%d too large (at most 8191)", nmax);
    const int eb = (n_sets + GC_EB - 1) / GC_EB;
    GB_REQUIRE(eb <= 65535, "gb_gravity_gradient_coefficients: at most %d sets per call", 65535 * GC_EB);
    GB_CUDA(cudaSetDevice(device));
    const int L = nmax + 1;
    const int per_set = 6 * (L + 2) * (L + 2);
    dim3 grid((per_set + 255) / 256, eb);
    gb_gravity_gradient_coefficients_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(d_anm, d_out, L,
                                                                                                 n_sets);
    GB_LAUNCH_CHECK();
    return GB_OK;
}

extern "C" int gb_rotate_tensor_to_local(double* d_v, const double* d_frame, int n_sets, int64_t n_points, int device,
                                         void* stream) {
    return rotate_sets<TensorToLocal>("gb_rotate_tensor_to_local", d_v, d_frame, n_sets, n_points, device, stream);
}

extern "C" int gb_gravity_gradient_coefficients_adjoint(const double* d_in, int n_sets, int nmax, double* d_anm,
                                                        int device, void* stream) {
    GB_REQUIRE(n_sets >= 0 && nmax >= 0, "gb_gravity_gradient_coefficients_adjoint: negative size (n_sets=%d, nmax=%d)",
               n_sets, nmax);
    if (n_sets == 0) return GB_OK;
    GB_REQUIRE(d_in && d_anm, "gb_gravity_gradient_coefficients_adjoint: NULL device pointer");
    GB_REQUIRE(nmax < 8192, "gb_gravity_gradient_coefficients_adjoint: nmax=%d too large (at most 8191)", nmax);
    const int eb = (n_sets + GC_EB - 1) / GC_EB;
    GB_REQUIRE(eb <= 65535, "gb_gravity_gradient_coefficients_adjoint: at most %d sets per call", 65535 * GC_EB);
    GB_CUDA(cudaSetDevice(device));
    const int L = nmax + 1;
    dim3 grid((L * L + 255) / 256, eb);
    gb_gravity_gradient_coefficients_adjoint_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(d_in, d_anm, L,
                                                                                                         n_sets);
    GB_LAUNCH_CHECK();
    return GB_OK;
}

extern "C" int gb_rotate_tensor_from_local(double* d_v, const double* d_frame, int n_sets, int64_t n_points, int device,
                                           void* stream) {
    return rotate_sets<TensorFromLocal>("gb_rotate_tensor_from_local", d_v, d_frame, n_sets, n_points, device, stream);
}
