// Factors of Cunningham's relation and the rotation to (east, north, up), shared by the gradient and gravity gradient
// transforms, their rotations and the transpose (gb_gradient.cu) and the Jacobian rows of the gradient covariance and
// normal equations (gb_points.cu): all must use the same expressions.
#pragma once
#include "gb_common.cuh"

namespace gbgrad {

constexpr double SQRT2 = 1.41421356237309504880;   // == sqrt(2.0) correctly rounded

// Factors in one fixed expression order, every operation rounded on its own (no contraction):
//   q  = (2n+1) / (2n+3)
//   f  = sqrt(p * q) * 0.5 [* sqrt2]   p = the integer product of the table, converted exactly to double
__device__ __forceinline__ double grad_q(int n) { return __ddiv_rn((double)(2 * n + 1), (double)(2 * n + 3)); }

__device__ __forceinline__ double grad_fz(int n, int m, double q) {
    return __dsqrt_rn(__dmul_rn((double)(n - m + 1) * (double)(n + m + 1), q));
}

__device__ __forceinline__ double grad_fp(int n, int m, double q) {
    const double f = __dmul_rn(__dsqrt_rn(__dmul_rn((double)(n + m + 1) * (double)(n + m + 2), q)), 0.5);
    return m == 0 ? __dmul_rn(f, SQRT2) : f;
}

__device__ __forceinline__ double grad_fm(int n, int m, double q) {
    const double f = __dmul_rn(__dsqrt_rn(__dmul_rn((double)(n - m + 1) * (double)(n - m + 2), q)), 0.5);
    return m == 1 ? __dmul_rn(f, SQRT2) : f;
}

// The outputs of component c (0 x, 1 y, 2 z) that the input (n, m, s) (s = 1: sine) reaches at degree n + 1, i.e. the
// transform read backwards: at most two terms f1 out(n+1, m1, s1) and f2 out(n+1, m2, s2) (the fp / fz term, then the fm
// term; has2 = false: none).  Every T-shaped product -- the transposed transform, the Jacobian rows F'_p T -- is
//   v = f1 x(m1, s1);  if (has2) v = v + f2 x(m2, s2)        (each product and sum rounded on its own)
//   z  -fz (n+1, m, s)
//   x  -fp (n+1, m+1, s)  + fm (n+1, m-1, s)            (m >= 1; a sine of order 0 does not exist)
//   y  cosine: -fp (n+1, m+1, S) - fm (n+1, m-1, S)      sine: +fp (n+1, m+1, C) + fm (n+1, m-1, C)
struct Terms {
    double f1, f2;
    int m1, s1, m2, s2;
    bool has2;
};

__device__ __forceinline__ Terms grad_terms(int c, int n, int m, int s, double q) {
    Terms t;
    t.f2 = 0.0;
    t.m2 = m - 1;
    t.has2 = false;
    if (c == 2) {
        t.f1 = -grad_fz(n, m, q);
        t.m1 = m;
        t.s1 = t.s2 = s;
        return t;
    }
    const double fp = grad_fp(n, m, q);
    t.m1 = m + 1;
    if (c == 0) {
        t.f1 = -fp;
        t.s1 = t.s2 = s;
        if (m >= 1 && (s == 0 || m >= 2)) { t.f2 = grad_fm(n, m, q); t.has2 = true; }
    } else if (s == 0) {
        t.f1 = -fp;
        t.s1 = t.s2 = 1;
        if (m >= 2) { t.f2 = -grad_fm(n, m, q); t.has2 = true; }
    } else {
        t.f1 = fp;
        t.s1 = t.s2 = 0;
        t.f2 = grad_fm(n, m, q);
        t.has2 = true;
    }
    return t;
}

// v = f1 x(m1, s1) [+ f2 x(m2, s2)] for a reader x(order, sine) of the degree-(n+1) values
template <class Read>
__device__ __forceinline__ double apply(const Terms& t, Read x) {
    double v = __dmul_rn(t.f1, x(t.m1, t.s1));
    if (t.has2) v = __dadd_rn(v, __dmul_rn(t.f2, x(t.m2, t.s2)));
    return v;
}

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

// The transpose: (east, north, up) -> (gx, gy, gz)
//   gx = -sl east - ct cl north + st cl up
//   gy =  cl east - ct sl north + st sl up
//   gz =            st north    + ct up          each product and sum rounded on its own, left to right
__device__ __forceinline__ void rotate_back(const Frame& f, double& east, double& north, double& up) {
    const double gx = __dadd_rn(__dadd_rn(__dmul_rn(-f.sl, east), __dmul_rn(__dmul_rn(-f.ct, f.cl), north)),
                                __dmul_rn(__dmul_rn(f.st, f.cl), up));
    const double gy = __dadd_rn(__dadd_rn(__dmul_rn(f.cl, east), __dmul_rn(__dmul_rn(-f.ct, f.sl), north)),
                                __dmul_rn(__dmul_rn(f.st, f.sl), up));
    const double gz = __dadd_rn(__dmul_rn(f.st, north), __dmul_rn(f.ct, up));
    east = gx;
    north = gy;
    up = gz;
}

template <bool TO_LOCAL>
__device__ __forceinline__ void rotate_dir(const Frame& f, double& a, double& b, double& c) {
    if constexpr (TO_LOCAL) rotate(f, a, b, c);
    else rotate_back(f, a, b, c);
}

// Q M Q' of a 3 x 3 matrix in place: rotate on the three columns of M, then on the three rows of the result.  Even for a
// symmetric M the result is symmetric only to rounding; callers keep one triangle or symmetrise.
__device__ __forceinline__ void rotate_matrix(const Frame& f, double (&M)[3][3]) {
#pragma unroll
    for (int j = 0; j < 3; ++j) rotate(f, M[0][j], M[1][j], M[2][j]);
#pragma unroll
    for (int j = 0; j < 3; ++j) rotate(f, M[j][0], M[j][1], M[j][2]);
}

}  // namespace gbgrad
