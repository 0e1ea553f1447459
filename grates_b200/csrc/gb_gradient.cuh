// Factors of Cunningham's relation and the rotation to (east, north, up), shared by the gradient transform
// (gb_gradient.cu) and the Jacobian tiles of the gradient covariance (gb_points.cu): both must use the same expressions.
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

}  // namespace gbgrad
