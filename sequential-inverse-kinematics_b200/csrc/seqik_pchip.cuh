// seqik_pchip.cuh -- the pchip slope rules and the interval search shared by the resampling kernel (seqik_kernels.cu)
// and its backward (seqik_pchip_grad.cu), so that the backward takes the forward's decisions and evaluates the forward's
// samples bit for bit.
#pragma once
#include <cuda_runtime.h>

__device__ __forceinline__ float pchip_div(float a, float b) { return __fdividef(a, b); }     // <= 2 ulp; |b| < 2^126 here
__device__ __forceinline__ double pchip_div(double a, double b) { return a / b; }
template <typename T> __device__ __forceinline__ T pchip_sign(T v) { return (T)((v > T(0)) - (v < T(0))); }
template <typename T> __device__ __forceinline__ T pchip_edge(T h0, T h1, T m0, T m1) {      // scipy PchipInterpolator._edge_case
    T d = pchip_div((T(2) * h0 + h1) * m0 - h0 * m1, h0 + h1);
    if (pchip_sign(d) != pchip_sign(m0)) d = T(0);
    else if (pchip_sign(m0) != pchip_sign(m1) && fabs(d) > T(3) * fabs(m0)) d = T(3) * m0;
    return d;
}
template <typename T> __device__ __forceinline__ T pchip_inner(T ma, T mb) {                 // _find_derivatives, interior point
    // uniform grid: w1 = w2 = 3 h, so 1 / ((w1 / ma + w2 / mb) / (w1 + w2)) is the harmonic mean 2 ma mb / (ma + mb)
    if (pchip_sign(ma) != pchip_sign(mb) || ma == T(0) || mb == T(0)) return T(0);
    return pchip_div(T(2) * ma * mb, ma + mb);
}

// Samples u of the new grid in interval k, xk = k ts <= u new_ts < xk1 = (k + 1) ts (the same comparisons as scipy's
// interval search, in float64), as [u_lo, u_hi); the last interval k = n - 2 also takes the samples past the last knot.
__device__ __forceinline__ void pchip_bounds(int k, int n, int m, double xk, double xk1, double new_ts, double inv_new_ts,
                                             int& lo, int& hi) {
    // (local copies: assigning through the references directly changed the forward kernel's register allocation)
    int u_lo = (int)ceil(xk * inv_new_ts), u_hi = (int)ceil(xk1 * inv_new_ts);
    while (u_lo > 0 && (double)(u_lo - 1) * new_ts >= xk) --u_lo;
    while ((double)u_lo * new_ts < xk) ++u_lo;
    while (u_hi > 0 && (double)(u_hi - 1) * new_ts >= xk1) --u_hi;
    while ((double)u_hi * new_ts < xk1) ++u_hi;
    if (k == n - 2) u_hi = m;                               // the last piece is extrapolated over the rest of the grid
    u_hi = min(u_hi, m); u_lo = min(u_lo, u_hi);
    lo = u_lo; hi = u_hi;
}

constexpr int PCHIP_STAGE_BYTES = 32768;
