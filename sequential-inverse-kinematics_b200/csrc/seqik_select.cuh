// seqik_select.cuh -- the order keys and the mid-quantile ranks and weights, shared by the statistics kernels of AlignPose
// (seqik_kernels.cu) and their backward (seqik_align_grad.cu), so that the backward selects on the forward's keys and ranks.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

__device__ __forceinline__ uint32_t order_key(float f) {
    // The bits go through an opaque move.  From __float_as_uint(f), the compiler turned `u | 0x80000000` into a float
    // negation of |f| (FADD -|f|, -0), which makes a NaN the canonical 0x7fffffff: a key just below +0's, inside any range
    // that straddles zero (the long kernel's NaN padding of its float4 sweeps included).
    uint32_t u;
    asm("mov.b32 %0, %1;" : "=r"(u) : "f"(f));
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_value(uint32_t k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// ranks of numpy.quantile(..., method="linear") at q = 0.45 and 0.55: floor(q (n-1)) and the next one
__device__ __forceinline__ void quantile_pos(double q, int64_t n, int64_t& lo, float& frac) {
    const double v = q * (double)(n - 1);
    lo = (int64_t)floor(v);
    if (lo > n - 1) lo = n - 1;
    frac = (float)(v - (double)lo);
}

// the four ranks of the mid-quantile of the m smallest keys, and the interpolation weights (numpy "linear").  The ranks
// come out non-decreasing, as warp_select4 and the long kernel's bin search require: for m = 2, 4, 6, 8, 10 both positions
// have the same lower neighbour (lo45 == lo55), and lo, lo + 1, lo, lo + 1 is selected as lo, lo, lo + 1, lo + 1.  The
// return value says so; mid_quantile_value puts the middle two back.
__device__ __forceinline__ bool mid_quantile_ranks(int64_t m, unsigned int* rank, float& f45, float& f55) {
    int64_t lo45, lo55;
    quantile_pos(0.45, m, lo45, f45); quantile_pos(0.55, m, lo55, f55);
#pragma unroll
    for (int k = 0; k < 4; ++k) { const int64_t r = (k < 2 ? lo45 : lo55) + (k & 1); rank[k] = (unsigned int)(r > m - 1 ? m - 1 : r); }
    const bool swap = rank[1] > rank[2];
    if (swap) { const unsigned int t = rank[1]; rank[1] = rank[2]; rank[2] = t; }
    return swap;
}
