// seqik_pchip_grad.cu -- seqik_pchip_resample_backward_f32/_f64 (include/seqik.h): the backward (vector-Jacobian product)
// of the pchip resampler.  A translation unit of its own, so that adding it leaves the code generated for seqik_kernels.cu
// unchanged.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <cuda_pipeline.h>

#include "../../include/seqik.h"
#include "seqik_common.h"
#include "seqik_pchip.cuh"

// Partial derivatives of the knot slopes on the branch the forward took (its decisions recomputed with its arithmetic).
// Interior knot, d = 2 a b / (a + b): dd/da = 2 b^2 / (a + b)^2, dd/db = 2 a^2 / (a + b)^2; 0 where the forward zeroed d.
template <typename T> __device__ __forceinline__ void pchip_inner_grad(T ma, T mb, T& ga, T& gb) {
    if (pchip_sign(ma) != pchip_sign(mb) || ma == T(0) || mb == T(0)) { ga = T(0); gb = T(0); return; }
    const T r = T(1) / (ma + mb), pa = ma * r, pb = mb * r;
    ga = T(2) * pb * pb; gb = T(2) * pa * pa;
}
// End knot, uniform grid: d = (3 m0 - m1) / 2; zeroed: 0; clamped to 3 m0: dd/dm0 = 3, dd/dm1 = 0.
template <typename T> __device__ __forceinline__ void pchip_edge_grad(T h, T m0, T m1, T& g0, T& g1) {
    const T d = pchip_div((T(2) * h + h) * m0 - h * m1, h + h);                          // pchip_edge(h, h, m0, m1)
    if (pchip_sign(d) != pchip_sign(m0)) { g0 = T(0); g1 = T(0); }
    else if (pchip_sign(m0) != pchip_sign(m1) && fabs(d) > T(3) * fabs(m0)) { g0 = T(3); g1 = T(0); }
    else { g0 = T(1.5); g1 = T(-0.5); }
}

// A sample at offset s in interval k is y_k + d_k s + c1 s^2 + c0 s^3 with m_k = (y_{k+1} - y_k) / h,
// c1 = (3 m_k - 2 d_k - d_{k+1}) / h, c0 = (d_k + d_{k+1} - 2 m_k) / h^2.  With the moments M_p = sum_u g_u s_u^p of the
// interval's samples, A = M2 / h and B = M3 / h^2:
//   dL/dy_k (direct) = M0,  dL/dd_k (left) = M1 - 2 A + B,  dL/dd_{k+1} (right) = B - A,  dL/dm_k (direct) = 3 A - 2 B.
// The knot slopes' partials chain these into G_m[k] = dL/dm_k, and dL/dy_i = M0[i] + (G_m[i-1] - G_m[i]) / h.  d_i depends
// on m_{i-1} and m_i (d_0 on m_0, m_1; d_{n-1} on m_{n-2}, m_{n-3}), so y_i needs the moments of intervals i-2 .. i+1.
//
// Mapping (that of the forward): one thread per (interval, channel) in four phases separated by barriers:
//   1. moments of one interval (its samples staged in shared memory like the forward's output, or read directly when the
//      range is too long for the buffer), and the slope partials of its left knot (interval n-2: also of knot n-1);
//   2. per knot, Gd = dL/dd (the right term of the interval on its left + the left term of its own) times the partials;
//   3. per interval, G_m = its direct term + the knot terms of its two knots (+ those of the end knots that reach it);
//   4. per owned knot, dL/dy.
// A CTA owns `owned` knots and works on owned + 3 intervals (2 to the left, 1 to the right), so no knot needs another
// CTA's result: one launch, no atomics, no scratch; the last CTA also writes knot n - 1.  Unlike the forward, a CTA
// whose intervals hold no sample (down-sampling) does not return: its knots still get the slope terms.
// Shared memory (dynamic): two staging buffers of stage_cap elements, then four per-interval arrays of S x width and two per-knot
// arrays of (S + 1) x width (S = owned + 3).
// Minimum CTAs per SM: without one, ptxas (CUDA 12.9) spilled the <float, 0> and <double, 1> instantiations at 64 and
// 40 registers; with it, 48 registers for W = 7 (five CTAs per SM) and at most 64 for the others, no spills.
template <typename T, int W>
__global__ void __launch_bounds__(256, W == 7 ? 5 : 4) pchip_backward_kernel(const T* __restrict__ in, const T* __restrict__ grad_out,
                                                             T* __restrict__ grad_in, int64_t n_block, int n, int m,
                                                             int width_rt, int owned, int stage_cap, double ts,
                                                             double new_ts, double inv_new_ts) {
    extern __shared__ __align__(16) unsigned char pchip_smem[];
    __shared__ int s_first, s_end;
    const int width = W ? W : width_rt;
    const int kpt = 256 / width;                                 // thread groups (one interval or knot each)
    const int S = owned + 3;
    T* stage = reinterpret_cast<T*>(pchip_smem);
    T* sM0 = stage + 2 * stage_cap;                              // per interval slot: M0, dL/dd left, dL/dd right, dL/dm
    T* sGl = sM0 + S * width;
    T* sGr = sGl + S * width;
    T* sGm = sGr + S * width;
    T* sLo = sGm + S * width;                                    // per knot slot: dd_k/dm_{k-1}, dd_k/dm_k (knot 0: dd/dm1
    T* sHi = sLo + (S + 1) * width;                              // in sLo; knot n-1: dd/dm_{n-3} in sHi), then x Gd
    const int kl = (int)threadIdx.x / width, j = (int)threadIdx.x - kl * width;
    const bool group = kl < kpt;
    const int k0 = (int)blockIdx.x * owned, kbase = k0 - 2;     // owned knots k0 .. k0 + owned - 1; slot t = k - kbase
    const bool last = blockIdx.x == gridDim.x - 1;
    const int n_own = min(owned, n - 1 - k0) + (last ? 1 : 0);
    if (threadIdx.x == 0) {
        int lo, hi, dummy;
        const int ka = max(kbase, 0), kb = min(kbase + S - 1, n - 2);
        pchip_bounds(ka, n, m, (double)ka * ts, (double)(ka + 1) * ts, new_ts, inv_new_ts, lo, dummy);
        pchip_bounds(kb, n, m, (double)kb * ts, (double)(kb + 1) * ts, new_ts, inv_new_ts, dummy, hi);
        s_first = lo; s_end = hi;
    }
    // the interval bounds of the thread's first slot, computed once (every slot when S <= kpt, i.e. width <= 64)
    int lo0 = 0, hi0 = 0;
    {
        const int k = kbase + kl;
        if (group && kl < S && k >= 0 && k <= n - 2)
            pchip_bounds(k, n, m, (double)k * ts, (double)(k + 1) * ts, new_ts, inv_new_ts, lo0, hi0);
    }
    __syncthreads();
    const int first = s_first, n_out = (s_end - first) * width;  // the CTA's grad_out range [first, s_end) x width
    constexpr int V = 16 / (int)sizeof(T);
    const bool staged = n_out + V - 1 <= stage_cap;
    const bool use_stage = staged && n_out > 0;
    const T h = (T)ts, rh = (T)(1.0 / ts);
    // grad_out range of block row bb -> buf, asynchronously (cp.async), coalesced and 128-bit where the source allows it:
    // element e goes to buf[off + e], so that the 16-byte lines of the source and of the buffer coincide
    auto stage_row = [&](int64_t bb, T* buf) {
        const T* src = grad_out + (bb * m + first) * width;
        const int off = (int)(((uintptr_t)src / sizeof(T)) % V);
        T* st = buf + off;
        const int head = min((V - off) % V, n_out), nv = (n_out - head) / V;
        for (int i = threadIdx.x; i < head; i += blockDim.x) __pipeline_memcpy_async(st + i, src + i, sizeof(T));
        for (int i = threadIdx.x; i < nv; i += blockDim.x) __pipeline_memcpy_async(st + head + i * V, src + head + i * V, 16);
        for (int i = head + nv * V + threadIdx.x; i < n_out; i += blockDim.x) __pipeline_memcpy_async(st + i, src + i, sizeof(T));
        __pipeline_commit();
    };
    // double buffer: the copy of the next block row this CTA handles is in flight while it works on the current one
    int cur = 0;
    if (use_stage && blockIdx.y < n_block) stage_row(blockIdx.y, stage);
    for (int64_t b = blockIdx.y; b < n_block; b += gridDim.y) {
        const T* y = in + b * n * width + j;
        const T* src = grad_out + (b * m + first) * width;
        const T* g = src;                                        // sample u of the range at g[(u - first) * width + j]
        if (use_stage) {
            if (b + gridDim.y < n_block) { stage_row(b + gridDim.y, stage + (cur ^ 1) * stage_cap); __pipeline_wait_prior(1); }
            else __pipeline_wait_prior(0);
            g = stage + cur * stage_cap + (int)(((uintptr_t)src / sizeof(T)) % V);
            __syncthreads();
        }
        // 1. moments and slope partials, per interval slot
        if (group) {
            for (int t = kl; t < S; t += kpt) {
                const int k = kbase + t;
                if (k < 0 || k > n - 2) continue;
                int u_lo = lo0, u_hi = hi0;
                const double xk = (double)k * ts;
                if (t != kl) pchip_bounds(k, n, m, xk, (double)(k + 1) * ts, new_ts, inv_new_ts, u_lo, u_hi);
                T M0 = T(0), M1 = T(0), M2 = T(0), M3 = T(0);
                const T* gp = g + (u_lo - first) * width + j;
                if (sizeof(T) == 4) {
                    // the forward's float32 offsets: the first in float64, then one multiply-add per sample
                    const float s0 = (float)((double)u_lo * new_ts - xk), dt = (float)new_ts;
                    float ur = 0.f;
                    for (int u = u_lo; u < u_hi; ++u, gp += width, ur += 1.f) {
                        const float s = fmaf(ur, dt, s0);
                        const float gv = (float)*gp, gs = gv * s, gss = gs * s;
                        M0 += gv; M1 += gs; M2 += gss; M3 += gss * s;
                    }
                } else {
                    for (int u = u_lo; u < u_hi; ++u, gp += width) {
                        const T s = (T)((double)u * new_ts - xk);
                        const T gv = *gp, gs = gv * s, gss = gs * s;
                        M0 += gv; M1 += gs; M2 += gss; M3 += gss * s;
                    }
                }
                const T A = M2 * rh, B = M3 * rh * rh;
                const int si = t * width + j;
                sM0[si] = M0;
                sGl[si] = M1 - T(2) * A + B;
                sGr[si] = B - A;
                sGm[si] = T(3) * A - T(2) * B;
                // the forward's secant slopes and the partials of the knot slopes it took
                const T* yk = y + (int64_t)k * width;
                const T y0 = __ldg(yk), y1 = __ldg(yk + width);
                const T slope = (y1 - y0) * rh;
                T lo, hi, lo_n = T(0), hi_n = T(0);                      // knot k; knot n-1 (k == n-2)
                if (n == 2) { lo = T(0); hi = T(1); lo_n = T(1); }
                else {
                    const T m_prev = (k > 0) ? (y0 - __ldg(yk - width)) * rh : T(0);
                    const T m_next = (k + 2 < n) ? (__ldg(yk + 2 * width) - y1) * rh : T(0);
                    if (k > 0) pchip_inner_grad(m_prev, slope, lo, hi);
                    else pchip_edge_grad(h, slope, m_next, hi, lo);
                    if (k + 2 == n) pchip_edge_grad(h, slope, m_prev, lo_n, hi_n);
                }
                sLo[si] = lo; sHi[si] = hi;
                if (k == n - 2) { sLo[si + width] = lo_n; sHi[si + width] = hi_n; }
            }
        }
        __syncthreads();
        // 2. per knot slot: Gd times the partials (knots 1 .. S - 1 of the slots, and knot 0 / n - 1 where they lie here)
        if (group) {
            for (int t = kl; t <= S; t += kpt) {
                const int k = kbase + t;
                if (k < 0 || k > n - 1 || (t == 0 && k != 0) || (t == S && k != n - 1)) continue;
                const int si = t * width + j;
                T gd = T(0);
                if (k >= 1) gd = sGr[si - width];
                if (k <= n - 2) gd += sGl[si];
                sLo[si] *= gd; sHi[si] *= gd;
            }
        }
        __syncthreads();
        // 3. per interval slot: G_m = direct + right partial of knot k + left partial of knot k + 1 (+ the end knots')
        if (group) {
            for (int t = kl; t <= owned + 1; t += kpt) {
                const int k = kbase + t;
                if (t == 0 || k < 0 || k > n - 2) continue;
                const int si = t * width + j;
                T gm = sGm[si] + sHi[si] + sLo[si + width];
                if (k == 1) gm += sLo[si - width];                      // d_0 depends on m_1
                if (k == n - 3) gm += sHi[si + 2 * width];              // d_{n-1} depends on m_{n-3}
                sGm[si] = gm;
            }
        }
        __syncthreads();
        // 4. per owned knot: dL/dy_i = M0[i] + (G_m[i-1] - G_m[i]) / h
        if (group) {
            for (int c = kl; c < n_own; c += kpt) {
                const int k = k0 + c, si = (c + 2) * width + j;
                T gy = T(0), gm = T(0);
                if (k >= 1) gm = sGm[si - width];
                if (k <= n - 2) { gy = sM0[si]; gm -= sGm[si]; }
                grad_in[(b * n + k) * width + j] = gy + gm * rh;
            }
        }
        __syncthreads();                                         // also: the buffer just read may be refilled next
        cur ^= 1;
    }
}

template <typename T>
static int pchip_backward_launch(const char* me, const T* in, const T* grad_out, T* grad_in, int64_t n_block, int64_t n,
                                 int64_t m, int64_t width, double original_ts, double new_ts, void* stream) {
    if (n_block < 0 || n < 0 || m < 0 || width < 0) return seqik_fail(SEQIK_EINVAL, "%s: negative size", me);
    if (n_block == 0 || width == 0) return SEQIK_OK;
    if (n < 2) return seqik_fail(SEQIK_EINVAL, "%s: at least 2 samples are needed", me);
    if (!in || !grad_out || !grad_in) return seqik_fail(SEQIK_EINVAL, "%s: NULL pointer", me);
    if (!(original_ts > 0.0) || !(new_ts > 0.0)) return seqik_fail(SEQIK_EINVAL, "%s: time steps must be positive", me);
    if (n * width > 2147483647LL || m * width > 2147483647LL) return seqik_fail(SEQIK_EINVAL, "%s: series too long for one launch", me);
    if (width > 256) return seqik_fail(SEQIK_EINVAL, "%s: at most 256 interleaved channels", me);
    const int64_t owned = 256 / width > 4 ? 256 / width - 3 : 1;
    const int64_t S = owned + 3;
    const int64_t gx = (n - 1 + owned - 1) / owned;
    int64_t gy = (1LL << 20) / (gx * 256);
    gy = gy < 1 ? 1 : (gy > n_block ? n_block : gy);
    if (gy > 65535) gy = 65535;
    // staging buffer: a CTA's grad_out range (S intervals and the extrapolated tail, one sample of slack each) + alignment
    // room, at most PCHIP_STAGE_BYTES; a longer range is read directly (same bits)
    constexpr int V = 16 / (int)sizeof(T), CAP = PCHIP_STAGE_BYTES / (int)sizeof(T);
    const double need = ((double)(S + 1) * (ceil(original_ts / new_ts) + 1.0) + 2.0) * (double)width + V;
    const int stage_cap = need >= CAP ? CAP : ((int)need + V - 1) / V * V;
    const size_t smem = ((size_t)2 * stage_cap + (size_t)(4 * S + 2 * (S + 1)) * (size_t)width) * sizeof(T);
    const dim3 grid((unsigned)gx, (unsigned)gy);
    const double inv_new = 1.0 / new_ts;
    cudaStream_t st = (cudaStream_t)stream;
    auto kernel = width == 7 ? pchip_backward_kernel<T, 7> : width == 1 ? pchip_backward_kernel<T, 1> : pchip_backward_kernel<T, 0>;
    if (smem > 48 * 1024) {                                      // wide run-time widths (up to 85 KB in float64)
        const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return seqik_check_launch(me);
    }
    kernel<<<grid, 256, smem, st>>>(in, grad_out, grad_in, n_block, (int)n, (int)m, (int)width, (int)owned, stage_cap,
                                    original_ts, new_ts, inv_new);
    return seqik_check_launch(me);
}
extern "C" int seqik_pchip_resample_backward_f32(const float* in, const float* grad_out, float* grad_in, int64_t n_block,
                                                 int64_t n, int64_t m, int64_t width, double original_ts, double new_ts,
                                                 void* stream) {
    return pchip_backward_launch<float>("seqik_pchip_resample_backward_f32", in, grad_out, grad_in, n_block, n, m, width,
                                        original_ts, new_ts, stream);
}
extern "C" int seqik_pchip_resample_backward_f64(const double* in, const double* grad_out, double* grad_in, int64_t n_block,
                                                 int64_t n, int64_t m, int64_t width, double original_ts, double new_ts,
                                                 void* stream) {
    return pchip_backward_launch<double>("seqik_pchip_resample_backward_f64", in, grad_out, grad_in, n_block, n, m, width,
                                         original_ts, new_ts, stream);
}
