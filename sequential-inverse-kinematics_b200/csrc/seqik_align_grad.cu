// seqik_align_grad.cu -- seqik_align_apply_backward_f32, seqik_leg_affine_backward_f32, seqik_head_apply_backward_f32 and
// seqik_head_affine_backward_f32/_f64 (include/seqik.h): the backward (vector-Jacobian products) of the leg and head
// alignment, i.e. of the affine maps of AlignPose.align_leg / align_head and of the mid-quantile statistics their rows come
// from.  A translation unit of its own, so that adding it leaves the code generated for seqik_kernels.cu unchanged.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/seqik.h"
#include "seqik_common.h"
#include "seqik_select.cuh"
#include "seqik_stream.cuh"

// ---- align_apply backward ---------------------------------------------------------------------------------------------------
// One leg-frame: p = its 15 pose floats, g = its 15 dL/dout floats, a = the chain's affine row -> gp = dL/dpose (15 floats) and
// part = its contribution to dL/daffine (8 floats), in the order the header states:
//   S_c = ((g1c + g2c) + g3c) + g4c,  D = ((d1 + d2) + d3) + d4 with d_i = ((p_ix - a0) g_ix + (p_iy - a1) g_iy) + (p_iz - a2) g_iz,
//   part = (-(a3 S_x), -(a3 S_y), -(a3 S_z), D, g0x + S_x, g0y + S_y, g0z + S_z, 0),  gp = (0, 0, 0, a3 g_1.., .., a3 g_4..)
__device__ __forceinline__ void apply_backward_row(const float* p, const float* g, const float* __restrict__ a, float* gp, float* part) {
    const float f0 = __ldg(a), f1 = __ldg(a + 1), f2 = __ldg(a + 2), sc = __ldg(a + 3);
    gp[0] = 0.f; gp[1] = 0.f; gp[2] = 0.f;
    float sx = 0.f, sy = 0.f, sz = 0.f, d = 0.f;
#pragma unroll
    for (int i = 1; i < 5; ++i) {
        const float gx = g[3 * i], gy = g[3 * i + 1], gz = g[3 * i + 2];
        gp[3 * i] = sc * gx; gp[3 * i + 1] = sc * gy; gp[3 * i + 2] = sc * gz;
        const float di = ((p[3 * i] - f0) * gx + (p[3 * i + 1] - f1) * gy) + (p[3 * i + 2] - f2) * gz;
        if (i == 1) { sx = gx; sy = gy; sz = gz; d = di; }
        else { sx = sx + gx; sy = sy + gy; sz = sz + gz; d = d + di; }
    }
    part[0] = -(sc * sx); part[1] = -(sc * sy); part[2] = -(sc * sz); part[3] = d;
    part[4] = g[0] + sx; part[5] = g[1] + sy; part[6] = g[2] + sz; part[7] = 0.f;
}

// Plain kernel (strided or unaligned pose, unaligned buffers, totals below one tile, the tail of the tile path): one thread per
// leg-frame, straight from global memory.  Every output is computed; the NULL ones are not stored.
__global__ void __launch_bounds__(TILE) align_apply_backward_kernel(const float* __restrict__ pose, int64_t cs, int64_t fs,
                                                                    const float* __restrict__ affine, const float* __restrict__ grad_out,
                                                                    float* __restrict__ grad_pose, float* __restrict__ part,
                                                                    int64_t n_chain, int64_t n_frame, int64_t first) {
    const int64_t lf = first + (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (lf >= n_chain * n_frame) return;
    const int64_t c = lf / n_frame, t = lf - c * n_frame;
    float p[15], g[15], gp[15], pa[8];
#pragma unroll
    for (int k = 0; k < 15; ++k) { p[k] = __ldg(pose + c * cs + t * fs + k); g[k] = __ldg(grad_out + lf * 15 + k); }
    apply_backward_row(p, g, affine + c * 8, gp, pa);
    if (grad_pose) {
#pragma unroll
        for (int k = 0; k < 15; ++k) grad_pose[lf * 15 + k] = gp[k];
    }
    if (part) {
#pragma unroll
        for (int k = 0; k < 8; ++k) part[lf * 8 + k] = pa[k];
    }
}

// Tile path (dense pose, 16-byte aligned buffers): pose and dL/dout in (30 KB a tile), dL/dpose and the partial rows out (23 KB);
// 53 KB a stage, two CTAs per SM.  A tile may straddle chains: each leg-frame reads its own chain's row.
struct AlignBackwardOp {
    const float* pose; const float* affine; const float* grad_out; float* grad_pose; float* part; int64_t n_frame;
    static constexpr int N_IN = 2, G_OFF = TILE * 15 * 4, OUT_OFF = TILE * 30 * 4, PART_OFF = TILE * 15 * 4;
    static constexpr int STAGE_BYTES = OUT_OFF + TILE * 23 * 4;
    static __device__ __forceinline__ int in_off(int i) { return i == 0 ? 0 : G_OFF; }
    __device__ __forceinline__ uint32_t in_bytes(int, int64_t) const { return TILE * 15 * 4; }
    __device__ __forceinline__ const void* in_src(int i, int64_t tile) const { return (i == 0 ? pose : grad_out) + tile * (TILE * 15); }
    __device__ __forceinline__ void compute(int tid, int64_t tile, unsigned char* stage) const {
        const float* s_p = reinterpret_cast<const float*>(stage);
        const float* s_g = reinterpret_cast<const float*>(stage + G_OFF);
        unsigned char* out = stage + OUT_OFF;
        float p[15], g[15], gp[15], pa[8];
#pragma unroll
        for (int k = 0; k < 15; ++k) { p[k] = s_p[tid * 15 + k]; g[k] = s_g[tid * 15 + k]; }   // stride 15 words: conflict-free
        apply_backward_row(p, g, affine + ((tile * TILE + tid) / n_frame) * 8, gp, pa);
        float* o = reinterpret_cast<float*>(out) + tid * 15;
#pragma unroll
        for (int k = 0; k < 15; ++k) o[k] = gp[k];
        float4* o4 = reinterpret_cast<float4*>(out + PART_OFF) + 2 * tid;
        o4[0] = make_float4(pa[0], pa[1], pa[2], pa[3]); o4[1] = make_float4(pa[4], pa[5], pa[6], pa[7]);
    }
    __device__ __forceinline__ void store(int64_t tile, const unsigned char* out) const {
        if (grad_pose) tma_store_1d_nocommit(grad_pose + tile * (TILE * 15), out, TILE * 15 * 4);
        if (part) tma_store_1d_nocommit(part + tile * (TILE * 8), out + PART_OFF, TILE * 8 * 4);
    }
};

extern "C" int seqik_align_apply_backward_f32(const float* pose, int64_t pose_chain_stride, int64_t pose_frame_stride,
                                              const float* affine, const float* grad_out, float* grad_pose, float* grad_affine_partial,
                                              int64_t n_chain, int64_t n_frame, void* stream) {
    if (n_chain < 0 || n_frame < 0) return seqik_fail(SEQIK_EINVAL, "seqik_align_apply_backward_f32: negative size");
    if (n_chain == 0 || n_frame == 0) return SEQIK_OK;
    if (!pose || !affine || !grad_out) return seqik_fail(SEQIK_EINVAL, "seqik_align_apply_backward_f32: NULL pointer");
    if (pose_frame_stride < 15)
        return seqik_fail(SEQIK_EINVAL, "seqik_align_apply_backward_f32: frame stride smaller than the innermost block");
    if (!grad_pose && !grad_affine_partial) return SEQIK_OK;
    const int64_t lf_total = n_chain * n_frame, full_tiles = lf_total / TILE, done = full_tiles * TILE;
    const bool dense = pose_frame_stride == 15 && pose_chain_stride == n_frame * 15;
    const bool aligned = ((((uintptr_t)pose) | ((uintptr_t)grad_out) | ((uintptr_t)grad_pose) | ((uintptr_t)grad_affine_partial)) & 15) == 0;
    cudaStream_t st = (cudaStream_t)stream;
    if (dense && aligned && full_tiles > 0) {
        launch_tiles(AlignBackwardOp{pose, affine, grad_out, grad_pose, grad_affine_partial, n_frame}, full_tiles, st);
        if (lf_total > done)
            align_apply_backward_kernel<<<(unsigned)((lf_total - done + TILE - 1) / TILE), TILE, 0, st>>>(
                pose, pose_chain_stride, pose_frame_stride, affine, grad_out, grad_pose, grad_affine_partial, n_chain, n_frame, done);
    } else {
        align_apply_backward_kernel<<<(unsigned)((lf_total + TILE - 1) / TILE), TILE, 0, st>>>(
            pose, pose_chain_stride, pose_frame_stride, affine, grad_out, grad_pose, grad_affine_partial, n_chain, n_frame, 0);
    }
    return seqik_check_launch("seqik_align_apply_backward_f32");
}

// ---- leg_affine backward ----------------------------------------------------------------------------------------------------
// The seven series of a chain are coxa x, y, z and the four SQUARED segment lengths, as order keys (the forward's keys: the
// fused kernel selects on the squares, and the square root is monotone, so the long path's order statistics are the same).
// Per series: the four keys of the mid-quantile's ranks (sorted, mid_quantile_ranks) by a radix select that also leaves each
// rank's j = rank - #{keys below its key}, then the frame of each rank under the
// tie rule: the j-th frame in ascending order among those whose key equals the rank's.
// Per series the result is 12 words: [0, 4) the keys, [4, 8) the j's, [8, 12) the frames.
constexpr int AG_RES = 12;

// The frames of the four keys val[k] (j[k]: see above; consumed) in key[0..n), by one warp, in one ascending sweep.
static __device__ void warp_find_frames(const uint32_t* __restrict__ key, int64_t n, const uint32_t* val, unsigned int* j,
                                 uint32_t* frame, int lane) {
    const unsigned full = 0xffffffffu;
    unsigned pending = 0xFu;
    for (int64_t i0 = 0; i0 < n && pending; i0 += 32) {
        const int64_t i = i0 + lane;
        const uint32_t kk = i < n ? key[i] : 0u;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const unsigned b = __ballot_sync(full, i < n && kk == val[k]);
            if ((pending >> k) & 1u) {
                const unsigned c = __popc(b);
                if (j[k] < c) {
                    unsigned m = b;
                    for (unsigned q = 0; q < j[k]; ++q) m &= m - 1u;             // drop the j lowest set bits
                    frame[k] = (uint32_t)(i0 + __ffs(m) - 1);
                    pending &= ~(1u << k);
                } else {
                    j[k] -= c;
                }
            }
        }
    }
}

// One writer per chain, in a fixed order (series 0..6, then sorted rank position 0..3; per segment its end point before its
// base point, x, y, z): the statistics' contributions are ADDED into grad_pose.  kf: the chain's seven result rows (stride
// AG_RES words).  The mid-quantiles and len are recomputed from the selected keys with the forward's float32 arithmetic.
static __device__ void chain_scatter(const float* __restrict__ p, int64_t fs, const float* __restrict__ k, int include_claw,
                              const float* __restrict__ a, const float* __restrict__ h, const uint32_t* kf, int64_t n_frame,
                              float* __restrict__ gp, float* __restrict__ gk) {
    unsigned int rank[4]; float f45, f55;
    const bool swap = mid_quantile_ranks(n_frame, rank, f45, f55);
    float w[4] = {0.5f * (1.f - f45), 0.5f * f45, 0.5f * (1.f - f55), 0.5f * f55};     // weights of ranks lo45, lo45+1, lo55, lo55+1
    if (swap) { const float t = w[1]; w[1] = w[2]; w[2] = t; }                          // ... by sorted position
    float m[7];
#pragma unroll
    for (int s = 0; s < 7; ++s) {
        float v4[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) { v4[t] = key_value(kf[s * AG_RES + t]); if (s >= 3) v4[t] = sqrtf(v4[t]); }
        if (swap) { const float t = v4[1]; v4[1] = v4[2]; v4[2] = t; }
        const float q0 = v4[0] + (v4[1] - v4[0]) * f45, q1 = v4[2] + (v4[3] - v4[2]) * f55;
        m[s] = 0.5f * (q0 + q1);
    }
    float len = m[3] + m[4] + m[5];
    if (include_claw) len += m[6];
    const float h3 = h[3];
    if (gk) { gk[0] = h[4]; gk[1] = h[5]; gk[2] = h[6]; gk[3] = h3 / len; }
    const float dlen = -(h3 * a[3]) / len;
    const int n_series = include_claw ? 7 : 6;
    for (int s = 0; s < n_series; ++s) {
        const float gs = s < 3 ? h[s] : dlen;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float share = gs * w[i];
            const int64_t t = kf[s * AG_RES + 8 + i];
            float* g = gp + t * 15;
            if (s < 3) { g[s] += share; continue; }
            const int jj = 3 * (s - 3);
            const float* q = p + t * fs + jj;
            const float dx = q[3] - q[0], dy = q[4] - q[1], dz = q[5] - q[2];
            const float sq = dx * dx + dy * dy + dz * dz;
            if (sq == 0.f) continue;                                   // the norm's subgradient at 0
            const float coef = share / sqrtf(sq);
            const float ux = coef * dx, uy = coef * dy, uz = coef * dz;
            g[jj + 3] += ux; g[jj + 4] += uy; g[jj + 5] += uz;
            g[jj] -= ux; g[jj + 1] -= uy; g[jj + 2] -= uz;
        }
    }
}

// The keys of the four (sorted) ranks of key[0..n) -> val, and rank - #{keys below each} -> rank (the j's), by ONE warp, n <= AG_N:
// a 4-pass MSB radix select with 8-bit digits; ranks that still share a prefix share a histogram (equal prefixes are adjacent),
// the histograms packed as 16-bit counters into 2 x 256 words of this warp.  The keys are only read.
constexpr int AG_WARPS = 7, AG_THREADS = 32 * AG_WARPS, AG_N = 1024;
static __device__ void warp_rank_select(const uint32_t* __restrict__ key, int n, unsigned int* rank, unsigned int (*hist)[256],
                                        int lane, uint32_t* val) {
    const unsigned full = 0xffffffffu;
    uint32_t prefix[4] = {0u, 0u, 0u, 0u}, mask = 0u;
#pragma unroll 1
    for (int shift = 24; shift >= 0; shift -= 8) {
        int h[4];
        h[0] = 0; h[1] = (prefix[1] == prefix[0]) ? 0 : 1;
        h[2] = (prefix[2] == prefix[1]) ? h[1] : h[1] + 1;
        h[3] = (prefix[3] == prefix[2]) ? h[2] : h[2] + 1;
        for (int k = lane; k < 512; k += 32) (&hist[0][0])[k] = 0u;
        __syncwarp(full);
        for (int i = lane; i < n; i += 32) {
            const uint32_t k = key[i], km = k & mask, d = (k >> shift) & 0xFFu;
            const int hh = (km == prefix[0]) ? 0 : (km == prefix[1]) ? h[1] : (km == prefix[2]) ? h[2] : (km == prefix[3]) ? h[3] : -1;
            if (hh >= 0) atomicAdd(&hist[hh >> 1][d], 1u << (16 * (hh & 1)));
        }
        __syncwarp(full);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            // each lane sums 8 bins, a warp scan finds the lane whose cumulative count first exceeds the rank, it walks its bins
            const unsigned int* hrow = &hist[h[k] >> 1][8 * lane];
            const int sh = 16 * (h[k] & 1);
            unsigned int own = 0;
#pragma unroll
            for (int d = 0; d < 8; ++d) own += (hrow[d] >> sh) & 0xFFFFu;
            unsigned int incl = own;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) { const unsigned int t = __shfl_up_sync(full, incl, off); if (lane >= off) incl += t; }
            const unsigned int hit = __ballot_sync(full, incl > rank[k]);
            const int sel = hit ? __ffs(hit) - 1 : 31;
            unsigned int acc = incl - own; int d = 0;
            for (; d < 8; ++d) { const unsigned int hv = (hrow[d] >> sh) & 0xFFFFu; if (acc + hv > rank[k]) break; acc += hv; }
            if (d > 7) d = 7;
            const uint32_t bin = (uint32_t)__shfl_sync(full, 8 * lane + d, sel);
            const unsigned int below = __shfl_sync(full, acc, sel);
            prefix[k] |= bin << shift; rank[k] -= below;
        }
        mask |= 0xFFu << shift;
        __syncwarp(full);                                              // every lane has read the histograms
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) val[k] = prefix[k];
}

// Recordings of up to AG_N frames: one CTA of seven warps per chain, like leg_affine_fused_kernel.  The key points pass through
// shared memory to the seven key rows; warp w selects the four keys of series w (warp_rank_select) and finds their frames
// (warp_find_frames); thread 0 scatters.
__global__ void __launch_bounds__(AG_THREADS) leg_affine_backward_fused_kernel(
        const float* __restrict__ pose, int64_t cs, int64_t fs, const float* __restrict__ consts, int include_claw,
        const float* __restrict__ affine, const float* __restrict__ grad_affine, float* __restrict__ grad_pose,
        float* __restrict__ grad_consts, int n_frame) {
    __shared__ __align__(16) uint32_t key[AG_WARPS][AG_N];
    __shared__ __align__(16) union { float stage[AG_THREADS * 15]; unsigned int hist[AG_WARPS][2][256]; } u;
    __shared__ uint32_t res[AG_WARPS][AG_RES];
    const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
    const int64_t c = blockIdx.x;
    const float* src = pose + c * cs;
    const bool vec = fs == 15 && ((((uintptr_t)src) & 15) == 0);
    for (int f0 = 0; f0 < n_frame; f0 += AG_THREADS) {
        const int nf = min(AG_THREADS, n_frame - f0);
        const float* tsrc = src + (int64_t)f0 * fs;
        if (vec) {                                                     // (f0 * 60 B is a multiple of 16)
            const int n4 = nf * 15 / 4;
            for (int i = tid; i < n4; i += AG_THREADS) reinterpret_cast<float4*>(u.stage)[i] = __ldg(reinterpret_cast<const float4*>(tsrc) + i);
            for (int i = 4 * n4 + tid; i < nf * 15; i += AG_THREADS) u.stage[i] = __ldg(tsrc + i);
        } else {
            for (int i = tid; i < nf * 15; i += AG_THREADS) u.stage[i] = __ldg(tsrc + (int64_t)(i / 15) * fs + i % 15);
        }
        __syncthreads();
        if (tid < nf) {
            const float* kp = u.stage + tid * 15;
            key[0][f0 + tid] = order_key(kp[0]); key[1][f0 + tid] = order_key(kp[1]); key[2][f0 + tid] = order_key(kp[2]);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float dx = kp[3 * j + 3] - kp[3 * j], dy = kp[3 * j + 4] - kp[3 * j + 1], dz = kp[3 * j + 5] - kp[3 * j + 2];
                key[3 + j][f0 + tid] = order_key(dx * dx + dy * dy + dz * dz);
            }
        }
        __syncthreads();
    }
    unsigned int j[4]; uint32_t val[4], frame[4]; float f45, f55;
    mid_quantile_ranks(n_frame, j, f45, f55);
    warp_rank_select(key[w], n_frame, j, u.hist[w], lane, val);
    warp_find_frames(key[w], n_frame, val, j, frame, lane);
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 4; ++k) { res[w][k] = val[k]; res[w][8 + k] = frame[k]; }
    }
    __syncthreads();
    if (tid == 0)
        chain_scatter(src, fs, consts + c * 4, include_claw, affine + c * 8, grad_affine + c * 8, &res[0][0], n_frame,
                      grad_pose + c * n_frame * 15, grad_consts ? grad_consts + c * 4 : nullptr);
}

// Longer recordings, through scratch: the keys of the seven series ([n_chain * 7][n_frame] words), a block per series selects
// the four keys by a 4-pass MSB radix select that also leaves each rank's j, a warp per series finds the frames in one sweep,
// and a thread per chain scatters.
__global__ void __launch_bounds__(256) leg_keys_kernel(const float* __restrict__ pose, int64_t cs, int64_t fs,
                                                       uint32_t* __restrict__ keys, int64_t n_chain, int64_t n_frame) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_chain * n_frame) return;
    const int64_t c = i / n_frame, t = i - c * n_frame;
    const float* p = pose + c * cs + t * fs;
    float kp[15];
#pragma unroll
    for (int j = 0; j < 15; ++j) kp[j] = __ldg(p + j);
    uint32_t* s = keys + c * 7 * n_frame + t;
    s[0] = order_key(kp[0]); s[n_frame] = order_key(kp[1]); s[2 * n_frame] = order_key(kp[2]);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float dx = kp[3 * j + 3] - kp[3 * j], dy = kp[3 * j + 4] - kp[3 * j + 1], dz = kp[3 * j + 5] - kp[3 * j + 2];
        s[(3 + j) * n_frame] = order_key(dx * dx + dy * dy + dz * dz);
    }
}

// counts: NULL (every key of a row takes part), or the number m of smallest keys per row that take part (the other keys of
// the row must be larger: the head series' +inf padding); a row with m <= 0 is left alone.
constexpr int KS_BLOCK = 256;
__global__ void __launch_bounds__(KS_BLOCK) key_select_kernel(const uint32_t* __restrict__ keys, int64_t n,
                                                              const int32_t* __restrict__ counts, uint32_t* __restrict__ res) {
    __shared__ unsigned int hist[4][256];
    __shared__ uint32_t s_prefix[4]; __shared__ unsigned int s_rank[4]; __shared__ int s_hist[4];
    const int64_t sidx = blockIdx.x;
    const uint32_t* v = keys + sidx * n;
    const int64_t m = counts ? (int64_t)counts[sidx] : n;
    if (m <= 0) return;                                                // (the whole block)
    if (threadIdx.x == 0) {
        unsigned int rank[4]; float f45, f55;
        mid_quantile_ranks(m, rank, f45, f55);
        for (int k = 0; k < 4; ++k) { s_rank[k] = rank[k]; s_prefix[k] = 0u; }
    }
    uint32_t mask = 0;
    for (int pass = 3; pass >= 0; --pass) {
        const int shift = 8 * pass;
        for (int k = threadIdx.x; k < 4 * 256; k += KS_BLOCK) (&hist[0][0])[k] = 0;
        __syncthreads();
        const uint32_t p0 = s_prefix[0], p1 = s_prefix[1], p2 = s_prefix[2], p3 = s_prefix[3];
        // ranks that still share a prefix share a histogram (the ranks are sorted: equal prefixes are adjacent)
        const int h1 = (p1 == p0) ? 0 : 1, h2 = (p2 == p0) ? 0 : (p2 == p1) ? 1 : 2;
        const int h3 = (p3 == p0) ? 0 : (p3 == p1) ? 1 : (p3 == p2) ? 2 : 3;
        if (threadIdx.x == 0) { s_hist[0] = 0; s_hist[1] = h1; s_hist[2] = h2; s_hist[3] = h3; }
        for (int64_t i = threadIdx.x; i < n; i += KS_BLOCK) {
            const uint32_t k = __ldg(v + i);
            const uint32_t km = k & mask, d = (k >> shift) & 0xFF;
            if (km == p0) atomicAdd(&hist[0][d], 1u);
            if (h1 == 1 && km == p1) atomicAdd(&hist[1][d], 1u);
            if (h2 == 2 && km == p2) atomicAdd(&hist[2][d], 1u);
            if (h3 == 3 && km == p3) atomicAdd(&hist[3][d], 1u);
        }
        __syncthreads();
        if (threadIdx.x < 4 * 32) {
            // warp w: the bin of rank s_rank[w] in its histogram (each lane sums 8 bins, a warp scan finds the lane whose
            // cumulative count first exceeds the rank, that lane walks its 8 bins)
            const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
            const unsigned int* hrow = &hist[s_hist[w]][8 * lane];
            unsigned int own = 0;
#pragma unroll
            for (int d = 0; d < 8; ++d) own += hrow[d];
            unsigned int incl = own;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) { const unsigned int t = __shfl_up_sync(0xffffffffu, incl, off); if (lane >= off) incl += t; }
            const unsigned int r = s_rank[w];
            const unsigned int hit = __ballot_sync(0xffffffffu, incl > r);
            const int sel = hit ? __ffs(hit) - 1 : 31;
            if (lane == sel) {
                unsigned int acc = incl - own; int d = 0;
                for (; d < 8; ++d) { if (acc + hrow[d] > r) break; acc += hrow[d]; }
                if (d > 7) d = 7;
                s_prefix[w] |= ((uint32_t)(8 * lane + d) << shift); s_rank[w] = r - acc;
            }
        }
        mask |= 0xFFu << shift;
        __syncthreads();
    }
    if (threadIdx.x < 4) {                                             // the keys, and rank - #{keys below} (the j's)
        res[sidx * AG_RES + threadIdx.x] = s_prefix[threadIdx.x];
        res[sidx * AG_RES + 4 + threadIdx.x] = s_rank[threadIdx.x];
    }
}

constexpr int KF_WARPS = 4;
__global__ void __launch_bounds__(32 * KF_WARPS) key_frames_kernel(const uint32_t* __restrict__ keys, int64_t n, int64_t n_series,
                                                                   const int32_t* __restrict__ counts, uint32_t* __restrict__ res) {
    const int lane = threadIdx.x & 31;
    const int64_t sidx = (int64_t)blockIdx.x * KF_WARPS + (threadIdx.x >> 5);
    if (sidx >= n_series || (counts && counts[sidx] <= 0)) return;    // whole warps leave
    uint32_t* r = res + sidx * AG_RES;
    uint32_t val[4], frame[4]; unsigned int j[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) { val[k] = r[k]; j[k] = r[4 + k]; }
    warp_find_frames(keys + sidx * n, n, val, j, frame, lane);
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 4; ++k) r[8 + k] = frame[k];
    }
}

__global__ void leg_affine_backward_finish_kernel(const float* __restrict__ pose, int64_t cs, int64_t fs, const float* __restrict__ consts,
                                                  int include_claw, const float* __restrict__ affine, const float* __restrict__ grad_affine,
                                                  const uint32_t* __restrict__ res, float* __restrict__ grad_pose,
                                                  float* __restrict__ grad_consts, int64_t n_chain, int64_t n_frame) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_chain) return;
    chain_scatter(pose + c * cs, fs, consts + c * 4, include_claw, affine + c * 8, grad_affine + c * 8, res + c * 7 * AG_RES, n_frame,
                  grad_pose + c * n_frame * 15, grad_consts ? grad_consts + c * 4 : nullptr);
}

extern "C" int seqik_leg_affine_backward_f32(const float* pose, int64_t pose_chain_stride, int64_t pose_frame_stride,
                                             const float* consts, int include_claw, const float* affine, const float* grad_affine,
                                             float* grad_pose, float* grad_consts, uint32_t* scratch,
                                             int64_t n_chain, int64_t n_frame, void* stream) {
    if (n_chain < 0 || n_frame < 0) return seqik_fail(SEQIK_EINVAL, "seqik_leg_affine_backward_f32: negative size");
    if (n_chain == 0) return SEQIK_OK;
    if (n_frame == 0) return seqik_fail(SEQIK_EINVAL, "seqik_leg_affine_backward_f32: empty recording");
    if (!pose || !consts || !affine || !grad_affine || !grad_pose) return seqik_fail(SEQIK_EINVAL, "seqik_leg_affine_backward_f32: NULL pointer");
    if (pose_frame_stride < 15) return seqik_fail(SEQIK_EINVAL, "seqik_leg_affine_backward_f32: frame stride smaller than the innermost block");
    if (n_chain > 2147483647LL) return seqik_fail(SEQIK_EINVAL, "seqik_leg_affine_backward_f32: too many chains");
    cudaStream_t st = (cudaStream_t)stream;
    if (n_frame <= AG_N) {
        leg_affine_backward_fused_kernel<<<(unsigned)n_chain, AG_THREADS, 0, st>>>(pose, pose_chain_stride, pose_frame_stride, consts,
                                                                                   include_claw, affine, grad_affine, grad_pose,
                                                                                   grad_consts, (int)n_frame);
        return seqik_check_launch("seqik_leg_affine_backward_f32");
    }
    if (!scratch) return seqik_fail(SEQIK_EINVAL, "seqik_leg_affine_backward_f32: recordings of more than 1024 frames need the scratch buffer");
    const int64_t n_series = n_chain * 7;
    uint32_t* keys = scratch;
    uint32_t* res = scratch + n_series * n_frame;
    leg_keys_kernel<<<(unsigned)((n_chain * n_frame + 255) / 256), 256, 0, st>>>(pose, pose_chain_stride, pose_frame_stride, keys,
                                                                                 n_chain, n_frame);
    key_select_kernel<<<(unsigned)n_series, KS_BLOCK, 0, st>>>(keys, n_frame, nullptr, res);
    key_frames_kernel<<<(unsigned)((n_series + KF_WARPS - 1) / KF_WARPS), 32 * KF_WARPS, 0, st>>>(keys, n_frame, n_series, nullptr, res);
    leg_affine_backward_finish_kernel<<<(unsigned)((n_chain + 127) / 128), 128, 0, st>>>(pose, pose_chain_stride, pose_frame_stride, consts,
                                                                                         include_claw, affine, grad_affine, res,
                                                                                         grad_pose, grad_consts, n_chain, n_frame);
    return seqik_check_launch("seqik_leg_affine_backward_f32");
}

// ---- head_apply backward ----------------------------------------------------------------------------------------------------
// One frame: h = (base xyz, tip xyz), g = their dL/dout, a = the trial's head row -> gh = dL/dhead (6 floats) and part = the
// frame's contribution to dL/daffine (8 floats), in the order the header states:
//   gh = (a3 G_b, a7 G_t),  part = (-((a3 G_b) + (a7 G_t)), P_b . G_b, G_b + G_t, P_t . G_t),  P = point - origin,
//   x . y = ((x0 y0 + x1 y1) + x2 y2)
__device__ __forceinline__ void head_apply_backward_frame(const float* h, const float* g, const float* __restrict__ a, float* gh,
                                                          float* part) {
    const float o0 = __ldg(a), o1 = __ldg(a + 1), o2 = __ldg(a + 2), sb = __ldg(a + 3), st = __ldg(a + 7);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        gh[c] = sb * g[c]; gh[3 + c] = st * g[3 + c];
        part[c] = -(gh[c] + gh[3 + c]); part[4 + c] = g[c] + g[3 + c];
    }
    part[3] = ((h[0] - o0) * g[0] + (h[1] - o1) * g[1]) + (h[2] - o2) * g[2];
    part[7] = ((h[3] - o0) * g[3] + (h[4] - o1) * g[4]) + (h[5] - o2) * g[5];
}

// Plain kernel (unaligned buffers, totals below one tile, the tail of the tile path): one thread per frame, straight from
// global memory.  Every output is computed; the NULL ones are not stored.
__global__ void __launch_bounds__(TILE) head_apply_backward_kernel(const float* __restrict__ head, const float* __restrict__ affine,
                                                                   const float* __restrict__ grad_out, float* __restrict__ grad_head,
                                                                   float* __restrict__ part, int64_t n_frame, int64_t total,
                                                                   int64_t first) {
    const int64_t f = first + (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (f >= total) return;
    float h[6], g[6], gh[6], pa[8];
#pragma unroll
    for (int k = 0; k < 6; ++k) { h[k] = __ldg(head + f * 6 + k); g[k] = __ldg(grad_out + f * 6 + k); }
    head_apply_backward_frame(h, g, affine + (f / n_frame) * 8, gh, pa);
    if (grad_head) {
#pragma unroll
        for (int k = 0; k < 6; ++k) grad_head[f * 6 + k] = gh[k];
    }
    if (part) {
#pragma unroll
        for (int k = 0; k < 8; ++k) part[f * 8 + k] = pa[k];
    }
}

// Tile path (16-byte aligned buffers): head and dL/dout in (12 KB a tile of 256 frames), dL/dhead and the partial rows out
// (14 KB); 26 KB a stage, four CTAs per SM.  A tile may straddle trials: each frame reads its own trial's row.
struct HeadApplyBackwardOp {
    const float* head; const float* affine; const float* grad_out; float* grad_head; float* part; int64_t n_frame;
    static constexpr int N_IN = 2, G_OFF = TILE * 6 * 4, OUT_OFF = TILE * 12 * 4, PART_OFF = TILE * 6 * 4;
    static constexpr int STAGE_BYTES = OUT_OFF + TILE * 14 * 4;
    static __device__ __forceinline__ int in_off(int i) { return i == 0 ? 0 : G_OFF; }
    __device__ __forceinline__ uint32_t in_bytes(int, int64_t) const { return TILE * 6 * 4; }
    __device__ __forceinline__ const void* in_src(int i, int64_t tile) const { return (i == 0 ? head : grad_out) + tile * (TILE * 6); }
    __device__ __forceinline__ void compute(int tid, int64_t tile, unsigned char* stage) const {
        const float* s_h = reinterpret_cast<const float*>(stage);
        const float* s_g = reinterpret_cast<const float*>(stage + G_OFF);
        unsigned char* out = stage + OUT_OFF;
        float h[6], g[6], gh[6], pa[8];
#pragma unroll
        for (int k = 0; k < 6; ++k) { h[k] = s_h[tid * 6 + k]; g[k] = s_g[tid * 6 + k]; }
        head_apply_backward_frame(h, g, affine + ((tile * TILE + tid) / n_frame) * 8, gh, pa);
        float2* o2 = reinterpret_cast<float2*>(out) + 3 * tid;
        o2[0] = make_float2(gh[0], gh[1]); o2[1] = make_float2(gh[2], gh[3]); o2[2] = make_float2(gh[4], gh[5]);
        float4* o4 = reinterpret_cast<float4*>(out + PART_OFF) + 2 * tid;
        o4[0] = make_float4(pa[0], pa[1], pa[2], pa[3]); o4[1] = make_float4(pa[4], pa[5], pa[6], pa[7]);
    }
    __device__ __forceinline__ void store(int64_t tile, const unsigned char* out) const {
        if (grad_head) tma_store_1d_nocommit(grad_head + tile * (TILE * 6), out, TILE * 6 * 4);
        if (part) tma_store_1d_nocommit(part + tile * (TILE * 8), out + PART_OFF, TILE * 8 * 4);
    }
};

extern "C" int seqik_head_apply_backward_f32(const float* head, const float* affine, const float* grad_out, float* grad_head,
                                             float* grad_affine_partial, int64_t n_trial, int64_t n_frame, void* stream) {
    if (n_trial < 0 || n_frame < 0) return seqik_fail(SEQIK_EINVAL, "seqik_head_apply_backward_f32: negative size");
    if (n_trial == 0 || n_frame == 0) return SEQIK_OK;
    if (!head || !affine || !grad_out) return seqik_fail(SEQIK_EINVAL, "seqik_head_apply_backward_f32: NULL pointer");
    if (!grad_head && !grad_affine_partial) return SEQIK_OK;
    const int64_t frames = n_trial * n_frame, full_tiles = frames / TILE, done = full_tiles * TILE;
    const bool aligned = ((((uintptr_t)head) | ((uintptr_t)grad_out) | ((uintptr_t)grad_head) | ((uintptr_t)grad_affine_partial)) & 15) == 0;
    cudaStream_t st = (cudaStream_t)stream;
    if (aligned && full_tiles > 0) {
        launch_tiles(HeadApplyBackwardOp{head, affine, grad_out, grad_head, grad_affine_partial, n_frame}, full_tiles, st);
        if (frames > done)
            head_apply_backward_kernel<<<(unsigned)((frames - done + TILE - 1) / TILE), TILE, 0, st>>>(
                head, affine, grad_out, grad_head, grad_affine_partial, n_frame, frames, done);
    } else {
        head_apply_backward_kernel<<<(unsigned)((frames + TILE - 1) / TILE), TILE, 0, st>>>(
            head, affine, grad_out, grad_head, grad_affine_partial, n_frame, frames, 0);
    }
    return seqik_check_launch("seqik_head_apply_backward_f32");
}

// ---- head_affine backward ---------------------------------------------------------------------------------------------------
// The five series of a trial are the rows seqik_head_series_* wrote: base x, y, z and d = |base - thorax_mid| at the
// stationary frames (+inf elsewhere, counts[0..3] of them), |tip - base| at every frame (counts[4] = n_frame).  Their keys
// are the order keys of those float32 values; the ranks are those of the m = counts[s] smallest, so the +inf padding, the
// largest key of a finite row, is never selected.  Per series the result is AG_RES words, as for the legs.

// The forward's mid-quantile of the four selected keys of a series of m values (mid_quantile_value, seqik_kernels.cu) and the
// weight of each sorted rank position in it.
__device__ __forceinline__ float selected_mid_quantile(const uint32_t* val, int64_t m, float* w) {
    unsigned int rank[4]; float f45, f55;
    const bool swap = mid_quantile_ranks(m, rank, f45, f55);
    w[0] = 0.5f * (1.f - f45); w[1] = 0.5f * f45; w[2] = 0.5f * (1.f - f55); w[3] = 0.5f * f55;
    if (swap) { const float t = w[1]; w[1] = w[2]; w[2] = t; }
    const float a0 = key_value(val[0]), a1 = key_value(val[swap ? 2 : 1]), b0 = key_value(val[swap ? 1 : 2]), b1 = key_value(val[3]);
    const float q0 = a0 + (a1 - a0) * f45, q1 = b0 + (b1 - b0) * f55;
    return 0.5f * (q0 + q1);
}

// One writer per trial, in a fixed order (series 0..4, then sorted rank position 0..3; series 3: base, thorax[0],
// thorax[k-1]; series 4: tip, base; x, y, z): the statistics' contributions are ADDED into gh (and gt unless NULL).
// kf: the trial's five result rows (stride AG_RES words).
template <typename T>
static __device__ void head_scatter(const T* __restrict__ head, const T* __restrict__ thorax, int64_t n_kp,
                                    const int32_t* __restrict__ counts, const float* __restrict__ a, const float* __restrict__ h,
                                    const uint32_t* kf, T* __restrict__ gh, T* __restrict__ gt, float* __restrict__ gk) {
    float s3 = 0.f, s4 = 0.f;
    for (int j = 0; j < 5; ++j) {
        const int64_t m = counts[j];
        float w[4];
        const float sj = m > 0 ? selected_mid_quantile(kf + j * AG_RES, m, w) : __int_as_float(0x7fffffff);
        if (j == 3) s3 = sj;
        if (j == 4) s4 = sj;
        const float ds = j < 3 ? h[j] : j == 3 ? -(h[3] * a[3]) / sj : -(h[7] * a[7]) / sj;     // dL/ds_j
        if (m <= 0) continue;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float share = ds * w[i];
            const int64_t t = kf[j * AG_RES + 8 + i];
            const T* b = head + t * 6;
            T* g = gh + t * 6;
            if (j < 3) { g[j] += (T)share; continue; }
            double dx, dy, dz;
            const T* t0 = thorax + t * n_kp * 3; const T* t1 = t0 + (n_kp - 1) * 3;
            if (j == 3) {                                              // base_to_thorax_mid's arithmetic
                dx = (double)b[0] - 0.5 * ((double)t0[0] + (double)t1[0]);
                dy = (double)b[1] - 0.5 * ((double)t0[1] + (double)t1[1]);
                dz = (double)b[2] - 0.5 * ((double)t0[2] + (double)t1[2]);
            } else {                                                   // head_series_kernel's |tip - base|
                dx = (double)b[3] - (double)b[0]; dy = (double)b[4] - (double)b[1]; dz = (double)b[5] - (double)b[2];
            }
            const double len = sqrt(dx * dx + dy * dy + dz * dz);
            if (len == 0.0) continue;                                  // the norm's subgradient at 0
            const T sh = (T)share;
            const T cx = sh * (T)(dx / len), cy = sh * (T)(dy / len), cz = sh * (T)(dz / len);
            if (j == 3) {
                g[0] += cx; g[1] += cy; g[2] += cz;
                if (gt) {
                    const T hx = (T)0.5 * cx, hy = (T)0.5 * cy, hz = (T)0.5 * cz;
                    T* q0 = gt + t * n_kp * 3; T* q1 = q0 + (n_kp - 1) * 3;
                    q0[0] -= hx; q0[1] -= hy; q0[2] -= hz;
                    q1[0] -= hx; q1[1] -= hy; q1[2] -= hz;
                }
            } else {
                g[3] += cx; g[4] += cy; g[5] += cz;
                g[0] -= cx; g[1] -= cy; g[2] -= cz;
            }
        }
    }
    if (gk) { gk[0] = h[4]; gk[1] = h[5]; gk[2] = h[6]; gk[3] = h[3] / s3; gk[4] = h[7] / s4; }
}

// Recordings of up to AG_N frames: one CTA of five warps per trial.  Warp w turns series row w into order keys in shared
// memory, selects the four keys of its ranks (warp_rank_select) and finds their frames (warp_find_frames); thread 0 scatters.
constexpr int HG_WARPS = 5, HG_THREADS = 32 * HG_WARPS;
template <typename T>
__global__ void __launch_bounds__(HG_THREADS) head_affine_backward_fused_kernel(
        const T* __restrict__ head, const T* __restrict__ thorax, int64_t n_kp, const float* __restrict__ series,
        const int32_t* __restrict__ counts, const float* __restrict__ affine, const float* __restrict__ grad_affine,
        T* __restrict__ grad_head, T* __restrict__ grad_thorax, float* __restrict__ grad_consts, int n_frame) {
    __shared__ __align__(16) uint32_t key[HG_WARPS][AG_N];
    __shared__ unsigned int hist[HG_WARPS][2][256];
    __shared__ uint32_t res[HG_WARPS][AG_RES];
    const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
    const int64_t tr = blockIdx.x;
    const int64_t m = counts[tr * 5 + w];
    if (m > 0) {                                                       // (warp-uniform)
        const float* row = series + (tr * 5 + w) * n_frame;
        for (int i = lane; i < n_frame; i += 32) key[w][i] = order_key(__ldg(row + i));
        __syncwarp();
        unsigned int j[4]; uint32_t val[4], frame[4]; float f45, f55;
        mid_quantile_ranks(m, j, f45, f55);
        warp_rank_select(key[w], n_frame, j, hist[w], lane, val);
        warp_find_frames(key[w], n_frame, val, j, frame, lane);
        if (lane == 0) {
#pragma unroll
            for (int k = 0; k < 4; ++k) { res[w][k] = val[k]; res[w][8 + k] = frame[k]; }
        }
    }
    __syncthreads();
    if (tid == 0)
        head_scatter<T>(head + tr * n_frame * 6, thorax + tr * n_frame * n_kp * 3, n_kp, counts + tr * 5, affine + tr * 8,
                        grad_affine + tr * 8, &res[0][0], grad_head + tr * n_frame * 6,
                        grad_thorax ? grad_thorax + tr * n_frame * n_kp * 3 : nullptr, grad_consts ? grad_consts + tr * 5 : nullptr);
}

// Longer recordings, through scratch: the keys of the series rows, then key_select_kernel and key_frames_kernel with the
// counts, then a thread per trial scatters.
__global__ void __launch_bounds__(256) head_keys_kernel(const float* __restrict__ series, uint32_t* __restrict__ keys, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) keys[i] = order_key(__ldg(series + i));
}

template <typename T>
__global__ void head_affine_backward_finish_kernel(const T* __restrict__ head, const T* __restrict__ thorax, int64_t n_kp,
                                                   const int32_t* __restrict__ counts, const float* __restrict__ affine,
                                                   const float* __restrict__ grad_affine, const uint32_t* __restrict__ res,
                                                   T* __restrict__ grad_head, T* __restrict__ grad_thorax,
                                                   float* __restrict__ grad_consts, int64_t n_trial, int64_t n_frame) {
    const int64_t tr = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (tr >= n_trial) return;
    head_scatter<T>(head + tr * n_frame * 6, thorax + tr * n_frame * n_kp * 3, n_kp, counts + tr * 5, affine + tr * 8,
                    grad_affine + tr * 8, res + tr * 5 * AG_RES, grad_head + tr * n_frame * 6,
                    grad_thorax ? grad_thorax + tr * n_frame * n_kp * 3 : nullptr, grad_consts ? grad_consts + tr * 5 : nullptr);
}

template <typename T>
static int head_affine_backward_launch(const char* name, const T* head, const T* thorax, int64_t n_kp, const float* series,
                                       const int32_t* counts, const float* consts, const float* affine, const float* grad_affine,
                                       T* grad_head, T* grad_thorax, float* grad_consts, uint32_t* scratch,
                                       int64_t n_trial, int64_t n_frame, void* stream) {
    if (n_trial < 0 || n_frame < 0) return seqik_fail(SEQIK_EINVAL, "%s: negative size", name);
    if (n_trial == 0) return SEQIK_OK;
    if (n_frame == 0) return seqik_fail(SEQIK_EINVAL, "%s: empty recording", name);
    if (!head || !thorax || !series || !counts || !consts || !affine || !grad_affine || !grad_head)
        return seqik_fail(SEQIK_EINVAL, "%s: NULL pointer", name);
    if (n_kp < 1) return seqik_fail(SEQIK_EINVAL, "%s: thorax needs at least one key point", name);
    if (n_frame > 2147483647LL) return seqik_fail(SEQIK_EINVAL, "%s: too many frames", name);
    if (n_trial > 429496729LL) return seqik_fail(SEQIK_EINVAL, "%s: too many trials", name);
    cudaStream_t st = (cudaStream_t)stream;
    if (n_frame <= AG_N) {
        head_affine_backward_fused_kernel<T><<<(unsigned)n_trial, HG_THREADS, 0, st>>>(head, thorax, n_kp, series, counts, affine,
                                                                                      grad_affine, grad_head, grad_thorax,
                                                                                      grad_consts, (int)n_frame);
        return seqik_check_launch(name);
    }
    if (!scratch) return seqik_fail(SEQIK_EINVAL, "%s: recordings of more than 1024 frames need the scratch buffer", name);
    const int64_t n_series = n_trial * 5;
    uint32_t* keys = scratch;
    uint32_t* res = scratch + n_series * n_frame;
    head_keys_kernel<<<(unsigned)((n_series * n_frame + 255) / 256), 256, 0, st>>>(series, keys, n_series * n_frame);
    key_select_kernel<<<(unsigned)n_series, KS_BLOCK, 0, st>>>(keys, n_frame, counts, res);
    key_frames_kernel<<<(unsigned)((n_series + KF_WARPS - 1) / KF_WARPS), 32 * KF_WARPS, 0, st>>>(keys, n_frame, n_series, counts, res);
    head_affine_backward_finish_kernel<T><<<(unsigned)((n_trial + 127) / 128), 128, 0, st>>>(head, thorax, n_kp, counts, affine,
                                                                                            grad_affine, res, grad_head, grad_thorax,
                                                                                            grad_consts, n_trial, n_frame);
    return seqik_check_launch(name);
}

extern "C" int seqik_head_affine_backward_f32(const float* head, const float* thorax, int64_t n_thorax_kp, const float* series,
                                              const int32_t* counts, const float* consts, const float* affine,
                                              const float* grad_affine, float* grad_head, float* grad_thorax, float* grad_consts,
                                              uint32_t* scratch, int64_t n_trial, int64_t n_frame, void* stream) {
    return head_affine_backward_launch<float>("seqik_head_affine_backward_f32", head, thorax, n_thorax_kp, series, counts, consts,
                                              affine, grad_affine, grad_head, grad_thorax, grad_consts, scratch, n_trial, n_frame,
                                              stream);
}
extern "C" int seqik_head_affine_backward_f64(const double* head, const double* thorax, int64_t n_thorax_kp, const float* series,
                                              const int32_t* counts, const float* consts, const float* affine,
                                              const float* grad_affine, double* grad_head, double* grad_thorax, float* grad_consts,
                                              uint32_t* scratch, int64_t n_trial, int64_t n_frame, void* stream) {
    return head_affine_backward_launch<double>("seqik_head_affine_backward_f64", head, thorax, n_thorax_kp, series, counts, consts,
                                               affine, grad_affine, grad_head, grad_thorax, grad_consts, scratch, n_trial, n_frame,
                                               stream);
}
