// seqik_fk_grad.cu -- seqik_fk_backward_f32 (include/seqik.h): the backward (vector-Jacobian product) of the stage-4 leg FK.
// A translation unit of its own, so that adding it leaves the code generated for seqik_kernels.cu unchanged.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/seqik.h"
#include "seqik_common.h"
#include "seqik_core.cuh"
#include "seqik_stream.cuh"

using namespace seqik;

// The forward is recomputed in registers with the arithmetic of fk_rows (seqik_kernels.cu) (same sincosv_, same rotate_frame); nothing of it is
// stored.  With d_k = -l_k A_k.c2 the vector of segment k (A_k = the frame after stage k) and S_k = the gradient summed over
// the joint rows at and past the end of segment k, one reverse sweep gives T_k = d_k x S_k + T_{k+1}; an angle of stage k
// turns segments k..4 about its world axis u, so dL/dangle = u . T_k, and dL/dl_k = -A_k.c2 . S_k.  No position enters, so
// the error does not grow with |origin| -- and the origin itself is not read: FK is a translation by it.
// q: 7 angles, g: 27 gradient floats (rows 0-8), ga: 7 out, go: 3 out, gl: 4 out.
__device__ __forceinline__ void fk_backward_rows(const float* q, const float* g, const float* __restrict__ prm,
                                                 float* ga, float* go, float* gl) {
    const float l[4] = {__ldg(prm), __ldg(prm + 1), __ldg(prm + 2), __ldg(prm + 3)};
    Mat3<float> A = {{1.f, 0.f, 0.f}, {0.f, 1.f, 0.f}, {0.f, 0.f, 1.f}};
    Vec3<float> c1[4], c2[4];                    // A_k.c1 (pitch axis of stage k) and A_k.c2 (segment direction)
    float sa, ca, sb, cb, v;
    Num<float>::sincosv_(q[0], &sa, &ca, &v); Num<float>::sincosv_(q[1], &sb, &cb, &v);
    A = rotate_frame(A, KIND_XY, sa, ca, sb, cb);
    c1[0] = A.c1; c2[0] = A.c2;
#pragma unroll
    for (int k = 1; k < 4; ++k) {
        if (k < 3) Num<float>::sincosv_(q[2 * k], &sa, &ca, &v);
        else { sa = 0.f; ca = 1.f; }
        Num<float>::sincosv_(q[2 * k + 1 - (k == 3)], &sb, &cb, &v);
        A = rotate_frame(A, KIND_ZY, sa, ca, sb, cb);
        c1[k] = A.c1; c2[k] = A.c2;
    }
    // reverse sweep: S_4 = g8, S_3 = g7 + S_4, S_2 = g6 + S_3, S_1 = (g4 + g5) + S_2
    Vec3<float> S = {0.f, 0.f, 0.f}, T = {0.f, 0.f, 0.f}, Tk[4];
    float dl[4];
#pragma unroll
    for (int k = 3; k >= 0; --k) {
        const float* h = g + 3 * (k + 5);
        Vec3<float> hk = {h[0], h[1], h[2]};
        if (k == 0) hk = {g[12] + g[15], g[13] + g[16], g[14] + g[17]};
        S = {hk.x + S.x, hk.y + S.y, hk.z + S.z};
        const Vec3<float> d = {-l[k] * c2[k].x, -l[k] * c2[k].y, -l[k] * c2[k].z};
        T = {fmaf(d.y, S.z, fmaf(-d.z, S.y, T.x)), fmaf(d.z, S.x, fmaf(-d.x, S.z, T.y)), fmaf(d.x, S.y, fmaf(-d.y, S.x, T.z))};
        Tk[k] = T;
        dl[k] = -dot(c2[k], S);
    }
    ga[0] = Tk[0].x;                             // yaw: world x
    ga[1] = dot(c1[0], Tk[0]);
    ga[2] = dot(c2[0], Tk[1]);                   // roll of stage k: A_{k-1}.c2
    ga[3] = dot(c1[1], Tk[1]);
    ga[4] = dot(c2[1], Tk[2]);
    ga[5] = dot(c1[2], Tk[2]);
    ga[6] = dot(c1[3], Tk[3]);
    go[0] = (((g[0] + g[3]) + g[6]) + g[9]) + S.x;
    go[1] = (((g[1] + g[4]) + g[7]) + g[10]) + S.y;
    go[2] = (((g[2] + g[5]) + g[8]) + g[11]) + S.z;
    gl[0] = dl[0]; gl[1] = dl[1]; gl[2] = dl[2]; gl[3] = dl[3];
}

// Plain kernel (unaligned pointers, totals below one tile, the tail of the tile path): one thread per leg-frame, staged
// through shared memory like fk_kernel.  Every output is computed; the NULL ones are not stored.
__global__ void __launch_bounds__(TILE) fk_backward_kernel(const float* __restrict__ angles, const float* __restrict__ params,
                                                               const float* __restrict__ grad_fk, float* __restrict__ grad_angles,
                                                               float* __restrict__ grad_origin, float* __restrict__ grad_lengths,
                                                               int64_t n_chain, int64_t n_frame, int64_t first) {
    __shared__ __align__(16) float s_in[TILE * 7];
    __shared__ __align__(16) float s_g[TILE * 27];
    __shared__ __align__(16) float s_ga[TILE * 7];
    __shared__ __align__(16) float s_go[TILE * 3];
    __shared__ __align__(16) float s_gl[TILE * 4];
    const int64_t total = n_chain * n_frame;
    const int64_t base = first + (int64_t)blockIdx.x * TILE;
    const int n_here = (int)min((int64_t)TILE, total - base);
    stage_in(s_in, angles + base * 7, n_here * 7);
    stage_in(s_g, grad_fk + base * 27, n_here * 27);
    __syncthreads();
    if (threadIdx.x < n_here) {
        const int64_t c = (base + threadIdx.x) / n_frame;
        const int t = threadIdx.x;
        fk_backward_rows(s_in + t * 7, s_g + t * 27, params + c * SEQIK_CHAIN_PARAM_FLOATS, s_ga + t * 7, s_go + t * 3, s_gl + t * 4);
    }
    __syncthreads();
    stage_out(grad_angles + base * 7, s_ga, n_here * 7);
    if (grad_origin) stage_out(grad_origin + base * 3, s_go, n_here * 3);
    if (grad_lengths) stage_out(grad_lengths + base * 4, s_gl, n_here * 4);
}

// Tile path: angles and grad_fk in (34 KB a tile), up to three output streams (14 KB); 48 KB a stage, two CTAs per SM
struct FkBackwardOp {
    const float* angles; const float* params; const float* grad_fk;
    float* grad_angles; float* grad_origin; float* grad_lengths; int64_t n_frame;
    static constexpr int N_IN = 2, G_OFF = TILE * 7 * 4, OUT_OFF = TILE * 34 * 4;
    static constexpr int GO_OFF = TILE * 7 * 4, GL_OFF = TILE * 10 * 4, STAGE_BYTES = OUT_OFF + TILE * 14 * 4;
    static __device__ __forceinline__ int in_off(int i) { return i == 0 ? 0 : G_OFF; }
    __device__ __forceinline__ uint32_t in_bytes(int i, int64_t) const { return i == 0 ? TILE * 7 * 4 : TILE * 27 * 4; }
    __device__ __forceinline__ const void* in_src(int i, int64_t tile) const { return i == 0 ? angles + tile * (TILE * 7) : grad_fk + tile * (TILE * 27); }
    __device__ __forceinline__ void compute(int tid, int64_t tile, unsigned char* stage) const {
        const float* s_in = reinterpret_cast<const float*>(stage);
        const float* s_g = reinterpret_cast<const float*>(stage + G_OFF);
        unsigned char* out = stage + OUT_OFF;
        const int64_t c = (tile * TILE + tid) / n_frame;
        float gl[4];
        fk_backward_rows(s_in + tid * 7, s_g + tid * 27, params + c * SEQIK_CHAIN_PARAM_FLOATS, reinterpret_cast<float*>(out) + tid * 7,
                         reinterpret_cast<float*>(out + GO_OFF) + tid * 3, gl);
        reinterpret_cast<float4*>(out + GL_OFF)[tid] = make_float4(gl[0], gl[1], gl[2], gl[3]);   // one 16-byte store: no bank conflicts
    }
    __device__ __forceinline__ void store(int64_t tile, const unsigned char* out) const {
        tma_store_1d_nocommit(grad_angles + tile * (TILE * 7), out, TILE * 7 * 4);
        if (grad_origin) tma_store_1d_nocommit(grad_origin + tile * (TILE * 3), out + GO_OFF, TILE * 3 * 4);
        if (grad_lengths) tma_store_1d_nocommit(grad_lengths + tile * (TILE * 4), out + GL_OFF, TILE * 4 * 4);
    }
};

extern "C" int seqik_fk_backward_f32(const float* angles, const float* origin, int64_t origin_frame_stride, const float* params,
                                     const float* grad_fk, float* grad_angles, float* grad_origin, float* grad_lengths,
                                     int64_t n_chain, int64_t n_frame, void* stream) {
    if (n_chain < 0 || n_frame < 0) return seqik_fail(SEQIK_EINVAL, "seqik_fk_backward_f32: negative size");
    if (n_chain == 0 || n_frame == 0) return SEQIK_OK;
    if (!angles || !origin || !params || !grad_fk || !grad_angles) return seqik_fail(SEQIK_EINVAL, "seqik_fk_backward_f32: NULL pointer");
    if (origin_frame_stride != 0 && origin_frame_stride != 3)
        return seqik_fail(SEQIK_EINVAL, "seqik_fk_backward_f32: origin_frame_stride must be 0 or 3");
    const int64_t total = n_chain * n_frame;
    const int64_t full_tiles = total / TILE, rest = total - full_tiles * TILE;
    const bool aligned = ((((uintptr_t)angles) | ((uintptr_t)grad_fk) | ((uintptr_t)grad_angles) | ((uintptr_t)grad_origin) |
                           ((uintptr_t)grad_lengths)) & 15) == 0;
    cudaStream_t st = (cudaStream_t)stream;
    if (aligned && full_tiles > 0) {
        launch_tiles(FkBackwardOp{angles, params, grad_fk, grad_angles, grad_origin, grad_lengths, n_frame}, full_tiles, st);
        if (rest)
            fk_backward_kernel<<<1, TILE, 0, st>>>(angles, params, grad_fk, grad_angles, grad_origin, grad_lengths, n_chain, n_frame,
                                                       full_tiles * TILE);
    } else {
        const int64_t grid = (total + TILE - 1) / TILE;
        fk_backward_kernel<<<(unsigned)grid, TILE, 0, st>>>(angles, params, grad_fk, grad_angles, grad_origin, grad_lengths,
                                                                n_chain, n_frame, 0);
    }
    return seqik_check_launch("seqik_fk_backward_f32");
}
