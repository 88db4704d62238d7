// seqik_kernels.cu -- sm_100a kernels + C ABI (include/seqik.h) of the SeqIKPy leg-IK hot path.
//
// Kernels
//   (the leg solver kernels live in seqik_solver.cu)
//   fk_kernel          angles -> 9x3 joint positions, HBM-bound streaming kernel (smem-staged, 128-bit I/O)
//   head_kernel        7 head/antenna angles per frame, HBM-bound elementwise
//   leg_series_kernel / mid_quantile_kernel / align_apply_kernel   AlignPose statistics + affine map
//
// No tensor cores: the work is scalar FP32 2x2 / 3x3 algebra (BASELINE.json north_star).
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <thread>
#include <vector>
#if defined(__SSE2__)
#include <immintrin.h>
#endif

#include "../../include/seqik.h"
#include "seqik_common.h"
#include "seqik_core.cuh"
#include "seqik_head.cuh"
#include "seqik_stream.cuh"

using namespace seqik;

// ---------------------------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

int seqik_fail(int code, const char* fmt, const char* a) {
    snprintf(g_err, sizeof(g_err), fmt, a);
    return code;
}
int seqik_check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
        return SEQIK_ECUDA;
    }
    return SEQIK_OK;
}
static inline int fail(int code, const char* fmt, const char* a = "") { return seqik_fail(code, fmt, a); }
static inline int check_launch(const char* what) { return seqik_check_launch(what); }

extern "C" int seqik_abi_version(void) { return SEQIK_ABI_VERSION; }

extern "C" int seqik_memcpy2d_async(void* dst, int64_t dst_pitch_bytes, const void* src, int64_t src_pitch_bytes,
                                    int64_t width_bytes, int64_t height, int direction, void* stream) {
    if (width_bytes < 0 || height < 0) return fail(SEQIK_EINVAL, "seqik_memcpy2d_async: negative size");
    if (width_bytes == 0 || height == 0) return SEQIK_OK;
    if (!dst || !src) return fail(SEQIK_EINVAL, "seqik_memcpy2d_async: NULL pointer");
    if (direction != 1 && direction != 2) return fail(SEQIK_EINVAL, "seqik_memcpy2d_async: direction must be 1 (H2D) or 2 (D2H)");
    if (dst_pitch_bytes < width_bytes || src_pitch_bytes < width_bytes) return fail(SEQIK_EINVAL, "seqik_memcpy2d_async: pitch smaller than width");
    cudaError_t e = cudaMemcpy2DAsync(dst, (size_t)dst_pitch_bytes, src, (size_t)src_pitch_bytes, (size_t)width_bytes, (size_t)height,
                                      direction == 1 ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost, (cudaStream_t)stream);
    if (e != cudaSuccess) { snprintf(g_err, sizeof(g_err), "seqik_memcpy2d_async: %s", cudaGetErrorString(e)); return SEQIK_ECUDA; }
    return SEQIK_OK;
}
extern "C" const char* seqik_last_error(void) { return g_err; }

// Device side of the joints-only wire format: the origin rows (key point 0) of frames [t0, t1) of every chain, compact
// ([n_chain][n_frame][3]), so that the host rebuilds rows 0-3 from 12 contiguous bytes per leg-frame instead of touching
// every cache line of its 60-byte-per-frame pose.
__global__ void __launch_bounds__(256) origin_rows_kernel(const float* __restrict__ pose, int64_t cs, int64_t fs, float* __restrict__ out,
                                                          int64_t out_cs, int64_t n_chain, int64_t t0, int64_t nt) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;          // one float of one origin row
    if (i >= n_chain * nt * 3) return;
    const int64_t c = i / (nt * 3), r = i - c * (nt * 3), t = r / 3, k = r - 3 * t;
    out[c * out_cs + (t0 + t) * 3 + k] = __ldg(pose + c * cs + (t0 + t) * fs + k);
}
extern "C" int seqik_origin_rows_f32(const float* pose, int64_t pose_chain_stride, int64_t pose_frame_stride, float* out,
                                     int64_t out_chain_stride, int64_t n_chain, int64_t t0, int64_t t1, void* stream) {
    if (n_chain < 0 || t0 < 0 || t1 < t0) return fail(SEQIK_EINVAL, "seqik_origin_rows_f32: bad range");
    if (n_chain == 0 || t1 == t0) return SEQIK_OK;
    if (!pose || !out) return fail(SEQIK_EINVAL, "seqik_origin_rows_f32: NULL pointer");
    if (pose_frame_stride < 3) return fail(SEQIK_EINVAL, "seqik_origin_rows_f32: frame stride too small");
    const int64_t total = n_chain * (t1 - t0) * 3;
    origin_rows_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(pose, pose_chain_stride, pose_frame_stride, out,
                                                                                         out_chain_stride, n_chain, t0, t1 - t0);
    return check_launch("seqik_origin_rows_f32");
}

// Host side of the joints-only wire format: the reference's nine-row FK layout rebuilt in HOST memory from the four joint rows
// that crossed the link and the origin row of the host-resident pose (rows 0-3 = origin, row 4 = row 5 = first joint).
// A memory-bound copy; chains are split over `n_threads` host threads.
extern "C" int seqik_fk_expand_host_f32(const float* joints, int64_t j_chain_stride, int64_t j_frame_stride,
                                        const float* pose, int64_t p_chain_stride, int64_t p_frame_stride,
                                        float* fk, int64_t f_chain_stride, int64_t f_frame_stride,
                                        int64_t n_chain, int64_t t0, int64_t t1, int n_threads) {
    if (n_chain < 0 || t0 < 0 || t1 < t0) return fail(SEQIK_EINVAL, "seqik_fk_expand_host_f32: bad range");
    if (n_chain == 0 || t1 == t0) return SEQIK_OK;
    if (!joints || !pose || !fk) return fail(SEQIK_EINVAL, "seqik_fk_expand_host_f32: NULL pointer");
    if (j_frame_stride < 12 || p_frame_stride < 3 || f_frame_stride < 27) return fail(SEQIK_EINVAL, "seqik_fk_expand_host_f32: frame stride too small");
    if (n_threads < 1) n_threads = 1;
    if ((int64_t)n_threads > n_chain) n_threads = (int)n_chain;
    auto work = [=](int64_t c0, int64_t c1) {
        for (int64_t c = c0; c < c1; ++c) {
            const float* j = joints + c * j_chain_stride + t0 * j_frame_stride;
            const float* p = pose + c * p_chain_stride + t0 * p_frame_stride;
            float* o = fk + c * f_chain_stride + t0 * f_frame_stride;
            int64_t t = t0;
#if defined(__SSE2__)
            // four frames = 108 floats = 27 x 16 bytes: assembled in registers / L1 and written with streaming stores, so that
            // the 648 MB of rows of a config-3 step are not first READ into the cache (write-allocate) before being overwritten
            if (f_frame_stride == 27 && ((((uintptr_t)o) & 15) == 0)) {
                alignas(16) float buf[108];
                for (; t + 4 <= t1; t += 4, o += 108) {
                    for (int f = 0; f < 4; ++f, j += j_frame_stride, p += p_frame_stride) {
                        float* b = buf + 27 * f;
                        const float x = p[0], y = p[1], z = p[2];
                        for (int r = 0; r < 4; ++r) { b[3 * r] = x; b[3 * r + 1] = y; b[3 * r + 2] = z; }
                        b[12] = j[0]; b[13] = j[1]; b[14] = j[2];
                        memcpy(b + 15, j, 12 * sizeof(float));
                    }
                    for (int k = 0; k < 27; ++k) _mm_stream_ps(o + 4 * k, _mm_load_ps(buf + 4 * k));
                }
                _mm_sfence();
            }
#endif
            for (; t < t1; ++t, j += j_frame_stride, p += p_frame_stride, o += f_frame_stride) {
                const float x = p[0], y = p[1], z = p[2];
                for (int r = 0; r < 4; ++r) { o[3 * r] = x; o[3 * r + 1] = y; o[3 * r + 2] = z; }
                o[12] = j[0]; o[13] = j[1]; o[14] = j[2];
                memcpy(o + 15, j, 12 * sizeof(float));
            }
        }
    };
    if (n_threads == 1) { work(0, n_chain); return SEQIK_OK; }
    std::vector<std::thread> pool;
    pool.reserve(n_threads);
    for (int k = 0; k < n_threads; ++k) pool.emplace_back(work, n_chain * k / n_threads, n_chain * (k + 1) / n_threads);
    for (auto& th : pool) th.join();
    return SEQIK_OK;
}

// ---------------------------------------------------------------------------------------------
// forward kinematics (streaming)
// ---------------------------------------------------------------------------------------------
// One thread per leg-frame; a block of 256 leg-frames stages its 256x7 angles through shared memory with
// coalesced loads and its 256x27 outputs back with coalesced stores.
constexpr int FK_BLOCK = 256;

// joint rows of one leg-frame: q = 7 angles, o = origin, out = 27 floats (shared by both FK kernels)
__device__ __forceinline__ void fk_rows(const float* q, const Vec3<float>& o, const float* __restrict__ prm, float* out) {
    const float l0 = __ldg(prm), l1 = __ldg(prm + 1), l2 = __ldg(prm + 2), l3 = __ldg(prm + 3);
    Mat3<float> A = {{1.f, 0.f, 0.f}, {0.f, 1.f, 0.f}, {0.f, 0.f, 1.f}};
    Vec3<float> p = o;
    float sa, ca, sb, cb, v;
#pragma unroll
    for (int r = 0; r < 4; ++r) { out[3 * r] = o.x; out[3 * r + 1] = o.y; out[3 * r + 2] = o.z; }
    // stage 1: Rx(yaw) Ry(pitch), coxa
    Num<float>::sincosv_(q[0], &sa, &ca, &v); Num<float>::sincosv_(q[1], &sb, &cb, &v);
    A = rotate_frame(A, KIND_XY, sa, ca, sb, cb);
    p = {fmaf(-l0, A.c2.x, p.x), fmaf(-l0, A.c2.y, p.y), fmaf(-l0, A.c2.z, p.z)};
    out[12] = out[15] = p.x; out[13] = out[16] = p.y; out[14] = out[17] = p.z;
    // stage 2: Rz(roll) Ry(CTr_pitch), femur
    Num<float>::sincosv_(q[2], &sa, &ca, &v); Num<float>::sincosv_(q[3], &sb, &cb, &v);
    A = rotate_frame(A, KIND_ZY, sa, ca, sb, cb);
    p = {fmaf(-l1, A.c2.x, p.x), fmaf(-l1, A.c2.y, p.y), fmaf(-l1, A.c2.z, p.z)};
    out[18] = p.x; out[19] = p.y; out[20] = p.z;
    // stage 3: Rz(CTr_roll) Ry(FTi_pitch), tibia
    Num<float>::sincosv_(q[4], &sa, &ca, &v); Num<float>::sincosv_(q[5], &sb, &cb, &v);
    A = rotate_frame(A, KIND_ZY, sa, ca, sb, cb);
    p = {fmaf(-l2, A.c2.x, p.x), fmaf(-l2, A.c2.y, p.y), fmaf(-l2, A.c2.z, p.z)};
    out[21] = p.x; out[22] = p.y; out[23] = p.z;
    // stage 4: Ry(TiTa_pitch), tarsus
    Num<float>::sincosv_(q[6], &sb, &cb, &v);
    A = rotate_frame(A, KIND_ZY, 0.f, 1.f, sb, cb);
    p = {fmaf(-l3, A.c2.x, p.x), fmaf(-l3, A.c2.y, p.y), fmaf(-l3, A.c2.z, p.z)};
    out[24] = p.x; out[25] = p.y; out[26] = p.z;
}

__global__ void __launch_bounds__(FK_BLOCK) fk_kernel(const float* __restrict__ angles, const float* __restrict__ origin,
                                                      int64_t origin_fs, const float* __restrict__ params,
                                                      float* __restrict__ fk, int64_t n_chain, int64_t n_frame, int64_t first) {
    __shared__ __align__(16) float s_in[FK_BLOCK * 7];
    __shared__ __align__(16) float s_org[FK_BLOCK * 3];
    __shared__ __align__(16) float s_out[FK_BLOCK * 27];
    const int64_t total = n_chain * n_frame;
    const int64_t base = first + (int64_t)blockIdx.x * FK_BLOCK;          // `first`: leg-frames already done by fk_tma_kernel
    const int n_here = (int)min((int64_t)FK_BLOCK, total - base);
    stage_in(s_in, angles + base * 7, n_here * 7);
    if (origin_fs) stage_in(s_org, origin + base * 3, n_here * 3);
    __syncthreads();
    if (threadIdx.x < n_here) {
        const int64_t lf = base + threadIdx.x;
        const int64_t c = lf / n_frame;
        const float* prm = params + c * SEQIK_CHAIN_PARAM_FLOATS;
        const float* op = origin_fs ? s_org + threadIdx.x * 3 : origin + c * 3;
        const Vec3<float> o = {op[0], op[1], op[2]};
        fk_rows(s_in + threadIdx.x * 7, o, prm, s_out + threadIdx.x * 27);
    }
    __syncthreads();
    stage_out(fk + base * 27, s_out, n_here * 27);
}

struct FkOp {
    const float* angles; const float* origin; int64_t origin_fs; const float* params; float* fk; int64_t n_frame;
    static constexpr int N_IN = 2, STAGE_BYTES = TILE * 37 * 4, OUT_OFF = TILE * 10 * 4;
    static __device__ __forceinline__ int in_off(int i) { return i == 0 ? 0 : TILE * 7 * 4; }
    __device__ __forceinline__ uint32_t in_bytes(int i, int64_t) const { return i == 0 ? TILE * 7 * 4 : (origin_fs ? TILE * 3 * 4 : 0); }
    __device__ __forceinline__ const void* in_src(int i, int64_t tile) const { return i == 0 ? angles + tile * (TILE * 7) : origin + tile * (TILE * 3); }
    __device__ __forceinline__ void compute(int tid, int64_t tile, unsigned char* stage) const {
        const float* s_in = reinterpret_cast<const float*>(stage);
        const float* s_org = reinterpret_cast<const float*>(stage + TILE * 7 * 4);
        float* s_out = reinterpret_cast<float*>(stage + OUT_OFF);
        const int64_t c = (tile * TILE + tid) / n_frame;
        const float* op = origin_fs ? s_org + tid * 3 : origin + c * 3;
        const Vec3<float> o = {op[0], op[1], op[2]};
        fk_rows(s_in + tid * 7, o, params + c * SEQIK_CHAIN_PARAM_FLOATS, s_out + tid * 27);
    }
    __device__ __forceinline__ void store(int64_t tile, const unsigned char* out) const { tma_store_1d_nocommit(fk + tile * (TILE * 27), out, TILE * 27 * 4); }
};

extern "C" int seqik_fk_f32(const float* angles, const float* origin, int64_t origin_frame_stride, const float* params,
                            float* fk, int64_t n_chain, int64_t n_frame, void* stream) {
    if (n_chain < 0 || n_frame < 0) return fail(SEQIK_EINVAL, "seqik_fk_f32: negative size");
    if (n_chain == 0 || n_frame == 0) return SEQIK_OK;
    if (!angles || !origin || !params || !fk) return fail(SEQIK_EINVAL, "seqik_fk_f32: NULL pointer");
    if (origin_frame_stride != 0 && origin_frame_stride != 3) return fail(SEQIK_EINVAL, "seqik_fk_f32: origin_frame_stride must be 0 or 3");
    const int64_t total = n_chain * n_frame;
    const int64_t full_tiles = total / FK_BLOCK, rest = total - full_tiles * FK_BLOCK;
    const bool aligned = ((((uintptr_t)angles) | ((uintptr_t)fk) | (origin_frame_stride ? (uintptr_t)origin : 0)) & 15) == 0;
    cudaStream_t st = (cudaStream_t)stream;
    if (aligned && full_tiles > 0) {
        // persistent TMA pipeline over the full tiles, the ragged tail by fk_kernel
        launch_tiles(FkOp{angles, origin, origin_frame_stride, params, fk, n_frame}, full_tiles, st);
        if (rest) {
            const int64_t done = full_tiles * FK_BLOCK;
            fk_kernel<<<1, FK_BLOCK, 0, st>>>(angles, origin, origin_frame_stride, params, fk, n_chain, n_frame, done);
        }
    } else {
        const int64_t grid = (total + FK_BLOCK - 1) / FK_BLOCK;
        fk_kernel<<<(unsigned)grid, FK_BLOCK, 0, st>>>(angles, origin, origin_frame_stride, params, fk, n_chain, n_frame, 0);
    }
    return check_launch("seqik_fk_f32");
}


// ---------------------------------------------------------------------------------------------
// head / antenna angles (elementwise; atan2_pos, signed_angle and head_point are in seqik_head.cuh)
// ---------------------------------------------------------------------------------------------
// one frame: rr / ll = (base xyz, tip xyz) of the right / left antenna, nk = neck; out7 = head roll, pitch, yaw, antenna yaw L,
// pitch L, yaw R, pitch R
__device__ __forceinline__ void head_frame(const float* rr, const float* ll, const float* nk, const float* __restrict__ ar,
                                           const float* __restrict__ al, float rest_head_pitch, float rest_ant_pitch, float* out7) {
    float rbx, rby, rbz, rtx, rty, rtz, lbx, lby, lbz, ltx, lty, ltz;
    head_point(rr, ar, false, rbx, rby, rbz); head_point(rr + 3, ar, true, rtx, rty, rtz);
    head_point(ll, al, false, lbx, lby, lbz); head_point(ll + 3, al, true, ltx, lty, ltz);
    const float nx = nk[0], ny = nk[1], nz = nk[2];
    const float hx = lbx - rbx, hy = lby - rby, hz = lbz - rbz;                                   // horizontal
    const float mx = (rbx + lbx) * 0.5f - nx, mz = (rbz + lbz) * 0.5f - nz;                      // mid - neck
    // roll: Y -> hor|x=0 about X; pitch: X -> mid|y=0 about Y (+rest); yaw: Y -> hor|z=0 about Z
    const float roll = signed_angle(hy, hz);
    out7[0] = roll; out7[1] = signed_angle(mx, -mz) + rest_head_pitch; out7[2] = signed_angle(hy, -hx);
    // derotation by -roll about X:  y' = y c + z s,  z' = -y s + z c
    float s, c, vers; Num<float>::sincosv_(roll, &s, &c, &vers);   // |roll| <= pi
    const float hdy = hy * c + hz * s, hdz = -hy * s + hz * c;                                    // derotated hor (x dropped)
#pragma unroll
    for (int side = 0; side < 2; ++side) {   // 0 = L, 1 = R  (reference loops ["L", "R"])
        const float bx = side ? rbx : lbx, by = side ? rby : lby, bz = side ? rbz : lbz;
        const float tx = side ? rtx : ltx, ty = side ? rty : lty, tz = side ? rtz : ltz;
        const float ax = tx - bx, ay = ty - by, az = tz - bz;                                     // antenna vector
        const float ady = ay * c + az * s, adz = -ay * s + az * c;
        // yaw: antenna|x=0 -> hor|x=0 about X ; det = X . (v1 x v2) = v1y v2z - v1z v2y
        float ayaw = signed_angle(ady * hdy + adz * hdz, ady * hdz - adz * hdy);
        if (side) ayaw = 3.14159265358979323846f - ayaw;
        // pitch: (neck - base)|y=0 -> antenna|y=0 about Y ; det = Y . (v1 x v2) = v1z v2x - v1x v2z
        const float gx = nx - bx, gy = ny - by, gz = nz - bz;
        const float gdz = -gy * s + gz * c;
        out7[3 + 2 * side] = ayaw;
        out7[4 + 2 * side] = signed_angle(gx * ax + gdz * adz, gdz * ax - gx * adz) - rest_ant_pitch;
    }
}

// kVec2: r_head and l_head are 8-byte aligned and read as 64-bit loads; otherwise (a view at an odd float offset) the same
// six floats are read one by one -- the arithmetic, hence the result, is the same
template <bool kVec2>
__global__ void __launch_bounds__(256) head_kernel(const float* __restrict__ r_head, const float* __restrict__ l_head,
                                                   const float* __restrict__ neck, int64_t neck_stride,
                                                   const float* __restrict__ affine_r, const float* __restrict__ affine_l,
                                                   const float* __restrict__ rest,
                                                   float* __restrict__ out, int64_t n_trial, int64_t n_frame) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_trial * n_frame) return;
    const int64_t tr = i / n_frame, t = i - tr * n_frame;
    const float* r = r_head + i * 6; const float* l = l_head + i * 6;        // 24-byte records: three 64-bit loads each
    float rr[6], ll[6];
    if (kVec2) {
        const float2 r01 = __ldg(reinterpret_cast<const float2*>(r)), r23 = __ldg(reinterpret_cast<const float2*>(r) + 1),
                     r45 = __ldg(reinterpret_cast<const float2*>(r) + 2);
        const float2 l01 = __ldg(reinterpret_cast<const float2*>(l)), l23 = __ldg(reinterpret_cast<const float2*>(l) + 1),
                     l45 = __ldg(reinterpret_cast<const float2*>(l) + 2);
        rr[0] = r01.x; rr[1] = r01.y; rr[2] = r23.x; rr[3] = r23.y; rr[4] = r45.x; rr[5] = r45.y;
        ll[0] = l01.x; ll[1] = l01.y; ll[2] = l23.x; ll[3] = l23.y; ll[4] = l45.x; ll[5] = l45.y;
    } else {
#pragma unroll
        for (int k = 0; k < 6; ++k) { rr[k] = __ldg(r + k); ll[k] = __ldg(l + k); }
    }
    float o7[7];
    head_frame(rr, ll, neck + (neck_stride ? i * 3 : tr * 3), affine_r ? affine_r + tr * 8 : nullptr,
               affine_l ? affine_l + tr * 8 : nullptr, rest[tr * 2], rest[tr * 2 + 1], o7);
    float* o = out + tr * 7 * n_frame + t;
#pragma unroll
    for (int k = 0; k < 7; ++k) o[k * n_frame] = o7[k];
}

extern "C" int seqik_head_angles_f32(const float* r_head, const float* l_head, const float* neck, int64_t neck_stride,
                                     const float* affine_r, const float* affine_l, const float* rest,
                                     float* out, int64_t n_trial, int64_t n_frame, void* stream) {
    if (n_trial < 0 || n_frame < 0) return fail(SEQIK_EINVAL, "seqik_head_angles_f32: negative size");
    if (n_trial == 0 || n_frame == 0) return SEQIK_OK;
    if (!r_head || !l_head || !neck || !rest || !out) return fail(SEQIK_EINVAL, "seqik_head_angles_f32: NULL pointer");
    if (neck_stride != 0 && neck_stride != 3) return fail(SEQIK_EINVAL, "seqik_head_angles_f32: neck_stride must be 0 or 3");
    if ((affine_r == nullptr) != (affine_l == nullptr))
        return fail(SEQIK_EINVAL, "seqik_head_angles_f32: affine_r and affine_l must both be given or both be NULL");
    const int64_t n = n_trial * n_frame;
    // (stays on plain loads: five atan2f and a sincos per 76-byte frame make this kernel issue-bound at ~0.57 of the HBM
    // peak with 2048 threads per SM; the 1024-thread TMA pipeline measured slower here, 0.37)
    // any 4-byte aligned head input is accepted: a view at an odd float offset takes the scalar-load instantiation
    const bool vec2 = ((((uintptr_t)r_head) | ((uintptr_t)l_head)) & 7) == 0;
    auto kernel = vec2 ? head_kernel<true> : head_kernel<false>;
    kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(r_head, l_head, neck, neck_stride, affine_r, affine_l,
                                                                         rest, out, n_trial, n_frame);
    return check_launch("seqik_head_angles_f32");
}

// ---------------------------------------------------------------------------------------------
// AlignPose: series, mid-quantiles, affine maps

// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) leg_series_kernel(const float* __restrict__ pose, int64_t cs, int64_t fs,
                                                         float* __restrict__ series, int64_t n_chain, int64_t n_frame) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_chain * n_frame) return;
    const int64_t c = i / n_frame, t = i - c * n_frame;
    const float* p = pose + c * cs + t * fs;
    float k[15];
#pragma unroll
    for (int j = 0; j < 15; ++j) k[j] = p[j];
    float* s = series + c * 7 * n_frame + t;
    s[0] = k[0]; s[n_frame] = k[1]; s[2 * n_frame] = k[2];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float dx = k[3 * j + 3] - k[3 * j], dy = k[3 * j + 4] - k[3 * j + 1], dz = k[3 * j + 5] - k[3 * j + 2];
        s[(3 + j) * n_frame] = sqrtf(dx * dx + dy * dy + dz * dz);
    }
}

extern "C" int seqik_leg_series_f32(const float* pose, int64_t pose_chain_stride, int64_t pose_frame_stride,
                                    float* series, int64_t n_chain, int64_t n_frame, void* stream) {
    if (n_chain < 0 || n_frame < 0) return fail(SEQIK_EINVAL, "seqik_leg_series_f32: negative size");
    if (n_chain == 0 || n_frame == 0) return SEQIK_OK;
    if (!pose || !series) return fail(SEQIK_EINVAL, "seqik_leg_series_f32: NULL pointer");
    const int64_t total = n_chain * n_frame;
    leg_series_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(pose, pose_chain_stride, pose_frame_stride,
                                                                                        series, n_chain, n_frame);
    return check_launch("seqik_leg_series_f32");
}

// Order statistic by 4-pass MSB radix select on order-preserving keys; one block per (series, rank).
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

constexpr int SEL_BLOCK = 256;
constexpr int SEL_CACHE = 8192;             // order keys of a series cached in shared memory up to this length

// ranks of numpy.quantile(..., method="linear") at q = 0.45 and 0.55: floor(q (n-1)) and the next one
__device__ __forceinline__ void quantile_pos(double q, int64_t n, int64_t& lo, float& frac) {
    const double v = q * (double)(n - 1);
    lo = (int64_t)floor(v);
    if (lo > n - 1) lo = n - 1;
    frac = (float)(v - (double)lo);
}

// One block per series: the four order statistics (two neighbours of each of the 0.45 / 0.55 quantile positions)
// are found together by a 4-pass MSB radix select -- per pass one sweep over the series (from shared memory when it
// fits, else re-read from global/L2) feeding four 256-bin histograms -- and combined into the mid-quantile.
constexpr uint32_t MQ_RETRY = 0x7fc00001u;   // NaN payload a fast kernel leaves in `out` for the series it hands to the general one
__global__ void __launch_bounds__(SEL_BLOCK) mid_quantile_kernel(const float* __restrict__ series, const int32_t* __restrict__ counts,
                                                                 int64_t n, float* __restrict__ out, int only_flagged) {
    __shared__ unsigned int hist[4][256];
    __shared__ uint32_t s_prefix[4]; __shared__ unsigned long long s_rank[4]; __shared__ int s_hist[4];
    __shared__ uint32_t cache[SEL_CACHE];
    const int64_t sidx = blockIdx.x;
    if (only_flagged && __float_as_uint(out[sidx]) != MQ_RETRY) return;       // (block-uniform)
    const float* v = series + sidx * n;
    const int64_t m = counts ? (int64_t)counts[sidx] : n;             // values that take part (the m smallest)
    if (m <= 0) { if (threadIdx.x == 0) out[sidx] = __int_as_float(0x7fc00000); return; }
    const bool cached = n <= SEL_CACHE;
    if (cached) for (int64_t i = threadIdx.x; i < n; i += SEL_BLOCK) cache[i] = order_key(__ldg(v + i));
    int64_t lo45, lo55; float f45, f55;
    quantile_pos(0.45, m, lo45, f45); quantile_pos(0.55, m, lo55, f55);
    if (threadIdx.x < 4) {
        int64_t r = (threadIdx.x < 2 ? lo45 : lo55) + (threadIdx.x & 1);
        s_rank[threadIdx.x] = (unsigned long long)(r > m - 1 ? m - 1 : r); s_prefix[threadIdx.x] = 0;
    }
    uint32_t mask = 0;
    for (int pass = 3; pass >= 0; --pass) {
        const int shift = 8 * pass;
        for (int k = threadIdx.x; k < 4 * 256; k += SEL_BLOCK) (&hist[0][0])[k] = 0;
        __syncthreads();
        const uint32_t p0 = s_prefix[0], p1 = s_prefix[1], p2 = s_prefix[2], p3 = s_prefix[3];
        // ranks that still share a prefix share a histogram (the four ranks are two adjacent pairs: they separate only in
        // the last passes), which removes most of the shared-memory atomics
        const int h1 = (p1 == p0) ? 0 : 1, h2 = (p2 == p0) ? 0 : (p2 == p1) ? 1 : 2;
        const int h3 = (p3 == p0) ? 0 : (p3 == p1) ? 1 : (p3 == p2) ? 2 : 3;
        if (threadIdx.x == 0) { s_hist[0] = 0; s_hist[1] = h1; s_hist[2] = h2; s_hist[3] = h3; }
        for (int64_t i = threadIdx.x; i < n; i += SEL_BLOCK) {
            const uint32_t k = cached ? cache[i] : order_key(__ldg(v + i));
            const uint32_t km = k & mask, d = (k >> shift) & 0xFF;
            if (km == p0) atomicAdd(&hist[0][d], 1u);
            if (h1 == 1 && km == p1) atomicAdd(&hist[1][d], 1u);
            if (h2 == 2 && km == p2) atomicAdd(&hist[2][d], 1u);
            if (h3 == 3 && km == p3) atomicAdd(&hist[3][d], 1u);
        }
        __syncthreads();
        if (threadIdx.x < 4 * 32) {
            // warp w locates the bin of rank s_rank[w] in hist[w]: each lane sums 8 bins, a warp scan finds the lane whose
            // cumulative count first exceeds the rank, that lane walks its 8 bins (a serial 256-bin walk per pass was 4/5
            // of this kernel's time)
            const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
            const unsigned int* hrow = &hist[s_hist[w]][8 * lane];
            unsigned int own = 0;
#pragma unroll
            for (int d = 0; d < 8; ++d) own += hrow[d];
            unsigned int incl = own;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) { const unsigned int t = __shfl_up_sync(0xffffffffu, incl, off); if (lane >= off) incl += t; }
            const unsigned long long r = s_rank[w];
            const unsigned int hit = __ballot_sync(0xffffffffu, (unsigned long long)incl > r);
            const int sel = hit ? __ffs(hit) - 1 : 31;                     // first lane whose cumulative count exceeds the rank
            if (lane == sel) {
                unsigned long long acc = (unsigned long long)(incl - own); int d = 0;
                for (; d < 8; ++d) { if (acc + hrow[d] > r) break; acc += hrow[d]; }
                if (d > 7) d = 7;
                s_prefix[w] |= ((uint32_t)(8 * lane + d) << shift); s_rank[w] = r - acc;
            }
        }
        mask |= 0xFFu << shift;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const float a0 = key_value(s_prefix[0]), a1 = key_value(s_prefix[1]), b0 = key_value(s_prefix[2]), b1 = key_value(s_prefix[3]);
        const float q0 = a0 + (a1 - a0) * f45, q1 = b0 + (b1 - b0) * f55;
        out[sidx] = 0.5f * (q0 + q1);
    }
}

// Short series (n <= WQ_N, e.g. the 1000-frame trials of the benchmark configurations): ONE WARP per series, no block
// barrier.  warp_mid_quantile() is shared with the fused per-chain kernel below.  Against a plain 4-pass radix select
// (5 700 warp instructions per 1000-sample series, profiles/r02_stream_ncu.txt) it
//   * starts at the first bit in which the series' keys differ (one min/max sweep): the leading passes, in which every key
//     fell into the same bin -- 32-way conflicts on one shared-memory counter -- no longer exist, and the first digit is spread
//     over its 256 bins;
//   * aggregates equal digits of a warp instruction before the atomic (match.any), so that what conflicts remain cost one add;
//   * after a pass, compacts the keys that still share a prefix with one of the four ranks to the front of the cache (a few
//     per rank): the next pass sweeps those only, and with 32 or fewer left the ranks are read off directly (each lane counts
//     the keys below its own);
//   * packs the four histograms into 256 words of two 16-bit pairs (counts <= 1024): 2 KB per warp.
// The order statistics are exact; the interpolation (mid_quantile_value) is a + (b - a) f in float32, like the kernel it
// replaces -- within 2 u |q| of np.quantile(..., method="linear") in float64 for same-sign statistics, not always its bits.
constexpr int WQ_N = 1024, WQ_WARPS = 4;
__device__ __forceinline__ uint32_t low_mask(int nb) { return nb >= 32 ? 0xffffffffu : ((1u << nb) - 1u); }

// The four keys of ranks rank[0] <= rank[1] <= rank[2] <= rank[3] (0-based, in sorted order) of key[0..n) -> val[0..3], by ONE
// warp.  key: shared memory, 16-byte aligned, overwritten; hist: 2 x 256 words of this warp.  n <= 4096 (16-bit counters
// once the ranks have separated).  Keys are handled as offsets from the smallest one, so that the digits of every pass --
// 8 bits starting at the top bit of the SPAN max - min -- are spread whatever the exponent the series lives in (a segment
// length that wanders around 0.5 differs from its neighbours in bit 24 of the raw keys and in nothing else).
__device__ void warp_select4(uint32_t* __restrict__ key, int n, unsigned int* rank, unsigned int (*hist)[256], int lane, uint32_t* val) {
    const unsigned full = 0xffffffffu;
    const unsigned lt = (1u << lane) - 1u;
    uint32_t prefix[4];                                             // warp-uniform
    const uint4* key4 = reinterpret_cast<const uint4*>(key);
    const int n4 = n >> 2;
    uint32_t kmin = 0xffffffffu, kmax = 0u;
    for (int i = lane; i < n4; i += 32) {
        const uint4 k = key4[i];
        kmin = min(min(kmin, k.x), min(min(k.y, k.z), k.w)); kmax = max(max(kmax, k.x), max(max(k.y, k.z), k.w));
    }
    if (4 * n4 + lane < n) { const uint32_t k = key[4 * n4 + lane]; kmin = min(kmin, k); kmax = max(kmax, k); }
    kmin = __reduce_min_sync(full, kmin); kmax = __reduce_max_sync(full, kmax);
    int hi = 32 - __clz((int)(kmax - kmin));                        // offsets need the bits [0, hi) (0: a constant series)
    uint32_t mask = ~low_mask(hi);
#pragma unroll
    for (int k = 0; k < 4; ++k) prefix[k] = 0u;
    uint32_t sub = kmin;                                            // key[] holds raw keys until the first compaction, offsets after it
    int cnt = n;                                                    // keys still in play: key[0..cnt)
    const uint32_t* fin = key;                                      // where the candidates of the direct finish sit (as offsets)
    bool direct = false;
#pragma unroll 1
    while (hi > 0) {
        const int lo = hi > 8 ? hi - 8 : 0;
        const uint32_t dm = (1u << (hi - lo)) - 1u;
        // ranks that still share a prefix share a histogram (h is non-decreasing: equal prefixes are adjacent)
        int h[4];
        h[0] = 0; h[1] = (prefix[1] == prefix[0]) ? 0 : 1;
        h[2] = (prefix[2] == prefix[1]) ? h[1] : h[1] + 1;
        h[3] = (prefix[3] == prefix[2]) ? h[2] : h[2] + 1;
        const bool one = h[3] == 0 && cnt == n;                     // every key shares the one prefix: the first pass
        {
            uint4* z = reinterpret_cast<uint4*>(&hist[0][0]);
            const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
            for (int k = lane; k < (one ? 256 : 512) / 4; k += 32) z[k] = zero;
        }
        __syncwarp(full);
        if (one) {
            // no prefix test, 128 keys per step, 32-bit counters
            for (int i = lane; i < n4; i += 32) {
                const uint4 k = key4[i];
                atomicAdd(&hist[0][((k.x - sub) >> lo) & dm], 1u); atomicAdd(&hist[0][((k.y - sub) >> lo) & dm], 1u);
                atomicAdd(&hist[0][((k.z - sub) >> lo) & dm], 1u); atomicAdd(&hist[0][((k.w - sub) >> lo) & dm], 1u);
            }
            if (4 * n4 + lane < n) atomicAdd(&hist[0][((key[4 * n4 + lane] - sub) >> lo) & dm], 1u);
        } else {
            for (int i0 = 0; i0 < cnt; i0 += 32) {
                const int i = i0 + lane;
                const uint32_t k = i < cnt ? key[i] - sub : 0u;
                const uint32_t km = k & mask, d = (k >> lo) & dm;
                int hh = -1;                                        // histogram this key counts in
                if (i < cnt) hh = (km == prefix[0]) ? 0 : (km == prefix[1]) ? h[1] : (km == prefix[2]) ? h[2] : (km == prefix[3]) ? h[3] : -1;
                if (hh >= 0) atomicAdd(&hist[hh >> 1][d], 1u << (16 * (hh & 1)));
            }
        }
        __syncwarp(full);
        unsigned int own = 0, incl = 0, in_bins = 0;                // in_bins: keys in the (distinct) bins the ranks fall into
        const unsigned int cmask = one ? 0xffffffffu : 0xffffu;
        int bins[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            // the bin of rank[k] in its histogram: each lane sums 8 bins, a warp scan finds the lane whose cumulative count first
            // exceeds the rank, that lane walks its 8 bins and broadcasts (bin, count below, count in the bin)
            const unsigned int* hrow = &hist[h[k] >> 1][8 * lane];
            const int sh16 = 16 * (h[k] & 1);
            if (k == 0 || h[k] != h[k - 1]) {
                own = 0;
#pragma unroll
                for (int d = 0; d < 8; ++d) own += (hrow[d] >> sh16) & cmask;
                incl = own;
#pragma unroll
                for (int off = 1; off < 32; off <<= 1) { const unsigned int t = __shfl_up_sync(full, incl, off); if (lane >= off) incl += t; }
            }
            const unsigned int hit = __ballot_sync(full, incl > rank[k]);
            const int sel = hit ? __ffs(hit) - 1 : 31;
            unsigned int acc = incl - own, hv = 0; int d = 0;
            for (; d < 8; ++d) { hv = (hrow[d] >> sh16) & cmask; if (acc + hv > rank[k]) break; acc += hv; }
            if (d > 7) d = 7;
            bins[k] = __shfl_sync(full, 8 * lane + d, sel);
            const unsigned int below = __shfl_sync(full, acc, sel);
            const unsigned int inbin = __shfl_sync(full, hv, sel);
            if (k == 0 || h[k] != h[k - 1] || bins[k] != bins[k - 1]) in_bins += inbin;
            prefix[k] |= ((uint32_t)bins[k] << lo); rank[k] -= below;
        }
        mask |= dm << lo;
        hi = lo;
        if (hi == 0) break;
        if (one && in_bins <= 64u) {
            // the usual end: a handful of keys share a bin with one of the ranks.  They are gathered (in any order) into the
            // unused half of the histogram storage and the ranks are read off directly
            uint32_t* list = hist[1];
            unsigned int* cursor = &hist[0][0];                     // (the first histogram has been read: its first word counts)
            __syncwarp(full);
            if (lane == 0) *cursor = 0u;
            __syncwarp(full);
            const int b0 = bins[0], b1 = bins[1], b2 = bins[2], b3 = bins[3];
            auto take = [&](uint32_t k) {
                k -= sub;
                const int d = (int)((k >> lo) & dm);
                if (d == b0 || d == b1 || d == b2 || d == b3) list[atomicAdd(cursor, 1u)] = k;
            };
            for (int i = lane; i < n4; i += 32) { const uint4 k = key4[i]; take(k.x); take(k.y); take(k.z); take(k.w); }
            if (4 * n4 + lane < n) take(key[4 * n4 + lane]);
            __syncwarp(full);
            cnt = (int)in_bins; fin = list; direct = true;
            break;
        }
        // compaction: the keys that still match one of the four prefixes move to the front, as offsets (pos <= i, and every lane
        // has read its key of this step before any lane writes: in-place is safe)
        int out = 0;
        for (int i0 = 0; i0 < cnt; i0 += 32) {
            const int i = i0 + lane;
            const uint32_t k = i < cnt ? key[i] - sub : 0u;
            const uint32_t km = k & mask;
            const bool keep = i < cnt && (km == prefix[0] || km == prefix[1] || km == prefix[2] || km == prefix[3]);
            const unsigned b = __ballot_sync(full, keep);
            __syncwarp(full);                                       // (every lane holds its key: the ballot already implies it)
            if (keep) key[out + __popc(b & lt)] = k;
            out += __popc(b);
            __syncwarp(full);
        }
        cnt = out; sub = 0u;
        if (cnt <= 64) { direct = true; break; }
    }
    if (direct) {
        // each lane holds up to two candidates and counts the candidates of the same prefix group that sort before each of
        // them (ties by position): their ranks within the group
        const bool va = lane < cnt, vb = lane + 32 < cnt;
        const uint32_t ka = va ? fin[lane] : 0u, kb = vb ? fin[lane + 32] : 0u;
        const uint32_t ga = ka & mask, gb = kb & mask;
        unsigned int ra = 0, rb = 0;
        for (int j = 0; j < cnt; ++j) {
            const uint32_t kj = fin[j], gj = kj & mask;
            ra += (gj == ga && (kj < ka || (kj == ka && j < lane))) ? 1u : 0u;
            rb += (gj == gb && (kj < kb || (kj == kb && j < lane + 32))) ? 1u : 0u;
        }
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const unsigned int hit_a = __ballot_sync(full, va && ga == prefix[t] && ra == rank[t]);
            const unsigned int hit_b = __ballot_sync(full, vb && gb == prefix[t] && rb == rank[t]);
            const uint32_t from_a = __shfl_sync(full, ka, hit_a ? __ffs(hit_a) - 1 : 0);
            const uint32_t from_b = __shfl_sync(full, kb, hit_b ? __ffs(hit_b) - 1 : 0);
            val[t] = (hit_a ? from_a : from_b) + kmin;
        }
    } else {
#pragma unroll
        for (int t = 0; t < 4; ++t) val[t] = prefix[t] + kmin;
    }
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
__device__ __forceinline__ float mid_quantile_value(const uint32_t* val, float f45, float f55, bool swap) {
    const float a0 = key_value(val[0]), a1 = key_value(val[swap ? 2 : 1]), b0 = key_value(val[swap ? 1 : 2]), b1 = key_value(val[3]);
    const float q0 = a0 + (a1 - a0) * f45, q1 = b0 + (b1 - b0) * f55;
    return 0.5f * (q0 + q1);
}
// key[0..n): order keys of the series (shared memory, 16-byte aligned, overwritten); m: the m smallest take part
__device__ float warp_mid_quantile(uint32_t* __restrict__ key, int n, int64_t m, unsigned int (*hist)[256], int lane) {
    unsigned int rank[4]; uint32_t val[4]; float f45, f55;
    const bool swap = mid_quantile_ranks(m, rank, f45, f55);
    warp_select4(key, n, rank, hist, lane, val);
    return mid_quantile_value(val, f45, f55, swap);
}

__global__ void __launch_bounds__(32 * WQ_WARPS) mid_quantile_warp_kernel(const float* __restrict__ series, const int32_t* __restrict__ counts,
                                                                          int64_t n_series, int n, float* __restrict__ out) {
    __shared__ __align__(16) uint32_t cache[WQ_WARPS][WQ_N];
    __shared__ __align__(16) unsigned int hist[WQ_WARPS][2][256];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t sidx = (int64_t)blockIdx.x * WQ_WARPS + w;
    if (sidx >= n_series) return;                                 // whole warps leave: no block-level barrier below
    const float* v = series + sidx * n;
    const int64_t m = counts ? (int64_t)counts[sidx] : n;
    if (m <= 0) { if (lane == 0) out[sidx] = __int_as_float(0x7fc00000); return; }
    uint32_t* key = cache[w];
    for (int i = lane; i < n; i += 32) key[i] = order_key(__ldg(v + i));
    __syncwarp(0xffffffffu);
    const float q = warp_mid_quantile(key, n, m, hist[w], lane);
    if (lane == 0) out[sidx] = q;
}

// AlignPose.align_leg statistics of one chain in ONE kernel (recordings of up to LA_N frames): a CTA of seven warps streams
// the chain's key points through shared memory once (60 B per leg-frame: the only DRAM traffic), builds the order keys of
// the seven series -- coxa x, y, z and the four segment lengths, alignment.py:392-415 -- in shared memory, each warp
// selects the mid-quantile of one series, and thread 0 writes the affine row (find_scale_leg + align_leg,
// alignment.py:417-423, 465-485).  The series never exist in global memory (the three-kernel path below wrote and re-read
// 56 B per leg-frame).
constexpr int LA_WARPS = 7, LA_THREADS = 32 * LA_WARPS, LA_N = 1024, LA_TILE = LA_THREADS;
__global__ void __launch_bounds__(LA_THREADS) leg_affine_fused_kernel(const float* __restrict__ pose, int64_t cs, int64_t fs,
                                                                      const float* __restrict__ consts, int include_claw,
                                                                      float* __restrict__ affine, int n_frame) {
    __shared__ __align__(16) uint32_t key[LA_WARPS][LA_N];
    __shared__ __align__(16) union { float stage[LA_TILE * 15]; unsigned int hist[LA_WARPS][2][256]; } u;
    __shared__ float stat[8];
    const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
    const int64_t c = blockIdx.x;
    const float* src = pose + c * cs;
    const bool vec = fs == 15 && ((((uintptr_t)src) & 15) == 0);
    // tile t + 1 is in flight (four 128-bit loads per thread, held in registers) while the keys of tile t are built
    float4 pre[4];
    auto prefetch = [&](int f0) {
        const int nf = min(LA_TILE, n_frame - f0);
        const int n4 = nf * 15 / 4;
        const float4* s4 = reinterpret_cast<const float4*>(src + (int64_t)f0 * 15);      // (f0 * 60 B is a multiple of 16)
#pragma unroll
        for (int k = 0; k < 4; ++k) { const int i = tid + k * LA_THREADS; if (i < n4) pre[k] = __ldg(s4 + i); }
    };
    if (vec) prefetch(0);
    for (int f0 = 0; f0 < n_frame; f0 += LA_TILE) {
        const int nf = min(LA_TILE, n_frame - f0);
        const float* tsrc = src + (int64_t)f0 * fs;
        if (vec) {
            const int n4 = nf * 15 / 4;
            float4* d4 = reinterpret_cast<float4*>(u.stage);
#pragma unroll
            for (int k = 0; k < 4; ++k) { const int i = tid + k * LA_THREADS; if (i < n4) d4[i] = pre[k]; }
            for (int i = 4 * n4 + tid; i < nf * 15; i += LA_THREADS) u.stage[i] = __ldg(tsrc + i);
        } else {
            for (int i = tid; i < nf * 15; i += LA_THREADS) u.stage[i] = __ldg(tsrc + (int64_t)(i / 15) * fs + i % 15);
        }
        __syncthreads();
        if (vec && f0 + LA_TILE < n_frame) prefetch(f0 + LA_TILE);
        if (tid < nf) {
            const float* k = u.stage + tid * 15;                   // stride 15 words: conflict-free
            key[0][f0 + tid] = order_key(k[0]); key[1][f0 + tid] = order_key(k[1]); key[2][f0 + tid] = order_key(k[2]);
            // the SQUARED segment lengths are selected (the square root is monotone: the order statistics of the lengths are
            // the roots of the order statistics of the squares, bit for bit); the root is taken of the four selected values only
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float dx = k[3 * j + 3] - k[3 * j], dy = k[3 * j + 4] - k[3 * j + 1], dz = k[3 * j + 5] - k[3 * j + 2];
                key[3 + j][f0 + tid] = order_key(dx * dx + dy * dy + dz * dz);
            }
        }
        __syncthreads();
    }
    {
        unsigned int rank[4]; uint32_t val[4]; float f45, f55;
        const bool swap = mid_quantile_ranks(n_frame, rank, f45, f55);
        warp_select4(key[w], n_frame, rank, u.hist[w], lane, val);
        if (lane == 0) {
            float v4[4];
#pragma unroll
            for (int t = 0; t < 4; ++t) { v4[t] = key_value(val[t]); if (w >= 3) v4[t] = sqrtf(v4[t]); }
            if (swap) { const float t = v4[1]; v4[1] = v4[2]; v4[2] = t; }
            const float q0 = v4[0] + (v4[1] - v4[0]) * f45, q1 = v4[2] + (v4[3] - v4[2]) * f55;
            stat[w] = 0.5f * (q0 + q1);
        }
    }
    __syncthreads();
    if (tid == 0) {
        const float* k = consts + c * 4;
        float len = stat[3] + stat[4] + stat[5];
        if (include_claw) len += stat[6];
        float* a = affine + c * 8;
        a[0] = stat[0]; a[1] = stat[1]; a[2] = stat[2]; a[3] = k[3] / len;
        a[4] = k[0]; a[5] = k[1]; a[6] = k[2]; a[7] = 0.f;
    }
}

// Long series (recordings of more than WQ_N frames; BASELINE config 5 has 100 000): one block per series, TWO sweeps over
// global memory instead of four, and hardly any conflicting atomics.  A strided sample of 2048 keys gives the range the
// bulk of the series lives in; sweep 1 bins every key of that range by the top 12 bits of its offset from the sample's
// minimum (4096 bins: the bins of the four ranks hold n / 4096-ish keys each) and counts the keys below the range;
// sweep 2 gathers the keys of those bins (a few hundred) into shared memory, where one warp finishes with warp_select4.
// A series the sample does not describe -- a rank outside its range, more than LQ_CAND candidates (heavy ties) -- is left to
// the general kernel (MQ_RETRY in `out`).  Series of up to LQ_CAND samples skip the sweeps: keys to shared memory, one warp.
constexpr int LQ_BLOCK = 256, LQ_BINS = 4096, LQ_CAND = 4096, LQ_SAMPLE = 2048;
constexpr uint32_t KEY_INF = 0xff800000u;     // order_key(+inf): padding of the head series, never part of the range
__global__ void __launch_bounds__(LQ_BLOCK) mid_quantile_long_kernel(const float* __restrict__ series, const int32_t* __restrict__ counts,
                                                                     int64_t n, float* __restrict__ out) {
    __shared__ __align__(16) unsigned int hist[LQ_BINS];           // (the first 512 words serve warp_select4 afterwards)
    __shared__ __align__(16) uint32_t cand[LQ_CAND];
    __shared__ uint32_t s_min, s_max;
    __shared__ unsigned int s_below, s_cnt, s_warp_tot[LQ_BLOCK / 32];
    __shared__ int s_bin[4]; __shared__ unsigned int s_binbelow[4], s_bincount[4];
    const unsigned full = 0xffffffffu;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int64_t sidx = blockIdx.x;
    const float* v = series + sidx * n;
    const int64_t m = counts ? (int64_t)counts[sidx] : n;
    if (m <= 0) { if (tid == 0) out[sidx] = __int_as_float(0x7fc00000); return; }
    unsigned int rank[4]; uint32_t val[4]; float f45, f55;
    const bool swap = mid_quantile_ranks(m, rank, f45, f55);
    if (n <= LQ_CAND) {
        for (int i = tid; i < (int)n; i += LQ_BLOCK) cand[i] = order_key(__ldg(v + i));
        __syncthreads();
        if (w == 0) {
            warp_select4(cand, (int)n, rank, reinterpret_cast<unsigned int (*)[256]>(hist), lane, val);
            if (lane == 0) out[sidx] = mid_quantile_value(val, f45, f55, swap);
        }
        return;
    }
    // ---- the range of a strided sample (+inf padding left out)
    if (tid == 0) { s_min = 0xffffffffu; s_max = 0u; s_below = 0u; s_cnt = 0u; }
    for (int k = tid; k < LQ_BINS; k += LQ_BLOCK) hist[k] = 0u;
    __syncthreads();
    {
        const int64_t stride = n / LQ_SAMPLE;
        uint32_t lo = 0xffffffffu, hi = 0u;
        for (int j = tid; j < LQ_SAMPLE; j += LQ_BLOCK) {
            const uint32_t k = order_key(__ldg(v + (int64_t)j * stride));
            if (k < KEY_INF) { lo = min(lo, k); hi = max(hi, k); }
        }
        lo = __reduce_min_sync(full, lo); hi = __reduce_max_sync(full, hi);
        if (lane == 0) { atomicMin(&s_min, lo); atomicMax(&s_max, hi); }
    }
    __syncthreads();
    const uint32_t smin = s_min, smax = s_max;
    if (smin > smax) { if (tid == 0) out[sidx] = __uint_as_float(MQ_RETRY); return; }       // nothing finite in the sample
    const int nb = 32 - __clz((int)(smax - smin));
    const int shift = nb > 12 ? nb - 12 : 0;
    // ---- sweep 1
    {
        unsigned int below = 0;
        auto count = [&](float x) {
            const uint32_t k = order_key(x);
            if (k < smin) ++below;
            else if (k <= smax) atomicAdd(&hist[(k - smin) >> shift], 1u);
        };
        if ((((uintptr_t)v) & 15) == 0) {
            // four independent 128-bit loads in flight per thread (the sweep is bound by load latency, not by the counting)
            const float4* v4 = reinterpret_cast<const float4*>(v);
            const int64_t n4 = n >> 2;
            const float4 none = make_float4(__int_as_float(0x7fc00000), __int_as_float(0x7fc00000), __int_as_float(0x7fc00000), __int_as_float(0x7fc00000));
            for (int64_t i = tid; i < n4; i += 4 * LQ_BLOCK) {
                float4 x[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) x[k] = (i + k * LQ_BLOCK < n4) ? __ldg(v4 + i + k * LQ_BLOCK) : none;      // (NaN: above every range)
#pragma unroll
                for (int k = 0; k < 4; ++k) { count(x[k].x); count(x[k].y); count(x[k].z); count(x[k].w); }
            }
            for (int64_t i = 4 * n4 + tid; i < n; i += LQ_BLOCK) count(__ldg(v + i));
        } else {
            for (int64_t i = tid; i < n; i += LQ_BLOCK) count(__ldg(v + i));
        }
        below = __reduce_add_sync(full, below);
        if (lane == 0 && below) atomicAdd(&s_below, below);
    }
    __syncthreads();
    // ---- the bins of the four ranks: every thread owns 16 bins, block-wide exclusive scan of the per-thread sums
    unsigned int own = 0;
#pragma unroll
    for (int d = 0; d < 16; ++d) own += hist[16 * tid + d];
    unsigned int incl = own;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) { const unsigned int t = __shfl_up_sync(full, incl, off); if (lane >= off) incl += t; }
    if (lane == 31) s_warp_tot[w] = incl;
    if (tid < 4) s_bin[tid] = -1;
    __syncthreads();
    unsigned int base = 0, n_in = 0;
#pragma unroll
    for (int k = 0; k < LQ_BLOCK / 32; ++k) { if (k < w) base += s_warp_tot[k]; n_in += s_warp_tot[k]; }
    const unsigned int excl = base + incl - own;
    const unsigned int below_all = s_below;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        if (rank[t] >= below_all && rank[t] - below_all < n_in) {
            const unsigned int r = rank[t] - below_all;
            if (r >= excl && r < excl + own) {                      // exactly one thread
                unsigned int acc = excl; int d = 0;
                for (; d < 16; ++d) { const unsigned int hv = hist[16 * tid + d]; if (acc + hv > r) break; acc += hv; }
                if (d > 15) d = 15;
                s_bin[t] = 16 * tid + d; s_binbelow[t] = acc; s_bincount[t] = hist[16 * tid + d];
            }
        }
    }
    __syncthreads();
    const int b0 = s_bin[0], b1 = s_bin[1], b2 = s_bin[2], b3 = s_bin[3];
    // candidates = the keys of the distinct bins (b0 <= b1 <= b2 <= b3); rank of each target within their sorted list
    unsigned int c = 0, lrank[4];
    {
        const int bb[4] = {b0, b1, b2, b3};
        unsigned int before = 0;
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            if (t > 0 && bb[t] != bb[t - 1]) before += s_bincount[t - 1];
            lrank[t] = before + (rank[t] - below_all - s_binbelow[t]);
        }
        c = before + s_bincount[3];
    }
    if (b0 < 0 || b1 < 0 || b2 < 0 || b3 < 0 || (shift > 0 && c > (unsigned int)LQ_CAND)) {
        if (tid == 0) out[sidx] = __uint_as_float(MQ_RETRY);
        return;
    }
    if (shift == 0) {
        // the range spans fewer than 4096 distinct keys (a constant or few-valued series): a bin IS a key value
        if (tid == 0) {
            val[0] = smin + (uint32_t)b0; val[1] = smin + (uint32_t)b1; val[2] = smin + (uint32_t)b2; val[3] = smin + (uint32_t)b3;
            out[sidx] = mid_quantile_value(val, f45, f55, swap);
        }
        return;
    }
    // ---- sweep 2
    {
        auto take = [&](float x) {
            const uint32_t k = order_key(x);
            if (k >= smin && k <= smax) {
                const int d = (int)((k - smin) >> shift);
                if (d == b0 || d == b1 || d == b2 || d == b3) cand[atomicAdd(&s_cnt, 1u)] = k;
            }
        };
        if ((((uintptr_t)v) & 15) == 0) {
            const float4* v4 = reinterpret_cast<const float4*>(v);
            const int64_t n4 = n >> 2;
            const float4 none = make_float4(__int_as_float(0x7fc00000), __int_as_float(0x7fc00000), __int_as_float(0x7fc00000), __int_as_float(0x7fc00000));
            for (int64_t i = tid; i < n4; i += 4 * LQ_BLOCK) {
                float4 x[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) x[k] = (i + k * LQ_BLOCK < n4) ? __ldg(v4 + i + k * LQ_BLOCK) : none;
#pragma unroll
                for (int k = 0; k < 4; ++k) { take(x[k].x); take(x[k].y); take(x[k].z); take(x[k].w); }
            }
            for (int64_t i = 4 * n4 + tid; i < n; i += LQ_BLOCK) take(__ldg(v + i));
        } else {
            for (int64_t i = tid; i < n; i += LQ_BLOCK) take(__ldg(v + i));
        }
    }
    __syncthreads();
    if (w == 0) {
        warp_select4(cand, (int)c, lrank, reinterpret_cast<unsigned int (*)[256]>(hist), lane, val);
        if (lane == 0) out[sidx] = mid_quantile_value(val, f45, f55, swap);
    }
}

extern "C" int seqik_mid_quantile_f32(const float* series, const int32_t* counts, float* scratch, float* out,
                                      int64_t n_series, int64_t n, void* stream) {
    (void)scratch;   // kept in the signature (ABI): the single-kernel select needs no scratch
    if (n_series < 0 || n < 0) return fail(SEQIK_EINVAL, "seqik_mid_quantile_f32: negative size");
    if (n_series == 0) return SEQIK_OK;
    if (n == 0) return fail(SEQIK_EINVAL, "seqik_mid_quantile_f32: empty series");
    if (!series || !out) return fail(SEQIK_EINVAL, "seqik_mid_quantile_f32: NULL pointer");
    if (n_series > 2147483647LL) return fail(SEQIK_EINVAL, "seqik_mid_quantile_f32: too many series");
    if (n <= WQ_N) {
        mid_quantile_warp_kernel<<<(unsigned)((n_series + WQ_WARPS - 1) / WQ_WARPS), 32 * WQ_WARPS, 0, (cudaStream_t)stream>>>(series, counts, n_series, (int)n, out);
    } else {
        // two sweeps from a sampled range; the series it could not settle that way (MQ_RETRY) go through the general kernel
        mid_quantile_long_kernel<<<(unsigned)n_series, LQ_BLOCK, 0, (cudaStream_t)stream>>>(series, counts, n, out);
        mid_quantile_kernel<<<(unsigned)n_series, SEL_BLOCK, 0, (cudaStream_t)stream>>>(series, counts, n, out, 1);
    }
    return check_launch("seqik_mid_quantile_f32");
}

__global__ void leg_affine_kernel(const float* __restrict__ stats, const float* __restrict__ consts, int include_claw,
                                  float* __restrict__ affine, int64_t n_chain) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_chain) return;
    const float* s = stats + c * 7; const float* k = consts + c * 4;
    float len = s[3] + s[4] + s[5];
    if (include_claw) len += s[6];
    float* a = affine + c * 8;
    a[0] = s[0]; a[1] = s[1]; a[2] = s[2]; a[3] = k[3] / len;
    a[4] = k[0]; a[5] = k[1]; a[6] = k[2]; a[7] = 0.f;
}

extern "C" int seqik_leg_affine_f32(const float* stats, const float* consts, int include_claw, float* affine,
                                    int64_t n_chain, void* stream) {
    if (n_chain < 0) return fail(SEQIK_EINVAL, "seqik_leg_affine_f32: negative size");
    if (n_chain == 0) return SEQIK_OK;
    if (!stats || !consts || !affine) return fail(SEQIK_EINVAL, "seqik_leg_affine_f32: NULL pointer");
    leg_affine_kernel<<<(unsigned)((n_chain + 127) / 128), 128, 0, (cudaStream_t)stream>>>(stats, consts, include_claw, affine, n_chain);
    return check_launch("seqik_leg_affine_f32");
}

// The whole statistics step of AlignPose.align_leg behind one call: key points -> affine rows.  Recordings of up to LA_N frames
// run the fused per-chain kernel (no scratch needed); longer ones the series / select / affine kernels with the series in
// `scratch` (n_chain * 7 * (n_frame + 1) floats).
extern "C" int seqik_leg_affine_from_pose_f32(const float* pose, int64_t pose_chain_stride, int64_t pose_frame_stride,
                                              const float* consts, int include_claw, float* scratch, float* affine,
                                              int64_t n_chain, int64_t n_frame, void* stream) {
    if (n_chain < 0 || n_frame < 0) return fail(SEQIK_EINVAL, "seqik_leg_affine_from_pose_f32: negative size");
    if (n_chain == 0) return SEQIK_OK;
    if (n_frame == 0) return fail(SEQIK_EINVAL, "seqik_leg_affine_from_pose_f32: empty recording");
    if (!pose || !consts || !affine) return fail(SEQIK_EINVAL, "seqik_leg_affine_from_pose_f32: NULL pointer");
    if (pose_frame_stride < 15) return fail(SEQIK_EINVAL, "seqik_leg_affine_from_pose_f32: frame stride smaller than the innermost block");
    if (n_chain > 2147483647LL) return fail(SEQIK_EINVAL, "seqik_leg_affine_from_pose_f32: too many chains");
    if (n_frame <= LA_N) {
        leg_affine_fused_kernel<<<(unsigned)n_chain, LA_THREADS, 0, (cudaStream_t)stream>>>(pose, pose_chain_stride, pose_frame_stride, consts,
                                                                                          include_claw, affine, (int)n_frame);
        return check_launch("seqik_leg_affine_from_pose_f32");
    }
    if (!scratch) return fail(SEQIK_EINVAL, "seqik_leg_affine_from_pose_f32: recordings of more than 1024 frames need the scratch buffer");
    float* series = scratch;
    float* stats = scratch + n_chain * 7 * n_frame;
    int rc = seqik_leg_series_f32(pose, pose_chain_stride, pose_frame_stride, series, n_chain, n_frame, stream);
    if (rc != SEQIK_OK) return rc;
    rc = seqik_mid_quantile_f32(series, nullptr, nullptr, stats, n_chain * 7, n_frame, stream);
    if (rc != SEQIK_OK) return rc;
    return seqik_leg_affine_f32(stats, consts, include_claw, affine, n_chain, stream);
}

__global__ void __launch_bounds__(256) align_apply_kernel(const float* __restrict__ pose, int64_t cs, int64_t fs,
                                                          const float* __restrict__ affine, float* __restrict__ out,
                                                          int64_t n_chain, int64_t n_frame, int64_t first) {
    const int64_t i = first + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // one thread per (leg-frame, key point)
    if (i >= n_chain * n_frame * 5) return;
    const int64_t lf = i / 5; const int kp = (int)(i - lf * 5);
    const int64_t c = lf / n_frame, t = lf - c * n_frame;
    const float* a = affine + c * 8;
    const float* p = pose + c * cs + t * fs + kp * 3;
    float* o = out + i * 3;
    if (kp == 0) { o[0] = a[4]; o[1] = a[5]; o[2] = a[6]; }
    else { o[0] = (p[0] - a[0]) * a[3] + a[4]; o[1] = (p[1] - a[1]) * a[3] + a[5]; o[2] = (p[2] - a[2]) * a[3] + a[6]; }
}

// TMA pipeline variant for a dense pose array: a tile = 256 leg-frames x 15 floats in, the same out
struct AlignOp {
    const float* pose; const float* affine; float* out; int64_t n_frame;
    static constexpr int N_IN = 1, STAGE_BYTES = TILE * 30 * 4, OUT_OFF = TILE * 15 * 4;
    static __device__ __forceinline__ int in_off(int) { return 0; }
    __device__ __forceinline__ uint32_t in_bytes(int, int64_t) const { return TILE * 15 * 4; }
    __device__ __forceinline__ const void* in_src(int, int64_t tile) const { return pose + tile * (TILE * 15); }
    __device__ __forceinline__ void compute(int tid, int64_t tile, unsigned char* stage) const {
        const float* s_in = reinterpret_cast<const float*>(stage);
        float* s_out = reinterpret_cast<float*>(stage + OUT_OFF);
        for (int e = tid; e < TILE * 5; e += TILE) {              // one (leg-frame, key point) per step: conflict-free 12-byte records
            const int lf = e / 5, kp = e - lf * 5;
            const float* a = affine + ((tile * TILE + lf) / n_frame) * 8;
            const float* p = s_in + e * 3;
            float* o = s_out + e * 3;
            if (kp == 0) { o[0] = __ldg(a + 4); o[1] = __ldg(a + 5); o[2] = __ldg(a + 6); }
            else {
                const float sc = __ldg(a + 3);
                o[0] = (p[0] - __ldg(a)) * sc + __ldg(a + 4); o[1] = (p[1] - __ldg(a + 1)) * sc + __ldg(a + 5); o[2] = (p[2] - __ldg(a + 2)) * sc + __ldg(a + 6);
            }
        }
    }
    __device__ __forceinline__ void store(int64_t tile, const unsigned char* o) const { tma_store_1d_nocommit(out + tile * (TILE * 15), o, TILE * 15 * 4); }
};

extern "C" int seqik_align_apply_f32(const float* pose, int64_t pose_chain_stride, int64_t pose_frame_stride,
                                     const float* affine, float* out, int64_t n_chain, int64_t n_frame, void* stream) {
    if (n_chain < 0 || n_frame < 0) return fail(SEQIK_EINVAL, "seqik_align_apply_f32: negative size");
    if (n_chain == 0 || n_frame == 0) return SEQIK_OK;
    if (!pose || !affine || !out) return fail(SEQIK_EINVAL, "seqik_align_apply_f32: NULL pointer");
    const int64_t lf_total = n_chain * n_frame, full_tiles = lf_total / TILE, done = full_tiles * TILE;
    const bool dense = pose_frame_stride == 15 && pose_chain_stride == n_frame * 15;
    const bool aligned = ((((uintptr_t)pose) | ((uintptr_t)out)) & 15) == 0;
    cudaStream_t st = (cudaStream_t)stream;
    if (dense && aligned && full_tiles > 0) {
        launch_tiles(AlignOp{pose, affine, out, n_frame}, full_tiles, st);
        if (lf_total > done)
            align_apply_kernel<<<(unsigned)(((lf_total - done) * 5 + 255) / 256), 256, 0, st>>>(pose, pose_chain_stride, pose_frame_stride,
                                                                                             affine, out, n_chain, n_frame, done * 5);
    } else {
        const int64_t total = lf_total * 5;
        align_apply_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(pose, pose_chain_stride, pose_frame_stride,
                                                                          affine, out, n_chain, n_frame, 0);
    }
    return check_launch("seqik_align_apply_f32");
}

// ---- antenna (AlignPose.align_head)
// The stationarity test thresholds a SECOND DIFFERENCE of distances (5e-5 against values ~1): it is evaluated in
// FP64 whatever the input type, because a single flipped frame moves the order statistics that follow by ~1e-4.
template <typename T>
__device__ __forceinline__ double base_to_thorax_mid(const T* __restrict__ head, const T* __restrict__ thorax,
                                                     int64_t n_kp, int64_t i) {
    const T* b = head + i * 6;
    const T* t0 = thorax + i * n_kp * 3; const T* t1 = t0 + (n_kp - 1) * 3;
    const double dx = (double)b[0] - 0.5 * ((double)t0[0] + (double)t1[0]);
    const double dy = (double)b[1] - 0.5 * ((double)t0[1] + (double)t1[1]);
    const double dz = (double)b[2] - 0.5 * ((double)t0[2] + (double)t1[2]);
    return sqrt(dx * dx + dy * dy + dz * dz);
}

template <typename T>
__global__ void __launch_bounds__(256) head_series_kernel(const T* __restrict__ head, const T* __restrict__ thorax,
                                                          int64_t n_kp, double threshold, float* __restrict__ series,
                                                          int32_t* __restrict__ counts, int64_t n_trial, int64_t n_frame) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool in = i < n_trial * n_frame;
    const int64_t tr = in ? i / n_frame : 0, t = in ? i - tr * n_frame : 0;
    bool stationary = false;
    if (in) {
        const T* b = head + i * 6;
        const double d0 = base_to_thorax_mid(head, thorax, n_kp, i);
        if (t + 2 < n_frame) {
            const double d1 = base_to_thorax_mid(head, thorax, n_kp, i + 1), d2 = base_to_thorax_mid(head, thorax, n_kp, i + 2);
            stationary = ((d2 - d1) - (d1 - d0)) < threshold;   // np.diff(np.diff(d)) < threshold, signed
        }
        const float inf = __int_as_float(0x7f800000);
        float* s = series + tr * 5 * n_frame + t;
        s[0] = stationary ? (float)b[0] : inf; s[n_frame] = stationary ? (float)b[1] : inf; s[2 * n_frame] = stationary ? (float)b[2] : inf;
        s[3 * n_frame] = stationary ? (float)d0 : inf;
        const double ax = (double)b[3] - (double)b[0], ay = (double)b[4] - (double)b[1], az = (double)b[5] - (double)b[2];
        s[4 * n_frame] = (float)sqrt(ax * ax + ay * ay + az * az);
    }
    // count stationary frames per trial: warp vote, one atomic per (warp, trial) when the warp sits in one trial
    const unsigned ballot = __ballot_sync(0xffffffffu, stationary);
    const int64_t tr0 = __shfl_sync(0xffffffffu, tr, 0);
    const bool uniform = __all_sync(0xffffffffu, !in || tr == tr0);
    if (uniform) {
        if ((threadIdx.x & 31) == 0 && ballot) atomicAdd(&counts[tr0 * 5], __popc(ballot));
    } else if (stationary) atomicAdd(&counts[tr * 5], 1);
}

__global__ void head_counts_finish_kernel(int32_t* __restrict__ counts, int64_t n_trial, int64_t n_frame) {
    const int64_t tr = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (tr >= n_trial) return;
    int32_t* c = counts + tr * 5;
    c[1] = c[0]; c[2] = c[0]; c[3] = c[0]; c[4] = (int32_t)n_frame;
}

template <typename T>
static int head_series_launch(const char* name, const T* head, const T* thorax, int64_t n_thorax_kp, double threshold,
                              float* series, int32_t* counts, int64_t n_trial, int64_t n_frame, void* stream) {
    if (n_trial < 0 || n_frame < 0) return fail(SEQIK_EINVAL, "%s: negative size", name);
    if (n_trial == 0 || n_frame == 0) return SEQIK_OK;
    if (!head || !thorax || !series || !counts) return fail(SEQIK_EINVAL, "%s: NULL pointer", name);
    if (n_thorax_kp < 1) return fail(SEQIK_EINVAL, "%s: thorax needs at least one key point", name);
    if (n_frame > 2147483647LL) return fail(SEQIK_EINVAL, "%s: too many frames", name);
    cudaStream_t st = (cudaStream_t)stream;
    if (cudaMemsetAsync(counts, 0, sizeof(int32_t) * 5 * n_trial, st) != cudaSuccess) return check_launch(name);
    const int64_t n = n_trial * n_frame;
    head_series_kernel<T><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(head, thorax, n_thorax_kp, threshold, series, counts, n_trial, n_frame);
    int rc = check_launch(name);
    if (rc) return rc;
    head_counts_finish_kernel<<<(unsigned)((n_trial + 127) / 128), 128, 0, st>>>(counts, n_trial, n_frame);
    return check_launch(name);
}

extern "C" int seqik_head_series_f32(const float* head, const float* thorax, int64_t n_thorax_kp, float threshold,
                                     float* series, int32_t* counts, int64_t n_trial, int64_t n_frame, void* stream) {
    return head_series_launch<float>("seqik_head_series_f32", head, thorax, n_thorax_kp, (double)threshold, series, counts,
                                     n_trial, n_frame, stream);
}
extern "C" int seqik_head_series_f64(const double* head, const double* thorax, int64_t n_thorax_kp, double threshold,
                                     float* series, int32_t* counts, int64_t n_trial, int64_t n_frame, void* stream) {
    return head_series_launch<double>("seqik_head_series_f64", head, thorax, n_thorax_kp, threshold, series, counts,
                                      n_trial, n_frame, stream);
}

__global__ void head_affine_kernel(const float* __restrict__ stats, const float* __restrict__ consts, float* __restrict__ affine,
                                   int64_t n_trial) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_trial) return;
    const float* s = stats + c * 5; const float* k = consts + c * 5;
    float* a = affine + c * 8;
    a[0] = s[0]; a[1] = s[1]; a[2] = s[2]; a[3] = k[3] / s[3];
    a[4] = k[0]; a[5] = k[1]; a[6] = k[2]; a[7] = k[4] / s[4];
}

extern "C" int seqik_head_affine_f32(const float* stats, const float* consts, float* affine, int64_t n_trial, void* stream) {
    if (n_trial < 0) return fail(SEQIK_EINVAL, "seqik_head_affine_f32: negative size");
    if (n_trial == 0) return SEQIK_OK;
    if (!stats || !consts || !affine) return fail(SEQIK_EINVAL, "seqik_head_affine_f32: NULL pointer");
    head_affine_kernel<<<(unsigned)((n_trial + 127) / 128), 128, 0, (cudaStream_t)stream>>>(stats, consts, affine, n_trial);
    return check_launch("seqik_head_affine_f32");
}

__global__ void __launch_bounds__(256) head_apply_kernel(const float* __restrict__ head, const float* __restrict__ affine,
                                                         float* __restrict__ out, int64_t n_trial, int64_t n_frame, int64_t first) {
    const int64_t i = first + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // one thread per (frame, key point)
    if (i >= n_trial * n_frame * 2) return;
    const int64_t tr = (i >> 1) / n_frame;
    float x, y, z;
    head_point(head + i * 3, affine + tr * 8, (i & 1) != 0, x, y, z);
    out[i * 3] = x; out[i * 3 + 1] = y; out[i * 3 + 2] = z;
}

// TMA pipeline variant: a tile = 1024 frames x 6 floats in, the same out (four frames per thread)
struct HeadApplyOp {
    const float* head; const float* affine; float* out; int64_t n_frame;
    static constexpr int FRAMES = 4 * TILE, N_IN = 1, STAGE_BYTES = FRAMES * 12 * 4, OUT_OFF = FRAMES * 6 * 4;
    static __device__ __forceinline__ int in_off(int) { return 0; }
    __device__ __forceinline__ uint32_t in_bytes(int, int64_t) const { return FRAMES * 6 * 4; }
    __device__ __forceinline__ const void* in_src(int, int64_t tile) const { return head + tile * (FRAMES * 6); }
    __device__ __forceinline__ void compute(int tid, int64_t tile, unsigned char* stage) const {
        const float* s_in = reinterpret_cast<const float*>(stage);
        float* s_out = reinterpret_cast<float*>(stage + OUT_OFF);
        for (int e = tid; e < FRAMES * 2; e += TILE) {            // one key point (base / tip) per step
            const int64_t tr = (tile * FRAMES + (e >> 1)) / n_frame;
            float x, y, z;
            head_point(s_in + e * 3, affine + tr * 8, (e & 1) != 0, x, y, z);
            s_out[e * 3] = x; s_out[e * 3 + 1] = y; s_out[e * 3 + 2] = z;
        }
    }
    __device__ __forceinline__ void store(int64_t tile, const unsigned char* o) const { tma_store_1d_nocommit(out + tile * (FRAMES * 6), o, FRAMES * 6 * 4); }
};

extern "C" int seqik_head_apply_f32(const float* head, const float* affine, float* out, int64_t n_trial, int64_t n_frame,
                                    void* stream) {
    if (n_trial < 0 || n_frame < 0) return fail(SEQIK_EINVAL, "seqik_head_apply_f32: negative size");
    if (n_trial == 0 || n_frame == 0) return SEQIK_OK;
    if (!head || !affine || !out) return fail(SEQIK_EINVAL, "seqik_head_apply_f32: NULL pointer");
    const int64_t frames = n_trial * n_frame, full_tiles = frames / HeadApplyOp::FRAMES, done = full_tiles * HeadApplyOp::FRAMES;
    const bool aligned = ((((uintptr_t)head) | ((uintptr_t)out)) & 15) == 0;
    cudaStream_t st = (cudaStream_t)stream;
    if (aligned && full_tiles > 0) {
        launch_tiles(HeadApplyOp{head, affine, out, n_frame}, full_tiles, st);
        if (frames > done)
            head_apply_kernel<<<(unsigned)(((frames - done) * 2 + 255) / 256), 256, 0, st>>>(head, affine, out, n_trial, n_frame, done * 2);
    } else {
        head_apply_kernel<<<(unsigned)((frames * 2 + 255) / 256), 256, 0, st>>>(head, affine, out, n_trial, n_frame, 0);
    }
    return check_launch("seqik_head_apply_f32");
}

// ---------------------------------------------------------------------------------------------
// pchip resampling of joint-angle series (the hand-off to a simulation time step)
// ---------------------------------------------------------------------------------------------
// utils.interpolate_signal (seqikpy/utils.py:332-349) = scipy.interpolate.pchip_interpolate(arange(0, n ts, ts), y,
// arange(0, n ts, new_ts)): Fritsch-Carlson derivatives (harmonic mean of the neighbouring secant slopes, 0 at a local
// extremum, the three-point rule with its two clamps at the ends), cubic Hermite pieces evaluated in the power basis
// about the left knot, and -- because the new grid runs past the last sample -- the last piece extrapolated.
// One thread per output sample; `width` interleaved channels ([block][sample][width], e.g. the 7 DOFs of an angles
// tensor) so that loads and stores of neighbouring threads are contiguous.  HBM-bound: (n + m) * width values per block.
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
// W = compile-time channel count (1 or 7: index arithmetic by multiply-shift), 0 = run-time `width` (<= 256).
// One thread per (interval k, channel j): the derivatives and the cubic's coefficients are computed once per interval and
// every sample of the new grid that falls into it is evaluated from them (10 samples per interval for 100 Hz -> 1 kHz);
// the samples past the last knot belong to the last interval.  A CTA owns floor(256 / width) whole intervals, hence one
// CONTIGUOUS range of the output, which it assembles in shared memory and writes with coalesced (128-bit) stores; ranges
// too long for the buffer (extreme up-sampling) are stored directly.  grid.x tiles the n - 1 intervals of one block row,
// grid.y strides over the block rows (the FP64 interval bounds are computed once per thread): no 64-bit division.
constexpr int PCHIP_STAGE_BYTES = 32768;
template <typename T, int W>
__global__ void __launch_bounds__(256) pchip_kernel(const T* __restrict__ in, T* __restrict__ out, int64_t n_block, int n,
                                                    int m, int width_rt, double ts, double new_ts, double inv_new_ts) {
    constexpr int CAP = PCHIP_STAGE_BYTES / (int)sizeof(T);
    __shared__ __align__(16) T stage[CAP];
    __shared__ int s_first, s_end;
    const int width = W ? W : width_rt;
    const int kpc = 256 / width;                                 // intervals per CTA
    const int kl = (int)threadIdx.x / width, j = (int)threadIdx.x - kl * width;
    const int k0 = (int)blockIdx.x * kpc, k1 = min(k0 + kpc, n - 1) - 1;     // this CTA's intervals
    const int k = k0 + kl;
    const bool active = kl < kpc && k <= k1;
    // samples u of the new grid with k ts <= u new_ts < (k + 1) ts  (same comparisons as scipy's interval search)
    const double xk = (double)k * ts, xk1 = (double)(k + 1) * ts;
    int u_lo = 0, u_hi = 0;
    if (active) {
        u_lo = (int)ceil(xk * inv_new_ts); u_hi = (int)ceil(xk1 * inv_new_ts);
        while (u_lo > 0 && (double)(u_lo - 1) * new_ts >= xk) --u_lo;
        while ((double)u_lo * new_ts < xk) ++u_lo;
        while (u_hi > 0 && (double)(u_hi - 1) * new_ts >= xk1) --u_hi;
        while ((double)u_hi * new_ts < xk1) ++u_hi;
        if (k == n - 2) u_hi = m;                               // the last piece is extrapolated over the rest of the grid
        u_hi = min(u_hi, m); u_lo = min(u_lo, u_hi);
        if (j == 0 && k == k0) s_first = u_lo;
        if (j == 0 && k == k1) s_end = u_hi;
    }
    __syncthreads();
    const int first = s_first, n_out = (s_end - first) * width;  // the CTA's output range [first, s_end) x width
    if (n_out <= 0) return;                                      // down-sampling: no sample in these intervals
    const bool staged = n_out <= CAP;
    const T h = (T)ts, rh = (T)(1.0 / ts);
    for (int64_t b = blockIdx.y; b < n_block; b += gridDim.y) {
        T* dst = out + (b * m + first) * width;
        if (active && u_lo < u_hi) {
            const T* y = in + (b * n + k) * width + j;
            const T y0 = __ldg(y), y1 = __ldg(y + width);
            const T slope = (y1 - y0) * rh;
            T d0, d1;
            if (n == 2) { d0 = slope; d1 = slope; }
            else {
                // secant slopes of the neighbouring intervals (where they exist)
                const T m_prev = (k > 0) ? (y0 - __ldg(y - width)) * rh : T(0);
                const T m_next = (k + 2 < n) ? (__ldg(y + 2 * width) - y1) * rh : T(0);
                d0 = (k > 0) ? pchip_inner(m_prev, slope) : pchip_edge(h, h, slope, m_next);
                d1 = (k + 2 < n) ? pchip_inner(slope, m_next) : pchip_edge(h, h, slope, m_prev);
            }
            // CubicHermiteSpline coefficients (power basis about the left knot), summed in ascending powers like PPoly
            const T t_ = (d0 + d1 - T(2) * slope) * rh;
            const T c0 = t_ * rh, c1 = (slope - d0) * rh - t_;
            T* o = (staged ? stage : dst) + (u_lo - first) * width + j;
            if (sizeof(T) == 4) {
                // float32: the offset of the first sample from the knot in float64, then one float32 multiply-add per sample
                // (s is rounded to float32 anyway; the error of the increment stays below half an ulp of the interval
                // length) -- four FP64-pipe instructions per output sample were the largest item of this kernel's issue budget
                const float s0 = (float)((double)u_lo * new_ts - xk), dt = (float)new_ts;
                float ur = 0.f;
                const float k0 = (float)y0, k1 = (float)d0, k2 = (float)c1, k3 = (float)c0;
                for (int u = u_lo; u < u_hi; ++u, o += width, ur += 1.f) {
                    const float s = fmaf(ur, dt, s0);
                    *o = (T)fmaf(fmaf(fmaf(k3, s, k2), s, k1), s, k0);      // Horner, three multiply-adds (float32 bound: 2e-6 relative)
                }
            } else {
                for (int u = u_lo; u < u_hi; ++u, o += width) {
                    const T s = (T)((double)u * new_ts - xk);
                    T res = y0, z = s;
                    res += d0 * z; z *= s;
                    res += c1 * z; z *= s;
                    res += c0 * z;
                    *o = res;
                }
            }
        }
        if (staged) {
            __syncthreads();
            // coalesced copy-out; 128-bit when the destination allows it
            constexpr int V = 16 / (int)sizeof(T);
            const int head = (int)(((16 - ((uintptr_t)dst & 15)) & 15) / sizeof(T));    // elements up to the first 16-byte boundary
            if (head == 0 && (n_out % V) == 0) {
                const float4* s4 = reinterpret_cast<const float4*>(stage); float4* d4 = reinterpret_cast<float4*>(dst);
                for (int i = threadIdx.x; i < n_out / V; i += blockDim.x) __stcs(d4 + i, s4[i]);
            } else {
                for (int i = threadIdx.x; i < n_out; i += blockDim.x) dst[i] = stage[i];
            }
            __syncthreads();
        }
    }
}
template <typename T>
static int pchip_launch(const char* me, const T* in, T* out, int64_t n_block, int64_t n, int64_t m, int64_t width,
                        double original_ts, double new_ts, void* stream) {
    if (n_block < 0 || n < 0 || m < 0 || width < 0) return seqik_fail(SEQIK_EINVAL, "%s: negative size", me);
    if (n_block == 0 || m == 0 || width == 0) return SEQIK_OK;
    if (n < 2) return seqik_fail(SEQIK_EINVAL, "%s: at least 2 samples are needed", me);
    if (!in || !out) return seqik_fail(SEQIK_EINVAL, "%s: NULL pointer", me);
    if (!(original_ts > 0.0) || !(new_ts > 0.0)) return seqik_fail(SEQIK_EINVAL, "%s: time steps must be positive", me);
    if (n * width > 2147483647LL || m * width > 2147483647LL) return seqik_fail(SEQIK_EINVAL, "%s: series too long for one launch", me);
    // ~1 M threads fill the machine; beyond that a thread walks over block rows (its interval bounds are computed once)
    if (width > 256) return seqik_fail(SEQIK_EINVAL, "%s: at most 256 interleaved channels", me);
    const int64_t kpc = 256 / width;
    const int64_t gx = (n - 1 + kpc - 1) / kpc;
    int64_t gy = (1LL << 20) / (gx * 256);
    gy = gy < 1 ? 1 : (gy > n_block ? n_block : gy);
    if (gy > 65535) gy = 65535;
    const dim3 grid((unsigned)gx, (unsigned)gy);
    const double inv_new = 1.0 / new_ts;
    cudaStream_t st = (cudaStream_t)stream;
    if (width == 7) pchip_kernel<T, 7><<<grid, 256, 0, st>>>(in, out, n_block, (int)n, (int)m, 7, original_ts, new_ts, inv_new);
    else if (width == 1) pchip_kernel<T, 1><<<grid, 256, 0, st>>>(in, out, n_block, (int)n, (int)m, 1, original_ts, new_ts, inv_new);
    else pchip_kernel<T, 0><<<grid, 256, 0, st>>>(in, out, n_block, (int)n, (int)m, (int)width, original_ts, new_ts, inv_new);
    return seqik_check_launch(me);
}
extern "C" int seqik_pchip_resample_f32(const float* in, float* out, int64_t n_block, int64_t n, int64_t m, int64_t width,
                                        double original_ts, double new_ts, void* stream) {
    return pchip_launch<float>("seqik_pchip_resample_f32", in, out, n_block, n, m, width, original_ts, new_ts, stream);
}
extern "C" int seqik_pchip_resample_f64(const double* in, double* out, int64_t n_block, int64_t n, int64_t m, int64_t width,
                                        double original_ts, double new_ts, void* stream) {
    return pchip_launch<double>("seqik_pchip_resample_f64", in, out, n_block, n, m, width, original_ts, new_ts, stream);
}
