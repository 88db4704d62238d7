// seqik_head_grad.cu -- seqik_head_angles_backward_f32 (include/seqik.h): the backward (vector-Jacobian product) of the
// head / antenna angles.  A translation unit of its own, so that adding it leaves the code generated for seqik_kernels.cu
// unchanged.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/seqik.h"
#include "seqik_common.h"
#include "seqik_core.cuh"
#include "seqik_head.cuh"

using namespace seqik;

// 1 / r2 of a squared length; 0 for r2 == 0 (the vector's terms then vanish: torch.atan2's gradient at (0, 0)).  A
// subnormal r2 is taken as FLT_MIN, so that a vector shorter than ~1e-19 still gives finite terms.
__device__ __forceinline__ float inv_sq(float r2) {
    float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(fmaxf(r2, 1.17549435e-38f)));
    return r2 > 0.f ? r : 0.f;
}

// One frame, the forward of head_frame (seqik_kernels.cu) recomputed with its arithmetic up to the roll's sin / cos, then
// one reverse pass.  Every angle is theta = atan2(e . (a x b), a . b), measured from a to b about the axis e, of vectors
// projected onto the plane normal to e; dtheta/db = (e x b) / |b|^2 and dtheta/da = -(e x a) / |a|^2.
//   roll   Y -> hor|x=0 about X:           dL/dhor += g0' (0, -hz, hy) / (hy^2 + hz^2), g0' = g0 + the antenna terms below
//   pitch  X -> mid|y=0 about Y:           dL/dmid = g1 (mz, 0, -mx) / (mx^2 + mz^2), mid = (rb + lb) / 2 - neck
//   yaw    Y -> hor|z=0 about Z:           dL/dhor += g2 (-hy, hx, 0) / (hx^2 + hy^2)
//   antenna yaw (per side) ad|x=0 -> hd|x=0 about X, antenna pitch gd|y=0 -> ad|y=0 about Y, where ad, hd, gd are the
//   antenna vector, hor and neck - base de-rotated by Rx(-roll): (y, z) -> (y c + z s, -y s + z c).  A de-rotated v has
//   dv/droll = (vz, -vy) in (y, z), so each of their terms also feeds the roll: dL/droll += G_vy vz - G_vz vy; and the
//   gradient of the raw vector is the transposed rotation of G_v: (c G_vy - s G_vz, s G_vy + c G_vz).  For the antenna
//   yaw both vectors are de-rotated about the angle's own axis and the two roll terms cancel in exact arithmetic (+g - g,
//   unless one vector is zero); the antenna pitch's do not.  The right antenna yaw is pi - theta: its gradient changes sign.
// The neck enters the head pitch (through mid - neck) and both antenna pitches (through neck - base).  Gradients with
// respect to the aligned points; the caller multiplies by the affine scale.
// g: 7 incoming gradients; grr / gll: (base xyz, tip xyz) out; gn: 3 out.
__device__ __forceinline__ void head_frame_backward(const float* rr, const float* ll, const float* nk, const float* __restrict__ ar,
                                                    const float* __restrict__ al, const float* g, float* grr, float* gll, float* gn) {
    float rbx, rby, rbz, rtx, rty, rtz, lbx, lby, lbz, ltx, lty, ltz;
    head_point(rr, ar, false, rbx, rby, rbz); head_point(rr + 3, ar, true, rtx, rty, rtz);
    head_point(ll, al, false, lbx, lby, lbz); head_point(ll + 3, al, true, ltx, lty, ltz);
    const float nx = nk[0], ny = nk[1], nz = nk[2];
    const float hx = lbx - rbx, hy = lby - rby, hz = lbz - rbz;
    const float mx = (rbx + lbx) * 0.5f - nx, mz = (rbz + lbz) * 0.5f - nz;
    const float roll = signed_angle(hy, hz);
    float s, c, vers; Num<float>::sincosv_(roll, &s, &c, &vers);
    const float hdy = hy * c + hz * s, hdz = -hy * s + hz * c;

    // head pitch and yaw
    const float wm = inv_sq(mx * mx + mz * mz);
    const float gmx = (mz * wm) * g[1], gmz = (-mx * wm) * g[1];
    const float wy = inv_sq(hx * hx + hy * hy);
    const float ghx = (-hy * wy) * g[2];
    float ghy = (hx * wy) * g[2], ghz = 0.f;
    float groll = g[0];
    const float whd = inv_sq(hdy * hdy + hdz * hdz);
    float ghdy = 0.f, ghdz = 0.f;                                            // dL/dhd, summed over both antenna yaws
    float gnx = -gmx, gny = 0.f, gnz = -gmz;
#pragma unroll
    for (int side = 0; side < 2; ++side) {   // 0 = L, 1 = R
        const float bx = side ? rbx : lbx, by = side ? rby : lby, bz = side ? rbz : lbz;
        const float tx = side ? rtx : ltx, ty = side ? rty : lty, tz = side ? rtz : ltz;
        const float ax = tx - bx, ay = ty - by, az = tz - bz;
        const float ady = ay * c + az * s, adz = -ay * s + az * c;
        const float gx = nx - bx, gy = ny - by, gz = nz - bz;
        const float gdz = -gy * s + gz * c;
        // antenna yaw: ad -> hd about X
        const float gyaw = side ? -g[5] : g[3];
        const float wa = inv_sq(ady * ady + adz * adz);
        float gady = (adz * wa) * gyaw, gadz = (-ady * wa) * gyaw;
        ghdy += (-hdz * whd) * gyaw; ghdz += (hdy * whd) * gyaw;
        // antenna pitch: gd -> ad about Y
        const float gp = g[4 + 2 * side];
        const float wp = inv_sq(ax * ax + adz * adz), wg = inv_sq(gx * gx + gdz * gdz);
        const float gax = (adz * wp) * gp;
        gadz += (-ax * wp) * gp;
        const float ggx = (-gdz * wg) * gp, ggdz = (gx * wg) * gp;
        // roll terms of the de-rotated antenna vector and neck - base (d gdz / droll = -gdy)
        const float gdy = gy * c + gz * s;
        groll += gady * adz - gadz * ady - ggdz * gdy;
        const float gay = c * gady - s * gadz, gaz = s * gady + c * gadz;
        const float ggy = -s * ggdz, ggz = c * ggdz;
        float* gb = side ? grr : gll;
        gb[3] = gax; gb[4] = gay; gb[5] = gaz;                               // tip
        gb[0] = -gax - ggx; gb[1] = -gay - ggy; gb[2] = -gaz - ggz;          // base: a = tip - base, neck - base
        gnx += ggx; gny += ggy; gnz += ggz;
    }
    groll += ghdy * hdz - ghdz * hdy;
    ghy += c * ghdy - s * ghdz; ghz += s * ghdy + c * ghdz;
    const float wr = inv_sq(hy * hy + hz * hz);
    ghy += (-hz * wr) * groll; ghz += (hy * wr) * groll;
    // hor = lb - rb, mid = (rb + lb) / 2 - neck
    const float hmx = 0.5f * gmx, hmz = 0.5f * gmz;
    grr[0] = (grr[0] - ghx) + hmx; grr[1] = grr[1] - ghy; grr[2] = (grr[2] - ghz) + hmz;
    gll[0] = (gll[0] + ghx) + hmx; gll[1] = gll[1] + ghy; gll[2] = (gll[2] + ghz) + hmz;
    gn[0] = gnx; gn[1] = gny; gn[2] = gnz;
}

// One thread per frame.  kVec2: r_head, l_head and both gradient records are 8-byte aligned and move as 64-bit loads /
// stores; otherwise as 32-bit ones -- the arithmetic, hence the result, is the same.
template <bool kVec2>
__global__ void __launch_bounds__(256) head_backward_kernel(const float* __restrict__ r_head, const float* __restrict__ l_head,
                                                            const float* __restrict__ neck, int64_t neck_stride,
                                                            const float* __restrict__ affine_r, const float* __restrict__ affine_l,
                                                            const float* __restrict__ grad_out, float* __restrict__ grad_r,
                                                            float* __restrict__ grad_l, float* __restrict__ grad_neck,
                                                            int64_t n_trial, int64_t n_frame) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_trial * n_frame) return;
    const int64_t tr = i / n_frame, t = i - tr * n_frame;
    const float* r = r_head + i * 6; const float* l = l_head + i * 6;
    float rr[6], ll[6], g[7];
    if (kVec2) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const float2 a = __ldg(reinterpret_cast<const float2*>(r) + k), b = __ldg(reinterpret_cast<const float2*>(l) + k);
            rr[2 * k] = a.x; rr[2 * k + 1] = a.y; ll[2 * k] = b.x; ll[2 * k + 1] = b.y;
        }
    } else {
#pragma unroll
        for (int k = 0; k < 6; ++k) { rr[k] = __ldg(r + k); ll[k] = __ldg(l + k); }
    }
    const float* gi = grad_out + tr * 7 * n_frame + t;                      // [n_trial][7][n_frame]: coalesced per angle
#pragma unroll
    for (int k = 0; k < 7; ++k) g[k] = __ldg(gi + k * n_frame);
    const float* ar = affine_r ? affine_r + tr * 8 : nullptr;
    const float* al = affine_l ? affine_l + tr * 8 : nullptr;
    float grr[6], gll[6], gn[3];
    head_frame_backward(rr, ll, neck + (neck_stride ? i * 3 : tr * 3), ar, al, g, grr, gll, gn);
    if (ar) {                                                               // d(aligned)/d(raw) = the row's scale, last
        const float rsb = ar[3], rst = ar[7], lsb = al[3], lst = al[7];
#pragma unroll
        for (int k = 0; k < 3; ++k) { grr[k] *= rsb; grr[k + 3] *= rst; gll[k] *= lsb; gll[k + 3] *= lst; }
    }
    float* orr = grad_r + i * 6; float* oll = grad_l + i * 6;
    if (kVec2) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            reinterpret_cast<float2*>(orr)[k] = make_float2(grr[2 * k], grr[2 * k + 1]);
            reinterpret_cast<float2*>(oll)[k] = make_float2(gll[2 * k], gll[2 * k + 1]);
        }
    } else {
#pragma unroll
        for (int k = 0; k < 6; ++k) { orr[k] = grr[k]; oll[k] = gll[k]; }
    }
    if (grad_neck) { float* on = grad_neck + i * 3; on[0] = gn[0]; on[1] = gn[1]; on[2] = gn[2]; }
}

extern "C" int seqik_head_angles_backward_f32(const float* r_head, const float* l_head, const float* neck, int64_t neck_stride,
                                              const float* affine_r, const float* affine_l, const float* grad_out,
                                              float* grad_r_head, float* grad_l_head, float* grad_neck,
                                              int64_t n_trial, int64_t n_frame, void* stream) {
    if (n_trial < 0 || n_frame < 0) return seqik_fail(SEQIK_EINVAL, "seqik_head_angles_backward_f32: negative size");
    if (n_trial == 0 || n_frame == 0) return SEQIK_OK;
    if (!r_head || !l_head || !neck || !grad_out || !grad_r_head || !grad_l_head)
        return seqik_fail(SEQIK_EINVAL, "seqik_head_angles_backward_f32: NULL pointer");
    if (neck_stride != 0 && neck_stride != 3)
        return seqik_fail(SEQIK_EINVAL, "seqik_head_angles_backward_f32: neck_stride must be 0 or 3");
    if ((affine_r == nullptr) != (affine_l == nullptr))
        return seqik_fail(SEQIK_EINVAL, "seqik_head_angles_backward_f32: affine_r and affine_l must both be given or both be NULL");
    const int64_t n = n_trial * n_frame;
    const bool vec2 = ((((uintptr_t)r_head) | ((uintptr_t)l_head) | ((uintptr_t)grad_r_head) | ((uintptr_t)grad_l_head)) & 7) == 0;
    auto kernel = vec2 ? head_backward_kernel<true> : head_backward_kernel<false>;
    kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(r_head, l_head, neck, neck_stride, affine_r, affine_l,
                                                                         grad_out, grad_r_head, grad_l_head, grad_neck, n_trial, n_frame);
    return seqik_check_launch("seqik_head_angles_backward_f32");
}
