// seqik_head.cuh -- the plane-angle arithmetic and the head-alignment map shared by the head-angle kernel
// (seqik_kernels.cu) and its backward (seqik_head_grad.cu), so that the backward recomputes the forward's exact bits.
#pragma once
#include <cuda_runtime.h>

// angle_between_segments (head_inverse_kinematics.py:163-183) for vectors that live in a coordinate plane:
// arccos(v1^.v2^) * (det > 0 ? 1 : -1), evaluated as atan2(|det|, dot) which keeps FP32 accuracy near 0 and pi.
// atan2(y, x) for y >= 0, result in [0, pi]: octant reduction to t = min/max in [0, 1], one more reduction at tan(pi/8)
// ((t - 1) / (t + 1)), then the degree-4 minimax polynomial in t^2 of Cephes' atanf (|error| < half an ulp of the result
// + 2e-7 rad including the two SFU reciprocals, i.e. < 3.2e-7 rad near pi, tests/test_gpu_stream.py; the parity bound of
// the head angles is 2e-5 rad).  Half the instructions of atan2f, no slow path:
// the head kernel is issue-bound on its five arctangents per frame.
__device__ __forceinline__ float atan2_pos(float y, float x) {
    const float ax = fabsf(x);
    const float mn = fminf(ax, y), mx = fmaxf(ax, y);
    float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(mx));
    const float t = mx > 0.f ? mn * r : 0.f;
    const bool big = t > 0.4142135679721832f;
    float q; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(q) : "f"(t + 1.0f));
    const float u = big ? (t - 1.0f) * q : t;
    const float z = u * u;
    float p = fmaf(8.05374449538e-2f, z, -1.38776856032e-1f);
    p = fmaf(p, z, 1.99777106478e-1f);
    p = fmaf(p, z, -3.33329491539e-1f);
    float a = fmaf(p * z, u, u);
    if (big) a += 0.78539816339744831f;
    if (y > ax) a = 1.57079632679489662f - a;
    if (x < 0.f) a = 3.14159265358979324f - a;
    return a;
}
__device__ __forceinline__ float signed_angle(float dotp, float det) {
    const float a = atan2_pos(fabsf(det), dotp);
    return det > 0.f ? a : -a;
}

// head-alignment row: (origin xyz, scale_base, template xyz, scale_tip)
__device__ __forceinline__ void head_point(const float* p, const float* __restrict__ aff, bool tip,
                                           float& x, float& y, float& z) {
    x = p[0]; y = p[1]; z = p[2];
    if (aff) {
        const float sc = tip ? aff[7] : aff[3];
        x = (x - aff[0]) * sc + aff[4]; y = (y - aff[1]) * sc + aff[5]; z = (z - aff[2]) * sc + aff[6];
    }
}
