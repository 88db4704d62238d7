// seqik_solver.cu -- the sequential leg-IK solver kernels (sm_100a) behind seqik_leg_solve_f32.
//
// Work decomposition.  A chain = one leg of one trial.  Inside a chain the reference's data dependences are
// kept exactly (leg_inverse_kinematics.py:259-282): the stage-s solve of frame t starts from the stage-s
// result of frame t-1 (warm start, :272) and from the frame built by stages 1..s-1 of frame t (frozen links).
// That dependence graph is a 4 x n_frame wavefront: solve(s+1, t) and solve(s, t+1) are independent.
//
//   schedule 1, "lane per chain"        one lane runs stages 1..4 of frame t, then frame t+1, ...
//                                       Fewest lanes per chain: the throughput schedule for very many chains.
//   schedule 2, "stage pipeline"        four adjacent lanes own one chain, lane s runs stage s+1 of every frame and
//                                       hands the frame (3x3 orientation + pivot) to lane s+1 through a small
//                                       shared-memory ring.  Chain latency drops from the sum of the four stages'
//                                       evaluations per frame to the slowest stage's.  The schedule for the
//                                       benchmark configurations (6 000 - 7 500 chains per GPU leave a B200 mostly
//                                       idle under schedule 1, whose run time is one chain's latency).
//
// Both run the same per-lane arithmetic (seqik_core.cuh: StageSolve::init / restart / trip), one function evaluation
// per loop trip, in a warp-convergent loop; lanes sit at different (frame, stage) positions ("decoupled" trips).
// Schedule 2 carries a solve from frame to frame (restart: no trigonometry), which is also what lets the closed-form
// warm step end most solves with their first evaluation (SEQIK_FLAG_CLOSED_FORM); schedule 1 starts every solve afresh.
// No tensor cores: the work is scalar FP32 2x2 / 3x3 algebra (BASELINE.json north_star).
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/seqik.h"
#include "seqik_common.h"
#include "seqik_core.cuh"
#include "seqik_block.cuh"
#include "seqik_tma.cuh"

using namespace seqik;

struct LegArgs {
    const float* pose; int64_t pose_cs, pose_fs;
    const float* affine; const float* params;
    float* angles; int64_t ang_cs, ang_fs;
    float* fk; int64_t fk_cs, fk_fs;
    const float* warm; int64_t warm_cs;
    int32_t* status; uint32_t* nfev;
    int64_t n_chain, n_frame;
    int stage_mask, gn_mask;
    int fk_joints;                          // SEQIK_FLAG_FK_JOINTS: fk holds the 4 joint rows only ([4][3] per leg-frame)
};

// alignment map applied on load (AlignPose.align_leg, alignment.py:471-485)
struct LoadMap {
    float fx, fy, fz, sc, tx, ty, tz; bool on;
    __device__ __forceinline__ void init(const float* affine, int64_t c) {
        on = affine != nullptr; fx = fy = fz = 0.f; sc = 1.f; tx = ty = tz = 0.f;
        if (on) { const float* q = affine + c * 8; fx = q[0]; fy = q[1]; fz = q[2]; sc = q[3]; tx = q[4]; ty = q[5]; tz = q[6]; }
    }
    __device__ __forceinline__ Vec3<float> apply(Vec3<float> v, int row) const {
        if (on) {
            if (row == 0) v = {tx, ty, tz};
            else v = {(v.x - fx) * sc + tx, (v.y - fy) * sc + ty, (v.z - fz) * sc + tz};
        }
        return v;
    }
};

// ---------------------------------------------------------------------------------------------
// schedule 1: one lane per chain
// ---------------------------------------------------------------------------------------------
// Global-memory IO policy of one chain.  Key points are read with plain (L1-cached) loads: a chain's
// frames are contiguous (60 B apart), so consecutive frames share 128 B lines.
struct DevIO {
    const float* pose; int64_t fs;          // base of this chain, frame stride
    const float* prm;                       // 32 floats
    float* ang; int64_t ang_fs;
    float* fk; int64_t fk_fs; bool fk_joints;
    LoadMap map;

    __device__ __forceinline__ Vec3<float> kp(int64_t t, int row) const {
        const float* p = pose + t * fs + row * 3;
        return map.apply({__ldg(p), __ldg(p + 1), __ldg(p + 2)}, row);
    }
    __device__ __forceinline__ void put_angles(int64_t t, const float* a, int i0, int i1) const {
        float* p = ang + t * ang_fs;
#pragma unroll
        for (int i = 0; i < 7; ++i) if (i >= i0 && i < i1) p[i] = a[i];
    }
    __device__ __forceinline__ float angle_in(int64_t t, int i) const { return ang[t * ang_fs + i]; }
    __device__ __forceinline__ void put_fk(int64_t t, int row, const Vec3<float>& v) const {
        if (fk_joints) { if (row < 5) return; row -= 5; }       // joints-only layout: rows 5..8 of the full one
        if (fk) { float* p = fk + t * fk_fs + row * 3; p[0] = v.x; p[1] = v.y; p[2] = v.z; }
    }
    __device__ __forceinline__ float seg(int i) const { return __ldg(prm + i); }
    __device__ __forceinline__ float lb(int i) const { return __ldg(prm + 4 + i); }
    __device__ __forceinline__ float ub(int i) const { return __ldg(prm + 11 + i); }
    __device__ __forceinline__ float null_sq(int i) const { return __ldg(prm + 25 + i); }
};

__global__ void __launch_bounds__(32) leg_solve_lane_kernel(LegArgs a) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= a.n_chain) return;
    DevIO io;
    io.pose = a.pose + c * a.pose_cs; io.fs = a.pose_fs;
    io.prm = a.params + c * SEQIK_CHAIN_PARAM_FLOATS;
    io.ang = a.angles + c * a.ang_cs; io.ang_fs = a.ang_fs;
    io.fk = a.fk ? a.fk + c * a.fk_cs : nullptr; io.fk_fs = a.fk_fs; io.fk_joints = a.fk_joints != 0;
    io.map.init(a.affine, c);
    float seed[7];
#pragma unroll
    for (int i = 0; i < 7; ++i) seed[i] = a.warm ? a.warm[c * a.warm_cs + i] : io.prm[18 + i];
    ChainRunner<float, DevIO> run;
    run.start(io, a.n_frame, seed, a.stage_mask, a.gn_mask);
    while (!run.finished()) run.step();
    if (a.status) a.status[c] = run.worst_status == ST_NONFINITE ? -1 : run.worst_status;
    if (a.nfev) { uint32_t* nf = a.nfev + c * 4; nf[0] = run.nf0; nf[1] = run.nf1; nf[2] = run.nf2; nf[3] = run.nf3; }
}

// ---------------------------------------------------------------------------------------------
// schedule 2: stage pipeline -- four adjacent lanes own one chain, lane s runs stage s+1 of every frame
// ---------------------------------------------------------------------------------------------
// One warp = `cpw` chains (1, 2, 4 or 8) x 4 stage lanes; lanes >= 4 cpw idle.  All lanes run the SAME straight-line
// code (StageSolve::trip is branch-free, the rotation kind is a per-lane select), so a warp iteration costs one trip
// whatever mix of positions its lanes are in.  Stage s hands frame t (orientation after its own rotation + the
// next pivot, 12 floats) to stage s+1 through a shared-memory ring of PIPE_DEPTH frames; progress counters travel
// by warp shuffle.  No block-level synchronisation: a block is one warp.
constexpr int PIPE_DEPTH = 4;               // frames a stage may run ahead of the next one
constexpr int PIPE_SLOT = 12;               // 3x3 frame (columns) + pivot
constexpr int PIPE_CHAINS = 8;              // chains per warp (maximum)

// kFull: all four stages solved and the nine-row FK layout written (the benchmark configurations and the dict API):
// the frozen-stage, partial-stage and output-layout decisions are compiled out.  Same arithmetic either way.
template <bool kFull>
__global__ void __launch_bounds__(32) leg_solve_pipe_kernel(LegArgs a, int cpw, int gate_period, int trip_period) {
    // hand-off ring: [stage][frame slot x 12 floats (+ 1 pad row)][chain].  Bank of an element = (8 (k + stage) + chain) mod 32:
    // the pad row shifts each stage's plane by 8 banks, so the 4 x 8 lanes of a warp, which all touch the same k at once,
    // hit 32 different banks (without it the four stage lanes of a chain collided: half of the kernel's shared-memory
    // wavefronts were bank-conflict replays, ncu l1tex__data_bank_conflicts_pipe_lsu_mem_shared).  [3] = identity
    // (stage 1's input)
    __shared__ float ring[4][PIPE_DEPTH * PIPE_SLOT + 1][PIPE_CHAINS];
    __shared__ float kpbuf[6][32];                                     // prefetched key points, one column per lane
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x;
    const int s = lane & 3;                                   // this lane's stage (0..3)
    const int cw = lane >> 2;                                 // chain within the warp
    const int64_t c = (int64_t)blockIdx.x * cpw + cw;
    int lo = 0, hi = 3;
    if (!kFull) {
        while (lo < 3 && !((a.stage_mask >> lo) & 1)) ++lo;
        while (hi > 0 && !((a.stage_mask >> hi) & 1)) --hi;
    }
    const bool owner = cw < cpw && c < a.n_chain;
    const bool live = owner && s <= hi;                       // lanes of stages after the last requested one idle
    const bool frozen = !kFull && s < lo;                     // DOFs read from the angles buffer, not solved
    const int n_frame = (int)a.n_frame;

    // per-lane constants of (chain, stage)
    const int64_t cc = owner ? c : 0;
    const float* prm = a.params + cc * SEQIK_CHAIN_PARAM_FLOATS;
    const float* pose = a.pose + cc * a.pose_cs;
    float* ang = a.angles + cc * a.ang_cs;
    float* fk = (kFull || a.fk) ? a.fk + cc * a.fk_cs : nullptr;
    const bool fk_joints = !kFull && a.fk_joints;
    LoadMap map; map.init(a.affine, cc);
    const int kind = (s == 0) ? KIND_XY : KIND_ZY;
    const float seg = __ldg(prm + s);
    const int ia = 2 * s, ib = (s == 3) ? 6 : 2 * s + 1;
    const float inf = Num<float>::inf();
    const float lb0 = (s == 3 || frozen) ? -inf : __ldg(prm + 4 + ia), ub0 = (s == 3 || frozen) ? inf : __ldg(prm + 11 + ia);
    const float lb1 = frozen ? -inf : __ldg(prm + 4 + ib), ub1 = frozen ? inf : __ldg(prm + 11 + ib);
    const float null_sq = frozen ? 0.f : __ldg(prm + 25 + s);
    const int n_full = (s == 0) ? 4 : (s == 1) ? 6 : (s == 2) ? 8 : 9;
    const int gn = stage_mode(a.gn_mask, s);                                  // StageSolve mode: Gauss-Newton, skip-confirm, Newton
    const bool esc = (a.gn_mask >> 4) & 1;
    const float has_a = (s == 3) ? 0.f : 1.f;
    const float* seed = a.warm ? a.warm + cc * a.warm_cs : prm + 18;
    float xa = (s == 3) ? 0.f : seed[ia], xb = seed[ib];                           // warm start, frame to frame

    // running output / input pointers of the frame this lane works on (advanced per frame: no 64-bit index math per access)
    float* pa_a = ang + ((s == 3) ? 6 : ia); float* pa_b = ang + ib;             // stage 4 has one DOF: both point at it
    float* pf = fk ? fk + 3 * s : nullptr;
    const float* pnext = pose;       // frame whose key points are prefetched next

    StageSolve<float> S;
    S.set_problem(kind, seg, has_a, null_sq, n_full, gn);
    if (live && !frozen) S.set_limit_trig(lb0, ub0);
    Mat3<float> A = {{1.f, 0.f, 0.f}, {0.f, 1.f, 0.f}, {0.f, 0.f, 1.f}};
    Vec3<float> piv = {0.f, 0.f, 0.f}, o = {0.f, 0.f, 0.f}, rel = {0.f, 0.f, 0.f};
    int t = 0;                       // frame this lane works on
    int started = 0, done = 0;       // frames whose hand-off was consumed / produced by this lane
    bool solving = false;
    uint32_t nf = 0; int worst = ST_GTOL;
    S.status = ST_GTOL;
    // stage 1 starts every frame from the identity frame at the origin: it reads them from a constant ring slot like
    // the other stages read their producer's, so that the hand-off read is the same instruction for all lanes
    if (lane < PIPE_CHAINS)
        for (int d = 0; d < PIPE_DEPTH; ++d)
            for (int k = 0; k < PIPE_SLOT; ++k) ring[3][d * PIPE_SLOT + k][lane] = (k == 0 || k == 4 || k == 8) ? 1.f : 0.f;
    __syncwarp(full);
    const int sp = (s + 3) & 3;      // ring this lane reads from
    // key points of frame t (origin + this stage's target, 6 floats), fetched one frame ahead with cp.async into
    // shared memory: the copy is in flight during the previous solve and does not hold a register scoreboard
    // (plain loads made the first dependent instruction of every open wait a full DRAM latency)
    const uint32_t kp_dst = (uint32_t)__cvta_generic_to_shared(&kpbuf[0][lane]);
    auto prefetch = [&]() {
        const float* p = pnext;
        const float* q = p + 3 * (s + 1);
        pnext += a.pose_fs;
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(kp_dst), "l"(p) : "memory");
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(kp_dst + 128), "l"(p + 1) : "memory");
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(kp_dst + 256), "l"(p + 2) : "memory");
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(kp_dst + 384), "l"(q) : "memory");
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(kp_dst + 512), "l"(q + 1) : "memory");
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(kp_dst + 640), "l"(q + 2) : "memory");
    };
    if (live && n_frame > 0) prefetch();
    bool carried = false;            // S holds the previous frame's solve of this (chain, stage)

    for (int gate_ctr = 1, trip_ctr = trip_period; __any_sync(full, live && t < n_frame);) {
        if (--gate_ctr == 0) {                          // open/close phases only every gate_period-th iteration (warp-uniform)
        gate_ctr = gate_period;
        __syncwarp(full);            // ring reads of the previous open phase are complete before a slot is written again
        const int started_next = __shfl_sync(full, started, (lane + 1) & 31);   // consumer's progress (lane + 1)
        // ---- optional singularity escape: a solve that ended on sin b = 0 may continue from a closed-form candidate
        if (esc && live && solving && !frozen && S.done() && S.escape_possible()) S.escape();
        // ---- close the converged solve: outputs + hand-off to the next stage (needs a free ring slot)
        if (live && t < n_frame && solving && S.done() && (s == hi || t < started_next + PIPE_DEPTH)) {
            if (!frozen) {
                xa = S.x0; xb = S.angle_b(); nf += (uint32_t)S.nfev;
                worst = (S.status == ST_MAXFEV && worst > ST_MAXFEV) ? ST_MAXFEV : worst;
                worst = (S.status == ST_NONFINITE) ? ST_NONFINITE : worst;
                const float xb_out = limit_clamp(xb, lb1, ub1);                        // (outputs inside the limits, seqik_core.cuh)
                *pa_a = (s == 3) ? xb_out : limit_clamp(xa, lb0, ub0);
                *pa_b = xb_out;
            }
            // joint position = pivot + A w(x) = target + A f   (q = A^T rel, f = w - q)
            const Vec3<float> Af = mul(A, S.res());
            const Vec3<float> np_ = {(piv.x + rel.x) + Af.x, (piv.y + rel.y) + Af.y, (piv.z + rel.z) + Af.z};
            if (kFull || fk) {
                // rows 0-3 repeat the origin, 4 and 5 are both the Coxa-Femur joint: lane s writes origin row s and its
                // own joint row(s), which spreads the 27 floats of a frame over the four lanes
                const Vec3<float> jw = {np_.x + o.x, np_.y + o.y, np_.z + o.z};
                if (fk_joints) {                                                         // joints-only layout: row s = this lane's joint
                    pf[0] = jw.x; pf[1] = jw.y; pf[2] = jw.z;
                } else {
                    pf[0] = o.x; pf[1] = o.y; pf[2] = o.z;                               // row s
                    pf[15] = jw.x; pf[16] = jw.y; pf[17] = jw.z;                         // row 5 + s
                    if (s == 0) { pf[12] = jw.x; pf[13] = jw.y; pf[14] = jw.z; }         // row 4
                    if (!kFull && s == hi && hi < 3) for (int r = 1; r < 4 - hi; ++r) { pf[3 * r] = o.x; pf[3 * r + 1] = o.y; pf[3 * r + 2] = o.z; }
                }
                pf += a.fk_fs;
            }
            pa_a += a.ang_fs; pa_b += a.ang_fs;
            if (s < hi) {
                const Mat3<float> B = rotate_frame_sel(A, kind, S.sa, S.ca, S.sin_b(), S.cos_b());   // lanes mix kinds: no branch
                float (*q)[PIPE_CHAINS] = &ring[s][(t & (PIPE_DEPTH - 1)) * PIPE_SLOT];
                q[0][cw] = B.c0.x; q[1][cw] = B.c0.y; q[2][cw] = B.c0.z; q[3][cw] = B.c1.x; q[4][cw] = B.c1.y; q[5][cw] = B.c1.z;
                q[6][cw] = B.c2.x; q[7][cw] = B.c2.y; q[8][cw] = B.c2.z; q[9][cw] = np_.x; q[10][cw] = np_.y; q[11][cw] = np_.z;
            }
            solving = false; ++t; done = t;
        }
        __syncwarp(full);            // ring writes above are visible to the reads below
        const int done_prev = __shfl_sync(full, done, (lane + 31) & 31);        // producer's progress (lane - 1)
        // ---- open the next solve when the previous stage has published this frame
        if (live && t < n_frame && !solving && (s == 0 || t < done_prev)) {
            {
                const float (*q)[PIPE_CHAINS] = &ring[sp][(t & (PIPE_DEPTH - 1)) * PIPE_SLOT];
                A.c0 = {q[0][cw], q[1][cw], q[2][cw]}; A.c1 = {q[3][cw], q[4][cw], q[5][cw]}; A.c2 = {q[6][cw], q[7][cw], q[8][cw]};
                piv = {q[9][cw], q[10][cw], q[11][cw]};
            }
            asm volatile("cp.async.wait_all;" ::: "memory");
            const Vec3<float> ko = {kpbuf[0][lane], kpbuf[1][lane], kpbuf[2][lane]};
            const Vec3<float> kt = {kpbuf[3][lane], kpbuf[4][lane], kpbuf[5][lane]};
            if (t + 1 < n_frame) prefetch();
            o = map.apply(ko, 0);
            const Vec3<float> k = map.apply(kt, s + 1);
            rel = {(k.x - o.x) - piv.x, (k.y - o.y) - piv.y, (k.z - o.z) - piv.z};
            const Vec3<float> q3 = mulT(A, rel);
            // a carried solve continues from its own final iterate; every SEQIK_RESYNC frames (and at the first frame of
            // a call) the iterate is re-derived from the angles.  Same code but for the trigonometry (restart's `fresh`).
            const bool fresh = !(carried && !frozen && (t & (SEQIK_RESYNC - 1)) != 0);
            if (fresh) {
                if (frozen) { xa = (s == 3) ? 0.f : *pa_a; xb = *pa_b; }
                S.set_iterate(xa, xb);
                carried = true;
            }
            S.restart(q3, lb0, ub0, lb1, ub1, fresh, !frozen && (t > 0 || a.warm != nullptr));   // frozen DOFs stay where they are
            if (frozen) S.status = ST_GTOL;
            solving = true; started = t + 1;
        }
        }   // gate
        // ---- one function evaluation (every trip_period-th iteration, warp-uniform)
        if (--trip_ctr == 0) {
            trip_ctr = trip_period;
            if (live && solving && !S.done()) S.trip();
        }
    }
    // per-chain statistics
    const int w1 = min(worst, __shfl_xor_sync(full, worst, 1));
    const int w2 = min(w1, __shfl_xor_sync(full, w1, 2));
    if (owner) {
        if (a.nfev) a.nfev[c * 4 + s] = nf;
        if (a.status && s == 0) a.status[c] = w2 == ST_NONFINITE ? -1 : w2;
    }
}

// ---------------------------------------------------------------------------------------------
// schedule 3: frame-parallel blocks -- one warp per chain, 32 consecutive frames per pass (lane = frame)
// ---------------------------------------------------------------------------------------------
// The algorithm and why its results are bit-identical to schedule 2 are described in seqik_block.cuh, which also holds the
// per-stage constants and the serial stage step of the replay and of the first frame: the host emulation of the schedule
// (tests/hostsim run_block) compiles the same code.  Per warp:
//   * the 32 x 60 B of key points of the NEXT block arrive by one bulk copy (cp.async.bulk -> mbarrier) while the current
//     block is solved; angles (32 x 28 B) and forward kinematics (32 x 108 B) are staged in shared memory and leave by two
//     bulk stores: every byte of the chain crosses the memory system once, in 128-byte lines (BASELINE.json north_star 2);
//   * pass / accumulate / verify / replay loop over the block; a block without a replay costs ~1 100 warp instructions
//     for 32 leg-frames, a replay one serial frame (StageSolve) and a recomputation of the lanes after it.
// A CTA is one warp (no block-level barrier); the launch shapes the number of resident warps per SM with dynamic shared
// memory so that the chains of a batch run in whole waves (seqik_leg_solve_f32).
constexpr int BLK = 32;
// serial_stage (seqik_block.cuh) as a real call (robust block kernel): the ~75 registers of the serial solver are then the
// callee's business and what the kernel keeps across it is saved at the -- cold -- call site instead of being spilled where it
// is defined, in the hot pass.
__device__ __noinline__ void serial_stage_call(int s, const SerialConst<float>& k, int gn_mask, bool esc, bool warm_ok, const Vec3<float>& kt,
                                               const Vec3<float>& o, Mat3<float>& A, Vec3<float>& piv, float& x0, float& x1,
                                               float& sa, float& ca, float& sb, float& cb, float& xb_out, Vec3<float>& w,
                                               uint32_t& nfev, int& worst) {
    serial_stage(s, k, gn_mask, esc, warm_ok, kt, o, A, piv, x0, x1, sa, ca, sb, cb, xb_out, w, nfev, worst);
}
enum : int { KC_L, KC_LB0, KC_UB0, KC_LB1S, KC_UB1S, KC_SL0, KC_CL0, KC_SU0, KC_CU0, KC_LB0P, KC_UB0P, KC_NSQ, KC_LB1, KC_UB1, KC_HAVE_BT, KC_N = 16 };
struct __align__(16) BlockShared {
    float pose[2][BLK * 15];           // key points of the current / next block (bulk-copy destination)
    float out_ang[BLK * 7];            // staged results (bulk-store source)
    float out_fk[BLK * 27];
    float2 acc_vk[7][BLK + 2];         // per angle series and frame: (v, k) of x <- k x + v   (+2: 16-byte rows, bank spread)
    float acc_x[7][BLK + 2];           // [l][t + 1]: placed angle BEFORE frame t of series l; [l][t + 2] after it ([0] unused)
    float kc[4][KC_N];                 // per-stage constants of the chain
    float P[4][4];                     // sin/cos (sa, ca, sb, cb) per stage of the state before the first lane of a pass
    float mapc[8];                     // alignment map applied on load (fixed xyz, scale, template xyz, on/off): rarely used, kept out of registers
    uint32_t nfx[4];                   // evaluations of replayed solves per stage (committed lanes count one each)
    uint64_t bar[2];
};

// The first frame of a recording is solved from the seed (never by the closed form): ~17 evaluations, 10 000 instructions that
// the block kernel would execute with ONE active lane per chain.  This kernel runs them for 32 chains per warp (lane = chain)
// before the block kernel starts and leaves, per chain, frame 0's results in the outputs and a record of the final state in the
// chain's angle rows 1..4 (they are overwritten with their own results later): 16 sin/cos, 7 placed angles, 4 evaluation
// counts, the status.  Same arithmetic as the replay path (serial_stage), so results do not depend on which of the two ran.
constexpr int FF_REC = 28;
template <int kFk>
__global__ void __launch_bounds__(BLK) leg_first_frame_kernel(LegArgs a) {
    const int64_t c = (int64_t)blockIdx.x * BLK + threadIdx.x;
    if (c >= a.n_chain) return;
    const float* prm = a.params + c * SEQIK_CHAIN_PARAM_FLOATS;
    const float* kp = a.pose + c * a.pose_cs;
    float* ang = a.angles + c * a.ang_cs;
    float* fk = kFk ? a.fk + c * a.fk_cs : nullptr;
    LoadMap map; map.init(a.affine, c);
    const bool esc = (a.gn_mask >> 4) & 1;
    const Vec3<float> o = map.apply({__ldg(kp), __ldg(kp + 1), __ldg(kp + 2)}, 0);
    Mat3<float> A = {{1.f, 0.f, 0.f}, {0.f, 1.f, 0.f}, {0.f, 0.f, 1.f}};
    Vec3<float> piv = {0.f, 0.f, 0.f};
    int worst = ST_GTOL;
#pragma unroll 1
    for (int s = 0; s < 4; ++s) {
        const StageConst<float> k = stage_const(prm, s);
        // the seed enters like a carried angle: set_iterate + place, sin/cos derived from the placed value
        float x0 = (s == 3) ? 0.f : place1(__ldg(prm + 18 + k.ia), k.lb0, k.ub0);
        float x1 = place1(__ldg(prm + 18 + k.ib) - k.shift, k.lb1s, k.ub1s);
        float sa = 0.f, ca = 1.f, sb, cb, v_;
        if (s < 3) Num<float>::sincosv_(x0, &sa, &ca, &v_);
        Num<float>::sincosv_(x1, &sb, &cb, &v_);
        const Vec3<float> kt = map.apply({__ldg(kp + 3 * s + 3), __ldg(kp + 3 * s + 4), __ldg(kp + 3 * s + 5)}, s + 1);
        float xb; Vec3<float> w; uint32_t ne = 0u;
        serial_stage(s, k, a.gn_mask, esc, false, kt, o, A, piv, x0, x1, sa, ca, sb, cb, xb, w, ne, worst);
        if (s < 3) ang[k.ia] = limit_clamp(x0, k.lb0, k.ub0);
        ang[k.ib] = limit_clamp(xb, k.lb1, k.ub1);
        put_fk_joint<kFk>(fk, s, o, w);
        auto rec = [&](int i) -> float& { return ang[(int64_t)(1 + i / 7) * a.ang_fs + i % 7]; };
        rec(4 * s) = sa; rec(4 * s + 1) = ca; rec(4 * s + 2) = sb; rec(4 * s + 3) = cb;
        if (s < 3) rec(16 + s) = place1(x0, k.lb0, k.ub0);
        rec(19 + s) = place1(x1, k.lb1s, k.ub1s);
        rec(23 + s) = __int_as_float((int)ne);
    }
    ang[(int64_t)4 * a.ang_fs + 6] = __int_as_float(worst);                  // record slot 27
}

// Two instantiations of the same source.  kRobust = false: the lean kernel for large batches -- a replay reruns the whole
// frame serially and the lanes after it are recomputed from stage 1; 96 registers, 18 resident warps per SM.  kRobust = true:
// for recordings that replay often (joint limits active, fast motion: 3-4 % of the frames of the bundled grooming trial) --
// a replay starts at the first failing stage, the lanes after it keep their earlier stages, and the one-variable stage
// sitting on its limit is decided exactly in the pass; 128 registers, 16 resident warps per SM.  Same results, bit for bit.
#ifndef SEQIK_BLOCK_MIN_CTAS
#define SEQIK_BLOCK_MIN_CTAS 16        // resident one-warp CTAs per SM the register allocation must allow: 128 registers, no spills (measured: 96 registers spill in the pass)
#endif
#ifndef SEQIK_BLOCK_MIN_CTAS_ROBUST
#define SEQIK_BLOCK_MIN_CTAS_ROBUST 16
#endif
template <int kFk, bool kRobust>       // kFk 0: no forward kinematics, 1: nine rows, 2: the four joint rows only
__global__ void __launch_bounds__(BLK, kRobust ? SEQIK_BLOCK_MIN_CTAS_ROBUST : SEQIK_BLOCK_MIN_CTAS)
leg_solve_block_kernel(LegArgs a, int bulk_in, int bulk_out, int first_done) {
    __shared__ __align__(128) BlockShared sh;
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x;
    const int64_t c = blockIdx.x;
    // (global pointers are rebuilt from the kernel arguments where they are used: a handful of places, and registers are scarce)
#define BLK_PRM (a.params + c * SEQIK_CHAIN_PARAM_FLOATS)
#define BLK_POSE (a.pose + c * a.pose_cs)
#define BLK_ANG (a.angles + c * a.ang_cs)
#define BLK_FK (a.fk + c * a.fk_cs)
    constexpr int FKF = kFk == 1 ? 27 : 12;                        // floats per leg-frame of the fk layout
    const int n_frame = (int)a.n_frame;
    const float inf = Num<float>::inf();
    const float half_pi = 1.57079632679489661923f;
    const bool esc = (a.gn_mask >> 4) & 1;
    const bool warm_given = a.warm != nullptr;
    const bool cf_all = (a.gn_mask & 0x8F) == 0x8F;                // closed-form warm step enabled in all four stages
    if (lane < 8) {
        float v = (lane == 3) ? 1.f : 0.f;
        if (a.affine != nullptr) v = (lane == 7) ? 1.f : __ldg(a.affine + c * 8 + lane);
        sh.mapc[lane] = v;
        if (lane < 4) sh.nfx[lane] = 0u;
    }
    const bool mapped = a.affine != nullptr;                       // (kernel argument: uniform, no shared-memory test per key point)
    auto map_apply = [&](Vec3<float> v, int row) -> Vec3<float> {  // AlignPose.align_leg on load (LoadMap), constants in shared memory
        if (mapped) {
            const float sc = sh.mapc[3];
            if (row == 0) v = {sh.mapc[4], sh.mapc[5], sh.mapc[6]};
            else v = {(v.x - sh.mapc[0]) * sc + sh.mapc[4], (v.y - sh.mapc[1]) * sc + sh.mapc[5], (v.z - sh.mapc[2]) * sc + sh.mapc[6]};
        }
        return v;
    };

    if (lane < 4) {                                                // per-(chain, stage) constants
        const StageConst<float> k = stage_const(BLK_PRM, lane);
        float* K = sh.kc[lane];
        K[KC_L] = k.L; K[KC_LB0] = k.lb0; K[KC_UB0] = k.ub0; K[KC_LB1S] = k.lb1s; K[KC_UB1S] = k.ub1s;
        K[KC_LB1] = k.lb1; K[KC_UB1] = k.ub1; K[KC_NSQ] = k.nsq;
        K[KC_SL0] = k.sl0; K[KC_CL0] = k.cl0; K[KC_SU0] = k.su0; K[KC_CU0] = k.cu0;
        K[KC_LB0P] = k.lb0p; K[KC_UB0P] = k.ub0p;
        K[KC_HAVE_BT] = (lane < 3 && k.cl0 * k.cl0 + k.sl0 * k.sl0 > 0.f) ? 1.f : 0.f;   // (the verification's have_bt, once per chain)
    }
    if (lane == 0) {
        mbar_init(&sh.bar[0], 1); mbar_init(&sh.bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp(full);
    // angle series: lanes 0..2 carry the first angle of stages 1..3, lanes 3..6 the second angle of stages 1..4
    const bool is_ser = lane < 7, is_a = lane < 3;
    const int sl_ = is_a ? lane : (is_ser ? lane - 3 : 0);
    const float ser_lb = sh.kc[sl_][is_a ? KC_LB0 : KC_LB1S], ser_ub = sh.kc[sl_][is_a ? KC_UB0 : KC_UB1S];
    const float ser_shift = (lane == 3) ? half_pi : 0.f;
    float xcar = 0.f;                                              // carried angle of this lane's series, caller's terms
    {
        const float* seed = warm_given ? a.warm + c * a.warm_cs : BLK_PRM + 18;
        if (is_ser) xcar = seed[is_a ? 2 * sl_ : (sl_ == 3 ? 6 : 2 * sl_ + 1)];
    }
    uint32_t n_commit = 0u; int worst = ST_GTOL;   // frames this lane committed from the pass (one evaluation per stage each)
    const int n_blk = (n_frame + BLK - 1) / BLK;
    auto frames_of = [&](int b) { const int r = n_frame - b * BLK; return r < BLK ? r : BLK; };
    auto bulk_load_ok = [&](int b) { return bulk_in && (frames_of(b) & 3) == 0; };
    auto issue_load = [&](int b) {                                 // lane 0
        const uint32_t bytes = (uint32_t)frames_of(b) * 60u;
        mbar_expect_tx(&sh.bar[b & 1], bytes);
        tma_load_1d(sh.pose[b & 1], BLK_POSE + (int64_t)b * (BLK * 15), bytes, &sh.bar[b & 1]);
    };
    if (lane == 0 && bulk_load_ok(0)) issue_load(0);

    for (int b = 0; b < n_blk; ++b) {
        const int cur = b & 1, nv = frames_of(b), t_abs0 = b * BLK;
        const float* kp = sh.pose[cur] + lane * 15;
        if (bulk_load_ok(b)) mbar_wait(&sh.bar[cur], (uint32_t)(b >> 1) & 1u);
        else {
            const float* src = BLK_POSE + (int64_t)t_abs0 * a.pose_fs;
            for (int i = lane; i < nv * 15; i += BLK) sh.pose[cur][i] = __ldg(src + (int64_t)(i / 15) * a.pose_fs + i % 15);
        }
        __syncwarp(full);
        if (lane == 0 && b + 1 < n_blk && bulk_load_ok(b + 1)) issue_load(b + 1);
        // ---- entry: the carried angles re-enter like set_iterate + place; their sin/cos are re-derived (SEQIK_RESYNC = 32)
        if (is_ser) {
            const float x = place1(xcar - ser_shift, ser_lb, ser_ub);
            float es, ec, v_;
            Num<float>::sincosv_(x, &es, &ec, &v_);
            sh.acc_x[lane][1] = x;
            if (is_a) { sh.P[sl_][0] = es; sh.P[sl_][1] = ec; } else { sh.P[sl_][2] = es; sh.P[sl_][3] = ec; }
            if (lane == 6) { sh.P[3][0] = 0.f; sh.P[3][1] = 1.f; }            // one-variable stage: first angle fixed at 0
        }
        __syncwarp(full);
        bool staged = false;
        int j0 = 0, s_start = 0;         // the pass covers lanes j0.. and stages s_start.. (earlier stages of those lanes stand)
        if (first_done && b == 0) {
            // frame 0 was solved by leg_first_frame_kernel: its record (final sin/cos, placed angles, counters) waits in the
            // chain's angle rows 1..4, its results in row 0 of the outputs; the block starts at lane 1 from that state
            float rec = 0.f;
            if (lane < FF_REC) rec = BLK_ANG[(int64_t)(1 + lane / 7) * a.ang_fs + lane % 7];
            if (lane < 16) sh.P[lane >> 2][lane & 3] = rec;
            const float vx = __shfl_sync(full, rec, 16 + (lane < 7 ? lane : 0));
            if (is_ser) sh.acc_vk[lane][0] = make_float2(vx, 0.f);
#pragma unroll
            if (lane >= 23 && lane < 27) sh.nfx[lane - 23] = (uint32_t)__float_as_int(rec);
            const int w0 = __float_as_int(__shfl_sync(full, rec, 27));
            if (lane == 0) worst = w0;
            if (lane < 7) sh.out_ang[lane] = BLK_ANG[lane];
            if (kFk && lane < FKF) sh.out_fk[lane] = BLK_FK[lane];
            staged = true;                                                     // (first block: no earlier bulk store to wait for)
            j0 = 1;
            __syncwarp(full);
        }
        const Vec3<float> o = map_apply({kp[0], kp[1], kp[2]}, 0);
        const bool enable_t = cf_all && (t_abs0 + lane > 0 || warm_given);
        // A replay that starts at stage sf leaves the stages before it valid for the lanes after it: those lanes park their
        // results of stages 0..2 in their own -- not yet committed -- rows of the staging area across the replay (31 floats)
        // and the next pass picks them up, so that the first pass of a block, the hot one, carries nothing over.
        float* const stash_f = sh.out_fk + lane * 27;
        float* const stash_a = sh.out_ang + lane * 7;
        for (; j0 < nv;) {
            const bool act = lane >= j0 && lane < nv;
            // results of the pass per lane and stage
            float Tsa[4], Tca[4], Tsb[4], Tcb[4];                  // final sin/cos per stage (speculated)
            float dA[4], dB[4]; uint32_t bits = 0u;                // per stage (byte s): bit 0 small_a & small_b & (cond or lim ok_q), 5-6 guess
            uint32_t lim_stages = 0u;                              // bit s: some active lane guessed a limit in stage s (warp-uniform)
            Vec3<float> npv[4];                                    // end point of each stage relative to the origin
            // ================= pass =================
            {
                Mat3<float> A = {{1.f, 0.f, 0.f}, {0.f, 1.f, 0.f}, {0.f, 0.f, 1.f}};
                Vec3<float> piv = {0.f, 0.f, 0.f};
#pragma unroll
                for (int s = 0; s < 4; ++s) {
                    const bool xy = s == 0, one_var = s == 3;
                    if (kRobust && s < s_start) {                  // (rare, warp-uniform) this stage's results of the previous pass stand
                        Tsa[s] = stash_f[9 * s]; Tca[s] = stash_f[9 * s + 1]; Tsb[s] = stash_f[9 * s + 2]; Tcb[s] = stash_f[9 * s + 3];
                        npv[s].x = stash_f[9 * s + 7]; npv[s].y = stash_f[9 * s + 8]; npv[s].z = stash_a[s < 3 ? s : 0];
                        if (s < 3) {
                            A = rotate_stage(A, s, Tsa[s], Tca[s], Tsb[s], Tcb[s]);
                            piv = npv[s];
                        }
                        continue;
                    }
                    const float* K = sh.kc[s];
                    const float L = K[KC_L];
                    // (the one-variable stage has no first angle: its sin/cos are the constants 0 and 1 in every state, so that
                    //  half of the move -- two shuffles, a rotation difference, an arcsine -- folds away at compile time)
                    const bool fold_a = one_var && !kRobust;          // (measured: the robust kernel, 600 chains, is 1.7 % slower with it)
                    const float Psa = fold_a ? 0.f : sh.P[s][0], Pca = fold_a ? 1.f : sh.P[s][1], Psb = sh.P[s][2], Pcb = sh.P[s][3];
                    const float sgn = (Psb < 0.f) ? -1.f : 1.f;
                    const Vec3<float> kt = map_apply({kp[3 * s + 3], kp[3 * s + 4], kp[3 * s + 5]}, s + 1);
                    const Vec3<float> rel = {(kt.x - o.x) - piv.x, (kt.y - o.y) - piv.y, (kt.z - o.z) - piv.z};
                    const Vec3<float> q3 = mulT(A, rel);
                    const Vec3<float> q = xy ? Vec3<float>{-q3.z, q3.y, q3.x} : q3;
                    const WarmCand<float> cd = warm_interior(q, L, one_var, sgn, Psa, Pca);
                    int g = WC_INTERIOR;
                    if (!one_var) g = warm_guess(cd.n_sa, cd.n_ca, K[KC_SL0], K[KC_CL0], K[KC_SU0], K[KC_CU0]);
                    float tsa = cd.n_sa, tca = cd.n_ca, tsb = cd.n_sb, tcb = cd.n_cb;
                    Vec3<float> f = cd.f;
                    bool cq = cd.cond;                             // the admission tests of this lane's candidate that depend on the target alone
                    const bool any_lim = !one_var && __any_sync(full, act && g != WC_INTERIOR);
                    if (any_lim) lim_stages |= 1u << s;
                    if (any_lim && g != WC_INTERIOR) {             // (warp-uniform outer test: the block is skipped when no lane needs it)
                        const bool lo = g == WC_LO;
                        tsa = lo ? K[KC_SL0] : K[KC_SU0]; tca = lo ? K[KC_CL0] : K[KC_CU0];
                        const WarmLimit<float> lc = warm_limit(q, L, lo, tsa, tca, sgn);
                        tsb = lc.c_sb; tcb = lc.c_cb; f = lc.f; cq = lc.ok_q;
                    }
                    if (kRobust && one_var) {
                        // The one-variable stage sitting ON a limit (TiTa_pitch = 0 for long stretches of a real recording): while
                        // the target keeps pushing it outward the serial solver's first evaluation meets a vanishing scaled
                        // gradient and the iterate stays where it is (status 1, one evaluation).  The lanes that follow the pass's
                        // starting state without a gap inherit that state unchanged, so the test is exact here -- no speculation.
                        const float xP = (j0 == 0) ? sh.acc_x[6][1] : sh.acc_vk[6][j0 - 1].x;          // placed angle before lane j0
                        float dl1 = xP - K[KC_LB1S], du1 = K[KC_UB1S] - xP;
                        if (dl1 <= 0.f) { dl1 = 1e-10f * fmaxf(1.f, fabsf(K[KC_LB1S])); du1 = (K[KC_UB1S] - K[KC_LB1S]) - dl1; }
                        if (du1 <= 0.f) { du1 = 1e-10f * fmaxf(1.f, fabsf(K[KC_UB1S])); dl1 = (K[KC_UB1S] - K[KC_LB1S]) - du1; }
                        if (fminf(dl1, du1) < 1e-6f) {             // (warp-uniform)
                            const WarmMove<float> mp = warm_move(cd.n_sa, cd.n_ca, cd.n_sb, cd.n_cb, Psa, Pca, Psb, Pcb);
                            const float nx1 = xP + mp.dB;
                            const bool in_b = (nx1 - K[KC_LB1S] > 1e-5f) & (K[KC_UB1S] - nx1 > 1e-5f);
                            const bool okP = enable_t & mp.small_a & mp.small_b & cd.cond & in_b;
                            const float Lsb = L * Psb, Lcb = L * Pcb;
                            const Vec3<float> fP = {-Lsb * Pca - q.x, -Lsb * Psa - q.y, -Lcb - q.z};
                            const float cost = 0.5f * dot(fP, fP);
                            const float g0 = 0.f * Lsb * fmaf(Psa, fP.x, -(Pca * fP.y));
                            const float g1 = fmaf(Lsb, fP.z, -(Lcb * fmaf(Pca, fP.x, Psa * fP.y)));
                            const float v1 = (g1 < 0.f && du1 < inf) ? du1 : (g1 > 0.f && dl1 < inf) ? dl1 : 1.f;
                            const bool stays = !okP && cost < inf && fmaxf(fabsf(g0), fabsf(g1 * v1)) < 1e-8f;
                            const unsigned run = __ballot_sync(full, act && stays) >> j0;            // bit k: lane j0 + k stays
                            const int n_stay = (run == 0xffffffffu) ? 32 : __ffs((int)~run) - 1;     // length of the run that starts at j0
                            if (act && lane < j0 + n_stay) { tsa = Psa; tca = Pca; tsb = Psb; tcb = Pcb; f = fP; g = WC_STAYS; }
                        }
                    }
                    Tsa[s] = tsa; Tca[s] = tca; Tsb[s] = tsb; Tcb[s] = tcb;
                    // the previous lane's state (the first lane of the pass: the state the pass starts from)
                    float psa = 0.f, pca = 1.f;
                    if (!fold_a) { psa = __shfl_up_sync(full, tsa, 1); pca = __shfl_up_sync(full, tca, 1); }
                    float psb = __shfl_up_sync(full, tsb, 1), pcb = __shfl_up_sync(full, tcb, 1);
                    if (lane == j0) { psa = Psa; pca = Pca; psb = Psb; pcb = Pcb; }
                    // The first angle's move is the interior candidate's in every case (warm_case tests it against the limits).
                    // The second angle's move is that of the lane's own candidate, (tsb, tcb): for an interior guess warm_step's
                    // interior move, for a limit guess its on-limit move (warm_limit_move is the same arithmetic) -- a lane
                    // uses only the one of its guess, in the series and in the verification alike.
                    const WarmMove<float> mv = warm_move(cd.n_sa, cd.n_ca, tsb, tcb, psa, pca, psb, pcb);
                    dA[s] = mv.dA; dB[s] = mv.dB;
                    // (what the verification needs of the tests that depend on the target alone: the half of warm_case that can
                    //  confirm the guess uses them only in the conjunction small_a & small_b & cq of the guessed candidate.  The
                    //  other half cannot confirm it whatever this bit says: a limit guess fails the interior half when the first
                    //  angle is inside its box (WC_INTERIOR or WC_NONE), and that half is false when it is not; an interior
                    //  guess never matches the limit half.)
                    bits |= (((mv.small_a & mv.small_b & cq) ? 1u : 0u) | ((uint32_t)g << 5)) << (8 * s);
                    if (act) {
                        float2 va = make_float2(mv.dA, 1.f), vb = make_float2(mv.dB, 1.f);
                        if (any_lim && (g == WC_LO || g == WC_HI))           // (rare: behind the warp-uniform test)
                            va = make_float2(g == WC_LO ? K[KC_LB0P] : K[KC_UB0P], 0.f);
                        if (kRobust && g == WC_STAYS) vb.x = 0.f;
                        if (!one_var) sh.acc_vk[s][lane] = va;
                        sh.acc_vk[3 + s][lane] = vb;
                    }
                    // end point, joint position, frame of the next stage
                    const Vec3<float> res = xy ? Vec3<float>{f.z, f.y, -f.x} : f;
                    const Vec3<float> Af = mul(A, res);
                    const Vec3<float> np_ = {(piv.x + rel.x) + Af.x, (piv.y + rel.y) + Af.y, (piv.z + rel.z) + Af.z};
                    npv[s] = np_;
                    if (s < 3) {
                        A = rotate_stage(A, s, tsa, tca, tsb, tcb);
                        piv = np_;
                    }
                }
            }
            __syncwarp(full);
            // ================= accumulate (frame order, one series per lane) =================
            // always from frame 0 (a replayed frame has left (its placed angle, 0) behind): one straight-line block
            // (the loads of the next group of 8 frames are in flight while the current group's dependent multiply-adds run)
            if (is_ser) {
                float x = sh.acc_x[lane][1];
                const float4* __restrict__ vk = reinterpret_cast<const float4*>(sh.acc_vk[lane]);
                float2* __restrict__ xo = reinterpret_cast<float2*>(sh.acc_x[lane] + 2);
                float4 p0 = vk[0], p1 = vk[1], p2 = vk[2], p3 = vk[3];
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    float4 n0 = p0, n1 = p1, n2 = p2, n3 = p3;
                    if (g < 3) { n0 = vk[4 * g + 4]; n1 = vk[4 * g + 5]; n2 = vk[4 * g + 6]; n3 = vk[4 * g + 7]; }
                    const float a0 = fmaf(p0.y, x, p0.x), a1 = fmaf(p0.w, a0, p0.z);
                    const float a2 = fmaf(p1.y, a1, p1.x), a3 = fmaf(p1.w, a2, p1.z);
                    const float a4 = fmaf(p2.y, a3, p2.x), a5 = fmaf(p2.w, a4, p2.z);
                    const float a6 = fmaf(p3.y, a5, p3.x), a7 = fmaf(p3.w, a6, p3.z);
                    xo[4 * g] = make_float2(a0, a1); xo[4 * g + 1] = make_float2(a2, a3);
                    xo[4 * g + 2] = make_float2(a4, a5); xo[4 * g + 3] = make_float2(a6, a7);
                    x = a7; p0 = n0; p1 = n1; p2 = n2; p3 = n3;
                }
            }
            __syncwarp(full);
            // ================= verify =================
            if (kRobust && s_start > 0) {                                     // (rare) the stages that stood: their verification data
#pragma unroll
                for (int s = 0; s < 3; ++s)
                    if (s < s_start) { dA[s] = stash_f[9 * s + 4]; dB[s] = stash_f[9 * s + 5]; }
                const uint32_t keep = 0xffffffffu << (8 * s_start);          // bytes of the stages this pass recomputed
                bits = (bits & keep) | (__float_as_uint(stash_a[3]) & ~keep);
                lim_stages |= (1u << s_start) - 1u;                           // (the whole decision for the stages that stood)
            }
            float ox0[4], ox1[4];
            int fs = 4;                                                       // first stage of this lane whose speculation does not hold
#pragma unroll
            for (int s = 3; s >= 0; --s) {
                const float* K = sh.kc[s];
                const uint32_t bs = bits >> (8 * s);
                const int g = (int)((bs >> 5) & 3u);
                const float xp0 = (s < 3) ? sh.acc_x[s < 3 ? s : 0][lane + 1] : 0.f, xp1 = sh.acc_x[3 + s][lane + 1];
                WarmMove<float> mv; mv.dA = (s < 3 || kRobust) ? dA[s] : 0.f; mv.dB = dB[s]; mv.small_a = bs & 1u; mv.small_b = true;
                const float lb0 = (s < 3 || kRobust) ? K[KC_LB0] : -inf, ub0 = (s < 3 || kRobust) ? K[KC_UB0] : inf;
                bool held;                                                    // the decision warm_step takes is the guessed one
                if (lim_stages & (1u << s))                                   // (warp-uniform) some lane guessed a limit: the whole decision
                    held = warm_case(enable_t, s < 3 && K[KC_HAVE_BT] != 0.f, s == 3, xp0, xp1, mv, true, lb0, ub0, K[KC_LB1S], K[KC_UB1S],
                                     g, dB[s], true, true, ox0[s], ox1[s]) == g;
                else                                                          // every active lane guessed interior: its half decides
                    held = warm_case_interior(enable_t, xp0, xp1, mv, true, lb0, ub0, K[KC_LB1S], K[KC_UB1S], ox0[s], ox1[s]) == WC_INTERIOR;
                if (kRobust && s == 3 && g == WC_STAYS) { held = true; ox0[s] = 0.f; ox1[s] = xp1; }      // decided exactly in the pass
                fs = held ? fs : s;
            }
            const unsigned failed = __ballot_sync(full, act && fs < 4);
            const int j = failed ? __ffs((int)failed) - 1 : nv;              // first lane whose speculation does not hold
            // ================= commit lanes j0 .. j-1 =================
            if (!staged) {                                                     // the previous block's bulk stores have read the staging area
                if (lane == 0) tma_store_wait_read<0>();
                __syncwarp(full);
                staged = true;
            }
            if (act && lane < j) {
                float* oa = sh.out_ang + lane * 7;
                oa[0] = ox0[0]; oa[1] = ox1[0] + half_pi; oa[2] = ox0[1]; oa[3] = ox1[1]; oa[4] = ox0[2]; oa[5] = ox1[2]; oa[6] = ox1[3];
                n_commit += 1u;
#pragma unroll
                for (int s = 0; s < 4; ++s) put_fk_joint<kFk>(sh.out_fk + lane * FKF, s, o, {npv[s].x + o.x, npv[s].y + o.y, npv[s].z + o.z});
            }
            if (j >= nv) break;
            // ================= replay lane j through the serial solver, from its first failing stage =================
            // state before frame j: the previous lane's (or the pass's starting state), angles from the accumulated series
            const int sf = __shfl_sync(full, fs, j);                         // (both kernels: the replaying lane keeps its verified stages)
            float qsa[4], qca[4], qsb[4], qcb[4];
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                qsa[s] = __shfl_sync(full, Tsa[s], (j + 31) & 31); qca[s] = __shfl_sync(full, Tca[s], (j + 31) & 31);
                qsb[s] = __shfl_sync(full, Tsb[s], (j + 31) & 31); qcb[s] = __shfl_sync(full, Tcb[s], (j + 31) & 31);
                if (j == j0) { qsa[s] = sh.P[s][0]; qca[s] = sh.P[s][1]; qsb[s] = sh.P[s][2]; qcb[s] = sh.P[s][3]; }
            }
            if (kRobust && act && lane > j && sf > 0) {                       // park stages 0..2 across the replay (see above)
#pragma unroll
                for (int s = 0; s < 3; ++s) {
                    stash_f[9 * s] = Tsa[s]; stash_f[9 * s + 1] = Tca[s]; stash_f[9 * s + 2] = Tsb[s]; stash_f[9 * s + 3] = Tcb[s];
                    stash_f[9 * s + 4] = dA[s]; stash_f[9 * s + 5] = dB[s];
                    stash_f[9 * s + 7] = npv[s].x; stash_f[9 * s + 8] = npv[s].y; stash_a[s] = npv[s].z;
                }
                stash_a[3] = __uint_as_float(bits);
            }
            __syncwarp(full);        // every lane has read sh.P before the replaying lane overwrites it
            if (lane == j) {
                Mat3<float> A = {{1.f, 0.f, 0.f}, {0.f, 1.f, 0.f}, {0.f, 0.f, 1.f}};
                Vec3<float> piv = {0.f, 0.f, 0.f};
                float* oa = sh.out_ang + lane * 7;
                float* of = sh.out_fk + lane * FKF;
                const bool warm_ok = t_abs0 + lane > 0 || warm_given;
                // the stages before the failing one stand as the pass left them: results out, frame rebuilt, state handed on
#pragma unroll
                for (int s = 0; s < 3; ++s) {
                    if (s < sf) {
                        oa[2 * s] = ox0[s]; oa[2 * s + 1] = (s == 0) ? ox1[s] + half_pi : ox1[s]; sh.nfx[s] += 1u;
                        put_fk_joint<kFk>(of, s, o, {npv[s].x + o.x, npv[s].y + o.y, npv[s].z + o.z});
                        A = rotate_stage(A, s, Tsa[s], Tca[s], Tsb[s], Tcb[s]);
                        piv = npv[s];
                        sh.P[s][0] = Tsa[s]; sh.P[s][1] = Tca[s]; sh.P[s][2] = Tsb[s]; sh.P[s][3] = Tcb[s];
                    }
                }
#pragma unroll 1
                for (int s = sf; s < 4; ++s) {
                    const float* K = sh.kc[s];
                    const SerialConst<float> k = {K[KC_L], K[KC_LB0], K[KC_UB0], K[KC_LB1], K[KC_UB1], K[KC_SL0], K[KC_CL0], K[KC_SU0], K[KC_CU0], K[KC_NSQ]};
                    float x0 = (s < 3) ? sh.acc_x[s < 3 ? s : 0][lane + 1] : 0.f, x1 = sh.acc_x[3 + s][lane + 1];
                    float sa = (s == 0) ? qsa[0] : (s == 1) ? qsa[1] : (s == 2) ? qsa[2] : qsa[3];
                    float ca = (s == 0) ? qca[0] : (s == 1) ? qca[1] : (s == 2) ? qca[2] : qca[3];
                    float sb = (s == 0) ? qsb[0] : (s == 1) ? qsb[1] : (s == 2) ? qsb[2] : qsb[3];
                    float cb = (s == 0) ? qcb[0] : (s == 1) ? qcb[1] : (s == 2) ? qcb[2] : qcb[3];
                    const Vec3<float> kt = map_apply({kp[3 * s + 3], kp[3 * s + 4], kp[3 * s + 5]}, s + 1);
                    float xb; Vec3<float> w; uint32_t ne = 0u;
                    if (kRobust) serial_stage_call(s, k, a.gn_mask, esc, warm_ok, kt, o, A, piv, x0, x1, sa, ca, sb, cb, xb, w, ne, worst);
                    else serial_stage(s, k, a.gn_mask, esc, warm_ok, kt, o, A, piv, x0, x1, sa, ca, sb, cb, xb, w, ne, worst);
                    // (outputs inside the limits, seqik_core.cuh limit_clamp: only the serial solver's iterates can sit an ulp
                    //  outside; the pass's closed-form angles are admitted 1e-5 inside and its on-limit angles are placed)
                    const float xb_out = limit_clamp(xb, K[KC_LB1], K[KC_UB1]);
                    if (s < 3) { oa[2 * s] = limit_clamp(x0, K[KC_LB0], K[KC_UB0]); oa[2 * s + 1] = xb_out; } else oa[6] = xb_out;
                    sh.nfx[s] += ne;
                    put_fk_joint<kFk>(of, s, o, w);
                    // hand the final state on: the next pass starts from it
                    sh.P[s][0] = sa; sh.P[s][1] = ca; sh.P[s][2] = sb; sh.P[s][3] = cb;
                    // ... and the angles, as a reset of their series: x <- 0 x + (placed angle)
                    if (s < 3) sh.acc_vk[s < 3 ? s : 0][lane] = make_float2(place1(x0, K[KC_LB0], K[KC_UB0]), 0.f);
                    sh.acc_vk[3 + s][lane] = make_float2(place1(x1, K[KC_LB1S], K[KC_UB1S]), 0.f);
                }
            }
            __syncwarp(full);
            j0 = j + 1;
            s_start = kRobust ? sf : 0;    // robust: the lanes after j keep their stages before sf (nothing those depend on has changed); lean: recomputed
            if (j0 >= nv) break;
        }
        // ---- carry the angles to the next block in the caller's terms (xa = x0, xb = x1 + shift)
        __syncwarp(full);
        if (j0 >= nv && nv > 0) {                                  // the block ended with a replay: run the series over its reset
            if (is_ser) {
                float x = sh.acc_x[lane][1];
                for (int t = 0; t < nv; ++t) { const float2 p = sh.acc_vk[lane][t]; x = fmaf(p.y, x, p.x); }
                sh.acc_x[lane][nv + 1] = x;
            }
            __syncwarp(full);
        }
        if (is_ser) xcar = sh.acc_x[lane][nv + 1] + ser_shift;
        // ---- results of the block leave: two bulk stores (or plain coalesced stores when sizes / addresses do not allow them)
        const bool bulk_store = bulk_out && (nv & 3) == 0;
        if (bulk_store) {
            fence_async_smem();
            __syncwarp(full);
            if (lane == 0) {
                tma_store_1d_nocommit(BLK_ANG + (int64_t)t_abs0 * 7, sh.out_ang, (uint32_t)nv * 28u);
                if (kFk) tma_store_1d_nocommit(BLK_FK + (int64_t)t_abs0 * FKF, sh.out_fk, (uint32_t)nv * (FKF * 4u));
                tma_commit();
            }
        } else {
            __syncwarp(full);
            float* da = BLK_ANG + (int64_t)t_abs0 * a.ang_fs;
            for (int i = lane; i < nv * 7; i += BLK) da[(int64_t)(i / 7) * a.ang_fs + i % 7] = sh.out_ang[i];
            if (kFk) {
                float* df = BLK_FK + (int64_t)t_abs0 * a.fk_fs;
                for (int i = lane; i < nv * FKF; i += BLK) df[(int64_t)(i / FKF) * a.fk_fs + i % FKF] = sh.out_fk[i];
            }
            __syncwarp(full);
        }
    }
    if (lane == 0) tma_store_wait_read<0>();
    // per-chain statistics
    n_commit = __reduce_add_sync(full, n_commit);
    const int w_all = __reduce_min_sync(full, worst);
    __syncwarp(full);
    if (lane == 0) {
        if (a.nfev) { uint32_t* p = a.nfev + c * 4; for (int s = 0; s < 4; ++s) p[s] = n_commit + sh.nfx[s]; }
        if (a.status) a.status[c] = w_all == ST_NONFINITE ? -1 : w_all;
    }
}

#undef BLK_PRM
#undef BLK_POSE
#undef BLK_ANG
#undef BLK_FK

// Launch of schedule 3.  One CTA (= one warp) per chain; the hardware block scheduler deals chains to SMs as warps
// retire.  Chains cost about the same, so the batch runs in "waves" of (resident warps per SM) x (SMs) chains and the
// time is ~ ceil(n_chain / (R n_sm)) * R: R is chosen to minimise that (a last wave that is nearly empty costs a full
// wave's latency; config 4's 7 500-chain shard: R = 13 -> 4 full waves instead of 3.2 at R = 16) and imposed through the
// dynamic shared memory size.  `forced` (1..32): tuning / tests.
template <int kFk, bool kRobust>
static int launch_block_kernel(const LegArgs& a, int bulk_in, int bulk_out, int forced, cudaStream_t st) {
    static thread_local int cached_dev = -1;
    static thread_local int n_sm = 148, r_max = 16, static_smem = 0, smem_sm = 227 * 1024;
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev != cached_dev) {
        cudaFuncAttributes at;
        if (cudaFuncGetAttributes(&at, leg_solve_block_kernel<kFk, kRobust>) != cudaSuccess) return seqik_check_launch("seqik_leg_solve_f32 (attributes)");
        cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
        cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev);
        static_smem = (int)at.sharedSizeBytes;
        int regs_sm = 65536;
        cudaDeviceGetAttribute(&regs_sm, cudaDevAttrMaxRegistersPerMultiprocessor, dev);
        const int by_regs = regs_sm / (((at.numRegs + 7) / 8 * 8) * BLK);            // registers are allocated per warp in units of 256
        const int by_smem = smem_sm / (static_smem + 1024);                            // 1 KB per CTA is reserved by the system
        r_max = by_regs < by_smem ? by_regs : by_smem;
        if (r_max > 32) r_max = 32;                                                    // CTAs per SM
        if (r_max < 1) r_max = 1;
        cudaFuncSetAttribute(leg_solve_block_kernel<kFk, kRobust>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_sm - static_smem - 1024);
        cudaFuncSetAttribute(leg_solve_block_kernel<kFk, kRobust>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        cached_dev = dev;
    }
    // resident warps per SM: as many as registers and shared memory allow -- measured faster than any "whole waves" choice
    // of fewer (latency hiding outweighs a partly filled last wave; profiles/r02_block_resident_sweep.jsonl)
    int r = r_max;
    if (forced) r = forced < r_max ? forced : r_max;
    // shared memory per CTA such that exactly r CTAs fit one SM
    int dyn = smem_sm / r - 1024 - static_smem;
    dyn = dyn < 0 ? 0 : dyn & ~127;
    if (r == r_max && !forced) dyn = 0;
    const int first_done = (a.warm == nullptr && a.n_frame >= 5) ? 1 : 0;
    if (first_done) leg_first_frame_kernel<kFk><<<(unsigned)((a.n_chain + BLK - 1) / BLK), BLK, 0, st>>>(a);
    leg_solve_block_kernel<kFk, kRobust><<<(unsigned)a.n_chain, BLK, (size_t)dyn, st>>>(a, bulk_in, bulk_out, first_done);
    return SEQIK_OK;
}
static int launch_block_schedule(const LegArgs& a, bool want_fk, bool fk_joints, int forced, int variant, cudaStream_t st) {
    const int fkf = fk_joints ? 12 : 27;
    const bool al_in = (((uintptr_t)a.pose) & 15) == 0 && (a.pose_cs & 3) == 0 && a.pose_fs == 15;
    const bool al_out = (((uintptr_t)a.angles) & 15) == 0 && (a.ang_cs & 3) == 0 && a.ang_fs == 7
                        && (!want_fk || ((((uintptr_t)a.fk) & 15) == 0 && (a.fk_cs & 3) == 0 && a.fk_fs == fkf));
    // variant: 1 lean, 2 robust, 0 automatic -- robust while the batch does not fill the robust kernel's resident warps anyway
    // (its lower occupancy then costs nothing and replay-heavy recordings, which typically come as a few long chains, gain
    // up to 2.5x); lean beyond (throughput regime; config 3: 0.335 against 0.372 ms)
    int n_sm = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    const bool robust = variant == 2 || (variant == 0 && a.n_chain <= (int64_t)SEQIK_BLOCK_MIN_CTAS_ROBUST * n_sm);
    if (robust) {
        if (!want_fk) return launch_block_kernel<0, true>(a, al_in, al_out, forced, st);
        return fk_joints ? launch_block_kernel<2, true>(a, al_in, al_out, forced, st) : launch_block_kernel<1, true>(a, al_in, al_out, forced, st);
    }
    if (!want_fk) return launch_block_kernel<0, false>(a, al_in, al_out, forced, st);
    return fk_joints ? launch_block_kernel<2, false>(a, al_in, al_out, forced, st) : launch_block_kernel<1, false>(a, al_in, al_out, forced, st);
}

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
extern "C" int seqik_leg_solve_f32(const float* pose, int64_t pose_chain_stride, int64_t pose_frame_stride,
                                   const float* affine, const float* params,
                                   float* angles, int64_t ang_chain_stride, int64_t ang_frame_stride,
                                   float* fk, int64_t fk_chain_stride, int64_t fk_frame_stride,
                                   const float* warm, int64_t warm_chain_stride,
                                   int32_t* status, uint32_t* nfev,
                                   int64_t n_chain, int64_t n_frame, uint32_t stage_mask, uint32_t flags, void* stream) {
    if (n_chain < 0 || n_frame < 0) return seqik_fail(SEQIK_EINVAL, "seqik_leg_solve_f32: negative size");
    if (n_chain == 0 || n_frame == 0) return SEQIK_OK;
    if (!pose || !params || !angles) return seqik_fail(SEQIK_EINVAL, "seqik_leg_solve_f32: pose, params and angles must not be NULL");
    {
        uint32_t m = stage_mask;
        while (m && !(m & 1u)) m >>= 1;
        if (stage_mask == 0 || stage_mask > 0xF || (m & (m + 1)) != 0)
            return seqik_fail(SEQIK_EINVAL, "seqik_leg_solve_f32: stage_mask must be a contiguous run of bits within 0xF");
    }
    const bool fk_joints = (flags & SEQIK_FLAG_FK_JOINTS) != 0;
    if (pose_frame_stride < 15 || ang_frame_stride < 7 || (fk && fk_frame_stride < (fk_joints ? 12 : 27)))
        return seqik_fail(SEQIK_EINVAL, "seqik_leg_solve_f32: frame stride smaller than the innermost block");
    if (n_frame > 2147483647LL) return seqik_fail(SEQIK_EINVAL, "seqik_leg_solve_f32: too many frames");
    uint32_t sched = (flags & SEQIK_FLAG_SCHED_MASK) >> SEQIK_FLAG_SCHED_SHIFT;
    if (sched > 3) return seqik_fail(SEQIK_EINVAL, "seqik_leg_solve_f32: unknown schedule");
    // automatic: frame-parallel blocks when every stage is solved with the closed-form warm step (the default flags) --
    // the schedule speculates on it; otherwise the stage pipeline (faster than one lane per chain at every size, DESIGN.md 7)
    const bool block_ok = stage_mask == 0xF && (flags & 0x8Fu) == 0x8Fu;
    if (sched == 3 && !block_ok)
        return seqik_fail(SEQIK_EINVAL, "seqik_leg_solve_f32: schedule 3 needs all four stages and SEQIK_FLAG_CLOSED_FORM with Gauss-Newton mode in every stage");
    if (sched == 0) sched = block_ok ? 3 : 2;
    LegArgs a;
    a.pose = pose; a.pose_cs = pose_chain_stride; a.pose_fs = pose_frame_stride;
    a.affine = affine; a.params = params;
    a.angles = angles; a.ang_cs = ang_chain_stride; a.ang_fs = ang_frame_stride;
    a.fk = fk; a.fk_cs = fk_chain_stride; a.fk_fs = fk_frame_stride;
    a.warm = warm; a.warm_cs = warm_chain_stride;
    a.status = status; a.nfev = nfev; a.n_chain = n_chain; a.n_frame = n_frame;
    a.fk_joints = fk_joints ? 1 : 0;
    a.stage_mask = (int)stage_mask; a.gn_mask = (int)(flags & 0xFF);   // bits 0-3 Gauss-Newton mode per stage, 4 escape, 5 skip-confirm, 6 Newton, 7 closed-form warm step
    if (sched == 3) {
        if (n_chain > 2147483647LL) return seqik_fail(SEQIK_EINVAL, "seqik_leg_solve_f32: too many chains");
        const int rc = launch_block_schedule(a, fk != nullptr, fk_joints, (flags >> SEQIK_FLAG_CPW_SHIFT) & 0x3F,
                                             (int)((flags >> SEQIK_FLAG_BLOCK_VARIANT_SHIFT) & 0x3u), (cudaStream_t)stream);
        if (rc != SEQIK_OK) return rc;
    } else if (sched == 1) {
        const int64_t grid = (n_chain + 31) / 32;
        leg_solve_lane_kernel<<<(unsigned)grid, 32, 0, (cudaStream_t)stream>>>(a);
    } else {
        // chains per warp (measured, DESIGN.md 7): spread the chains over one warp per SM sub-partition (4 x 148) while
        // that is possible, then fill the warps -- up to 5 chains (20 lanes) while the warps still fit the SMs in about two
        // waves (a warp runs the iteration block for all its lanes whenever ONE lane needs it, so less-than-full warps
        // execute fewer instructions per chain: 6 000 / 7 500 / 15 000 chains are 3 / 6 / 18 % faster at 4 - 5 chains per
        // warp than at 8), 6 beyond that (18 000 - 60 000 chains: 6 is 15 - 22 % faster than 8; `scripts/sweep.py big`).
        // Small batches run at pure chain latency whatever the packing.
        int dev = 0, n_sm = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
        int cpw = (int)((n_chain + 4LL * n_sm - 1) / (4LL * n_sm));
        // (with the iterating flag sets nearly every lane needs the iteration block anyway: full warps are best there)
        const int cap = !(flags & SEQIK_FLAG_CLOSED_FORM) ? PIPE_CHAINS : (n_chain <= 27LL * 4 * n_sm) ? 5 : 6;
        cpw = cpw < 1 ? 1 : (cpw > cap ? cap : cpw);
        const uint32_t forced = (flags >> SEQIK_FLAG_CPW_SHIFT) & 0x3F;     // tuning / tests
        if (forced) cpw = (int)forced;
        if (cpw < 1 || cpw > PIPE_CHAINS) return seqik_fail(SEQIK_EINVAL, "seqik_leg_solve_f32: chains per warp must be 1..8");
        const int64_t grid = (n_chain + cpw - 1) / cpw;
        // Period of the open/close phases.  A phase costs the warp about two trips whatever the number of lanes that take
        // part, so it pays to let nearly all lanes of the warp finish their solves and then close / open together: every
        // 6th iteration for the reference's iterates (3 - 6 trips per solve; config 3, ms per 1000 frames at period
        // 1 / 2 / 4 / 6 / 8 = 5.8 / 4.4 / 3.9 / 3.6 / 3.6), every 4th with Newton steps (2 - 3 trips), every 2nd with the
        // closed-form warm step every iteration for up to 7 000 chains (latency regime: a lane then handles one frame per
        // iteration) and every 3rd beyond (throughput regime: fewer instructions; 60 000 chains: 6.1 / 5.7 / 5.2 ms at
        // period 1 / 2 / 3, `profiles/r01_ab_merged_phase.txt`).  Scheduling only: results are unchanged.
        const uint32_t gate_sel = (flags >> SEQIK_FLAG_GATE_SHIFT) & 0xFu;    // 0 auto, else the period in iterations
        const int gate_period = gate_sel ? (int)gate_sel
                              : (flags & SEQIK_FLAG_CLOSED_FORM) ? (n_chain <= 7000 ? 1 : 3) : (flags & SEQIK_FLAG_NEWTON) ? 4 : 6;
        const uint32_t trip_sel = (flags >> SEQIK_FLAG_TRIP_SHIFT) & 0x7u;
        const int trip_period = trip_sel ? (int)trip_sel : 1;
        if (stage_mask == 0xF && fk && !fk_joints) leg_solve_pipe_kernel<true><<<(unsigned)grid, 32, 0, (cudaStream_t)stream>>>(a, cpw, gate_period, trip_period);
        else leg_solve_pipe_kernel<false><<<(unsigned)grid, 32, 0, (cudaStream_t)stream>>>(a, cpw, gate_period, trip_period);
    }
    return seqik_check_launch("seqik_leg_solve_f32");
}
