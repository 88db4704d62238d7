// Host build of csrc/seqik_core.cuh, seqik_generic.cuh and seqik_block.cuh for CPU-side algorithm tests (tests/ only).
// The block schedule's emulation (run_block) runs the kernels' own replay and first-frame arithmetic (serial_stage).
// TEST INFRASTRUCTURE: compiled by tests/hostsim_build.py with g++, loaded via ctypes by
// tests; the product package never loads it.
#include "seqik_core.cuh"
#include "seqik_generic.cuh"
#include "seqik_block.cuh"
#include <cstdint>

using namespace seqik;

template <typename R>
static void run_chain(const R* pose, int64_t n_frame, const R* seg, const R* lb, const R* ub,
                      const R* null_sq, const R* seed, R* angles, R* fk, int32_t* nfev, int32_t* status,
                      int stage_mask, int gn_mask, double* iterates = nullptr) {
    ChainParams<R> P;
    for (int i = 0; i < 4; ++i) { P.seg[i] = seg[i]; P.null_sq[i] = null_sq[i]; }
    for (int i = 0; i < 7; ++i) { P.lb[i] = lb[i]; P.ub[i] = ub[i]; }
    R ang[7];
    for (int i = 0; i < 7; ++i) ang[i] = seed[i];
    for (int64_t t = 0; t < n_frame; ++t) {
        FrameStats fs;
        solve_frame<R>(P, pose + t * 15, ang, fk ? fk + t * 27 : nullptr, &fs, stage_mask, gn_mask);
        for (int i = 0; i < 7; ++i) angles[t * 7 + i] = ang[i];
        if (nfev) for (int s = 0; s < 4; ++s) { nfev[t * 4 + s] = fs.nfev[s]; status[t * 4 + s] = fs.status[s]; }
        if (iterates) for (int i = 0; i < 7; ++i) iterates[t * 7 + i] = fs.iterate[i];
    }
}

// ---- the decoupled per-lane runner, driven serially (one step() at a time) ----
template <typename R> struct HostIO {
    const R* pose; const R* seg_; const R* lb_; const R* ub_; const R* nsq_; R* angles; R* fk;
    Vec3<R> kp(int64_t t, int row) const { const R* p = pose + t * 15 + row * 3; return {p[0], p[1], p[2]}; }
    void put_angles(int64_t t, const R* a, int i0, int i1) const { for (int i = i0; i < i1; ++i) angles[t * 7 + i] = a[i]; }
    R angle_in(int64_t t, int i) const { return angles[t * 7 + i]; }
    void put_fk(int64_t t, int row, const Vec3<R>& v) const { R* p = fk + t * 27 + row * 3; p[0] = v.x; p[1] = v.y; p[2] = v.z; }
    R seg(int i) const { return seg_[i]; }
    R lb(int i) const { return lb_[i]; }
    R ub(int i) const { return ub_[i]; }
    R null_sq(int i) const { return nsq_[i]; }
};
template <typename R>
static int64_t run_runner(const R* pose, int64_t n_frame, const R* seg, const R* lb, const R* ub, const R* null_sq,
                          const R* seed, R* angles, R* fk, uint32_t* nfev_sum, int stage_mask, int gn_mask) {
    HostIO<R> io{pose, seg, lb, ub, null_sq, angles, fk};
    ChainRunner<R, HostIO<R>> run;
    run.start(io, n_frame, seed, stage_mask, gn_mask);
    int64_t steps = 0;
    while (!run.finished()) { run.step(); ++steps; }
    nfev_sum[0] = run.nf0; nfev_sum[1] = run.nf1; nfev_sum[2] = run.nf2; nfev_sum[3] = run.nf3;
    return steps;
}

extern "C" {
int64_t hostsim_runner_f32(const float* pose, int64_t n_frame, const float* seg, const float* lb, const float* ub,
                           const float* null_sq, const float* seed, float* angles, float* fk, uint32_t* nfev_sum,
                           int stage_mask, int gn_mask) {
    return run_runner<float>(pose, n_frame, seg, lb, ub, null_sq, seed, angles, fk, nfev_sum, stage_mask, gn_mask);
}
void hostsim_chain_f32(const float* pose, int64_t n_frame, const float* seg, const float* lb, const float* ub,
                       const float* null_sq, const float* seed, float* angles, float* fk, int32_t* nfev,
                       int32_t* status, int stage_mask, int gn_mask) {
    run_chain<float>(pose, n_frame, seg, lb, ub, null_sq, seed, angles, fk, nfev, status, stage_mask, gn_mask);
}
// the same with the final iterates of every stage before the output clamp (core limit_clamp), as doubles
void hostsim_chain_iterates_f32(const float* pose, int64_t n_frame, const float* seg, const float* lb, const float* ub,
                                const float* null_sq, const float* seed, float* angles, double* iterates, int gn_mask) {
    run_chain<float>(pose, n_frame, seg, lb, ub, null_sq, seed, angles, nullptr, nullptr, nullptr, 0xF, gn_mask, iterates);
}
void hostsim_chain_f64(const double* pose, int64_t n_frame, const double* seg, const double* lb, const double* ub,
                       const double* null_sq, const double* seed, double* angles, double* fk, int32_t* nfev,
                       int32_t* status, int stage_mask, int gn_mask) {
    run_chain<double>(pose, n_frame, seg, lb, ub, null_sq, seed, angles, fk, nfev, status, stage_mask, gn_mask);
}
}

// ---- the stage-pipeline kernel's per-lane arithmetic, run serially: the solve of (stage, frame) is carried from
// (stage, frame - 1) by StageSolve::restart and re-derived by init every SEQIK_RESYNC frames, exactly as
// leg_solve_pipe_kernel does (csrc/seqik_solver.cu); scheduling does not change the arithmetic.
static void run_carried(const float* pose, int64_t n_frame, const float* prm, float* angles, float* fk, int32_t* nfev,
                        int gn_mask) {
    typedef float R;
    StageSolve<R> S[4];
    bool carried[4] = {false, false, false, false};
    R xa[4], xb[4];
    for (int s = 0; s < 4; ++s) { xa[s] = (s == 3) ? 0.f : prm[18 + 2 * s]; xb[s] = prm[18 + ((s == 3) ? 6 : 2 * s + 1)]; }
    const R inf = Num<R>::inf();
    const bool esc = (gn_mask >> 4) & 1;
    for (int64_t t = 0; t < n_frame; ++t) {
        const R* kp = pose + t * 15;
        const Vec3<R> o = {kp[0], kp[1], kp[2]};
        Mat3<R> A = {{1.f, 0.f, 0.f}, {0.f, 1.f, 0.f}, {0.f, 0.f, 1.f}};
        Vec3<R> piv = {0.f, 0.f, 0.f};
        R* f9 = fk + t * 27;
        for (int s = 0; s < 4; ++s) {
            const int kind = (s == 0) ? KIND_XY : KIND_ZY;
            const int ia = 2 * s, ib = (s == 3) ? 6 : 2 * s + 1;
            const R lb0 = (s == 3) ? -inf : prm[4 + ia], ub0 = (s == 3) ? inf : prm[11 + ia];
            const R lb1 = prm[4 + ib], ub1 = prm[11 + ib];
            const int n_full = (s == 0) ? 4 : (s == 1) ? 6 : (s == 2) ? 8 : 9;
            const int gn = stage_mode(gn_mask, s);
            const Vec3<R> k = {kp[3 * (s + 1)], kp[3 * (s + 1) + 1], kp[3 * (s + 1) + 2]};
            const Vec3<R> rel = {(k.x - o.x) - piv.x, (k.y - o.y) - piv.y, (k.z - o.z) - piv.z};
            const Vec3<R> q3 = mulT(A, rel);
            const bool fresh = !(carried[s] && (t & (SEQIK_RESYNC - 1)) != 0);
            if (fresh) {
                const bool had = S[s].have_bt && carried[s];
                const float l0 = S[s].sl0, l1 = S[s].cl0, u0 = S[s].su0, u1 = S[s].cu0;
                S[s].set_problem(kind, prm[s], (s == 3) ? 0.f : 1.f, prm[25 + s], n_full, gn);
                if (!carried[s]) S[s].set_limit_trig(lb0, ub0);          // once per (chain, stage), like the kernel
                else { S[s].have_bt = had; S[s].sl0 = l0; S[s].cl0 = l1; S[s].su0 = u0; S[s].cu0 = u1; }
                S[s].set_iterate(xa[s], xb[s]); carried[s] = true;
            }
            S[s].restart(q3, lb0, ub0, lb1, ub1, fresh, t > 0);
            for (;;) {
                while (!S[s].done()) S[s].trip();
                if (!(esc && S[s].escape())) break;
            }
            xa[s] = S[s].x0; xb[s] = S[s].angle_b();
            if (s != 3) angles[t * 7 + ia] = limit_clamp(xa[s], lb0, ub0);
            angles[t * 7 + ib] = limit_clamp(xb[s], lb1, ub1);
            nfev[t * 4 + s] = S[s].nfev;
            const Vec3<R> Af = mul(A, S[s].res());
            const Vec3<R> np_ = {(piv.x + rel.x) + Af.x, (piv.y + rel.y) + Af.y, (piv.z + rel.z) + Af.z};
            const Vec3<R> jw = {np_.x + o.x, np_.y + o.y, np_.z + o.z};
            f9[3 * s] = o.x; f9[3 * s + 1] = o.y; f9[3 * s + 2] = o.z;
            f9[15 + 3 * s] = jw.x; f9[16 + 3 * s] = jw.y; f9[17 + 3 * s] = jw.z;
            if (s == 0) { f9[12] = jw.x; f9[13] = jw.y; f9[14] = jw.z; }
            A = rotate_frame(A, kind, S[s].sa, S[s].ca, S[s].sin_b(), S[s].cos_b());
            piv = np_;
        }
    }
}
extern "C" void hostsim_carried_f32(const float* pose, int64_t n_frame, const float* prm, float* angles, float* fk,
                                    int32_t* nfev, int gn_mask) {
    run_carried(pose, n_frame, prm, angles, fk, nfev, gn_mask);
}

// ---- the frame-parallel block schedule (csrc/seqik_block.cuh, leg_solve_block_kernel), emulated lane by lane: 32 frames of
// a chain per pass (lane = frame, all four stages in the lane), closed-form candidates speculated from each frame's own key
// points, angle increments accumulated in frame order, warm_step's admission tests verified with the exact angles, the first
// lane that fails replayed through the serial solver.  Must equal run_carried bit for bit.  The per-stage constants
// (stage_const), the replay (serial_stage), the frame rotation and the forward-kinematics rows are the kernels' own code.
// stats: [0] blocks, [1] passes, [2] serial frames, [3] serial frames by reason: first frame, [4] not admitted
static void run_block(const float* pose, int64_t n_frame, const float* prm, const float* warm, float* angles, float* fk,
                      int32_t* nfev, int gn_mask, int64_t* stats) {
    typedef float R;
    const int W = 32;
    const bool esc = (gn_mask >> 4) & 1;
    StageConst<R> K[4];
    for (int s = 0; s < 4; ++s) K[s] = stage_const(prm, s);
    // series l: 0..2 first angle of stages 1..3, 3..6 second angle of stages 1..4; carried in the caller's terms
    R xcar[7];
    const float* seed = warm ? warm : prm + 18;
    for (int s = 0; s < 3; ++s) xcar[s] = seed[K[s].ia];
    for (int s = 0; s < 4; ++s) xcar[3 + s] = seed[K[s].ib];
    auto ser_lb = [&](int l) { return l < 3 ? K[l].lb0 : K[l - 3].lb1s; };
    auto ser_ub = [&](int l) { return l < 3 ? K[l].ub0 : K[l - 3].ub1s; };
    struct Trig { R sa, ca, sb, cb; };
    for (int64_t t0 = 0; t0 < n_frame; t0 += W) {
        const int nv = (int)((n_frame - t0 < W) ? n_frame - t0 : W);
        stats[0]++;
        // ---- entry: the carried angles re-enter like StageSolve::set_iterate + place, their sin/cos are re-derived
        R acc_x[7][W + 1], acc_v[7][W], acc_k[7][W];
        Trig P[4];                                   // state before the first lane of the pass
        R es[7], ec[7];
        for (int l = 0; l < 7; ++l) {
            const R x = (l >= 3) ? xcar[l] - K[l - 3].shift : xcar[l];
            acc_x[l][0] = place1(x, ser_lb(l), ser_ub(l));
            R v_; Num<R>::sincosv_(acc_x[l][0], &es[l], &ec[l], &v_);
        }
        for (int s = 0; s < 4; ++s) {
            if (s < 3) { P[s].sa = es[s]; P[s].ca = ec[s]; }
            else { R v_; Num<R>::sincosv_(R(0), &P[s].sa, &P[s].ca, &v_); }
            P[s].sb = es[3 + s]; P[s].cb = ec[3 + s];
        }
        Trig T[4][W];
        Vec3<R> jw[4][W], org[W];
        R outx0[4][W], outx1[4][W];
        int j0 = 0;
        for (;;) {
            stats[1]++;
            // ---- pass: lanes j0 .. nv-1
            R dA[4][W], dB[4][W], dB2[4][W]; bool sm_a[4][W], sm_b[4][W], sm_b2[4][W], cond[4][W], limq[4][W]; int guess[4][W];
            Mat3<R> A[W]; Vec3<R> piv[W];
            for (int t = j0; t < nv; ++t) {
                A[t] = {{1.f, 0.f, 0.f}, {0.f, 1.f, 0.f}, {0.f, 0.f, 1.f}}; piv[t] = {0.f, 0.f, 0.f};
                const R* kp = pose + (t0 + t) * 15; org[t] = {kp[0], kp[1], kp[2]};
            }
            for (int s = 0; s < 4; ++s) {
                const StageConst<R>& k = K[s];
                const bool xy = s == 0, one_var = s == 3;
                const R sgn = (P[s].sb < R(0)) ? R(-1) : R(1);
                Vec3<R> res[W], rel[W];
                for (int t = j0; t < nv; ++t) {
                    const R* kp = pose + (t0 + t) * 15;
                    const Vec3<R> kt = {kp[3 * (s + 1)], kp[3 * (s + 1) + 1], kp[3 * (s + 1) + 2]};
                    rel[t] = {(kt.x - org[t].x) - piv[t].x, (kt.y - org[t].y) - piv[t].y, (kt.z - org[t].z) - piv[t].z};
                    const Vec3<R> q3 = mulT(A[t], rel[t]);
                    const Vec3<R> q = xy ? Vec3<R>{-q3.z, q3.y, q3.x} : q3;
                    const WarmCand<R> c = warm_interior(q, k.L, one_var, sgn, P[s].sa, P[s].ca);
                    cond[s][t] = c.cond;
                    int g = WC_INTERIOR;
                    if (k.have_bt() && !one_var) g = warm_guess(c.n_sa, c.n_ca, k.sl0, k.cl0, k.su0, k.cu0);
                    guess[s][t] = g;
                    Vec3<R> f = c.f;
                    T[s][t] = {c.n_sa, c.n_ca, c.n_sb, c.n_cb};
                    limq[s][t] = false;
                    if (g != WC_INTERIOR) {
                        const bool lo = g == WC_LO;
                        const R b_sa = lo ? k.sl0 : k.su0, b_ca = lo ? k.cl0 : k.cu0;
                        const WarmLimit<R> lc = warm_limit(q, k.L, lo, b_sa, b_ca, sgn);
                        limq[s][t] = lc.ok_q; f = lc.f;
                        // the interior candidate's sin/cos are still needed for the admission tests (warm_move below)
                        dA[s][t] = c.n_sa; dB[s][t] = c.n_ca; dB2[s][t] = c.n_sb;      // parked; overwritten below
                        outx0[s][t] = c.n_cb;
                        T[s][t] = {b_sa, b_ca, lc.c_sb, lc.c_cb};
                    }
                    res[t] = xy ? Vec3<R>{f.z, f.y, -f.x} : f;
                }
                for (int t = nv - 1; t >= j0; --t) {          // (descending: T[s][t-1] is read before lane t-1 parks anything)
                    const Trig pv = (t == j0) ? P[s] : T[s][t - 1];
                    Trig in = T[s][t];
                    if (guess[s][t] != WC_INTERIOR) in = {dA[s][t], dB[s][t], dB2[s][t], outx0[s][t]};
                    const WarmMove<R> mv = warm_move(in.sa, in.ca, in.sb, in.cb, pv.sa, pv.ca, pv.sb, pv.cb);
                    dA[s][t] = mv.dA; dB[s][t] = mv.dB; sm_a[s][t] = mv.small_a; sm_b[s][t] = mv.small_b;
                    dB2[s][t] = 0.f; sm_b2[s][t] = false;
                    if (guess[s][t] != WC_INTERIOR) warm_limit_move(T[s][t].sb, T[s][t].cb, pv.sb, pv.cb, dB2[s][t], sm_b2[s][t]);
                    const bool lim = guess[s][t] != WC_INTERIOR;
                    if (s < 3) { acc_v[s][t] = lim ? (guess[s][t] == WC_LO ? k.lb0p : k.ub0p) : mv.dA; acc_k[s][t] = lim ? 0.f : 1.f; }
                    acc_v[3 + s][t] = lim ? dB2[s][t] : mv.dB; acc_k[3 + s][t] = 1.f;
                }
                for (int t = j0; t < nv; ++t) {
                    const Vec3<R> Af = mul(A[t], res[t]);
                    const Vec3<R> np_ = {(piv[t].x + rel[t].x) + Af.x, (piv[t].y + rel[t].y) + Af.y, (piv[t].z + rel[t].z) + Af.z};
                    jw[s][t] = {np_.x + org[t].x, np_.y + org[t].y, np_.z + org[t].z};
                    A[t] = rotate_stage(A[t], s, T[s][t].sa, T[s][t].ca, T[s][t].sb, T[s][t].cb);
                    piv[t] = np_;
                }
            }
            // ---- accumulate in frame order: x = k x + v, one series per lane
            for (int l = 0; l < 7; ++l) {
                R x = acc_x[l][j0];
                for (int t = j0; t < nv; ++t) { x = Num<R>::fma_(acc_k[l][t], x, acc_v[l][t]); acc_x[l][t + 1] = x; }
            }
            // ---- verify
            int fail = nv;
            for (int t = j0; t < nv && fail == nv; ++t) {
                const bool enable_t = (t0 + t > 0) || warm != nullptr;
                for (int s = 0; s < 4; ++s) {
                    const StageConst<R>& k = K[s];
                    const int mode = stage_mode(gn_mask, s);
                    const bool enable = enable_t && (mode & 8) && (mode & 1);
                    const R xp0 = (s < 3) ? acc_x[s][t] : R(0), xp1 = acc_x[3 + s][t];
                    WarmMove<R> mv; mv.dA = dA[s][t]; mv.dB = dB[s][t]; mv.small_a = sm_a[s][t]; mv.small_b = sm_b[s][t];
                    const int wc = warm_case(enable, k.have_bt(), s == 3, xp0, xp1, mv, cond[s][t], k.lb0, k.ub0, k.lb1s, k.ub1s,
                                             guess[s][t], dB2[s][t], sm_b2[s][t], limq[s][t], outx0[s][t], outx1[s][t]);
                    if (wc != guess[s][t]) { fail = t; break; }
                }
            }
            // ---- commit lanes j0 .. fail-1
            for (int t = j0; t < fail; ++t) {
                const int64_t ta = t0 + t;
                for (int s = 0; s < 4; ++s) {
                    if (s != 3) angles[ta * 7 + K[s].ia] = outx0[s][t];
                    angles[ta * 7 + K[s].ib] = outx1[s][t] + K[s].shift;
                    nfev[ta * 4 + s] = 1;
                    put_fk_joint<1>(fk + ta * 27, s, org[t], jw[s][t]);
                }
            }
            if (fail == nv) break;
            // ---- replay lane `fail` through the serial solver, from the previous lane's state
            {
                const int j = fail; const int64_t ta = t0 + j;
                stats[2]++; stats[(ta == 0 && !warm) ? 3 : 4]++;
                const R* kp = pose + ta * 15;
                const Vec3<R> o = {kp[0], kp[1], kp[2]};
                Mat3<R> Aj = {{1.f, 0.f, 0.f}, {0.f, 1.f, 0.f}, {0.f, 0.f, 1.f}};
                Vec3<R> pj = {0.f, 0.f, 0.f};
                for (int s = 0; s < 4; ++s) {
                    const Trig pv = (j == j0) ? P[s] : T[s][j - 1];
                    R x0 = (s < 3) ? acc_x[s][j] : R(0), x1 = acc_x[3 + s][j];
                    R sa = pv.sa, ca = pv.ca, sb = pv.sb, cb = pv.cb, xb;
                    const Vec3<R> kt = {kp[3 * (s + 1)], kp[3 * (s + 1) + 1], kp[3 * (s + 1) + 2]};
                    Vec3<R> w; uint32_t ne = 0u; int worst = ST_GTOL;
                    serial_stage(s, K[s], gn_mask, esc, ta > 0 || warm != nullptr, kt, o, Aj, pj, x0, x1, sa, ca, sb, cb, xb, w, ne, worst);
                    if (s != 3) angles[ta * 7 + K[s].ia] = limit_clamp(x0, K[s].lb0, K[s].ub0);
                    angles[ta * 7 + K[s].ib] = limit_clamp(xb, K[s].lb1, K[s].ub1);
                    nfev[ta * 4 + s] = (int32_t)ne;
                    put_fk_joint<1>(fk + ta * 27, s, o, w);
                    T[s][j] = {sa, ca, sb, cb};
                    if (s < 3) acc_x[s][j + 1] = place1(x0, K[s].lb0, K[s].ub0);
                    acc_x[3 + s][j + 1] = place1(x1, K[s].lb1s, K[s].ub1s);
                }
                for (int s = 0; s < 4; ++s) P[s] = T[s][j];
                j0 = j + 1;
                if (j0 >= nv) break;
            }
        }
        // ---- carry the angles to the next block in the caller's terms (xa = x0, xb = x1 + shift)
        for (int l = 0; l < 7; ++l) xcar[l] = (l >= 3) ? acc_x[l][nv] + K[l - 3].shift : acc_x[l][nv];
    }
}
extern "C" void hostsim_block_f32(const float* pose, int64_t n_frame, const float* prm, const float* warm, float* angles,
                                  float* fk, int32_t* nfev, int gn_mask, int64_t* stats) {
    run_block(pose, n_frame, prm, warm, angles, fk, nfev, gn_mask, stats);
}

// ---- generic 7-DOF solve (csrc/seqik_generic.cuh): pose (N,2,3) = ThC origin + claw per frame; prm = 32-float row
// (seg 0..3, lb 4..10, ub 11..17, seed 18..24, null_sq 25; joints in generic chain order).  teacher: NULL, or (N,7)
// seeds that replace the warm start of every frame (teacher-forced single solves).
template <typename R>
static void run_generic(const R* pose, int64_t n_frame, const R* prm, const R* teacher, R* angles, R* fk,
                        int32_t* nfev, int32_t* status) {
    GenericSolve<R> S;
    for (int i = 0; i < 7; ++i) S.x[i] = prm[18 + i];
    for (int64_t t = 0; t < n_frame; ++t) {
        const R* p = pose + t * 6;
        if (teacher) for (int i = 0; i < 7; ++i) S.x[i] = teacher[t * 7 + i];
        S.start(prm, Vec3<R>{p[3] - p[0], p[4] - p[1], p[5] - p[2]}, prm[25]);
        while (!S.done()) S.trip();
        for (int i = 0; i < 7; ++i) angles[t * 7 + i] = S.x[i];
        nfev[t] = S.nfev; status[t] = S.status;
        if (fk) {
            Vec3<R> org[3], claw;
            S.joints(org, &claw);
            R* o = fk + t * 27;
            for (int r = 0; r < 4; ++r) { o[3 * r] = p[0]; o[3 * r + 1] = p[1]; o[3 * r + 2] = p[2]; }
            const Vec3<R> rows[5] = {org[0], org[0], org[1], org[2], claw};
            for (int r = 0; r < 5; ++r) { o[12 + 3 * r] = rows[r].x + p[0]; o[13 + 3 * r] = rows[r].y + p[1]; o[14 + 3 * r] = rows[r].z + p[2]; }
        }
    }
}

// n independent single solves, each with its own constants row prm (n,32) (seed from 18..24), target (n,3) as the kernel
// forms it (key point minus origin, already rounded) -> angles (n,7), fk rows relative to the origin (n,9,3), nfev, status
template <typename R>
static void run_generic_solves(int64_t n, const R* prm, const R* target, R* angles, R* fk, int32_t* nfev, int32_t* status) {
    for (int64_t k = 0; k < n; ++k) {
        const R* pk = prm + k * 32;
        GenericSolve<R> S;
        for (int i = 0; i < 7; ++i) S.x[i] = pk[18 + i];
        S.start(pk, Vec3<R>{target[3 * k], target[3 * k + 1], target[3 * k + 2]}, pk[25]);
        while (!S.done()) S.trip();
        for (int i = 0; i < 7; ++i) angles[k * 7 + i] = S.x[i];
        nfev[k] = S.nfev; status[k] = S.status;
        Vec3<R> org[3], claw;
        S.joints(org, &claw);
        R* o = fk + k * 27;
        for (int r = 0; r < 12; ++r) o[r] = R(0);
        const Vec3<R> rows[5] = {org[0], org[0], org[1], org[2], claw};
        for (int r = 0; r < 5; ++r) { o[12 + 3 * r] = rows[r].x; o[13 + 3 * r] = rows[r].y; o[14 + 3 * r] = rows[r].z; }
    }
}

extern "C" {
void hostsim_generic_f32(const float* pose, int64_t n_frame, const float* prm, const float* teacher, float* angles,
                         float* fk, int32_t* nfev, int32_t* status) {
    run_generic<float>(pose, n_frame, prm, teacher, angles, fk, nfev, status);
}
void hostsim_generic_f64(const double* pose, int64_t n_frame, const double* prm, const double* teacher, double* angles,
                         double* fk, int32_t* nfev, int32_t* status) {
    run_generic<double>(pose, n_frame, prm, teacher, angles, fk, nfev, status);
}
void hostsim_generic_solves_f32(int64_t n, const float* prm, const float* target, float* angles, float* fk, int32_t* nfev,
                                int32_t* status) {
    run_generic_solves<float>(n, prm, target, angles, fk, nfev, status);
}
void hostsim_generic_solves_f64(int64_t n, const double* prm, const double* target, double* angles, double* fk,
                                int32_t* nfev, int32_t* status) {
    run_generic_solves<double>(n, prm, target, angles, fk, nfev, status);
}
}

// ---- self-checks of refactors that are otherwise only visible on the GPU: the select-based frame rotation equals the
// branching one bit for bit, and restart() equals its three pieces.  Returns the number of mismatches.
extern "C" int hostsim_selfcheck(const float* rnd, int n) {
    int bad = 0;
    for (int i = 0; i + 16 <= n; i += 16) {
        const float* r = rnd + i;
        const Mat3<float> A = {{r[0], r[1], r[2]}, {r[3], r[4], r[5]}, {r[6], r[7], r[8]}};
        for (int kind = 0; kind < 2; ++kind) {
            const Mat3<float> X = rotate_frame(A, kind, r[9], r[10], r[11], r[12]);
            const Mat3<float> Y = rotate_frame_sel(A, kind, r[9], r[10], r[11], r[12]);
            const float* x = &X.c0.x; const float* y = &Y.c0.x;
            for (int k = 0; k < 9; ++k) bad += !(x[k] == y[k]);
        }
        for (int fresh = 0; fresh < 2; ++fresh) {
            StageSolve<float> S1, S2;
            const Vec3<float> q0 = {0.3f * r[0], 0.3f * r[1], -0.4f + 0.1f * r[2]};
            S1.init(KIND_ZY, 0.4f, 1.f, q0, 0.2f * r[3], -0.8f + 0.2f * r[4], -1.f, 1.f, -2.f, 0.f, 1.5f, 6, 15);
            while (!S1.done()) S1.trip();
            S2 = S1;
            const Vec3<float> q1 = {q0.x + 0.02f * r[5], q0.y + 0.02f * r[6], q0.z + 0.02f * r[7]};
            S1.restart(q1, -1.f, 1.f, -2.f, 0.f, fresh != 0, true);
            const Vec3<float> q = S2.restart_a(q1, -1.f, 1.f, -2.f, 0.f, fresh != 0);
            S2.warm_step(q, -1.f, 1.f, -2.f - S2.shift, 0.f - S2.shift, S2.closed_form && S2.gn_mode);
            S2.restart_b(q, -1.f, 1.f, -2.f, 0.f);
            bad += !(S1.x0 == S2.x0 && S1.x1 == S2.x1 && S1.status == S2.status && S1.cost == S2.cost && S1.sa == S2.sa && S1.cb == S2.cb);
        }
    }
    return bad;
}

// ---- the closed-form warm step on its own: a Rz(a) Ry(b) stage (two variables, or one with has_a = 0) carried at
// (a, b) meets target q; out = (a', b', seeded, seed_at, cost at the new point).
extern "C" void hostsim_warm_step_f64(double L, double has_a, const double* ab, const double* q, const double* lbub, double* out) {
    StageSolve<double> S;
    S.set_problem(KIND_ZY, L, has_a, 1.0, 6, 15);
    S.set_limit_trig(lbub[0], lbub[1]);
    S.set_iterate(ab[0], ab[1]);
    const Vec3<double> qq = {q[0], q[1], q[2]};
    S.restart(qq, lbub[0], lbub[1], lbub[2], lbub[3], true, true);
    out[0] = S.x0; out[1] = S.angle_b(); out[2] = S.seeded ? 1.0 : 0.0; out[3] = S.seed_at; out[4] = S.cost;
}

// ---- one solve step on its own: init at (a, b) against q, then `n_trip` evaluations; out = (a', b', cost, nfev, status)
extern "C" void hostsim_trips_f64(double L, const double* ab, const double* q, const double* lbub, int mode, int n_trip, double* out) {
    StageSolve<double> S;
    const Vec3<double> qq = {q[0], q[1], q[2]};
    S.init(KIND_ZY, L, 1.0, qq, ab[0], ab[1], lbub[0], lbub[1], lbub[2], lbub[3], 1.0, 6, mode);
    for (int i = 0; i < n_trip && !S.done(); ++i) S.trip();
    out[0] = S.x0; out[1] = S.angle_b(); out[2] = S.cost; out[3] = S.nfev; out[4] = S.status;
}
