// seqik_block.cuh -- building blocks of the frame-parallel ("block") schedule of the sequential leg-IK solver.
//
// Why frames can run in parallel at all.  The reference's frame loop is serial because every solve is warm-started
// from the previous frame's solution (seqikpy/leg_inverse_kinematics.py:272).  With the closed-form warm step
// (StageSolve::warm_step, seqik_core.cuh) a carried solve usually ENDS at the point of the sphere |w| = L nearest to the
// new target, on the warm start's branch -- and that point is a function of the frame's own target and of ONE bit of
// history (the sign of sin b).  What the previous frame still contributes is small and cheap:
//   (1) the sin/cos of its solution: the new angles are the old ones plus the small rotation between the two (deltas),
//   (2) the accumulated angles themselves: the strictly-inside-the-box admission tests and the reported values,
//   (3) the decision between the interior minimiser and the one with the first angle on a limit.
// So a warp takes 32 consecutive frames of one chain, lane = frame, all four stages in the lane:
//   pass        every lane computes its closed-form candidates from its own key points (speculating (3) from the
//               candidate's direction relative to the limits), its end point, frame rotation and forward kinematics;
//               the previous lane's sin/cos arrive by shuffle and give the deltas of (1);
//   accumulate  seven lanes add the deltas up in FRAME ORDER, one angle series each (x = k x + v: v = delta, k = 1;
//               for a frame on a limit v = that limit, k = 0) -- the same float additions the serial solver performs;
//   verify      every lane re-evaluates warm_step's admission tests with the exact accumulated angles of (2);
//   replay      the first lane whose speculation does not hold runs the frame through the serial solver
//               (StageSolve::restart / trip / escape: iterating solves, first frame of a recording, near-singular
//               targets, ...), hands its final state on, and the lanes after it are recomputed.
// Every lane that commits has taken exactly the decisions and performed exactly the float operations of the serial
// carried solve (tests/hostsim run_carried, leg_solve_pipe_kernel), so results are BIT-IDENTICAL to schedule 2; the
// functions below restate warm_step() piecewise and are pinned to it by tests/test_host_core.py (host emulation of this
// schedule against the serial one) and tests/test_gpu_parity.py (kernel against kernel).
// The per-stage constants (stage_const), the serial stage step of the replay and of the first frame (serial_stage), the
// frame rotation (rotate_stage) and the forward-kinematics rows (put_fk_joint) below are the kernels' code and the host
// emulation's (tests/hostsim run_block) alike, so the CPU suite compiles and runs the same arithmetic as the GPU.
#pragma once
#include "seqik_core.cuh"

namespace seqik {

// make_strictly_feasible of one variable, exactly as StageSolve::place does it (a value ON a bound moves 1e-10 inside)
template <typename R> SK_HD R place1(R x, R lb, R ub) {
    typedef Num<R> N;
    R dl = x - lb, du = ub - x;
    const R rs = R(1e-10);
    if (dl <= R(0)) { dl = rs * N::max_(R(1), N::abs_(lb)); x = lb + dl; du = (ub - lb) - dl; }
    if (du <= R(0)) { du = rs * N::max_(R(1), N::abs_(ub)); x = ub - du; }
    return x;
}

template <typename R> SK_HD R asin_small_(R s) { return StageSolve<R>::asin_small(s); }
template <typename R> SK_HD R ws_hs_max_() { return StageSolve<R>::ws_hs_max(); }

// ---- warm_step(), piece 1: the interior candidate -- the point of the sphere nearest to the target q (already mapped into
// the Rz Ry form), on the branch `sgn` of the warm start.  (sa, ca): the warm start's first-angle trigonometry, used by the
// one-variable stage only.  `cond`: the admission tests that depend on the target alone.
template <typename R> struct WarmCand { R n_sa, n_ca, n_sb, n_cb; Vec3<R> f; bool cond; };
template <typename R> SK_HD WarmCand<R> warm_interior(const Vec3<R>& q, R L, bool one_var, R sgn, R sa, R ca) {
    typedef Num<R> N;
    WarmCand<R> c;
    const R rho2 = one_var ? q.x * q.x : N::fma_(q.y, q.y, q.x * q.x);
    const R qn2 = N::fma_(q.z, q.z, rho2);
    const R rn = N::rsqrt_(qn2), rr = N::rsqrt_(rho2);
    const R t_ = sgn * rr;
    c.n_sb = one_var ? -(q.x * rn) : sgn * (rho2 * rr) * rn; c.n_cb = -(q.z * rn);
    c.n_ca = one_var ? ca : -(q.x * t_); c.n_sa = one_var ? sa : -(q.y * t_);
    c.cond = (one_var | (rho2 > R(0.01) * qn2)) & (qn2 > R(0.25) * L * L) & (qn2 < N::inf());
    const R k = N::fma_(L, rn, R(-1));
    c.f = {q.x * k, one_var ? -q.y : q.y * k, q.z * k};
    return c;
}

// ---- piece 2: the move from the warm start (sa, ca, sb, cb) to a candidate: angle increments by the half-angle form
template <typename R> struct WarmMove { R dA, dB; bool small_a, small_b; };
template <typename R> SK_HD WarmMove<R> warm_move(R n_sa, R n_ca, R n_sb, R n_cb, R sa, R ca, R sb, R cb) {
    typedef Num<R> N;
    WarmMove<R> m;
    const R sda = N::fma_(n_sa, ca, -(n_ca * sa)), cda = N::fma_(n_ca, ca, n_sa * sa);
    const R sdb = N::fma_(n_sb, cb, -(n_cb * sb)), cdb = N::fma_(n_cb, cb, n_sb * sb);
    const R hsa = sda * N::rsqrt_(R(2) + R(2) * cda), hsb = sdb * N::rsqrt_(R(2) + R(2) * cdb);
    m.dA = R(2) * asin_small_(hsa); m.dB = R(2) * asin_small_(hsb);
    m.small_a = (N::abs_(hsa) < ws_hs_max_<R>()) & (cda > R(0)); m.small_b = (N::abs_(hsb) < ws_hs_max_<R>()) & (cdb > R(0));
    return m;
}

// ---- piece 3: the candidate with the first angle ON a limit (lo: the lower one).  (b_sa, b_ca) = sin/cos of that limit.
// `ok_q`: the admission tests that depend on the target alone (branch, conditioning in the plane, KKT sign).
template <typename R> struct WarmLimit { R c_sb, c_cb; Vec3<R> f; bool ok_q; };
template <typename R> SK_HD WarmLimit<R> warm_limit(const Vec3<R>& q, R L, bool lo, R b_sa, R b_ca, R sgn) {
    typedef Num<R> N;
    WarmLimit<R> c;
    const R qe = N::fma_(q.y, b_sa, q.x * b_ca), pn2 = N::fma_(q.z, q.z, qe * qe);
    const R rp = N::rsqrt_(pn2);
    c.c_sb = -(qe * rp); c.c_cb = -(q.z * rp);
    const R ga = c.c_sb * N::fma_(b_ca, q.y, -(b_sa * q.x));
    const bool kkt = lo ? (ga > R(0)) : (ga < R(0));
    c.ok_q = (c.c_sb * sgn > R(0.1)) & (pn2 > R(0.25) * L * L) & (pn2 < N::inf()) & kkt;
    const R Lsb_c = L * c.c_sb;
    c.f = {-(Lsb_c * b_ca) - q.x, -(Lsb_c * b_sa) - q.y, -(L * c.c_cb) - q.z};
    return c;
}
template <typename R> SK_HD void warm_limit_move(R c_sb, R c_cb, R sb, R cb, R& dB2, bool& small_b2) {
    typedef Num<R> N;
    const R sdb2 = N::fma_(c_sb, cb, -(c_cb * sb)), cdb2 = N::fma_(c_cb, cb, c_sb * sb);
    const R hsb2 = sdb2 * N::rsqrt_(R(2) + R(2) * cdb2);
    dB2 = R(2) * asin_small_(hsb2);
    small_b2 = (N::abs_(hsb2) < ws_hs_max_<R>()) & (cdb2 > R(0));
}

// ---- speculation of the case from the candidate's direction alone: 1 / 2 when it lies just outside the lower / upper
// limit of the first angle, else 0 (interior).  Only a guess -- warm_case() below decides with the exact angles.
enum : int { WC_INTERIOR = 0, WC_LO = 1, WC_HI = 2, WC_STAYS = 3, WC_NONE = -1 };   // WC_STAYS: one-variable stage parked on a limit (block kernel)
template <typename R> SK_HD int warm_guess(R n_sa, R n_ca, R sl0, R cl0, R su0, R cu0) {
    typedef Num<R> N;
    const R s_lo = N::fma_(n_sa, cl0, -(n_ca * sl0)), c_lo = N::fma_(n_ca, cl0, n_sa * sl0);   // sin / cos (a - lb)
    const R s_hi = N::fma_(su0, n_ca, -(cu0 * n_sa)), c_hi = N::fma_(cu0, n_ca, su0 * n_sa);   // sin / cos (ub - a)
    const bool below = (c_lo > R(0.5)) & (s_lo <= R(1e-5)), above = (c_hi > R(0.5)) & (s_hi <= R(1e-5));
    return (below == above) ? WC_INTERIOR : below ? WC_LO : WC_HI;
}

// ---- piece 4: the decision warm_step() takes, given the exact placed warm-start angles (xp0, xp1).  `guess`: the case the
// candidate data (dB2, small_b2, lim_ok_q) was prepared for.  Returns WC_INTERIOR / WC_LO / WC_HI when the serial solver ends
// at that candidate, WC_NONE when it would not (or when it would take a limit the data was not prepared for): the caller
// then runs the frame through the serial solver.  x0 / x1: the solve's final angles in that case.
template <typename R>
SK_HD int warm_case(bool enable, bool have_bt, bool one_var, R xp0, R xp1, const WarmMove<R>& mv, bool cond,
                    R lb0, R ub0, R lb1s, R ub1s, int guess, R dB2, bool small_b2, bool lim_ok_q, R& x0, R& x1) {
    typedef Num<R> N;
    const R m = R(1e-5);
    const R nx0 = xp0 + mv.dA, nx1 = xp1 + mv.dB;
    const bool in_a = (nx0 - lb0 > m) & (ub0 - nx0 > m), in_b = (nx1 - lb1s > m) & (ub1s - nx1 > m);
    const bool ok = enable & mv.small_a & mv.small_b & cond & in_a & in_b;
    x0 = nx0; x1 = nx1;
    if (ok) return WC_INTERIOR;
    const bool below = nx0 - lb0 <= m, above = ub0 - nx0 <= m;
    if (!(enable & have_bt & !one_var & (below != above) & mv.small_a)) return WC_NONE;
    const bool lo = below;
    if (guess != (lo ? WC_LO : WC_HI)) return WC_NONE;
    const R b_x0 = lo ? lb0 : ub0;
    const R cx1 = xp1 + dB2;
    const bool ok_b = (N::abs_(b_x0 - xp0) < StageSolve<R>::ws_move_max()) & small_b2 & lim_ok_q & (cx1 - lb1s > m) & (ub1s - cx1 > m);
    x0 = b_x0; x1 = cx1;
    return ok_b ? (lo ? WC_LO : WC_HI) : WC_NONE;
}

// ---- the constants of one (chain, stage), derived from the chain's 32-float parameter row (include/seqik.h: segment
// lengths 0..3, lower / upper limits 4..10 / 11..17, seed 18..24, null_sq 25..28).  SerialConst: what serial_stage() reads.
// It stays these ten floats: the robust block kernel hands them to its out-of-line serial_stage_call through memory.
template <typename R> struct SerialConst {
    R L, lb0, ub0, lb1, ub1;            // segment length, limits of the first / second angle in the caller's terms
    R sl0, cl0, su0, cu0;               // sin/cos of the first angle's limits (all zero without both: warm_guess says interior)
    R nsq;                              // squared norm of the inert slots (StageSolve::null_sq)
    SK_HD bool have_bt() const { return lb0 > -Num<R>::inf() && ub0 < Num<R>::inf(); }
};
template <typename R> struct StageConst : SerialConst<R> {
    int ia, ib;                         // row indices of the first / second angle (stage 4 has one: ia = ib = 6)
    R shift;                            // stage 1 is solved in the Rz Ry form: second angle x1 = b - pi/2
    R lb1s, ub1s;                       // second angle's limits in that form
    R lb0p, ub0p;                       // the first angle's limits as place1 leaves them (the value of a frame on a limit)
};
template <typename R> SK_HD R ld_param(const R* p) {
#if defined(__CUDA_ARCH__)
    return __ldg(p);
#else
    return *p;
#endif
}
template <typename R> SK_HD StageConst<R> stage_const(const R* prm, int s) {
    typedef Num<R> N;
    const R inf = N::inf();
    StageConst<R> k;
    k.ia = 2 * s; k.ib = (s == 3) ? 6 : 2 * s + 1;
    k.shift = (s == 0) ? R(1.57079632679489661923) : R(0);
    k.lb0 = (s == 3) ? -inf : ld_param(prm + 4 + k.ia); k.ub0 = (s == 3) ? inf : ld_param(prm + 11 + k.ia);
    k.lb1 = ld_param(prm + 4 + k.ib); k.ub1 = ld_param(prm + 11 + k.ib);
    k.L = ld_param(prm + s); k.nsq = ld_param(prm + 25 + s);
    k.lb1s = k.lb1 - k.shift; k.ub1s = k.ub1 - k.shift;
    k.sl0 = k.cl0 = k.su0 = k.cu0 = R(0);
    R v_;
    if (k.have_bt()) { N::sincosv_(k.lb0, &k.sl0, &k.cl0, &v_); N::sincosv_(k.ub0, &k.su0, &k.cu0, &v_); }
    k.lb0p = place1(k.lb0, k.lb0, k.ub0); k.ub0p = place1(k.ub0, k.lb0, k.ub0);
    return k;
}

// ---- A <- A Rot_a(a) Ry(b) of stage s, from the sin/cos of its iterate in the Rz Ry form (stage 1: b = x1 + pi/2, so
// sin b = cos x1 and cos b = -sin x1, as StageSolve::sin_b / cos_b)
template <typename R> SK_HD Mat3<R> rotate_stage(const Mat3<R>& A, int s, R sa, R ca, R sb, R cb) {
    const bool xy = s == 0;
    return rotate_frame_sel(A, xy ? KIND_XY : KIND_ZY, sa, ca, xy ? cb : sb, xy ? -sb : cb);
}

// ---- the forward-kinematics rows of stage s's joint w in one leg-frame.  kFk 1, nine rows: 0-3 the origin o, 4 repeats 5,
// 5 + s the joint of stage s (stage s writes rows s and 5 + s, stage 1 also row 4).  kFk 2, the joints only: row s.
template <int kFk, typename R> SK_HD void put_fk_joint(R* fk, int s, const Vec3<R>& o, const Vec3<R>& w) {
    if (kFk == 1) {
        fk[3 * s] = o.x; fk[3 * s + 1] = o.y; fk[3 * s + 2] = o.z;
        fk[15 + 3 * s] = w.x; fk[16 + 3 * s] = w.y; fk[17 + 3 * s] = w.z;
        if (s == 0) { fk[12] = w.x; fk[13] = w.y; fk[14] = w.z; }
    } else if (kFk == 2) { fk[3 * s] = w.x; fk[3 * s + 1] = w.y; fk[3 * s + 2] = w.z; }
}

// ---- one stage of one frame through the serial solver, exactly as run_carried / leg_solve_pipe_kernel run it for a carried
// solve: the iterate (x0, x1: placed angles; sa..cb: their sin/cos) meets the target kt in the frame (A, piv) the earlier
// stages of this frame built.  On return the iterate is the solve's final one, (A, piv) are those of the next stage, w is the
// joint position, xb_out the second angle in the caller's terms.  The replay of the block kernel, the first-frame kernel and
// the host emulation of the schedule run this code.
template <typename R>
SK_HD void serial_stage(int s, const SerialConst<R>& k, int gn_mask, bool esc, bool warm_ok, const Vec3<R>& kt, const Vec3<R>& o,
                        Mat3<R>& A, Vec3<R>& piv, R& x0, R& x1, R& sa, R& ca, R& sb, R& cb, R& xb_out, Vec3<R>& w,
                        uint32_t& nfev, int& worst) {
    StageSolve<R> S;
    S.set_problem(s == 0 ? KIND_XY : KIND_ZY, k.L, s == 3 ? R(0) : R(1), k.nsq, (s == 0) ? 4 : (s == 1) ? 6 : (s == 2) ? 8 : 9, stage_mode(gn_mask, s));
    S.sl0 = k.sl0; S.cl0 = k.cl0; S.su0 = k.su0; S.cu0 = k.cu0;
    S.have_bt = k.have_bt();
    S.x0 = x0; S.x1 = x1; S.sa = sa; S.ca = ca; S.sb = sb; S.cb = cb;
    const Vec3<R> rel = {(kt.x - o.x) - piv.x, (kt.y - o.y) - piv.y, (kt.z - o.z) - piv.z};
    const Vec3<R> q3 = mulT(A, rel);
    S.restart(q3, k.lb0, k.ub0, k.lb1, k.ub1, false, warm_ok);
    for (;;) {
        while (!S.done()) S.trip();
        if (!(esc && S.escape())) break;
    }
    nfev += (uint32_t)S.nfev;
    worst = (S.status == ST_MAXFEV && worst > ST_MAXFEV) ? ST_MAXFEV : worst;
    worst = (S.status == ST_NONFINITE) ? ST_NONFINITE : worst;
    const Vec3<R> Af = mul(A, S.res());
    const Vec3<R> np_ = {(piv.x + rel.x) + Af.x, (piv.y + rel.y) + Af.y, (piv.z + rel.z) + Af.z};
    w = {np_.x + o.x, np_.y + o.y, np_.z + o.z};
    A = rotate_stage(A, s, S.sa, S.ca, S.sb, S.cb);
    piv = np_;
    x0 = S.x0; x1 = S.x1; sa = S.sa; ca = S.ca; sb = S.sb; cb = S.cb; xb_out = S.angle_b();
}

}  // namespace seqik
