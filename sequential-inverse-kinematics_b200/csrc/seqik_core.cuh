// seqik_core.cuh -- per-lane solver core of the sequential leg-IK path.
//
// One "stage solve" of SeqIKPy (reference: seqikpy/leg_inverse_kinematics.py:259-282,
// ikpy Chain.inverse_kinematics -> scipy.optimize.least_squares, method "trf") is a
// bounded nonlinear least-squares problem with 3 residuals and at most TWO variables
// that move the end point (SURVEY.md 3.2/3.4): every other chain slot (Base link,
// frozen links, the last link) has an identically-zero Jacobian column.
//
// This header restates scipy's Trust-Region-Reflective iteration
// (scipy/optimize/_lsq/trf.py:206-413, common.py) on that active pair, in the pivot
// frame of the stage, so that the whole solve is closed-form scalar arithmetic that
// lives in registers:
//   * in the pivot frame the two Jacobian columns are ORTHOGONAL (ja.jb = 0, |jb| = L,
//     |ja| = L |cos b| or L |sin b|), so J^T J + diag is diagonal and the SVD of the
//     augmented Jacobian (trf.py:296-303) is the identity: no 2x2 eigen-solve;
//   * the inert slots enter only through `null_sq` (their squared norm: initial trust
//     radius trf.py:236 and the xtol test common.py:705-718) and `max_nfev = 100 n`;
//   * m = 3 < n always, so solve_lsq_trust_region (common.py:57-168) always takes its
//     rank-deficient branch -- restated literally, including the final rescale of the
//     step to the trust radius and the Levenberg parameter carried between iterations.
//
// FP32 specifics (none change the FP64 instantiation's results beyond rounding):
//   * distances to the bounds (dl, du) are carried as separate scalars and updated
//     incrementally, so Coleman-Li scaling near an active bound keeps full relative
//     accuracy (scipy iterates sit 1e-14 inside the bounds);
//   * a trial point is evaluated through the angle-addition form (sin/cos/versine of the
//     STEP), which yields the change of the end point, hence the actual cost reduction,
//     with relative accuracy ~1e-6 even when it is 1e-9 of the cost (ftol = 1e-8);
//   * device arithmetic: reciprocal / square root through the SFU approximations
//     (rcp/sqrt/rsqrt.approx, <= 2 ulp), sin/cos by an in-line Cody-Waite reduction valid for
//     |x| <= 2 pi (all angles are bounded by the joint limits), multiply-adds written as
//     explicit fma so that every kernel that includes this header rounds identically
//     (the library is compiled with -fmad=false).
//
// One trip() = one function evaluation.  Nothing is kept between trips except the iterate:
// the scaling / model quantities are recomputed from it (they are cheap and it makes a trip
// one straight-line block, which is what a warp of lanes at different positions needs).
//
// On top of that restatement (flags of include/seqik.h, all optional, see DESIGN.md 2):
//   * Newton steps (plan()): the residual-curvature term of the two-angle segment is closed
//     form, so the Newton step of the same scaled model is a 2x2 solve -- taken where the full
//     Hessian is safely positive definite and the step is admissible, else the step above;
//   * closed-form warm step (warm_step()): a stage points a segment at its target, so the
//     box-free minimiser is the point of the sphere |w| = L nearest to the target (on the
//     warm start's branch), and with the first angle on a limit it is the nearest point of a
//     circle; for the next frame of a carried solve the iterate is moved there when that is a
//     short, interior, well-conditioned move and the solve ends with that one evaluation.
// The reference's own iterates are what runs when the flags are off and wherever the
// admission tests fail.
//
// The same header is compiled by nvcc for the kernels and by g++ for the host-side
// test harness in tests/hostsim (test infrastructure; never loaded by the product).
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define SK_HD __host__ __device__ __forceinline__
#define SK_HD_COLD __host__ __device__ __noinline__     // rare paths: one out-of-line copy instead of one per call site
#else
#define SK_HD inline
#define SK_HD_COLD inline
#endif

namespace seqik {

// ---------------------------------------------------------------------------------
// scalar helpers
// ---------------------------------------------------------------------------------
template <typename R> struct Num;
template <> struct Num<float> {
    static SK_HD float fma_(float a, float b, float c) { return fmaf(a, b, c); }
    static SK_HD float abs_(float x) { return fabsf(x); }
    static SK_HD float max_(float a, float b) { return fmaxf(a, b); }
    static SK_HD float min_(float a, float b) { return fminf(a, b); }
    static SK_HD float copysign_(float a, float b) { return copysignf(a, b); }
    static SK_HD float rcp_(float x) {
#if defined(__CUDA_ARCH__)
        float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r;
#else
        return 1.0f / x;
#endif
    }
    static SK_HD float sqrt_(float x) {
#if defined(__CUDA_ARCH__)
        float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r;
#else
        return sqrtf(x);
#endif
    }
    static SK_HD float rsqrt_(float x) {
#if defined(__CUDA_ARCH__)
        float r; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r;
#else
        return 1.0f / sqrtf(x);
#endif
    }
    // sin, cos and versine (1 - cos) of x, |x| <= 2 pi: quadrant reduction + minimax polynomials on
    // [-pi/4, pi/4]; the versine keeps full relative accuracy for tiny x (no 1 - cos cancellation).
    static SK_HD void sincosv_(float x, float* s, float* c, float* v) {
        if (fabsf(x) < 0.78f) {          // quadrant 0 (the usual case for a STEP): same polynomials, no reduction
            const float z = x * x;
            float sp = fmaf(z, -1.9515295891e-4f, 8.3321608736e-3f);
            sp = fmaf(sp, z, -1.6666654611e-1f);
            float cp = fmaf(z, 2.443315711809948e-5f, -1.388731625493765e-3f);
            cp = fmaf(cp, z, 4.166664568298827e-2f);
            *s = fmaf(sp * z, x, x);
            *v = fmaf(-cp * z, z, 0.5f * z);
            *c = 1.0f - *v;
            return;
        }
        const float kf = rintf(x * 0.636619772367581343f);                 // x * 2/pi
        float r = fmaf(kf, -1.57079601287841796875f, x);                   // Cody-Waite, pi/2 = hi + mid + lo
        r = fmaf(kf, -3.1391647326017846e-07f, r);
        r = fmaf(kf, -5.390302529957764e-15f, r);
        const float z = r * r;
        float sp = fmaf(z, -1.9515295891e-4f, 8.3321608736e-3f);
        sp = fmaf(sp, z, -1.6666654611e-1f);
        const float sn = fmaf(sp * z, r, r);                               // sin r
        float cp = fmaf(z, 2.443315711809948e-5f, -1.388731625493765e-3f);
        cp = fmaf(cp, z, 4.166664568298827e-2f);
        const float vr = fmaf(-cp * z, z, 0.5f * z);                       // 1 - cos r = z/2 - z^2 (...)
        const float cs = 1.0f - vr;                                        // cos r
        const int q = ((int)kf) & 3;
        const float ss = (q & 1) ? cs : sn, cc = (q & 1) ? sn : cs;
        *s = (q & 2) ? -ss : ss;
        *c = ((q + 1) & 2) ? -cc : cc;
        *v = (q == 0) ? vr : 1.0f - *c;
    }
    // the same for two angles at once: ONE branch for the pair (both in quadrant 0, the usual case for a step), and the
    // two polynomial chains in one basic block so that they interleave.  Bitwise equal to two sincosv_ calls.
    static SK_HD void sincosv2_(float x, float y, float* sx, float* cx, float* vx, float* sy, float* cy, float* vy) {
        if (fmaxf(fabsf(x), fabsf(y)) < 0.78f) {
            const float zx = x * x, zy = y * y;
            float spx = fmaf(zx, -1.9515295891e-4f, 8.3321608736e-3f), spy = fmaf(zy, -1.9515295891e-4f, 8.3321608736e-3f);
            spx = fmaf(spx, zx, -1.6666654611e-1f); spy = fmaf(spy, zy, -1.6666654611e-1f);
            float cpx = fmaf(zx, 2.443315711809948e-5f, -1.388731625493765e-3f), cpy = fmaf(zy, 2.443315711809948e-5f, -1.388731625493765e-3f);
            cpx = fmaf(cpx, zx, 4.166664568298827e-2f); cpy = fmaf(cpy, zy, 4.166664568298827e-2f);
            *sx = fmaf(spx * zx, x, x); *sy = fmaf(spy * zy, y, y);
            *vx = fmaf(-cpx * zx, zx, 0.5f * zx); *vy = fmaf(-cpy * zy, zy, 0.5f * zy);
            *cx = 1.0f - *vx; *cy = 1.0f - *vy;
            return;
        }
        sincosv_(x, sx, cx, vx); sincosv_(y, sy, cy, vy);
    }
    static SK_HD float inf() { return INFINITY; }
    static SK_HD float tiny() { return 1.17549435e-38f; }     // stands in for nextafter(0, .)
    static SK_HD float eps_in() { return 2.220446e-16f; }     // fp64 ulp: strict-feasibility gap
};
template <> struct Num<double> {
    static SK_HD double fma_(double a, double b, double c) { return fma(a, b, c); }
    static SK_HD double abs_(double x) { return fabs(x); }
    static SK_HD double max_(double a, double b) { return fmax(a, b); }
    static SK_HD double min_(double a, double b) { return fmin(a, b); }
    static SK_HD double copysign_(double a, double b) { return copysign(a, b); }
    static SK_HD double rcp_(double x) { return 1.0 / x; }
    static SK_HD double sqrt_(double x) { return sqrt(x); }
    static SK_HD double rsqrt_(double x) { return 1.0 / sqrt(x); }
    static SK_HD void sincosv_(double x, double* s, double* c, double* v) {
        *s = sin(x); *c = cos(x);
        const double h = sin(0.5 * x);
        *v = 2.0 * h * h;
    }
    static SK_HD void sincosv2_(double x, double y, double* sx, double* cx, double* vx, double* sy, double* cy, double* vy) {
        sincosv_(x, sx, cx, vx); sincosv_(y, sy, cy, vy);
    }
    static SK_HD double inf() { return (double)INFINITY; }
    static SK_HD double tiny() { return 4.9406564584124654e-324; }
    static SK_HD double eps_in() { return 2.220446049250313e-16; }
};

constexpr int SEQIK_RESYNC = 32;
// StageSolve mode of stage s (0..3) from the solver flags (include/seqik.h): bit 0 Gauss-Newton mode of that stage,
// bit 1 skip-confirm, bit 2 Newton steps, bit 3 closed-form warm step
inline
#if defined(__CUDACC__)
__host__ __device__
#endif
int stage_mode(int flags, int s) { return ((flags >> s) & 1) | (((flags >> 5) & 1) << 1) | (((flags >> 6) & 1) << 2) | (((flags >> 7) & 1) << 3); }
          // frames between full re-initialisations of a carried solve

enum : int { KIND_XY = 0, KIND_ZY = 1 };   // Rx(a)Ry(b) (stage 1)  |  Rz(a)Ry(b) (stages 2-4)

enum : int {
    ST_MAXFEV = 0, ST_GTOL = 1, ST_FTOL = 2, ST_XTOL = 3, ST_BOTH = 4, ST_RUNNING = -1,
    ST_NONFINITE = -2      // residual not finite at the start of a solve (scipy raises there): the solve is skipped
};

// An angle is written out clamped to its limits.  The iterate itself can sit one float32 ulp (or, on a limit at 0, one
// FLT_MIN) outside the box: the bound distances are carried as separate scalars and x + step rounds on its own.  A value
// outside a limit, and that limit itself, both re-enter the next solve through place()'s nudge to the same point, so the
// clamp changes no later iterate.  NaN passes through.  The clamp also hides how far an iterate left the box: the tests
// see the iterate before the clamp through the host build (FrameStats::iterate, tests/test_stage_model_cpu.py).
template <typename R> SK_HD R limit_clamp(R x, R lo, R hi) { return x < lo ? lo : (x > hi ? hi : x); }

template <typename R> struct Vec3 { R x, y, z; };
template <typename R> SK_HD R dot(const Vec3<R>& a, const Vec3<R>& b) {
    return Num<R>::fma_(a.z, b.z, Num<R>::fma_(a.y, b.y, a.x * b.x));
}

// ---------------------------------------------------------------------------------
// One stage solve: the iterate + one evaluation per trip()
// ---------------------------------------------------------------------------------
// Internally every stage is solved in the Rz(a) Ry(b) form.  Stage 1 (Rx(a) Ry(b)) is mapped onto it by the constant
// rotation P = Ry(pi/2): Rx(a) Ry(b) (0,0,-L) = P Rz(a) Ry(b - pi/2) (0,0,-L), i.e. target q' = P^T q = (-q.z, q.y, q.x),
// pitch variable b' = b - pi/2 with its bounds shifted alike (`xy`, `shift`).  One code path for all lanes of a warp.
template <typename R>
struct StageSolve {
    // problem
    bool xy; R shift;                   // stage-1 mapping: b = x1 + shift
    R L, has_a; R span0, span1;         // span = ub - lb (inf if unbounded)
    R null_sq; int max_nfev;
    bool gn_mode;   // true: take the Gauss-Newton step when it fits the trust region (see trip())
    // iterate
    R x0, x1, dl0, dl1, du0, du1;      // angles and distances to the bounds (inf = no bound)
    R sa, ca, sb, cb;                   // sin/cos of the iterate
    Vec3<R> f; R cost, g0, g1;         // residual w(x) - q, 0.5 |f|^2, gradient J^T f
    R Delta, alpha; int nfev, status;
    bool escaped;                       // escape() already used in this solve
    R last_ratio;                       // actual/predicted reduction of the previous evaluation of this solve (0: none yet)
    R st0, st1, step_h_sq, pred;        // the step plan() chose for the next evaluation, its hat-space length^2, its predicted reduction
    bool skip_confirm;                  // SEQIK_FLAG_SKIP_CONFIRM, see trip()
    bool newton;                        // SEQIK_FLAG_NEWTON, see plan()
    bool closed_form;                   // SEQIK_FLAG_CLOSED_FORM, see warm_step()
    bool seeded;                        // this solve started (and ended) at warm_step()'s point
    Vec3<R> seed_f;                     // residual at that point
    int seed_at;                        // 0 interior, 1 / 2: first angle on its lower / upper limit
    bool have_bt; R sl0, cl0, su0, cu0; // sin/cos of the first angle's limits (set_limit_trig)

    typedef Num<R> N;
    SK_HD int kind_() const { return xy ? KIND_XY : KIND_ZY; }
    SK_HD R has_a_() const { return has_a; }
    // results in the caller's (un-mapped) terms
    SK_HD R angle_b() const { return x1 + shift; }
    SK_HD R sin_b() const { return xy ? cb : sb; }                      // sin(b' + pi/2) = cos b'
    SK_HD R cos_b() const { return xy ? -sb : cb; }                     // cos(b' + pi/2) = -sin b'
    SK_HD Vec3<R> res() const { return xy ? Vec3<R>{f.z, f.y, -f.x} : f; }   // residual w - q = P f'

    // end point w = Rot_a Ry(b) (0,0,-L) of the solved segment in the pivot frame
    SK_HD Vec3<R> point() const {
        const R Lsb = L * sb, Lcb = L * cb;
        return {-Lsb * ca, -Lsb * sa, -Lcb};
    }
    // gradient g = J^T f with the two Jacobian columns of w:  ja = has_a (Lsb sa, -Lsb ca, 0),  jb = (-Lcb ca, -Lcb sa, Lsb)
    SK_HD void gradient() {
        const R Lsb = L * sb, Lcb = L * cb;
        g0 = has_a * Lsb * N::fma_(sa, f.x, -(ca * f.y));
        g1 = N::fma_(Lsb, f.z, -(Lcb * N::fma_(ca, f.x, sa * f.y)));
    }
    // |ja|^2 (|jb|^2 = L^2, ja.jb = 0)
    SK_HD R ja_sq() const { return has_a * (L * sb) * (L * sb); }

    // Coleman-Li scaling (common.py CL_scaling_vector): v = distance to the bound the anti-gradient points at
    SK_HD void cl_scaling(R& v0, R& v1, R& dv0, R& dv1) const {
        const R inf = N::inf();
        v0 = R(1); dv0 = R(0); v1 = R(1); dv1 = R(0);
        if (g0 < R(0) && du0 < inf) { v0 = du0; dv0 = R(-1); } else if (g0 > R(0) && dl0 < inf) { v0 = dl0; dv0 = R(1); }
        if (g1 < R(0) && du1 < inf) { v1 = du1; dv1 = R(-1); } else if (g1 > R(0) && dl1 < inf) { v1 = dl1; dv1 = R(1); }
    }

    // x0 and its distances to the bounds; a seed ON a bound (legal) is nudged inside (make_strictly_feasible, rstep 1e-10)
    SK_HD void place(R a, R b, R lb0, R ub0, R lb1, R ub1) {
        span0 = ub0 - lb0; span1 = ub1 - lb1;
        x0 = a; x1 = b;
        dl0 = a - lb0; du0 = ub0 - a; dl1 = b - lb1; du1 = ub1 - b;
        if (N::min_(N::min_(dl0, du0), N::min_(dl1, du1)) <= R(0)) {
            const R rs = R(1e-10);
            if (dl0 <= R(0)) { dl0 = rs * N::max_(R(1), N::abs_(lb0)); x0 = lb0 + dl0; du0 = span0 - dl0; }
            if (du0 <= R(0)) { du0 = rs * N::max_(R(1), N::abs_(ub0)); x0 = ub0 - du0; dl0 = span0 - du0; }
            if (dl1 <= R(0)) { dl1 = rs * N::max_(R(1), N::abs_(lb1)); x1 = lb1 + dl1; du1 = span1 - dl1; }
            if (du1 <= R(0)) { du1 = rs * N::max_(R(1), N::abs_(ub1)); x1 = ub1 - du1; dl1 = span1 - du1; }
        }
    }

    // the constants of a (chain, stage) problem / the seed of a new solve in the caller's terms
    SK_HD void set_problem(int kind_in, R L_, R has_a_in, R null_sq_, int n_full, int mode) {
        gn_mode = (mode & 1) != 0; skip_confirm = (mode & 2) != 0; newton = (mode & 4) != 0; closed_form = (mode & 8) != 0;   // see stage_mode()
        seeded = false;
        xy = kind_in == KIND_XY; shift = xy ? R(1.57079632679489661923) : R(0);
        L = L_; has_a = has_a_in; null_sq = null_sq_; max_nfev = 100 * n_full;
        have_bt = false; seed_at = 0; sl0 = cl0 = su0 = cu0 = R(0);
    }
    SK_HD void set_iterate(R a, R b) { x0 = a; x1 = b - shift; }

    // least_squares prologue: x0 made strictly feasible (rstep 1e-10), f, g, Delta0
    SK_HD void init(int kind_in, R L_, R has_a_in, const Vec3<R>& q_in, R a, R b,
                    R lb0, R ub0, R lb1, R ub1, R null_sq_, int n_full, int mode = 0) {
        set_problem(kind_in, L_, has_a_in, null_sq_, n_full, mode);
        set_iterate(a, b);
        restart(q_in, lb0, ub0, lb1, ub1, true, false);
    }

    // The prologue proper.  `fresh`: the sin/cos of the iterate are derived from the angles (a new solve, init()).
    // Otherwise this is the next frame of the same (chain, stage): the warm start IS the previous solve's final iterate,
    // so its sin/cos are carried over and only the bound distances and the residual against the new target are rebuilt
    // (least_squares prologue without the trigonometry).  Callers pass fresh = true every SEQIK_RESYNC frames so that the
    // carried sin/cos cannot drift from the angle (float32 random walk, ~1e-6 rad over 32 frames).  One code path for
    // both, so that lanes of a warp that re-derive and lanes that carry run the same instructions but the trigonometry.
    // asin for |s| <= WS_HS_MAX (series through s^15: truncation < 3e-8 at 0.44)
    static SK_HD R asin_small(R s) {
        const R z = s * s;
        R p = N::fma_(z, R(0.013964843750000000), R(0.017352764423076924));
        p = N::fma_(p, z, R(0.022372159090909092)); p = N::fma_(p, z, R(0.030381944444444444));
        p = N::fma_(p, z, R(0.044642857142857144));
        p = N::fma_(p, z, R(0.075)); p = N::fma_(p, z, R(0.16666666666666666));
        return N::fma_(p * z, s, s);
    }
    // largest half-angle sine of a closed-form move: both rotations of a warm step stay below 2 asin(0.44) = 0.91 rad
    static SK_HD R ws_hs_max() { return R(0.44); }
    static SK_HD R ws_move_max() { return R(0.91); }

    // Optional (SEQIK_FLAG_CLOSED_FORM): the closed-form warm step.  A stage points a segment of fixed length at its
    // target: without the box, the minimiser of |w(a, b) - q|^2 is the point of the sphere |w| = L nearest to q, i.e.
    // (sb ca, sb sa, cb) = -q / |q| on the branch (sign of sb) of the warm start -- the minimiser the reference's
    // iteration converges to from that warm start when it is a short step away.  So for the next frame of a carried
    // solve the iterate is MOVED there before the prologue (sin/cos directly from q, the angles by the small rotation
    // from the carried iterate); the prologue then finds a vanishing gradient and the solve ends with its first
    // evaluation, or Newton's iteration polishes it.  Taken only when the move is small (both rotations below
    // 0.5 rad), stays strictly inside the box and away from the sin b = 0 singularity, and the minimum is well
    // conditioned (its Hessian is |q| / L times the Gauss-Newton one: |q| > L / 2, Newton's own admission test -- closer
    // targets leave the direction ill-determined and the reference crawls there); in every other case -- first
    // frame of a call, re-derivation frames, active bounds, large moves -- the solve runs from the warm start exactly
    // as without the flag.  One-variable stage 4: the same in the plane of its single rotation.
    SK_HD void warm_step(const Vec3<R>& q, R lb0, R ub0, R lb1, R ub1, bool enable = true) {
        const bool one_var = has_a == R(0);
        const R rho2 = one_var ? q.x * q.x : N::fma_(q.y, q.y, q.x * q.x);
        const R qn2 = N::fma_(q.z, q.z, rho2);
        const R rn = N::rsqrt_(qn2), rr = N::rsqrt_(rho2);
        const R sgn = (sb < R(0)) ? R(-1) : R(1);
        const R t_ = sgn * rr;
        const R n_sb = one_var ? -(q.x * rn) : sgn * (rho2 * rr) * rn, n_cb = -(q.z * rn);
        const R n_ca = one_var ? ca : -(q.x * t_), n_sa = one_var ? sa : -(q.y * t_);
        const R sda = N::fma_(n_sa, ca, -(n_ca * sa)), cda = N::fma_(n_ca, ca, n_sa * sa);
        const R sdb = N::fma_(n_sb, cb, -(n_cb * sb)), cdb = N::fma_(n_cb, cb, n_sb * sb);
        // rotation angles by the half-angle form: sin(d / 2) = sin d / sqrt(2 (1 + cos d)), |d| < 0.5 rad
        const R hsa = sda * N::rsqrt_(R(2) + R(2) * cda), hsb = sdb * N::rsqrt_(R(2) + R(2) * cdb);
        const R nx0 = x0 + R(2) * asin_small(hsa), nx1 = x1 + R(2) * asin_small(hsb);
        const R m = R(1e-5);
        // (bitwise &: every test is evaluated, no short-circuit branches in this block)
        const bool in_a = (nx0 - lb0 > m) & (ub0 - nx0 > m), in_b = (nx1 - lb1 > m) & (ub1 - nx1 > m);
        const bool small_a = (N::abs_(hsa) < ws_hs_max()) & (cda > R(0)), small_b = (N::abs_(hsb) < ws_hs_max()) & (cdb > R(0));
        const bool ok = enable & small_a & small_b & (one_var | (rho2 > R(0.01) * qn2)) & (qn2 > R(0.25) * L * L) & (qn2 < N::inf())
                        & in_a & in_b;
        // residual there: w = L q / |q| (in the rotation's plane for one variable), f = w - q
        const R k = N::fma_(L, rn, R(-1));
        seed_f = {q.x * k, one_var ? -q.y : q.y * k, q.z * k};
        // ---- the same with the first angle ON its limit: when the free minimiser lies beyond a limit of `a` (and only
        // then), the box-constrained minimiser has a = that limit and b the minimiser in the plane of the b rotation
        // at that a: (sb, cb) = -(q_e, q_z) / |.|, q_e = q . (ca, sa, 0).  Admitted under the same tests (small moves,
        // same branch, conditioning in that plane, b strictly interior) plus the KKT sign of the a-gradient there.
        // One block behind one branch: only lanes whose free minimiser left the box through a limit of `a` enter it
        // (a few per cent of the solves of the benchmark workload, none on most recordings).
        x0 = ok ? nx0 : x0; x1 = ok ? nx1 : x1;
        sa = ok ? n_sa : sa; ca = ok ? n_ca : ca; sb = ok ? n_sb : sb; cb = ok ? n_cb : cb;
        seeded = ok; seed_at = 0;
        const bool below = nx0 - lb0 <= m, above = ub0 - nx0 <= m;
        if (enable & have_bt & !one_var & !ok & (below != above) & small_a) {
            const bool lo = below;
            const R b_sa = lo ? sl0 : su0, b_ca = lo ? cl0 : cu0, b_x0 = lo ? lb0 : ub0;
            const R qe = N::fma_(q.y, b_sa, q.x * b_ca), pn2 = N::fma_(q.z, q.z, qe * qe);
            const R rp = N::rsqrt_(pn2);
            const R c_sb = -(qe * rp), c_cb = -(q.z * rp);
            const R sdb2 = N::fma_(c_sb, cb, -(c_cb * sb)), cdb2 = N::fma_(c_cb, cb, c_sb * sb);
            const R hsb2 = sdb2 * N::rsqrt_(R(2) + R(2) * cdb2);
            const R cx1 = x1 + R(2) * asin_small(hsb2);
            const R ga = c_sb * N::fma_(b_ca, q.y, -(b_sa * q.x));      // sign of d cost / d a at the candidate (times L > 0)
            const bool kkt = lo ? (ga > R(0)) : (ga < R(0));
            const bool ok_b = (N::abs_(b_x0 - x0) < ws_move_max())
                              & (N::abs_(hsb2) < ws_hs_max()) & (cdb2 > R(0)) & (c_sb * sgn > R(0.1)) & (pn2 > R(0.25) * L * L) & (pn2 < N::inf())
                              & (cx1 - lb1 > m) & (ub1 - cx1 > m) & kkt;
            if (ok_b) {
                x0 = b_x0; x1 = cx1; sa = b_sa; ca = b_ca; sb = c_sb; cb = c_cb;
                seeded = true; seed_at = lo ? 1 : 2;
                const R Lsb_c = L * c_sb;
                seed_f = {-(Lsb_c * b_ca) - q.x, -(Lsb_c * b_sa) - q.y, -(L * c_cb) - q.z};
            }
        }
    }
    // sin/cos of the first angle's limits, for warm_step()'s on-the-limit case (once per (chain, stage))
    SK_HD void set_limit_trig(R lb0, R ub0) {
        R v_;
        have_bt = lb0 > -N::inf() && ub0 < N::inf();
        if (have_bt) { N::sincosv_(lb0, &sl0, &cl0, &v_); N::sincosv_(ub0, &su0, &cu0, &v_); }
    }

    // `warm`: the iterate is a previous frame's solution (false only for the seed of a recording's first frame), i.e.
    // the closed-form warm step may be taken.
    SK_HD void restart(const Vec3<R>& q_in, R lb0, R ub0, R lb1, R ub1, bool fresh = false, bool warm = true) {
        const Vec3<R> q = restart_a(q_in, lb0, ub0, lb1, ub1, fresh);
        warm_step(q, lb0, ub0, lb1 - shift, ub1 - shift, closed_form && gn_mode && warm);
        restart_b(q, lb0, ub0, lb1, ub1);
    }
    // The same in three pieces, so that a kernel can put independent work of its own next to the straight-line middle
    // one (warm_step) and have the two instruction streams interleave:
    // (a) target into the solve's own frame, bound distances, trigonometry of a fresh iterate
    SK_HD Vec3<R> restart_a(const Vec3<R>& q_in, R lb0, R ub0, R lb1, R ub1, bool fresh) {
        const Vec3<R> q = xy ? Vec3<R>{-q_in.z, q_in.y, q_in.x} : q_in;
        place(x0, x1, lb0, ub0, lb1 - shift, ub1 - shift);   // bound distances (re-)derived from the angle
        if (fresh) { R va, vb; N::sincosv_(x0, &sa, &ca, &va); N::sincosv_(x1, &sb, &cb, &vb); }
        return q;
    }
    // (b) after warm_step(): the solve ends at the seeded point, or the least_squares prologue runs
    SK_HD void restart_b(const Vec3<R>& q, R lb0, R ub0, R lb1, R ub1) {
        alpha = R(0); nfev = 1; escaped = false; last_ratio = R(0);
        if (seeded) {
            // the minimiser itself: the gradient vanishes by construction (w is parallel to q, both Jacobian columns are
            // orthogonal to w; on a limit the first one points out of the box), so the solve ends with this evaluation
            dl0 = x0 - lb0; du0 = ub0 - x0; dl1 = x1 - (lb1 - shift); du1 = (ub1 - shift) - x1;   // strictly inside: no nudge
            if (seed_at != 0) {                  // on a limit: one fp64 ulp inside, like the iterates that land there
                const R gap = inner_gap(x0);
                dl0 = (seed_at == 1) ? gap : span0 - gap; du0 = (seed_at == 1) ? span0 - gap : gap;
            }
            f = seed_f; cost = R(0.5) * dot(f, f); g0 = R(0); g1 = R(0);
            status = (cost < N::inf()) ? ST_GTOL : ST_NONFINITE;
            return;
        }
        const Vec3<R> w = point();
        f = {w.x - q.x, w.y - q.y, w.z - q.z};
        cost = R(0.5) * dot(f, f);
        gradient();
        R v0, v1, dv0, dv1; cl_scaling(v0, v1, dv0, dv1);
        // v can be ~1e-38 (an iterate parked on a bound at 0): there x = +-v, the term x^2 / v = v is negligible
        // against null_sq >= 1 and x * x underflows, so it is dropped instead of evaluating 0 * rcp(tiny) = 0 * inf
        const R xb_ = x1 + shift;
        const R q0 = (v0 > R(1e-30)) ? x0 * x0 * N::rcp_(v0) : R(0), q1 = (v1 > R(1e-30)) ? xb_ * xb_ * N::rcp_(v1) : R(0);
        Delta = N::sqrt_(null_sq + q0 + q1);
        if (Delta == R(0)) Delta = R(1);
        status = (cost < N::inf()) ? ST_RUNNING : ST_NONFINITE;      // false for NaN and inf
        plan(status == ST_RUNNING);
    }

    // Singularity escape (optional, SEQIK_FLAG_ESCAPE).  For the Rz(a) Ry(b) stages the end point does not depend on
    // `a` when sin b = 0: a solve that ends there (typically with `a` parked on a bound) has a vanishing gradient
    // although a far better point may exist.  The reference leaves such a corner only through the rounding noise of
    // its finite-difference Jacobian (SURVEY.md finding 4), i.e. frames later and irreproducibly.  Here the two
    // closed-form mirror solutions of "point a segment at the target" (SURVEY.md 3.4), clamped to the box, are
    // evaluated; if one is clearly better the solve continues from it.  At most once per solve.
    SK_HD bool escape_possible() const { return !(escaped || xy || has_a == R(0) || sb * sb > R(1e-8)); }
    SK_HD bool escape() {
        if (!escape_possible()) return false;
        escaped = true;
        const Vec3<R> w = point();
        const Vec3<R> q = {w.x - f.x, w.y - f.y, w.z - f.z};
        const R rho2 = N::fma_(q.y, q.y, q.x * q.x), qn = N::sqrt_(rho2 + q.z * q.z);
        if (rho2 < R(1e-10) * L * L) return false;            // target on the axis: `a` really is irrelevant
        const R pi = R(3.14159265358979323846);
        const R phi = atan2(q.y, q.x), bs = acos(N::max_(R(-1), N::min_(R(1), -q.z * N::rcp_(qn))));
        const R lb0 = x0 - dl0, ub0 = x0 + du0, lb1 = x1 - dl1, ub1 = x1 + du1;
        R best = cost, ba = x0, bb = x1;
        for (int k = 0; k < 2; ++k) {
            R aa = k ? phi : phi + pi, b2 = k ? -bs : bs;
            if (aa > pi) aa -= R(2) * pi;
            aa = N::max_(lb0, N::min_(ub0, aa)); b2 = N::max_(lb1, N::min_(ub1, b2));
            R s_a, c_a, s_b, c_b, v_;
            N::sincosv_(aa, &s_a, &c_a, &v_); N::sincosv_(b2, &s_b, &c_b, &v_);
            const R dx = -L * s_b * c_a - q.x, dy = -L * s_b * s_a - q.y, dz = -L * c_b - q.z;
            const R cst = R(0.5) * N::fma_(dz, dz, N::fma_(dy, dy, dx * dx));
            if (cst < best) { best = cst; ba = aa; bb = b2; }
        }
        nfev += 2;
        if (!(best < R(0.98) * cost - R(5e-7))) return false;  // clearly better: > 2 % and > (1e-3 mm)^2 / 2
        const R nsq = null_sq; const int mx = max_nfev; const int nf = nfev;
        const int md = (gn_mode ? 1 : 0) | (skip_confirm ? 2 : 0) | (newton ? 4 : 0) | (closed_form ? 8 : 0);
        const bool bt = have_bt; const R t0 = sl0, t1 = cl0, t2 = su0, t3 = cu0;    // per-(chain, stage) constants survive
        init(KIND_ZY, L, has_a, q, ba, bb, lb0, ub0, lb1, ub1, nsq, 1, md);
        max_nfev = mx; nfev = nf; escaped = true;
        have_bt = bt; sl0 = t0; cl0 = t1; su0 = t2; cu0 = t3;
        return true;
    }

    SK_HD bool done() const { return status != ST_RUNNING; }

    // step_size_to_bound from distances (dl, du) along p; hit flags.  rcp(0) = inf gives +inf for a zero component.
    static SK_HD R to_bound(R dl0_, R du0_, R dl1_, R du1_, R p0, R p1, bool& h0, bool& h1) {
        const R r0 = N::rcp_(p0), r1 = N::rcp_(p1);
        const R s0 = (p0 != R(0)) ? N::max_(-dl0_ * r0, du0_ * r0) : N::inf();
        const R s1 = (p1 != R(0)) ? N::max_(-dl1_ * r1, du1_ * r1) : N::inf();
        const R m = N::min_(s0, s1);
        h0 = (p0 != R(0)) && (s0 == m); h1 = (p1 != R(0)) && (s1 == m);
        return m;
    }

    // minimize_quadratic_1d(a, b, lo, hi, c): straight-line (selects only)
    static SK_HD void minq(R a, R b, R lo, R hi, R c, R& t_best, R& y_best) {
        const R yl = N::fma_(lo, N::fma_(a, lo, b), c), yh = N::fma_(hi, N::fma_(a, hi, b), c);
        const R e = R(-0.5) * b * N::rcp_(a);
        const R ye = N::fma_(e, N::fma_(a, e, b), c);
        t_best = lo; y_best = yl;
        if (yh < y_best) { y_best = yh; t_best = hi; }
        if (a != R(0) && lo < e && e < hi && ye < y_best) { y_best = ye; t_best = e; }
    }

    // Quantities of one outer iteration in the scaled ("hat") variables: B = Jh^T Jh + diag (diagonal), gh
    struct Hat { R d0, d1, B0, B1, gh0, gh1, theta; };

    // value of the hat-space quadratic model at s (evaluate_quadratic, common.py)
    static SK_HD R model(const Hat& h, R s0, R s1) {
        return N::fma_(s1, h.gh1, N::fma_(s0, h.gh0, R(0.5) * N::fma_(h.B1 * s1, s1, h.B0 * s0 * s0)));
    }

    // select_step (trf.py:129-203) restricted to the active pair.
    static SK_HD void select_step(const Hat& h, R dl0, R du0, R dl1, R du1, R Delta, R p0, R p1, R ph0, R ph1,
                                  R& st0, R& st1, R& sh0, R& sh1, R& pred) {
        const bool inb = (dl0 + p0 >= R(0)) && (du0 - p0 >= R(0)) && (dl1 + p1 >= R(0)) && (du1 - p1 >= R(0));
        // in_bounds: scipy returns the plain step.  By far the common case once the trust region has adapted; the
        // three-candidate search below is straight-line code that only runs for lanes whose step leaves the box.
        if (inb) { st0 = p0; st1 = p1; sh0 = ph0; sh1 = ph1; pred = -model(h, ph0, ph1); return; }
        bool h0, h1;
        const R p_stride = to_bound(dl0, du0, dl1, du1, p0, p1, h0, h1);
        R rh0 = h0 ? -ph0 : ph0, rh1 = h1 ? -ph1 : ph1;
        R r0 = h.d0 * rh0, r1 = h.d1 * rh1;
        p0 *= p_stride; p1 *= p_stride; ph0 *= p_stride; ph1 *= p_stride;
        // intersect_trust_region(ph, rh, Delta): positive root
        R to_tr;
        {
            const R a = N::fma_(rh1, rh1, rh0 * rh0), b = N::fma_(ph1, rh1, ph0 * rh0);
            const R c = N::min_(N::fma_(ph1, ph1, ph0 * ph0) - Delta * Delta, R(0));
            const R disc = N::sqrt_(N::max_(N::fma_(b, b, -(a * c)), R(0)));
            const R qq = -(b + N::copysign_(disc, b));
            const R t1 = (qq != R(0)) ? qq * N::rcp_(a) : R(0), t2 = (qq != R(0)) ? c * N::rcp_(qq) : R(0);
            to_tr = N::max_(t1, t2);
        }
        bool u0, u1;
        const R to_bd = to_bound(dl0 + p0, du0 - p0, dl1 + p1, du1 - p1, r0, r1, u0, u1);
        const R r_stride = N::min_(to_bd, to_tr);
        const bool rpos = r_stride > R(0);
        const R r_l = rpos ? (R(1) - h.theta) * p_stride * N::rcp_(r_stride) : R(0);
        const R r_u = rpos ? ((r_stride == to_bd) ? h.theta * to_bd : to_tr) : R(-1);
        R r_value = N::inf();
        {
            // build_quadratic_1d(Jh, gh, rh, s0=ph, diag=dh) with the diagonal B
            const R a = R(0.5) * N::fma_(h.B1 * rh1, rh1, h.B0 * rh0 * rh0);
            const R b = N::fma_(h.gh1, rh1, h.gh0 * rh0) + N::fma_(h.B1 * ph1, rh1, h.B0 * ph0 * rh0);
            const R c = model(h, ph0, ph1);
            R rs, rv; minq(a, b, r_l, r_u, c, rs, rv);
            if (r_l <= r_u) {
                r_value = rv;
                rh0 = N::fma_(rh0, rs, ph0); rh1 = N::fma_(rh1, rs, ph1);
                r0 = rh0 * h.d0; r1 = rh1 * h.d1;
            }
        }
        // strictly interior truncated step
        p0 *= h.theta; p1 *= h.theta; ph0 *= h.theta; ph1 *= h.theta;
        const R p_value = model(h, ph0, ph1);
        // scaled anti-gradient
        const R ah0 = -h.gh0, ah1 = -h.gh1;
        const R a0 = h.d0 * ah0, a1 = h.d1 * ah1;
        const R to_tr2 = Delta * N::rsqrt_(N::fma_(ah1, ah1, ah0 * ah0));
        const R to_bd2 = to_bound(dl0, du0, dl1, du1, a0, a1, u0, u1);
        const R ag_hi = (to_bd2 < to_tr2) ? h.theta * to_bd2 : to_tr2;
        R ag_value, ags;
        {
            const R a = R(0.5) * N::fma_(h.B1 * ah1, ah1, h.B0 * ah0 * ah0);
            const R b = N::fma_(h.gh1, ah1, h.gh0 * ah0);
            minq(a, b, R(0), ag_hi, R(0), ags, ag_value);
        }
        const bool take_p = p_value < r_value && p_value < ag_value;
        const bool take_r = !take_p && r_value < p_value && r_value < ag_value;
        st0 = take_p ? p0 : take_r ? r0 : a0 * ags; st1 = take_p ? p1 : take_r ? r1 : a1 * ags;
        sh0 = take_p ? ph0 : take_r ? rh0 : ah0 * ags; sh1 = take_p ? ph1 : take_r ? rh1 : ah1 * ags;
        pred = -(take_p ? p_value : take_r ? r_value : ag_value);
    }

    // The general step of plan(): Levenberg iteration when the Gauss-Newton step does not fit the trust region, then
    // select_step's three-candidate search when the step leaves the box.  Rare once the trust region has adapted
    // (< 0.1 % of the evaluations of the benchmark workload), so it lives out of line.
    struct Step { R st0, st1, sh_sq, pred, alpha; };
    static SK_HD_COLD Step slow_step(Hat h, R tg0, R tg1, bool gn_taken, bool one_var, R Delta, R alpha,
                                     R dl0, R du0, R dl1, R du1) {
        R t0 = tg0, t1 = tg1;
        if (gn_taken) alpha = R(0);
        if (!gn_taken) {
            if (one_var) {
                // one variable: whatever the Levenberg parameter, the step is rescaled to the trust radius below,
                // i.e. p_h = -sign(gh1) Delta (the parameter is never used again for this stage)
                t0 = R(0); t1 = h.gh1;
            } else {
                const R rDelta = N::rcp_(Delta);
                R a_up = N::sqrt_(N::fma_(h.gh1, h.gh1, h.gh0 * h.gh0)) * rDelta, a_lo = R(0);
                if (alpha == R(0)) alpha = R(0.001) * a_up;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
                for (int it = 0; it < 10; ++it) {
                    if (alpha < a_lo || alpha > a_up) alpha = N::max_(R(0.001) * a_up, N::sqrt_(a_lo * a_up));
                    const R e0 = h.B0 + alpha, e1 = h.B1 + alpha;
                    const R r0 = (e0 != R(0)) ? N::rcp_(e0) : R(0), r1 = (e1 != R(0)) ? N::rcp_(e1) : R(0);
                    t0 = (h.gh0 != R(0)) ? h.gh0 * r0 : R(0); t1 = (h.gh1 != R(0)) ? h.gh1 * r1 : R(0);
                    const R pn = N::sqrt_(N::fma_(t1, t1, t0 * t0));
                    const R phi = pn - Delta;
                    const R dd = N::fma_(t1 * t1, r1, t0 * t0 * r0);        // -phi' * pn
                    if (phi < R(0)) a_up = alpha;
                    const R ratio = (dd > R(0)) ? -(phi * pn) * N::rcp_(dd) : R(0);   // phi / phi'
                    a_lo = N::max_(a_lo, alpha - ratio);
                    alpha -= pn * ratio * rDelta;                            // (phi + Delta) * ratio / Delta
                    if (N::abs_(phi) < R(0.01) * Delta) break;
                }
                const R e0 = h.B0 + alpha, e1 = h.B1 + alpha;
                t0 = (e0 != R(0) && h.gh0 != R(0)) ? h.gh0 * N::rcp_(e0) : R(0);
                t1 = (e1 != R(0) && h.gh1 != R(0)) ? h.gh1 * N::rcp_(e1) : R(0);
            }
        }
        const R sc = gn_taken ? R(1) : Delta * N::rsqrt_(N::fma_(t1, t1, t0 * t0));
        const R ph0 = -t0 * sc, ph1 = -t1 * sc;
        Step o; R sh0, sh1;
        select_step(h, dl0, du0, dl1, du1, Delta, h.d0 * ph0, h.d1 * ph1, ph0, ph1, o.st0, o.st1, sh0, sh1, o.pred);
        o.sh_sq = N::fma_(sh1, sh1, sh0 * sh0); o.alpha = alpha;
        return o;
    }

    // plan(): the head of scipy's outer iteration for the CURRENT iterate -- scaling, termination tests that need no
    // evaluation (gtol, max_nfev, skip-confirm), trust-region step -- leaving the step to evaluate in (st0, st1,
    // step_h_sq, pred).  It runs at the end of init()/restart() and at the end of every trip(), so a solve costs
    // exactly one loop trip per function evaluation and its termination is known in the trip that produced it.
    // (After a rejected step the iterate is unchanged and only Delta/alpha differ: plan() recomputes the same head.)
    SK_HD void plan(bool active = true) {
        const R gtol = R(1e-8), ftol = R(1e-8);
        R v0, v1, dv0, dv1; cl_scaling(v0, v1, dv0, dv1);
        const R g_norm = N::max_(N::abs_(g0 * v0), N::abs_(g1 * v1));
        // straight-line code: the termination tests that need no evaluation are folded into selects at the end, so that
        // a trip is one basic block but for the rare general step (lanes that are not `active` change nothing)
        const bool stop_g = g_norm < gtol, stop_n = nfev >= max_nfev;
        const bool run = active && !stop_g && !stop_n;
        const bool one_var = has_a_() == R(0);
        const R B0 = N::fma_(v0, ja_sq(), g0 * dv0), B1 = N::fma_(v1, L * L, g1 * dv1);   // Jh^T Jh + diag(g dv), diagonal
        R n_st0 = R(0), n_st1 = R(0), n_sh = R(0), n_pred = R(0), n_alpha = R(0);
        bool take = false, gn_taken = false;
        // Optional (SEQIK_FLAG_NEWTON): the Newton step of the same scaled model with the residual-curvature term
        // sum_i f_i Hess(w_i) added -- closed form for the two-angle segment: w_aa = (Lsb ca, Lsb sa, 0), w_bb = -w,
        // w_ab = (Lcb sa, -Lcb ca, 0).  The targets are noisy key points, so the residual does not vanish at the solution
        // and Gauss-Newton converges only linearly (3.3 - 4.8 evaluations per warm-started solve); Newton's iteration
        // reaches the same minimiser (to ~1e-6 rad of where the reference's ftol stop leaves it) in 2 - 3.  Taken only
        // where the full Hessian is safely positive definite and close to the Gauss-Newton one, the step fits the trust
        // region and stays inside the box; every other case falls through to the reference's step below.  Written in
        // terms of v = d^2 (no square roots): with r = H^-1-weighted gradient, the step is p = -v r, its hat-space
        // length^2 is sum v r^2 and the model's predicted reduction is sum v g r - 0.5 (p_h^T H p_h).
        if (newton && gn_mode) {
            const R Lsb = L * sb, Lcb = L * cb;
            const R u = N::fma_(ca, f.x, sa * f.y), w_ = N::fma_(sa, f.x, -(ca * f.y));
            const R e00 = has_a * Lsb * u, e11 = N::fma_(Lsb, u, Lcb * f.z), e01 = has_a * Lcb * w_;
            const R B0_ = one_var ? R(1) : B0;
            const R H00 = one_var ? R(1) : N::fma_(v0, e00, B0), H11 = N::fma_(v1, e11, B1);
            const R ve = v0 * v1 * e01;                                   // H01^2 = ve * e01
            const R det = N::fma_(H00, H11, -(ve * e01));
            const bool pd = H00 > R(0.5) * B0_ && H11 > R(0.5) * B1 && det > R(0.25) * B0_ * B1;
            const R rdet = N::rcp_(det);
            const R r0 = N::fma_(H11, g0, -(v1 * e01 * g1)) * rdet, r1 = N::fma_(H00, g1, -(v0 * e01 * g0)) * rdet;
            const R q0_ = -(v0 * r0), q1_ = -(v1 * r1);
            const R nsq = N::fma_(v1 * r1, r1, v0 * r0 * r0);
            const bool n_inb = (dl0 + q0_ >= R(0)) && (du0 - q0_ >= R(0)) && (dl1 + q1_ >= R(0)) && (du1 - q1_ >= R(0));
            take = pd && n_inb && nsq <= Delta * Delta;
            const R quad = N::fma_(H11 * v1 * r1, r1, N::fma_(R(2) * ve * r0, r1, H00 * v0 * r0 * r0));
            n_st0 = q0_; n_st1 = q1_; n_sh = nsq; n_pred = N::fma_(v1 * g1, r1, v0 * g0 * r0) - R(0.5) * quad;
        }
        if (run && !take) {
            Hat h;
            h.d0 = N::sqrt_(v0); h.d1 = N::sqrt_(v1);
            h.gh0 = h.d0 * g0; h.gh1 = h.d1 * g1;
            h.B0 = B0; h.B1 = B1;
            h.theta = N::max_(R(0.995), R(1) - g_norm);
            // ---- solve_lsq_trust_region, rank-deficient branch; singular values^2 = (B0, B1), V = I
            // gn_mode: scipy's SVD of the full chain leaves ~1e-17 singular values on the inert slots; the Levenberg
            // parameter then decays to ~1e-20 and that null-space noise absorbs the trust-region norm, i.e. the active
            // pair receives the plain Gauss-Newton step whenever it fits in Delta.  Measured against the reference's
            // shipped angles (6000 frames x 2 legs) this reproduces the reference's evaluation counts and termination
            // statuses; the literal rank-deficient branch below is kept for the steps that do not fit.
            const R tg0 = one_var ? R(0) : h.gh0 * N::rcp_(h.B0), tg1 = h.gh1 * N::rcp_(h.B1);
            gn_taken = gn_mode && (one_var || h.B0 > R(0)) && h.B1 > R(0) && (N::fma_(tg1, tg1, tg0 * tg0) <= Delta * Delta);
            // fast path: the Gauss-Newton step fits the trust region and stays inside the box (select_step's in_bounds case)
            const R ph0 = -tg0, ph1 = -tg1, p0 = h.d0 * ph0, p1 = h.d1 * ph1;
            const bool inb = (dl0 + p0 >= R(0)) && (du0 - p0 >= R(0)) && (dl1 + p1 >= R(0)) && (du1 - p1 >= R(0));
            n_st0 = p0; n_st1 = p1; n_sh = N::fma_(ph1, ph1, ph0 * ph0); n_pred = -model(h, ph0, ph1);
            if (!(gn_taken && inb)) {
                const Step o = slow_step(h, tg0, tg1, gn_taken, one_var, Delta, alpha, dl0, du0, dl1, du1);
                n_st0 = o.st0; n_st1 = o.st1; n_sh = o.sh_sq; n_pred = o.pred; n_alpha = o.alpha;
            }
        }
        st0 = run ? n_st0 : st0; st1 = run ? n_st1 : st1; step_h_sq = run ? n_sh : step_h_sq; pred = run ? n_pred : pred;
        alpha = run ? n_alpha : alpha;
        // Optional (SEQIK_FLAG_SKIP_CONFIRM): do not evaluate a step that would only CONFIRM convergence.  When the model
        // has just been accurate (previous actual/predicted within 25 % of 1) and now predicts a reduction below
        // ftol * cost for a plain Gauss-Newton (or Newton) step, the reference evaluates that step, accepts it and stops
        // on ftol; the step is below sqrt(2 ftol cost) / L ~ 3e-6 rad.  Saves one of the ~5 evaluations of a solve.
        const bool confirm_only = skip_confirm && (take || gn_taken) && n_pred < ftol * cost && n_pred >= R(0) && N::abs_(last_ratio - R(1)) < R(0.25);
        const int st_new = stop_g ? ST_GTOL : stop_n ? ST_MAXFEV : confirm_only ? ST_FTOL : ST_RUNNING;
        status = active ? st_new : status;
    }

    // One function evaluation: one pass of scipy's inner `while actual_reduction <= 0` loop on the step plan() left,
    // then plan() for the next one.
    SK_HD void trip() {
        const R ftol = R(1e-8), xtol = R(1e-8);
        // ---- trial point: strictly feasible, evaluated through the step's sin/cos/versine
        R nx0 = x0 + st0, nx1 = x1 + st1;
        R ndl0 = dl0 + st0, ndu0 = du0 - st0, ndl1 = dl1 + st1, ndu1 = du1 - st1;
        R e0 = st0, e1 = st1;   // applied step
        if (N::min_(N::min_(ndl0, ndu0), N::min_(ndl1, ndu1)) <= R(0)) {   // landed on a bound: pull one fp64 ulp inside
            if (ndl0 <= R(0)) { const R gap = inner_gap(nx0 - ndl0); e0 = gap - dl0; ndl0 = gap; ndu0 = span0 - gap; nx0 = x0 + e0; }
            if (ndu0 <= R(0)) { const R gap = inner_gap(nx0 + ndu0); e0 = du0 - gap; ndu0 = gap; ndl0 = span0 - gap; nx0 = x0 + e0; }
            if (ndl1 <= R(0)) { const R gap = inner_gap(nx1 - ndl1); e1 = gap - dl1; ndl1 = gap; ndu1 = span1 - gap; nx1 = x1 + e1; }
            if (ndu1 <= R(0)) { const R gap = inner_gap(nx1 + ndu1); e1 = du1 - gap; ndu1 = gap; ndl1 = span1 - gap; nx1 = x1 + e1; }
        }
        R sda, cda, va, sdb, cdb, vb;
        N::sincosv2_(e0, e1, &sda, &cda, &va, &sdb, &cdb, &vb);
        const R dsa = N::fma_(ca, sda, -(sa * va)), dca = -N::fma_(sa, sda, ca * va);   // sin/cos(a + e0) - sin/cos(a)
        const R dsb = N::fma_(cb, sdb, -(sb * vb)), dcb = -N::fma_(sb, sdb, cb * vb);
        const R nsa = sa + dsa, nca = ca + dca, nsb = sb + dsb, ncb = cb + dcb;
        const Vec3<R> dw = {-L * N::fma_(dsb, nca, sb * dca), -L * N::fma_(dsb, nsa, sb * dsa), -L * dcb};   // w(x + e) - w(x)
        nfev += 1;
        const R actual = -N::fma_(R(0.5), dot(dw, dw), dot(f, dw));
        // update_tr_radius
        const R ratio_pos = (actual != R(0)) ? actual * N::rcp_(pred) : R(0);
        const R ratio = (pred > R(0)) ? ratio_pos : ((pred == R(0) && actual == R(0)) ? R(1) : R(0));
        last_ratio = ratio;
        const bool shrink = ratio < R(0.25), grow = !shrink && ratio > R(0.75) && step_h_sq > R(0.9025) * Delta * Delta;
        const R Delta_new = shrink ? R(0.25) * N::sqrt_(step_h_sq) : grow ? R(2) * Delta : Delta;
        // check_termination
        const R step_sq = N::fma_(st1, st1, st0 * st0);
        const R xb_ = x1 + shift;
        const R x_norm = N::sqrt_(N::fma_(xb_, xb_, N::fma_(x0, x0, null_sq)));
        const R xt_rhs = xtol * (xtol + x_norm);
        const bool ft = (actual < ftol * cost) && (ratio > R(0.25));
        const bool xt = step_sq < xt_rhs * xt_rhs;
        const int term = (ft && xt) ? ST_BOTH : ft ? ST_FTOL : xt ? ST_XTOL : ST_RUNNING;
        const bool go_on = term == ST_RUNNING;
        alpha = go_on ? alpha * (Delta * N::rcp_(Delta_new)) : alpha; Delta = go_on ? Delta_new : Delta;
        // accept / reject by selects (the gradient of an unchanged iterate is recomputed to the same bits)
        const bool acc = actual > R(0);
        x0 = acc ? nx0 : x0; x1 = acc ? nx1 : x1;
        dl0 = acc ? ndl0 : dl0; du0 = acc ? ndu0 : du0; dl1 = acc ? ndl1 : dl1; du1 = acc ? ndu1 : du1;
        sa = acc ? nsa : sa; ca = acc ? nca : ca; sb = acc ? nsb : sb; cb = acc ? ncb : cb;
        f = {acc ? f.x + dw.x : f.x, acc ? f.y + dw.y : f.y, acc ? f.z + dw.z : f.z};
        cost = acc ? cost - actual : cost;
        gradient();
        status = term;
        plan(go_on);
    }

    // make_strictly_feasible(x, lb, ub, rstep=0): one fp64 ulp inside the bound `b`
    static SK_HD R inner_gap(R b) {
        const R ab = N::abs_(b);
        return (ab > R(0)) ? N::eps_in() * ab : N::tiny();
    }
};

// ---------------------------------------------------------------------------------
// 3x3 frame algebra for the stage hand-off
// ---------------------------------------------------------------------------------
template <typename R> struct Mat3 { Vec3<R> c0, c1, c2; };   // columns

template <typename R> SK_HD Vec3<R> mulT(const Mat3<R>& A, const Vec3<R>& v) {   // A^T v
    return {dot(A.c0, v), dot(A.c1, v), dot(A.c2, v)};
}
template <typename R> SK_HD Vec3<R> mul(const Mat3<R>& A, const Vec3<R>& v) {    // A v
    typedef Num<R> N;
    return {N::fma_(A.c2.x, v.z, N::fma_(A.c1.x, v.y, A.c0.x * v.x)),
            N::fma_(A.c2.y, v.z, N::fma_(A.c1.y, v.y, A.c0.y * v.x)),
            N::fma_(A.c2.z, v.z, N::fma_(A.c1.z, v.y, A.c0.z * v.x))};
}
template <typename R> SK_HD Vec3<R> lin(const Vec3<R>& a, R s, const Vec3<R>& b, R t) {
    typedef Num<R> N;
    return {N::fma_(b.x, t, a.x * s), N::fma_(b.y, t, a.y * s), N::fma_(b.z, t, a.z * s)};
}
// A <- A * Rot_a(a) * Ry(b), Rot_a = Rx (KIND_XY) or Rz (KIND_ZY)
template <typename R> SK_HD Mat3<R> rotate_frame(const Mat3<R>& A, int kind, R sa, R ca, R sb, R cb) {
    Mat3<R> B;
    if (kind == KIND_XY) { B.c0 = A.c0; B.c1 = lin(A.c1, ca, A.c2, sa); B.c2 = lin(A.c1, -sa, A.c2, ca); }
    else { B.c0 = lin(A.c0, ca, A.c1, sa); B.c1 = lin(A.c0, -sa, A.c1, ca); B.c2 = A.c2; }
    Mat3<R> C;
    C.c0 = lin(B.c0, cb, B.c2, -sb); C.c1 = B.c1; C.c2 = lin(B.c0, sb, B.c2, cb);
    return C;
}

// the same without a branch on `kind` (selects on the columns; identical arithmetic): for callers whose lanes mix kinds
template <typename R> SK_HD Mat3<R> rotate_frame_sel(const Mat3<R>& A, int kind, R sa, R ca, R sb, R cb) {
    const bool xy = kind == KIND_XY;
    const Vec3<R> U = xy ? A.c1 : A.c0, V = xy ? A.c2 : A.c1, W = xy ? A.c0 : A.c2;
    const Vec3<R> P = lin(U, ca, V, sa), Q = lin(U, -sa, V, ca);
    Mat3<R> B;
    B.c0 = xy ? W : P; B.c1 = xy ? P : Q; B.c2 = xy ? Q : W;
    Mat3<R> C;
    C.c0 = lin(B.c0, cb, B.c2, -sb); C.c1 = B.c1; C.c2 = lin(B.c0, sb, B.c2, cb);
    return C;
}

// ---------------------------------------------------------------------------------
// ChainRunner: one (trial, leg) chain advanced ONE function evaluation per step().
//
// The kernels give every lane one runner and call step() in a convergent loop: lanes of a
// warp then sit at different (frame, stage) positions of their own chains ("decoupled"
// schedule), so a slow solve delays only its own chain instead of the whole warp.  The
// data dependences of the reference are kept exactly: stage s of frame t starts from the
// stage-s angles of frame t-1 (leg_inverse_kinematics.py:272) and from the frame built by
// stages 1..s-1 of frame t (kinematic_chain.py stage builders).
//
// IO is a policy: kp(t,row) -> key point (already aligned), put_angles(t, ang7),
// put_fk(t,row,v), and chain constants.
// ---------------------------------------------------------------------------------
template <typename R, typename IO>
struct ChainRunner {
    IO io;
    int64_t t, n_frame;
    int s;                       // current stage 0..3
    int lo, hi, gn_mask;         // stages lo..hi are solved; stages < lo are frozen at the angles read from io
    Mat3<R> A; Vec3<R> piv, o, rel;
    R ang0, ang1, ang2, ang3, ang4, ang5, ang6;   // scalars, not an array: `s` is a run-time index
    StageSolve<R> S;
    uint32_t nf0, nf1, nf2, nf3; int worst_status;

    SK_HD void begin_frame() {
        A = {{R(1), R(0), R(0)}, {R(0), R(1), R(0)}, {R(0), R(0), R(1)}};
        piv = {R(0), R(0), R(0)};
        o = io.kp(t, 0);
        for (int r = 0; r < 4; ++r) io.put_fk(t, r, o);
        s = 0;
    }
    SK_HD void begin_stage() {
        const Vec3<R> k = io.kp(t, s + 1);
        rel = {(k.x - o.x) - piv.x, (k.y - o.y) - piv.y, (k.z - o.z) - piv.z};
        const Vec3<R> q = mulT(A, rel);
        const R inf = Num<R>::inf();
        const int n_full = (s == 0) ? 4 : (s == 1) ? 6 : (s == 2) ? 8 : 9;
        const int gn = stage_mode(gn_mask, s);
        const bool frozen = s < lo;
        if (frozen) {   // kinematic_chain.py: earlier-stage DOFs are `fixed` links at angles[...][t]
            if (s == 0) { ang0 = io.angle_in(t, 0); ang1 = io.angle_in(t, 1); }
            else if (s == 1) { ang2 = io.angle_in(t, 2); ang3 = io.angle_in(t, 3); }
            else { ang4 = io.angle_in(t, 4); ang5 = io.angle_in(t, 5); }
        }
        if (s == 3) S.init(KIND_ZY, io.seg(3), R(0), q, R(0), ang6, -inf, inf, io.lb(6), io.ub(6), io.null_sq(3), n_full, gn);
        else {
            const int ia = 2 * s, ib = 2 * s + 1;
            const R a = (s == 0) ? ang0 : (s == 1) ? ang2 : ang4;
            const R b = (s == 0) ? ang1 : (s == 1) ? ang3 : ang5;
            if (frozen) S.init(s == 0 ? KIND_XY : KIND_ZY, io.seg(s), R(1), q, a, b, -inf, inf, -inf, inf, R(0), n_full, gn);
            else S.init(s == 0 ? KIND_XY : KIND_ZY, io.seg(s), R(1), q, a, b, io.lb(ia), io.ub(ia), io.lb(ib), io.ub(ib),
                        io.null_sq(s), n_full, gn);
        }
        if (frozen) S.status = ST_GTOL;
    }
    // stage_mask: contiguous bits lo..hi
    SK_HD void start(const IO& io_, int64_t n_frame_, const R* seed, int stage_mask_, int gn_mask_) {
        io = io_; n_frame = n_frame_; t = 0; s = 0; gn_mask = gn_mask_;
        lo = 0; while (lo < 3 && !((stage_mask_ >> lo) & 1)) ++lo;
        hi = 3; while (hi > 0 && !((stage_mask_ >> hi) & 1)) --hi;
        ang0 = seed[0]; ang1 = seed[1]; ang2 = seed[2]; ang3 = seed[3]; ang4 = seed[4]; ang5 = seed[5]; ang6 = seed[6];
        nf0 = nf1 = nf2 = nf3 = 0;
        worst_status = ST_GTOL;
        if (n_frame > 0) { begin_frame(); begin_stage(); }
    }
    SK_HD bool finished() const { return t >= n_frame; }

    // close the converged stage, open the next one (possibly of the next frame)
    SK_HD void advance() {
        if (s >= lo) {
            if (s == 0) { ang0 = S.x0; ang1 = S.angle_b(); nf0 += (uint32_t)S.nfev; }
            else if (s == 1) { ang2 = S.x0; ang3 = S.angle_b(); nf1 += (uint32_t)S.nfev; }
            else if (s == 2) { ang4 = S.x0; ang5 = S.angle_b(); nf2 += (uint32_t)S.nfev; }
            else { ang6 = S.angle_b(); nf3 += (uint32_t)S.nfev; }
            if (S.status == ST_MAXFEV && worst_status > ST_MAXFEV) worst_status = ST_MAXFEV;
            if (S.status == ST_NONFINITE) worst_status = ST_NONFINITE;
        }
        // next pivot = pivot + A w(x) = target + A f   (q = A^T rel, f = w - q)
        const Vec3<R> Af = mul(A, S.res());
        piv = {(piv.x + rel.x) + Af.x, (piv.y + rel.y) + Af.y, (piv.z + rel.z) + Af.z};
        const Vec3<R> jw = {piv.x + o.x, piv.y + o.y, piv.z + o.z};
        if (s == 0) { io.put_fk(t, 4, jw); io.put_fk(t, 5, jw); } else io.put_fk(t, 5 + s, jw);
        if (s < hi) {
            A = rotate_frame(A, S.kind_(), S.sa, S.ca, S.sin_b(), S.cos_b());
            ++s;
            begin_stage();
        } else {
            const R out7[7] = {limit_clamp(ang0, io.lb(0), io.ub(0)), limit_clamp(ang1, io.lb(1), io.ub(1)),
                               limit_clamp(ang2, io.lb(2), io.ub(2)), limit_clamp(ang3, io.lb(3), io.ub(3)),
                               limit_clamp(ang4, io.lb(4), io.ub(4)), limit_clamp(ang5, io.lb(5), io.ub(5)),
                               limit_clamp(ang6, io.lb(6), io.ub(6))};
            io.put_angles(t, out7, 2 * lo, hi == 3 ? 7 : 2 * hi + 2);
            ++t;
            if (t < n_frame) { begin_frame(); begin_stage(); }
        }
    }
    // one evaluation for this lane (no-op when the chain is finished)
    SK_HD void step() {
        if (finished()) return;
        if (S.done() && (gn_mask & 16) && s >= lo && S.escape()) { /* solve continues from the escape point */ }
        if (S.done()) advance();
        if (!finished() && !S.done()) S.trip();
    }
};

// Per-chain constants (one leg of one trial)
template <typename R> struct ChainParams {
    R seg[4];        // Coxa, Femur, Tibia, Tarsus lengths
    R lb[7], ub[7];  // DOF order: ThC_yaw, ThC_pitch, ThC_roll, CTr_pitch, CTr_roll, FTi_pitch, TiTa_pitch
    R null_sq[4];    // squared norm of the inert seed slots of stages 1-4
};

struct FrameStats { int nfev[4]; int status[4]; double iterate[7]; };   // iterate: the angles before limit_clamp

// Reference (serial) composition of the four stage solves of one frame; the kernels use
// the same pieces but interleave them across lanes.  `ang` in/out: previous frame's
// angles (warm start, leg_inverse_kinematics.py:272) -> this frame's.
// `kp`: 5 key points (row 0 = ThC origin).  `fk`: 9x3 output rows (may be null).
template <typename R>
SK_HD void solve_frame(const ChainParams<R>& P, const R* kp, R* ang, R* fk, FrameStats* fs, int stage_mask = 0xF, int gn_mask = 0) {
    const int n_full[4] = {4, 6, 8, 9};
    const Vec3<R> o = {kp[0], kp[1], kp[2]};
    Mat3<R> A = {{R(1), R(0), R(0)}, {R(0), R(1), R(0)}, {R(0), R(0), R(1)}};
    Vec3<R> piv = {R(0), R(0), R(0)};
    Vec3<R> joint[4];
    for (int s = 0; s < 4; ++s) {
        const Vec3<R> tgt = {kp[3 * (s + 1)] - o.x, kp[3 * (s + 1) + 1] - o.y, kp[3 * (s + 1) + 2] - o.z};
        const Vec3<R> rel = {tgt.x - piv.x, tgt.y - piv.y, tgt.z - piv.z};
        const Vec3<R> q = mulT(A, rel);
        const int kind = (s == 0) ? KIND_XY : KIND_ZY;
        const int ia = (s == 3) ? -1 : 2 * s, ib = (s == 3) ? 6 : 2 * s + 1;
        StageSolve<R> S;
        const R inf = Num<R>::inf();
        if (s == 3) S.init(kind, P.seg[s], R(0), q, R(0), ang[ib], -inf, inf, P.lb[ib], P.ub[ib], P.null_sq[s], n_full[s], stage_mode(gn_mask, s));
        else S.init(kind, P.seg[s], R(1), q, ang[ia], ang[ib], P.lb[ia], P.ub[ia], P.lb[ib], P.ub[ib], P.null_sq[s], n_full[s], stage_mode(gn_mask, s));
        if (stage_mask & (1 << s)) {
            while (!S.done()) S.trip();
            if ((gn_mask & 16) && S.escape()) while (!S.done()) S.trip();
        }
        if (s != 3) ang[ia] = limit_clamp(S.x0, P.lb[ia], P.ub[ia]);
        ang[ib] = limit_clamp(S.angle_b(), P.lb[ib], P.ub[ib]);
        if (fs) {
            fs->nfev[s] = S.nfev; fs->status[s] = S.status;
            if (s != 3) fs->iterate[ia] = (double)S.x0;
            fs->iterate[ib] = (double)S.angle_b();
        }
        // next pivot = pivot + A w = target + A f
        const Vec3<R> Af = mul(A, S.res());
        piv = {(piv.x + rel.x) + Af.x, (piv.y + rel.y) + Af.y, (piv.z + rel.z) + Af.z};
        joint[s] = piv;
        A = rotate_frame(A, kind, S.sa, S.ca, S.sin_b(), S.cos_b());
    }
    if (fk) {
        for (int r = 0; r < 4; ++r) { fk[3 * r] = o.x; fk[3 * r + 1] = o.y; fk[3 * r + 2] = o.z; }
        const int row[5] = {4, 5, 6, 7, 8};
        const int src[5] = {0, 0, 1, 2, 3};
        for (int k = 0; k < 5; ++k) {
            fk[3 * row[k]] = joint[src[k]].x + o.x; fk[3 * row[k] + 1] = joint[src[k]].y + o.y; fk[3 * row[k] + 2] = joint[src[k]].z + o.z;
        }
    }
}

}  // namespace seqik
