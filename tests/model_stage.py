"""Float64 model of one stage solve of the leg solver, vectorised over leg-frames.  TEST TOOL.

A stage points one segment of length L, on a two-axis gimbal about a fixed pivot, at a target q: it minimises
f(a, b) = 0.5 |w(a, b) - q|^2 over the box lb <= (a, b) <= ub, with w the end point of ``model_trf2.stage_w``
(kind 0: Rx(a) Ry(b) (0,0,-L), stage 1; kind 1: Rz(a) Ry(b) (0,0,-L), stages 2-3; kind 2: Ry(b) (0,0,-L), stage 4,
`a` inert).  The frames are those of ``oracle.seqik_oracle.fk_closed_form``.

The model is TEACHER-FORCED: the pivot and rotation of stage k are built in float64 from the solver's own float32
angles of stages < k, and the target is the float32 key point the kernel read, cast to float64.  Each stage solve is
then checked against its own problem, and errors do not compound across stages.

The error bound the tests apply (u = 2^-24, float32 unit roundoff; x* the polished point; t the key point relative to
the ThC origin and p the pivot, so that the kernel's target is A^T (t - p); sigma = 1 + (|t| + |p|) / L):

  * cost:    f(x) - f(x*) <= ftol_term + C u sigma L (L + |q|),                      C = 2 K
  * angles:  |b - b*| <= K u sigma + theta,  |a - a*| <= K u sigma / |sin b*| + theta   (conditioned frames),
             theta = theta_ftol + theta_gtol
  * limits:  lb <= x <= ub in float32, no slack;
  * stationarity: the polish moves no angle by more than max(1e-3 rad, sqrt(2 ftol_term / max(lambda_min, 1e-2 L^2)))
    -- more means that the solver's answer is not a stationary point at all.  Where sin b* < 0.05 the move of `a`
    counts scaled by |sin b*| / 0.05: at sin b* = 0 any `a` is a minimiser.  The second term is the ftol gap in angle
    in a flat valley (an ftol stop there is legitimately that far from the minimiser); lambda_min is floored at
    1e-2 L^2 so that the limit stays finite on singular and negative-curvature frames: it never exceeds
    sqrt(2 ftol f / (1 - 0.995^2) / (1e-2 L^2)) ~ 0.014 sqrt(f) / L rad, f the cost.

K = 64 follows from the float32 error sources of one stage, each stated as a multiple of u:
  - the target q = A^T ((k - o) - p), k the key point: 2 roundings of |t| + |p| for rel, 3 for the product with A; the pivot p is an
    accumulation of one product A w (3 u) per earlier stage, <= 9 u; the frame A went through <= 3 rotate_frame products
    (2 u per column each) with sin/cos that are re-derived (Cody-Waite + minimax polynomial, <= 2 u) or carried for at
    most SEQIK_RESYNC = 32 frames (one angle-addition update per frame, a random walk of ~1 u per update, <= 6 u):
    3 (2 + 2) + 6 = 18 u.  Together 2 + 3 + 9 + 18 = 32 u of |t| + |p|.  The minimiser's direction moves by
    |dq| / |q| <= 2 |dq| / L on conditioned frames (|q| >= L / 2), i.e. by <= 64 u (|t| + |p|) / L = 64 u (sigma - 1);
  - the solve itself: the closed-form warm step's three rsqrt.approx (<= 2 ulp each) on sin(d / 2), |d| <= 0.91 rad,
    ~6 u; the s^15 truncation of the arcsine series below |s| < 0.44 (< 3e-8, doubled: 1 u); the float32 angle
    (<= 0.5 u |x|, |x| <= pi: 2 u) and its sin/cos (2 u); a gtol stop away from limits (the gradient below 1e-8, i.e.
    < 1e-8 / L^2 ~ 2 u on L >= 0.3): 13 u <= 64 u.
  So the angle error is below 64 u (sigma - 1) + 64 u = K u sigma.
The cost bound is first order: at an active limit the gradient does not vanish, |g| <= L (L + |q|), and the angle
error above multiplies it; the factor 2 covers the second-order term 0.5 lambda_max |dx|^2 with lambda_max <= L (L + |q|).

ftol_term covers solves that iterate and stop on scipy's ftol = 1e-8, as the reference does: the last step reduced the
cost by less than ftol f; with the Gauss-Newton iteration contracting the cost gap by rho^2 per step (rho the spectral
radius of I - G^-1 H at x*, G the Gauss-Newton matrix, H the exact Hessian, capped at 0.995 - scipy's theta) the
remaining gap is below ftol f / (1 - rho^2).  theta_ftol = sqrt(2 ftol_term / lambda_min) is the same gap in angle.

Conditioned frames: the reduced Hessian at x* is at least a quarter of the Gauss-Newton one in every free direction
(Newton's admission test in plan()), |sin b*| >= 0.05 where `a` is free, and |q| >= L / 2 (the assumption of the
derivation of K below).  Elsewhere (the CTr_pitch = 0 episodes,
negative curvature, targets closer than L / 2 to the pivot) only the cost bound and the stationarity test apply.
theta_gtol = gtol / (v lambda_min), v = min(1, distance to a limit), is added to the bound of a free angle: scipy's
gtol = 1e-8 test is on the Coleman-Li scaled gradient |g| v, so near a limit it stops with |g| up to gtol / v, as the
reference does; an angle whose minimiser lies ON a limit is allowed to stop gtol / |g| short of it for the same reason.
"""
import numpy as np

U32 = 2.0 ** -24
K_ANGLE = 64.0
C_COST = 2.0 * K_ANGLE
FTOL = 1e-8
RHO_MAX = 0.995
POLISH_MOVE_MAX = 1e-3
SNAP = 1e-9
SIN_B_MIN = 0.05
LAM_FLOOR = 1e-2
GTOL = 1e-8
CURV_MIN = 0.25
KINDS = (0, 1, 1, 2)


def _rx(t):
    c, s = np.cos(t), np.sin(t)
    o, z = np.ones_like(t), np.zeros_like(t)
    return np.stack([np.stack([o, z, z], -1), np.stack([z, c, -s], -1), np.stack([z, s, c], -1)], -2)


def _ry(t):
    c, s = np.cos(t), np.sin(t)
    o, z = np.ones_like(t), np.zeros_like(t)
    return np.stack([np.stack([c, z, s], -1), np.stack([z, o, z], -1), np.stack([-s, z, c], -1)], -2)


def _rz(t):
    c, s = np.cos(t), np.sin(t)
    o, z = np.ones_like(t), np.zeros_like(t)
    return np.stack([np.stack([c, -s, z], -1), np.stack([s, c, z], -1), np.stack([z, z, o], -1)], -2)


def stage_w(kind, L, a, b):
    """Vectorised ``model_trf2.stage_w`` + second derivatives: w, w_a, w_b, w_aa, w_ab, w_bb, each (..., 3)."""
    sa, ca, sb, cb = np.sin(a), np.cos(a), np.sin(b), np.cos(b)
    z = np.zeros_like(a * b)
    st = lambda *c: np.stack(np.broadcast_arrays(*c), -1)
    if kind == 0:
        w = st(-L * sb, L * cb * sa, -L * cb * ca)
        wa = st(z, L * cb * ca, L * cb * sa)
        wb = st(-L * cb, -L * sb * sa, L * sb * ca)
        waa = st(z, -L * cb * sa, L * cb * ca)
        wab = st(z, -L * sb * ca, -L * sb * sa)
        wbb = st(L * sb, -L * cb * sa, L * cb * ca)
    elif kind == 1:
        w = st(-L * sb * ca, -L * sb * sa, -L * cb)
        wa = st(L * sb * sa, -L * sb * ca, z)
        wb = st(-L * cb * ca, -L * cb * sa, L * sb)
        waa = st(L * sb * ca, L * sb * sa, z)
        wab = st(L * cb * sa, -L * cb * ca, z)
        wbb = -w
    else:
        w = st(-L * sb, z, -L * cb)
        wa = st(z, z, z)
        wb = st(-L * cb, z, L * sb)
        waa = wab = st(z, z, z)
        wbb = -w
    return w, wa, wb, waa, wab, wbb


def derivs(kind, L, q, a, b):
    """cost (M,), gradient (M, 2), exact Hessian (M, 2, 2), Gauss-Newton matrix (M, 2, 2) of 0.5 |w - q|^2."""
    w, wa, wb, waa, wab, wbb = stage_w(kind, L, a, b)
    f = w - q
    cost = 0.5 * np.einsum("...i,...i", f, f)
    g = np.stack([np.einsum("...i,...i", wa, f), np.einsum("...i,...i", wb, f)], -1)
    J = np.stack([wa, wb], -1)                                           # (M, 3, 2)
    G = np.einsum("...ki,...kj->...ij", J, J)
    C = np.stack([np.stack([np.einsum("...i,...i", waa, f), np.einsum("...i,...i", wab, f)], -1),
                  np.stack([np.einsum("...i,...i", wab, f), np.einsum("...i,...i", wbb, f)], -1)], -2)
    return cost, g, G + C, G


def frames(pose, ang, seg):
    """Teacher-forced problems of the four stages.  pose (M, 5, 3), ang (M, 7) as the kernel read / wrote them,
    seg (M, 4) or (4,).  Returns a list of four dicts: q (M, 3), x (M, 2) the solver's (a, b), t and p (M, 3)."""
    pose = np.asarray(pose, dtype=np.float64)
    ang = np.asarray(ang, dtype=np.float64)
    seg = np.broadcast_to(np.asarray(seg, dtype=np.float64), (pose.shape[0], 4))
    t = pose[:, 1:5] - pose[:, None, 0]
    down = lambda L: np.stack([np.zeros_like(L), np.zeros_like(L), -L], -1)
    R = np.broadcast_to(np.eye(3), (pose.shape[0], 3, 3))
    p = np.zeros((pose.shape[0], 3))
    gimbal = ((_rx, _ry, 0, 1), (_rz, _ry, 2, 3), (_rz, _ry, 4, 5), (None, _ry, None, 6))
    out = []
    for k in range(4):
        q = np.einsum("mji,mj->mi", R, t[:, k] - p)
        ra, rb, ia, ib = gimbal[k]
        a = np.zeros(pose.shape[0]) if ia is None else ang[:, ia]
        out.append(dict(q=q, x=np.stack([a, ang[:, ib]], -1), t=t[:, k], p=p.copy(), L=seg[:, k]))
        R = R @ rb(ang[:, ib]) if ra is None else R @ ra(a) @ rb(ang[:, ib])
        p = p + np.einsum("mij,mj->mi", R, down(seg[:, k]))
    return out


def polish(kind, L, q, x0, lb, ub, tol=1e-14, max_iter=200):
    """Projected damped Newton / Levenberg-Marquardt on the box from x0, to a step below `tol`: returns x* (M, 2).
    Variables on a limit with the gradient pointing out of the box are held; the free block takes the Newton step of the
    exact Hessian, shifted to positive definite and damped until the cost decreases.  A zero gradient gives a zero step,
    so a first-order KKT point (a saddle on the CTr_pitch = 0 singularity included) stays where it is, as with TRF."""
    x = np.clip(np.array(x0, dtype=np.float64), lb, ub)
    M = x.shape[0]
    free_a = np.full(M, kind != 2)
    mu = np.zeros(M)
    live = np.ones(M, dtype=bool)
    for _ in range(max_iter):
        if not live.any():
            break
        i = np.where(live)[0]
        Li = L[i] if np.ndim(L) else L
        cost, g, H, G = derivs(kind, Li, q[i], x[i, 0], x[i, 1])
        held = ((x[i] <= lb[i]) & (g > 0)) | ((x[i] >= ub[i]) & (g < 0))
        held[:, 0] |= ~free_a[i]
        fr = ~held
        Hf = H * (fr[:, :, None] & fr[:, None, :]) + np.eye(2) * (~fr)[:, :, None]
        gf = np.where(fr, g, 0.0)
        lmin = np.linalg.eigvalsh(Hf)[:, 0]
        scale = np.abs(np.einsum("mii->mi", Hf)).max(1) + 1e-300
        shift = np.maximum(0.0, -lmin) + mu[i] + (lmin <= 0) * 1e-9 * scale
        step = -np.linalg.solve(Hf + shift[:, None, None] * np.eye(2), gf[..., None])[..., 0]
        xn = np.clip(x[i] + step, lb[i], ub[i])
        cn = derivs(kind, Li, q[i], xn[:, 0], xn[:, 1])[0]
        ok = cn <= cost
        moved = np.abs(xn - x[i]).max(1)
        x[i[ok]] = xn[ok]
        mu[i[ok]] = 0.0
        mu[i[~ok]] = np.maximum(10.0 * mu[i[~ok]], 1e-6 * scale[~ok])
        live[i[ok & (moved < tol)]] = False
        live[i[~ok & (mu[i] > 1e6 * scale)]] = False
    return x


def analyse(kind, L, q, x_dev, lb, ub, t, p):
    """Everything the bound needs for one stage: the polished point, cost gap, per-angle errors and their bounds,
    conditioning and the flags.  All arrays (M,) or (M, 2)."""
    L = np.asarray(L, dtype=np.float64)
    # the solver parks an angle that reached a limit 1e-10 (make_strictly_feasible) or one float64 ulp inside it: the
    # polish starts from the limit itself, so that a CTr_pitch = 0 corner has an exactly vanishing `a`-gradient
    snap, snap_u = SNAP * np.maximum(1.0, np.abs(lb)), SNAP * np.maximum(1.0, np.abs(ub))
    x0 = np.where(np.abs(x_dev - lb) <= snap, lb, np.where(np.abs(ub - x_dev) <= snap_u, ub, x_dev))
    xs = polish(kind, L, q, x0, lb, ub)
    f_dev, _, _, _ = derivs(kind, L, q, x_dev[:, 0], x_dev[:, 1])
    f_st, g, H, G = derivs(kind, L, q, xs[:, 0], xs[:, 1])
    held = ((xs <= lb) & (g > 0)) | ((xs >= ub) & (g < 0))
    held[:, 0] |= kind == 2
    fr = ~held
    Hf = H * (fr[:, :, None] & fr[:, None, :]) + np.eye(2) * (~fr)[:, :, None]
    lam = np.linalg.eigvalsh(Hf)
    # internal-frame sin b: |d w / d a| = L |sin b'| (stage 1: b' = b - pi/2)
    sin_b = np.abs(np.cos(xs[:, 1])) if kind == 0 else np.abs(np.sin(xs[:, 1]))
    d = np.sqrt(np.maximum(np.einsum("mii->mi", G), 1e-300))
    S = Hf / (np.where(fr, d, 1.0)[:, :, None] * np.where(fr, d, 1.0)[:, None, :])
    ls = np.linalg.eigvalsh(S)
    rho = np.minimum(np.abs(1.0 - ls).max(1), RHO_MAX)
    ftol_term = FTOL * np.maximum(f_dev, 0.0) / (1.0 - rho * rho)
    lam_min = lam[:, 0]
    theta_ftol = np.sqrt(2.0 * ftol_term / np.maximum(lam_min, 1e-300))
    neg_curv = lam_min < 0
    qn = np.linalg.norm(q, axis=1)
    sigma = 1.0 + (np.linalg.norm(t, axis=1) + np.linalg.norm(p, axis=1)) / L
    conditioned = ~neg_curv & (ls[:, 0] >= CURV_MIN) & (held[:, 0] | (sin_b >= SIN_B_MIN)) & (qn >= 0.5 * L)
    # scipy's gtol test is on the Coleman-Li scaled gradient |g_i| v_i, v_i the distance to the limit the anti-gradient
    # points at (1 without one): near a limit it admits |g_i| up to gtol / v_i, an angle gtol / (v_i lambda_min) short
    v = np.minimum(np.minimum(np.minimum(xs - lb, ub - xs), np.minimum(x_dev - lb, ub - x_dev)), 1.0)
    # ... and an angle whose minimiser is ON a limit stops short of it by up to gtol / |g_i| (there |g_i| v_i < gtol)
    theta_gtol = np.where(fr, GTOL / np.maximum(v * np.maximum(lam_min, 1e-300)[:, None], 1e-300),
                          np.where(held & (np.arange(2) >= (kind == 2)), GTOL / np.maximum(np.abs(g), 1e-300), 0.0))
    ang_bound_b = K_ANGLE * U32 * sigma + theta_ftol + theta_gtol[:, 1]
    ang_bound_a = K_ANGLE * U32 * sigma / np.maximum(sin_b, 1e-300) + theta_ftol + theta_gtol[:, 0]
    cost_bound = ftol_term + C_COST * U32 * sigma * L * (L + qn)
    return dict(x_star=xs, gap=f_dev - f_st, cost_bound=cost_bound, err=np.abs(x_dev - xs),
                bound=np.stack([ang_bound_a, ang_bound_b], -1), conditioned=conditioned, singular=~conditioned,
                neg_curv=neg_curv, sin_b=sin_b, sigma=sigma, lam_min=lam_min, cost=f_dev,
                # `a` is undetermined where sin b* -> 0 (the CTr_pitch / FTi_pitch = 0 corners): its move there counts by
                # the end point's motion it causes, |da| |sin b*|, relative to that at |sin b*| = 0.05
                moved=np.maximum(np.abs(x_dev - xs)[:, 1], np.abs(x_dev - xs)[:, 0] * np.minimum(1.0, sin_b / SIN_B_MIN)),
                move_max=np.maximum(POLISH_MOVE_MAX, np.sqrt(2.0 * ftol_term / np.maximum(lam_min, LAM_FLOOR * L * L))))


def check_chain(pose, ang, prm, stages=(1, 2, 3, 4)):
    """All stage checks of one chain's frames: pose (F, 5, 3) and ang (F, 7) as float32 arrays the kernel read and
    wrote, prm the float32 params row.  Returns per stage a dict of worst ratios and counts (see `worst`), and raises
    AssertionError with the offending frames when a bound is broken."""
    pose = np.asarray(pose)
    ang32 = np.asarray(ang, dtype=np.float32)
    prm = np.asarray(prm, dtype=np.float32)
    lb32, ub32 = prm[4:11], prm[11:18]
    assert ((ang32 >= lb32) & (ang32 <= ub32)).all(), np.argwhere(~((ang32 >= lb32) & (ang32 <= ub32)))[:5]
    pr = frames(pose, ang32, prm[0:4])
    lb, ub = lb32.astype(np.float64), ub32.astype(np.float64)
    out = {}
    for s in stages:
        k = s - 1
        st = pr[k]
        if s == 4:
            blo, bhi = np.array([0.0, lb[6]]), np.array([0.0, ub[6]])
        else:
            blo, bhi = lb[2 * k:2 * k + 2], ub[2 * k:2 * k + 2]
        M = pose.shape[0]
        r = analyse(KINDS[k], st["L"], st["q"], st["x"], np.broadcast_to(blo, (M, 2)), np.broadcast_to(bhi, (M, 2)),
                    st["t"], st["p"])
        out[s] = r
    return out


def worst(res):
    """Largest ratios to the bounds over a check_chain result (or a list of them), and the frame counts."""
    res = res if isinstance(res, list) else [res]
    w = dict(cost=0.0, angle=0.0, moved=0.0, frames=0, singular=0, stage={})
    for r in res:
        for s, a in r.items():
            c = a["conditioned"]
            w["cost"] = max(w["cost"], float((a["gap"] / a["cost_bound"]).max(initial=0.0)))
            rat = a["err"] / a["bound"]
            if s == 4:
                rat = rat[:, 1:]
            w["angle"] = max(w["angle"], float(rat[c].max(initial=0.0)))
            # per stage: the largest angle ratio and the median rounding part of the b bound (K u sigma, rad) -- what an
            # error must exceed to be seen on that stage
            ws = w["stage"].setdefault(s, dict(angle=0.0, bound=[]))
            ws["angle"] = max(ws["angle"], float(rat[c].max(initial=0.0)))
            ws["bound"].append(np.median(K_ANGLE * U32 * a["sigma"]) if len(c) else np.nan)
            w["moved"] = max(w["moved"], float((a["moved"] / a["move_max"]).max(initial=0.0)))
            w["frames"] += len(c)
            w["singular"] += int((~c).sum())
    return w


def merge(ws):
    """Worst of several `worst` results; per stage the largest angle ratio and the median rounding bound."""
    out = dict(cost=0.0, angle=0.0, moved=0.0, frames=0, singular=0, stage={})
    for w in ws:
        for k in ("cost", "angle", "moved"):
            out[k] = max(out[k], w[k])
        out["frames"] += w["frames"]; out["singular"] += w["singular"]
        for s, v in w["stage"].items():
            o = out["stage"].setdefault(s, dict(angle=0.0, bound=[]))
            o["angle"] = max(o["angle"], v["angle"]); o["bound"] += v["bound"]
    return out


def report(label, w):
    """One line per workload: worst ratios, then per stage the largest angle ratio / median K u sigma."""
    st = "  ".join(f"s{s} {v['angle']:.2f}/{np.nanmedian(v['bound']):.1e}" for s, v in sorted(w["stage"].items()))
    return (f"{label:44s} cost {w['cost']:.3g}  angle {w['angle']:.3g}  stationarity {w['moved']:.3g}  "
            f"frames {w['frames']}  unconditioned {w['singular']}  |  {st}")


def assert_within(res, label=""):
    """Every bound of a check_chain result holds; returns `worst` of it."""
    for s, a in res.items():
        bad = np.where(a["gap"] > a["cost_bound"])[0]
        assert len(bad) == 0, (label, "cost", s, bad[:5], a["gap"][bad[:5]], a["cost_bound"][bad[:5]])
        rat = a["err"] / a["bound"]
        if s == 4:
            rat = rat[:, 1:]
        bad = np.where(a["conditioned"] & (rat > 1).any(1))[0]
        assert len(bad) == 0, (label, "angle", s, bad[:5], a["err"][bad[:5]], a["bound"][bad[:5]])
        bad = np.where(a["moved"] > a["move_max"])[0]
        assert len(bad) == 0, (label, "stationarity", s, bad[:5], a["moved"][bad[:5]])
    return worst(res)
