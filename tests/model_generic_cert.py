"""Stability classifier and float64 certificate of the generic 7-DOF solve (csrc/seqik_generic.cuh).  TEST TOOL.

Why a classifier.  The generic solve crawls through near-tied candidate steps (trf.py select_step), so the last bits of
its inputs can decide which iterates it visits.  Two builds of the same source that round a few operations differently
can therefore disagree on a solve without either being wrong.  The builds here differ in exactly two ways in float64:
  * the device's ``sincos`` and glibc's ``sin``/``cos`` may round the same argument 1 ulp apart;
  * the eight-lanes-per-chain mapping (seqik_generic_group.cuh) sums over the joints in butterfly order.
Every other operation is an explicit ``fma`` or an IEEE-rounded ``+ - * / sqrt`` on both (the library is compiled with
-fmad=false, the host build with -ffp-contract=off).  A 1-ulp change of one sine moves the claw of one evaluation by
about u64 |claw|; through the seven rotations of the chain such changes add up to some ten ulps, i.e. a relative
perturbation of ~2e-15 of the residual.  So a solve is called STABLE when the float64 host build, re-run with the
target moved by relative amounts of DELTA = 3e-15 and 6e-15 in both directions and in four directions in space (and the
seed, on joints strictly inside the box, scaled by 1 +- DELTA), gives the same status, the same number of evaluations
and angles within EPS_STABLE = 1e-11 rad of the unperturbed solve.  On a stable solve any two faithful builds must agree
to EPS = 1e-10 rad: ten times the spread the classifier admits, so a solve just inside the classifier's cut cannot make
a correct build fail.  (Measured on the grooming fixture: the angles of same-nfev copies differ by 2e-14 rad at the
median and 1.3e-11 rad at the 90th percentile; the tail comes from xtol endings, where the last step is 1e-8 |x|.)

Why a certificate.  Float32 cannot be held to a trace: its crawl ends by xtol in rounding noise (no grooming solve is
stable under a 2^-22 perturbation).  A returned float32 solve is therefore checked in float64 at the angles as
returned, against the target as the kernel formed it, fl32(kt - ko):
  * ``feasible``: lb < x < ub in working precision, no slack;
  * ``fk_err``: the returned FK rows against the float64 FK of the returned angles.  Bound
    FK_C u (|o| + L), L = sum of the segment lengths: the sin/cos of each joint carry a few ulps, each of the seven
    rotations and four segment offsets adds a few more, and the origin is added last (an ulp of |o|);
  * ``resid``: the claw residual |claw(x) - t|, on targets built as reachable that the float64 host build reaches
    (within REACHED; from a random seed the crawl can also end in a local minimum 0.2 - 1.5 mm away, in every
    build).  The float32 rounding floor is ~u L (the residual is formed from ~L-sized coordinates), but the crawl
    stops by ftol or xtol, and neither gives a rigorous bound: ftol ("the cost fell by less than 1e-8 of itself")
    fires on a linearly converging crawl wherever its contraction comes close to 1, and in float32 a cost decrease
    below ~u cost is lost to rounding, so the trust radius shrinks until xtol fires wherever the crawl has stalled.
    The bound is therefore empirical: RESID_MARGIN times the float64 host build's largest residual on the same
    workload, plus RESID_C u L.  The float32 host build stalls up to 4.7e-5 mm (~350 u L, a far-origin solve) from
    such targets; RESID_C = 1024 leaves a margin of about 3;
  * ``gscaled``: the Coleman-Li scaled gradient max |v * g|, v the distances to the bound the gradient points at.
    The gtol test the kernel applied saw g with an error of ~u |J| |f| + u |J| L (|J| <= L per column), so on a
    gtol ending the float64 value is at most gtol + GRAD_C u L^2 max v, on every target.  ftol and xtol endings
    have no gradient bound of their own (same reason as above; on a far or a zero target the float32 crawl stalls
    where the gradient is still 1e-4 - 1e-1).  On reached targets they get GRAD_MARGIN times the float64 host
    build's largest value on the workload plus the same rounding term (the float32 host build needs up to 12 times
    the float64 value: GRAD_MARGIN = 16).
The same checks with u = 2^-53 certify a float64 solve that is not stable.
"""
import numpy as np

import hostsim_build as H
import model_generic as MG

DELTA = 3e-15          # relative target / seed perturbation of the classifier (see the docstring)
EPS_STABLE = 1e-11     # rad: spread of the perturbed copies a stable solve may show
EPS = 1e-10            # rad: agreement required of two builds on a stable solve
U32, U64 = 2.0 ** -24, 2.0 ** -53
FK_C = 16              # FK rows: FK_C u (|o| + L)
RESID_C = 1024         # residual floor: RESID_C u L
GRAD_C = 64            # scaled gradient: GRAD_C u L^2 max v
RESID_MARGIN = 4.0     # margin on the float64 host build's largest residual of a workload
GRAD_MARGIN = 16.0     # margin on the float64 host build's largest scaled gradient of a workload (reached targets)
GTOL = 1e-8
UNKNOWN = -9           # status argument of check() where the termination status of each solve is not reported
REACHED = 1e-5         # mm: a target built as reachable counts as reached where the float64 host build gets this close

_DIRS = np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0], [0.0, 0.0, 1.0], [1.0, 1.0, 1.0]]) / np.array([[1], [1], [1], [3 ** 0.5]])


def perturbed_copies(prm, target):
    """The classifier's copies of a batch: [(prm, target)] * 6 (four target moves, two seed scalings)."""
    prm = np.asarray(prm, dtype=np.float64)
    target = np.asarray(target, dtype=np.float64)
    L = prm[:, 0:4].sum(axis=1)
    size = np.maximum(np.linalg.norm(target, axis=1), L)[:, None]
    out = []
    for k, e in zip((1, -1, 2, -2), _DIRS):
        out.append((prm, target * (1 + k * DELTA) + k * DELTA * size * e))
    seed, lb, ub = prm[:, 18:25], prm[:, 4:11], prm[:, 11:18]
    inner = (seed - lb > 1e-6) & (ub - seed > 1e-6)
    for k in (1, -1):
        p = prm.copy()
        p[:, 18:25] = np.where(inner, seed * (1 + k * DELTA), seed)
        out.append((p, target))
    return out


def host(prm, target, dtype=np.float64):
    """Host build of the one-lane solve: dict of angles, fk (relative to the origin), nfev, status."""
    a, fk, nf, st = H.solve_generic_many(prm, target, dtype=dtype)
    return dict(angles=a, fk=fk, nfev=nf, status=st)


def classify(prm, target):
    """float64 host solves of a batch and their stability: (result dict, stable mask (n,), spread (n,))."""
    base = host(prm, target)
    stable = np.ones(len(base["nfev"]), dtype=bool)
    spread = np.zeros(len(base["nfev"]))
    for p, t in perturbed_copies(prm, target):
        r = host(p, t)
        with np.errstate(invalid="ignore"):
            d = np.abs(r["angles"] - base["angles"]).max(axis=1)
        d = np.where(np.isnan(d), np.inf, d)
        spread = np.maximum(spread, d)
        stable &= (r["status"] == base["status"]) & (r["nfev"] == base["nfev"]) & (d <= EPS_STABLE)
    return base, stable, spread


def formed_target(origin, claw, dtype):
    """The target as the kernel forms it: key point minus origin, both in working precision (returned in float64)."""
    return (np.asarray(claw).astype(dtype) - np.asarray(origin).astype(dtype)).astype(np.float64)


def certificate(x, prm, target):
    """float64 quantities of returned solves x (n,7) for constants rows prm (n,32) and targets (n,3) (as formed)."""
    x = np.asarray(x, dtype=np.float64)
    prm = np.asarray(prm, dtype=np.float64)
    n = x.shape[0]
    cost, gs, resid, vmax = np.zeros(n), np.zeros(n), np.zeros(n), np.zeros(n)
    fk = np.zeros((n, 9, 3))
    for k in range(n):
        seg, lb, ub = prm[k, 0:4], prm[k, 4:11], prm[k, 11:18]
        if not np.isfinite(x[k]).all():
            cost[k] = gs[k] = resid[k] = np.nan
            fk[k] = np.nan
            continue
        f, J = MG.residual_jacobian(x[k], seg, target[k])
        g = J.T @ f
        v = np.where(g < 0, ub - x[k], np.where(g > 0, x[k] - lb, 1.0))
        cost[k] = 0.5 * f @ f
        gs[k] = np.abs(v * g).max()
        vmax[k] = np.abs(v).max()
        resid[k] = np.linalg.norm(f)
        fk[k] = MG.fk_rows(x[k], seg)
    return dict(cost=cost, gscaled=gs, resid=resid, fk=fk, vmax=vmax)


def feasible(x, prm, dtype):
    """lb < x < ub in working precision, no slack, per solve."""
    x = np.asarray(x).astype(dtype)
    prm = np.asarray(prm).astype(dtype)
    return ((x > prm[:, 4:11]) & (x < prm[:, 11:18])).all(axis=1)


def reference(host64, prm, target, reachable):
    """What the certificate needs from the float64 host solves of a workload: per-solve residual, the largest residual
    over the reachable targets it reached, and the largest scaled gradient."""
    c = certificate(host64["angles"], prm, target)
    reached = np.asarray(reachable, dtype=bool) & (c["resid"] <= REACHED)
    return dict(resid=c["resid"], resid_max=float(c["resid"][reached].max()) if reached.any() else 0.0,
                gscaled_max=float(c["gscaled"][reached].max()) if reached.any() else 0.0)


def check(x, fk, status, prm, origin, target, reachable, ref, dtype):
    """Certificate of returned solves (angles x, FK rows fk with the origin added, status) in working precision `dtype`
    against the float64 host references `ref` (``reference``) of the same workload.  Returns
    (dict of boolean masks of the solves that FAIL each check, dict of the largest ratio to each bound).  `status` is the
    termination status of each solve (1 = gtol) or UNKNOWN: the device reports only a per-chain summary, so there the
    scaled gradient is checked on reached targets only."""
    u = U32 if dtype == np.float32 else U64
    prm64 = np.asarray(prm).astype(dtype).astype(np.float64)
    origin = np.asarray(origin, dtype=np.float64)
    L = prm64[:, 0:4].sum(axis=1)
    c = certificate(x, prm64, target)
    fk_ref = c["fk"] + origin.astype(dtype).astype(np.float64)[:, None, :]
    fk_err = np.abs(np.asarray(fk, dtype=np.float64) - fk_ref).max(axis=(1, 2))
    fk_bound = FK_C * u * (np.abs(origin).max(axis=1) + L)
    resid_bound = RESID_MARGIN * ref["resid_max"] + RESID_C * u * L
    g_round = GRAD_C * u * L * L * c["vmax"]
    gtol_end = np.asarray(status) == 1
    g_bound = np.where(gtol_end, GTOL, GRAD_MARGIN * ref["gscaled_max"]) + g_round
    reachable = np.asarray(reachable, dtype=bool) & (ref["resid"] <= REACHED)
    fails = dict(
        feasible=~feasible(x, prm, dtype),
        fk=~(fk_err <= fk_bound),
        resid=reachable & ~(c["resid"] <= resid_bound),
        gscaled=(gtol_end | reachable) & ~(c["gscaled"] <= g_bound),
    )
    ratios = dict(fk=float(np.max(fk_err / fk_bound)),
                  resid=float(np.max(np.where(reachable, c["resid"] / resid_bound, 0.0))),
                  gscaled=float(np.max(np.where(gtol_end | reachable, c["gscaled"] / g_bound, 0.0))))
    return fails, ratios


# ----------------------------------------------------------------------------------------------------------
# workloads: one-frame solves as (prm (n,32), origin (n,3), claw key point (n,3), reachable (n,)), all float64
def _posture(rng, lb, ub, n):
    return lb + (ub - lb) * rng.uniform(0.05, 0.95, size=(n, 7))


def _claw(x, seg):
    return np.array([MG.chain_points(xi, seg)[1] for xi in x])


def _unit(rng, n):
    v = rng.normal(size=(n, 3))
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def edge_workloads(seg, lb, ub, seed7, n=24, rng_seed=0):
    """The edge families of the generic solve for one leg's constants, n solves each."""
    rng = np.random.default_rng(rng_seed)
    seg, lb, ub, seed7 = (np.asarray(a, dtype=np.float64) for a in (seg, lb, ub, seed7))
    L = seg.sum()

    def rows(seeds, null_sq=0.0):
        p = np.zeros((len(seeds), 32))
        p[:, 0:4], p[:, 4:11], p[:, 11:18], p[:, 18:25], p[:, 25] = seg, lb, ub, seeds, null_sq
        return p

    zero = np.zeros((n, 3))
    stage4 = np.tile(seed7, (n, 1))
    out = {}
    out["reach_1.3"] = (rows(stage4), zero, 1.3 * L * _unit(rng, n), np.zeros(n, bool))
    out["reach_100"] = (rows(stage4), zero, 100 * L * _unit(rng, n), np.zeros(n, bool))
    out["target_0"] = (rows(_posture(rng, lb, ub, n)), zero, zero.copy(), np.zeros(n, bool))
    out["target_1e-3"] = (rows(_posture(rng, lb, ub, n)), zero, 1e-3 * _unit(rng, n), np.zeros(n, bool))
    # postures with 1-4 joints on their limits (limits of 0 included: four of the seven are 0)
    post = _posture(rng, lb, ub, n)
    for k in range(n):
        j = rng.choice(7, size=1 + k % 4, replace=False)
        post[k, j] = np.where(rng.uniform(size=len(j)) < 0.5, lb[j], ub[j])
    out["limit_posture"] = (rows(_posture(rng, lb, ub, n)), zero, _claw(post, seg), np.zeros(n, bool))
    # seeds on a bound, within 1e-10 of one, and outside the box (the make_strictly_feasible midpoint path)
    seeds = _posture(rng, lb, ub, n)
    for k in range(n):
        j = rng.choice(7, size=1 + k % 3, replace=False)
        side = np.where(rng.uniform(size=len(j)) < 0.5, lb[j], ub[j])
        kind = k % 3
        if kind == 0:
            seeds[k, j] = side
        elif kind == 1:
            seeds[k, j] = side + np.where(side == lb[j], 1, -1) * 1e-10 * rng.uniform(0.1, 1.0, size=len(j))
        else:
            seeds[k, j] = side + np.where(side == lb[j], -1, 1) * rng.uniform(1e-3, 0.5, size=len(j))
    out["seed_bound"] = (rows(seeds), zero, _claw(_posture(rng, lb, ub, n), seg), np.ones(n, bool))
    out["null_sq"] = (rows(_posture(rng, lb, ub, n), null_sq=rng.uniform(0.01, 4.0, size=n)), zero,
                      _claw(_posture(rng, lb, ub, n), seg), np.ones(n, bool))
    o = 1e3 * _unit(rng, n)
    out["origin_1e3"] = (rows(_posture(rng, lb, ub, n)), o, o + _claw(_posture(rng, lb, ub, n), seg), np.ones(n, bool))
    return out


def grooming_workload(gold, grooming, li, seg, lb, ub, seed9):
    """Every solve of the generic fixture as a one-frame solve from the oracle's own seed (teacher forced)."""
    n = int(gold["n_frame"])
    teacher = np.vstack([np.asarray(seed9, dtype=np.float64)[None], gold["oracle_angles"][li][:-1]])
    prm = np.zeros((n, 32))
    prm[:, 0:4], prm[:, 4:11], prm[:, 11:18], prm[:, 18:25] = seg, lb, ub, teacher[:, 1:8]
    prm[:, 25] = teacher[:, 0] ** 2 + teacher[:, 8] ** 2
    pose = grooming["pose"][li][:n]
    return prm, pose[:, 0].astype(np.float64), pose[:, 4].astype(np.float64), np.ones(n, bool)


def maxfev_workload(seg, lb, ub, n=200, rng_seed=5):
    """Targets 1e-3 mm from the ThC from random interior seeds: most crawls run into the evaluation limit (status 0),
    and a few of those do so stably (the ending is reproducible to the last evaluation)."""
    rng = np.random.default_rng(rng_seed)
    seg, lb, ub = (np.asarray(a, dtype=np.float64) for a in (seg, lb, ub))
    prm = np.zeros((n, 32))
    prm[:, 0:4], prm[:, 4:11], prm[:, 11:18], prm[:, 18:25] = seg, lb, ub, _posture(rng, lb, ub, n)
    return prm, np.zeros((n, 3)), 1e-3 * _unit(rng, n), np.zeros(n, bool)
