"""The generic 7-DOF solve (csrc/seqik_generic.cuh) held to its float64 specification without a GPU.

tests/model_generic.py is the executable float64 specification; tests/hostsim runs the same .cuh source on the host.
On every solve the stability classifier of tests/model_generic_cert.py calls stable -- one that a perturbation of the
target and seed far below any tolerance does not move -- the two must take the same iterates: same status, same number
of evaluations, angles within EPS.  That is the link between the specification and the source the kernels compile.
The float32 host build is held to the float64 certificate on every solve, which validates the certificate's bounds
before they are applied to the device (tests/test_gpu_generic_cert.py).
"""
import numpy as np
import pytest

import model_generic as MG
import model_generic_cert as C
from test_generic_cpu import LEGS, consts

# measured stable fractions of the teacher-forced grooming solves (float64 host build): RF 0.874, LF 0.820
STABLE_FLOOR = {"RF": 0.85, "LF": 0.80}


def leg_workloads(leg, gold, grooming):
    _, seg, lb, ub, seed = consts(leg)
    w = C.edge_workloads(seg, lb, ub, seed[1:8])
    w["grooming"] = C.grooming_workload(gold, grooming, LEGS.index(leg), seg, lb, ub, seed)
    return w


@pytest.fixture(scope="module")
def classified(generic_gold, grooming_leg):
    """(leg, family) -> (workload, float64 host result, stable mask, spread)."""
    out = {}
    for leg in LEGS:
        for name, (prm, o, kp, reach) in leg_workloads(leg, generic_gold, grooming_leg).items():
            t = C.formed_target(o, kp, np.float64)
            base, stable, spread = C.classify(prm, t)
            out[leg, name] = ((prm, o, kp, reach, t), base, stable, spread)
    return out


def model_solve(prm, t):
    return MG.trf7(prm[0:4], t, prm[18:25], prm[4:11], prm[11:18], null_sq=prm[25])


def test_model_equals_host_on_stable_solves(classified):
    """Every stable solve of every workload (all 500 grooming frames of both legs, 24 solves of each edge family):
    the float64 model and the float64 host build return the same status, evaluation count and angles within EPS."""
    report = []
    for (leg, name), ((prm, o, kp, reach, t), base, stable, spread) in classified.items():
        for k in np.where(stable)[0]:
            x, st, nf, _ = model_solve(prm[k], t[k])
            assert st == base["status"][k] and nf == base["nfev"][k], (leg, name, k, st, nf, base["status"][k], base["nfev"][k])
            assert np.abs(x - base["angles"][k]).max() <= C.EPS, (leg, name, k, np.abs(x - base["angles"][k]).max())
        report.append(f"{leg} {name}: {stable.sum()}/{len(stable)} stable")
    print("\n".join(report))


@pytest.mark.parametrize("leg", LEGS)
def test_grooming_stable_fraction(classified, leg):
    """Most teacher-forced grooming solves are stable, so the trace equality of the GPU tests is not vacuous."""
    stable = classified[leg, "grooming"][2]
    print(f"{leg}: stable fraction {stable.mean():.3f}")
    assert stable.mean() >= STABLE_FLOOR[leg]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_host_meets_certificate(classified, dtype):
    """The host build in float32 (and float64) meets the certificate on every solve of every workload: angles strictly
    inside the box in working precision, FK rows, residual and scaled gradient within their bounds."""
    worst = {}
    for (leg, name), ((prm, o, kp, reach, t64), base, _, _) in classified.items():
        t = C.formed_target(o, kp, dtype)
        h = C.host(prm.astype(dtype), t.astype(dtype), dtype=dtype)
        assert np.isfinite(h["angles"]).all() and np.isfinite(h["fk"]).all()
        assert (h["status"] >= 0).all()
        fk = h["fk"].astype(np.float64) + o.astype(dtype).astype(np.float64)[:, None]
        fails, ratios = C.check(h["angles"], fk, h["status"], prm, o, t, reach, C.reference(base, prm, t64, reach), dtype)
        for key, bad in fails.items():
            assert not bad.any(), (leg, name, key, np.where(bad)[0], ratios)
        for key, r in ratios.items():
            worst[key] = max(worst.get(key, 0.0), r)
    print(f"{np.dtype(dtype).name} host build, largest ratio to each bound: " + ", ".join(f"{k} {v:.3g}" for k, v in worst.items()))


def test_classifier_flags_a_near_tie(classified):
    """A target placed on the boundary between two outcomes (bisected to the last bits between a solve and a perturbed
    copy that ends differently) is classified unstable, and the classifier is deterministic."""
    (prm, o, kp, reach, t), base, stable, _ = classified["RF", "grooming"]
    k = int(np.where(~stable)[0][0])
    p1 = prm[k:k + 1]
    ref = C.host(p1, t[k:k + 1])
    far = None
    for p, tc in C.perturbed_copies(p1, t[k:k + 1]):
        r = C.host(p, tc)
        if p is p1 and (r["nfev"][0] != ref["nfev"][0] or np.abs(r["angles"] - ref["angles"]).max() > C.EPS_STABLE):
            far = tc
            break
    assert far is not None
    lo, hi = t[k:k + 1].copy(), far.copy()
    for _ in range(60):
        mid = 0.5 * (lo + hi)
        if np.array_equal(mid, lo) or np.array_equal(mid, hi):
            break
        r = C.host(p1, mid)
        same = r["nfev"][0] == ref["nfev"][0] and np.abs(r["angles"] - ref["angles"]).max() <= C.EPS_STABLE
        lo, hi = (mid, hi) if same else (lo, mid)
    _, st, _ = C.classify(p1, lo)
    assert not st[0]
    _, st2, _ = C.classify(p1, hi)
    assert not st2[0]
    again, stable2, _ = C.classify(prm, t)
    assert np.array_equal(stable2, stable) and np.array_equal(again["angles"], base["angles"])


@pytest.mark.parametrize("status", [0, 2, 3])
def test_model_and_host_agree_on_endings(classified, status):
    """The MAXFEV (0), ftol (2) and xtol (3) endings: each occurs stably, and there the model ends the same way as the
    host build, at the same evaluation (900 for MAXFEV) with the same angles."""
    if status == 0:
        _, seg, lb, ub, _ = consts("RF")
        prm, o, kp, _ = C.maxfev_workload(seg, lb, ub)
        t = C.formed_target(o, kp, np.float64)
        base, stable, _ = C.classify(prm, t)
        cases = [(prm, t, base, k) for k in np.where(stable & (base["status"] == 0))[0]]
    else:
        cases = [(w[0], w[4], base, k) for (w, base, stable, _) in classified.values()
                 for k in np.where(stable & (base["status"] == status))[0]][:20]
    assert cases, f"no stable solve ends with status {status}"
    for prm, t, base, k in cases:
        x, st, nf, _ = model_solve(prm[k], t[k])
        assert st == status and nf == base["nfev"][k] and np.abs(x - base["angles"][k]).max() <= C.EPS
    print(f"status {status}: {len(cases)} stable solves")
