"""The float64 stage model (tests/model_stage.py) against the oracle and scipy, and its error bound calibrated on the float32
host build of csrc/seqik_core.cuh -- the arithmetic of every solver kernel but for the approximate reciprocal and square
root of the device (<= 2 ulp), so that the bound is shown to hold before it is applied to the B200's results."""
import numpy as np
import pytest
from scipy.optimize import least_squares

import hostsim_build as H
import model_stage as MS
from oracle import seqik_oracle as O

GN = 0b11111111       # SEQIK_FLAG_DEFAULT
GN_REF = 0b0111111    # SEQIK_FLAG_REFERENCE_ITERATES


def test_stage_residual_equals_the_oracle_chain():
    """|w(a, b) - q| of every teacher-forced stage equals |FK - target| of the oracle's build_chain + forward_kinematics
    for that stage (earlier DOFs as fixed links), to 1e-12, on random angles inside the limits."""
    from seqikpy_b200 import synthetic as S
    size, bounds, init = S.chain_constants()
    rng = np.random.default_rng(3)
    leg = "RM"
    lb = np.array([bounds[f"{leg}_{d}"][0] for d in O.DOF_ORDER])
    ub = np.array([bounds[f"{leg}_{d}"][1] for d in O.DOF_ORDER])
    seg = np.array([size[f"{leg}_{s}"] for s in O.SEGMENTS])
    n = 40
    ang = rng.uniform(lb, ub, (n, 7))
    pose = np.zeros((n, 5, 3))
    pose[:, 0] = rng.normal(0, 1, (n, 3))
    pose[:, 1:] = pose[:, None, 0] + rng.normal(0, 1.0, (n, 4, 3))
    probs = MS.frames(pose, ang, seg)
    angles = {f"Angle_{leg}_{d}": ang[:, i] for i, d in enumerate(O.DOF_ORDER)}
    for s in (1, 2, 3, 4):
        p = probs[s - 1]
        w = MS.stage_w(MS.KINDS[s - 1], seg[s - 1], p["x"][:, 0], p["x"][:, 1])[0]
        ours = np.linalg.norm(w - p["q"], axis=1)
        for t in range(n):
            links = O.build_chain(s, leg, size, bounds, angles, t)
            x = np.zeros(len(links))
            for dof in O.STAGE_DOFS[s]:
                x[[l.name for l in links].index(f"{leg}_{dof}")] = angles[f"Angle_{leg}_{dof}"][t]
            ref = O.forward_kinematics(links, x)[:3, 3] - (pose[t, s] - pose[t, 0])
            assert abs(np.linalg.norm(ref) - ours[t]) < 1e-12, (s, t)


def _scipy_stage(kind, L, q, x0, lb, ub):
    na = 0 if kind == 2 else 2
    sl = slice(1, 2) if kind == 2 else slice(0, 2)

    def fun(z):
        x = np.array([0.0, z[0]]) if kind == 2 else z
        return MS.stage_w(kind, L, np.array([x[0]]), np.array([x[1]]))[0][0] - q
    r = least_squares(fun, x0[sl], bounds=(lb[sl], ub[sl]), xtol=1e-15, ftol=1e-15, gtol=1e-15, method="trf")
    return (np.array([0.0, r.x[0]]) if na == 0 else r.x), r.cost


@pytest.mark.parametrize("kind, case", [(k, c) for k in (0, 1) for c in ("interior", "a_on_limit", "b_on_limit", "both_on_limits")]
                         + [(2, "interior"), (2, "b_on_limit")])
def test_polish_equals_scipy(kind, case):
    """The polish lands where scipy's TRF with tolerances 1e-15 lands, from the same start, on random boxes."""
    rng = np.random.default_rng(100 + 7 * kind + len(case))
    L = 0.6
    n, xs, cs, ref_x, ref_c = 60, [], [], [], []
    lbs, ubs = [], []
    for _ in range(n):
        x_true = np.array([rng.uniform(-1.2, 1.2), rng.uniform(-2.4, -0.4)])
        if kind == 2:
            x_true[0] = 0.0
        w = MS.stage_w(kind, L, x_true[:1], x_true[1:])[0][0]
        q = w * rng.uniform(0.8, 1.3) + rng.normal(0, 0.05, 3)
        half = np.array([rng.uniform(0.3, 0.8), rng.uniform(0.3, 0.8)])
        lb, ub = x_true - half, x_true + half
        if case in ("a_on_limit", "both_on_limits"):                  # the box cuts the minimiser off in `a`
            lb[0], ub[0] = x_true[0] + 0.1, x_true[0] + 0.9
        if case in ("b_on_limit", "both_on_limits"):
            lb[1], ub[1] = x_true[1] - 0.9, x_true[1] - 0.1
        if kind == 2:
            lb[0] = ub[0] = 0.0
        x0 = lb + rng.uniform(0.2, 0.8, 2) * (ub - lb)
        rx, rc = _scipy_stage(kind, L, q, x0, lb, ub)
        xp = MS.polish(kind, np.array([L]), q[None], x0[None], lb[None], ub[None])[0]
        xs.append(xp); ref_x.append(rx); ref_c.append(rc)
        cs.append(MS.derivs(kind, L, q[None], xp[:1], xp[1:])[0][0])
        lbs.append(lb); ubs.append(ub)
    xs, ref_x, cs, ref_c = map(np.asarray, (xs, ref_x, cs, ref_c))
    # both are local methods: from a start between two basins they may settle in different ones (a few per cent)
    same = (np.abs(cs - ref_c) < 1e-12) & (np.abs(xs - ref_x).max(1) < 1e-7)
    assert same.mean() >= 0.9, (same.mean(), np.abs(xs - ref_x).max(0))
    on = (np.isclose(xs, np.asarray(lbs), atol=1e-12) | np.isclose(xs, np.asarray(ubs), atol=1e-12))[same]
    on[:, 0] &= kind != 2                                              # (kind 2: `a` is inert, its box is [0, 0])
    if case in ("a_on_limit", "both_on_limits"):
        assert on[:, 0].mean() > 0.5
    if case in ("b_on_limit", "both_on_limits"):
        assert on[:, 1].mean() > 0.5
    if case == "interior":
        assert on.mean() < 0.2


def _report(label, ws):
    print(MS.report(label, MS.merge(ws)))


def test_host_build_stays_within_the_bound(grooming_leg, locomotion):
    """The bound of model_stage.py on the float32 host build: the frame-parallel block schedule (default flags) on the
    48 synthetic chains x 1000 frames, both grooming legs and the locomotion recording; the frame-by-frame solves on one
    synthetic trial; the serial solves with the reference-iterates flags (scipy's iteration throughout) on the grooming
    legs.  Every angle inside its limits with no slack, every stage's cost and angles within the bound, no polish move
    beyond the stationarity limit.  Run with -s for the worst ratios, per workload and per stage."""
    from seqikpy_b200 import data as D, synthetic as S
    from seqikpy_b200.kinematic_chain import KinematicChainSeq
    from seqikpy_b200.utils import calculate_body_size
    size, bounds, init = S.chain_constants()
    chain = KinematicChainSeq(bounds, list(S.LEGS), size)
    res = []
    for tr in range(8):
        pose = S.make_trial(tr, 1000).astype(np.float32)
        for li, leg in enumerate(S.LEGS):
            row = chain.pack_chain_params(leg, init[leg]).astype(np.float32)
            a, _, _, _ = H.run_block_f32(pose[:, li], row, GN)
            res.append(MS.assert_within(MS.check_chain(pose[:, li], a, row), ("synthetic", tr, leg)))
    _report("synthetic 48 x 1000", res)
    res = []                                       # frame-by-frame solves (the one-lane-per-chain kernel's arithmetic)
    pose = S.make_trial(0, 1000).astype(np.float32)
    for li, leg in enumerate(S.LEGS):
        row = chain.pack_chain_params(leg, init[leg]).astype(np.float32)
        a = H.solve_chain(pose[:, li], row[0:4], row[4:11], row[11:18], row[25:29], row[18:25], gn_mask=GN)[0]
        res.append(MS.assert_within(MS.check_chain(pose[:, li], a, row), ("synthetic, serial", leg)))
    _report("synthetic 6 x 1000, serial", res)
    chain_g = KinematicChainSeq(D.BOUNDS, ["RF", "LF"], None)
    for flags, name in ((GN, "block"), (GN_REF, "serial, reference iterates")):
        res = []
        for li, leg in enumerate(("RF", "LF")):
            row = chain_g.pack_chain_params(leg, D.INITIAL_ANGLES[leg]).astype(np.float32)
            pose = grooming_leg["pose"][li].astype(np.float32)
            if flags == GN:
                a = H.run_block_f32(pose, row, GN)[0]
            else:
                a = H.solve_chain(pose, row[0:4], row[4:11], row[11:18], row[25:29], row[18:25], gn_mask=flags)[0]
            res.append(MS.assert_within(MS.check_chain(pose, a, row), ("grooming", name, leg)))
        _report(f"grooming, {name}", res)
    legs = list(locomotion["legs"])
    chain_l = KinematicChainSeq(D.BOUNDS_LOCOMOTION, legs, calculate_body_size(D.TEMPLATE_NMF_LOCOMOTION, legs))
    res = []
    for i, leg in enumerate(legs):
        row = chain_l.pack_chain_params(leg, D.INITIAL_ANGLES_LOCOMOTION[leg]).astype(np.float32)
        pose = locomotion["aligned"][i].astype(np.float32)
        a = H.run_block_f32(pose, row, GN)[0]
        res.append(MS.assert_within(MS.check_chain(pose, a, row), ("locomotion", leg)))
    _report("locomotion", res)



def test_iterates_before_the_output_clamp(grooming_leg):
    """The solver's final iterates before the output clamp (seqik_core.cuh limit_clamp), through the host build.  An
    iterate that reaches a limit is pulled one float64 ulp inside it, which float32 cannot represent; and the angle and
    its distance to the limit are updated apart at every accepted step, half an ulp of rounding each.  So an iterate may
    end a few float32 ulps beyond a limit (on the grooming legs: at most 2), or FLT_MIN beyond a limit at 0
    (make_strictly_feasible's smallest gap); this test allows 4 ulps, so that trip()'s pull onto the limit cannot go
    wrong by more unseen behind the clamp.  The written angle is the iterate clamped; on the grooming legs the clamp acts
    on a few dozen angles."""
    from seqikpy_b200 import data as D
    from seqikpy_b200.kinematic_chain import KinematicChainSeq
    chain = KinematicChainSeq(D.BOUNDS, ["RF", "LF"], None)
    n_clamped = 0
    for flags in (GN, GN_REF):
        for li, leg in enumerate(("RF", "LF")):
            row = chain.pack_chain_params(leg, D.INITIAL_ANGLES[leg]).astype(np.float32)
            lb, ub = row[4:11], row[11:18]
            ang, it = H.chain_iterates_f32(grooming_leg["pose"][li], row[0:4], lb, ub, row[25:29], row[18:25], gn_mask=flags)
            it32 = it.astype(np.float32)
            assert np.array_equal(it32.astype(np.float64), it)
            assert np.array_equal(ang, np.minimum(np.maximum(it32, lb), ub))
            tiny = np.float32(1.17549435e-38)
            lo = np.where(lb == 0, -tiny, lb - 4 * np.spacing(np.abs(lb)))
            hi = np.where(ub == 0, tiny, ub + 4 * np.spacing(np.abs(ub)))
            assert ((it32 >= lo) & (it32 <= hi)).all(), np.argwhere(~((it32 >= lo) & (it32 <= hi)))[:5]
            n_clamped += int((ang != it32).sum())
    assert n_clamped > 0
