"""The generic 7-DOF solve on the B200 against its float64 specification, on both kernel mappings.

Float64: on every solve the stability classifier (tests/model_generic_cert.py) calls stable the device equals the host
build of the same source (tests/hostsim, which tests/test_generic_cert_cpu.py ties to the numpy specification): same
status, same evaluation count, angles within EPS, FK rows to rounding, rows 0-3 the origin and row 4 row 5 bit for bit.
Unstable float64 solves and every float32 solve meet the float64 certificate.  Workloads: one-frame chains (per-solve
status and evaluation count) of both grooming legs teacher-forced from the oracle's seeds and of the edge families
(unreachable, zero and 1e-3 mm targets, postures with joints on their limits, seeds on / next to / outside the box,
null_sq > 0, an origin 1e3 mm away, evaluation-limit crawls), and free-running recordings replayed on the host frame by
frame from the device's own previous angles.  Then the per-chain status, the skipped-frame contract, and the scheduling:
chains per warp, groups per warp and the automatic choice of the mapping are bit-identical within a mapping.
"""
import numpy as np
import pytest

import model_generic_cert as C
from test_generic_cert_cpu import leg_workloads
from test_generic_cpu import LEGS, consts, params_row

pytestmark = pytest.mark.gpu

SCHEDULES = (1, 2)


@pytest.fixture(scope="module")
def api():
    import torch
    assert torch.cuda.is_available(), "these tests need the B200"
    from seqikpy_b200 import _native, engine
    _native.load_library()
    return torch, engine


def device(api, prm, origin, claw, dtype, schedule, cpw=0):
    """One-frame chains on the device -> angles (n,7), fk (n,9,3) as float64 arrays of working-precision values, status, nfev."""
    torch, engine = api
    td = torch.float32 if dtype == np.float32 else torch.float64
    pose = np.stack([origin, claw], axis=1)[:, None].astype(dtype)
    out = engine.leg_solve_generic(torch.tensor(pose, device="cuda"), torch.tensor(prm.astype(dtype), device="cuda"),
                                   schedule=schedule, chains_per_warp=cpw)
    a, fk, st, nf = (o.cpu().numpy() for o in out)
    return a[:, 0].astype(np.float64), fk[:, 0].astype(np.float64), st, nf


@pytest.fixture(scope="module")
def work(generic_gold, grooming_leg):
    """(leg, family) -> (prm, origin, claw, reachable, float64 host result, stable, certificate reference); the float64
    host replay is computed once here."""
    out = {}
    for leg in LEGS:
        w = leg_workloads(leg, generic_gold, grooming_leg)
        _, seg, lb, ub, _ = consts(leg)
        w["maxfev"] = tuple(a[:40] for a in C.maxfev_workload(seg, lb, ub))
        for name, (prm, o, kp, reach) in w.items():
            t = C.formed_target(o, kp, np.float64)
            base, stable, _ = C.classify(prm, t)
            out[leg, name] = (prm, o, kp, reach, base, stable, C.reference(base, prm, t, reach))
    return out


def check_f64(prm, o, kp, reach, base, stable, ref, a, fk, st, nf, where):
    """Device float64 one-frame solves against the host build (stable) or the certificate (unstable)."""
    t = C.formed_target(o, kp, np.float64)
    L = prm[:, 0:4].sum(axis=1)
    assert np.isfinite(a).all() and np.isfinite(fk).all(), where
    assert C.feasible(a, prm, np.float64).all(), (where, np.where(~C.feasible(a, prm, np.float64))[0])
    assert (fk[:, :4] == o[:, None]).all() and (fk[:, 4] == fk[:, 5]).all(), where
    s = np.where(stable)[0]
    want_st = np.where(base["status"] == 0, 0, 1)
    bad_st = s[(st[s] != want_st[s]) | (nf[s] != base["nfev"][s])]
    assert not len(bad_st), (where, "status/nfev", [(k, st[k], nf[k], base["status"][k], base["nfev"][k]) for k in bad_st[:5]])
    dev = np.abs(a - base["angles"]).max(axis=1)
    assert (dev[s] <= C.EPS).all(), (where, "angles", [(k, dev[k]) for k in s[dev[s] > C.EPS][:5]])
    fk_err = np.abs(fk - (C.certificate(a, prm, t)["fk"] + o[:, None])).max(axis=(1, 2))     # float64 FK of the returned angles
    bound = C.FK_C * C.U64 * (np.abs(o).max(axis=1) + L)
    assert (fk_err[s] <= bound[s]).all(), (where, "fk", float(np.max(fk_err[s] / bound[s])))
    u = ~stable
    ref_u = dict(ref, resid=ref["resid"][u])                   # the per-solve entries of the unstable solves
    fails, _ = C.check(a[u], fk[u], np.full(int(u.sum()), C.UNKNOWN), prm[u], o[u], t[u], reach[u], ref_u, np.float64)
    for key, bad in fails.items():
        assert not bad.any(), (where, "certificate", key, np.where(u)[0][bad])
    return int(stable.sum())


@pytest.mark.parametrize("schedule", SCHEDULES)
def test_f64_one_frame_solves(api, work, schedule):
    """Float64, every workload: stable solves equal the host build, unstable ones meet the certificate."""
    report = []
    for (leg, name), (prm, o, kp, reach, base, stable, ref) in work.items():
        a, fk, st, nf = device(api, prm, o, kp, np.float64, schedule)
        n_st = check_f64(prm, o, kp, reach, base, stable, ref, a, fk, st, nf, (leg, name, schedule))
        report.append(f"{leg} {name}: {n_st}/{len(stable)} stable")
    print(f"schedule {schedule}: " + "; ".join(report))


@pytest.mark.parametrize("schedule", SCHEDULES)
def test_f32_one_frame_certificate(api, work, schedule):
    """Float32, every workload: every solve meets the float64 certificate; prints the largest ratio to each bound."""
    worst = {}
    for (leg, name), (prm, o, kp, reach, base, stable, ref) in work.items():
        a, fk, st, nf = device(api, prm, o, kp, np.float32, schedule)
        assert np.isfinite(a).all() and np.isfinite(fk).all()
        assert (st >= 0).all()
        f32 = fk.astype(np.float32)
        assert (f32[:, :4] == o.astype(np.float32)[:, None]).all() and (f32[:, 4] == f32[:, 5]).all()
        t = C.formed_target(o, kp, np.float32)
        fails, ratios = C.check(a, fk, np.full(len(st), C.UNKNOWN), prm, o, t, reach, ref, np.float32)
        for key, bad in fails.items():
            assert not bad.any(), (leg, name, schedule, key, np.where(bad)[0], ratios)
        for key, r in ratios.items():
            worst[key] = max(worst.get(key, 0.0), r)
    print(f"float32 schedule {schedule}, largest ratio to each bound: " + ", ".join(f"{k} {v:.3g}" for k, v in worst.items()))


# ---------------------------------------------------------------------------------------------------------------------
# free-running recordings, replayed on the host frame by frame from the device's own previous angles
def recordings(grooming_leg, n_long=500, n_short=60, len_short=4):
    """Per leg: one long recording and n_short short ones -> list of (leg, pose (n_chain, n_frame, 5, 3))."""
    out = []
    for li, leg in enumerate(LEGS):
        p = grooming_leg["pose"][li]
        out.append((leg, p[None, :n_long]))
        out.append((leg, np.stack([p[50 * k:50 * k + len_short] for k in range(n_short)])))
    return out


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("schedule", SCHEDULES)
def test_free_running_replayed(api, grooming_leg, dtype, schedule):
    """Warm-started chains on the device; each frame re-solved on the host from the device's previous angles.  Float64:
    stable frames equal the host, unstable ones meet the certificate, and a chain whose frames are all stable reports the
    sum of the host's evaluation counts.  Float32: every frame meets the certificate."""
    torch, engine = api
    td = torch.float32 if dtype == np.float32 else torch.float64
    n_stable = n_all = n_chain_eq = 0
    for leg, pose in recordings(grooming_leg):
        _, seg, lb, ub, seed = consts(leg)
        row = params_row(seg, lb, ub, seed)
        n_chain, n_frame = pose.shape[:2]
        out = engine.leg_solve_generic(torch.tensor(pose.astype(dtype), device="cuda"),
                                       torch.tensor(np.tile(row, (n_chain, 1)).astype(dtype), device="cuda"), schedule=schedule)
        a, fk, st, nf = (x.cpu().numpy() for x in out)
        a64, fk64 = a.astype(np.float64), fk.astype(np.float64)
        seeds = np.concatenate([np.tile(row[18:25].astype(dtype), (n_chain, 1, 1)), a[:, :-1]], axis=1).astype(np.float64)
        prm = np.tile(row, (n_chain * n_frame, 1))
        prm[:, 18:25] = seeds.reshape(-1, 7)
        o, kp = pose[:, :, 0].reshape(-1, 3).astype(np.float64), pose[:, :, 4].reshape(-1, 3).astype(np.float64)
        reach = np.ones(len(prm), bool)
        A, FK = a64.reshape(-1, 7), fk64.reshape(-1, 9, 3)
        if dtype == np.float64:
            t = C.formed_target(o, kp, np.float64)
            base, stable, _ = C.classify(prm, t)
            ref = C.reference(base, prm, t, reach)
            # per-frame status and nfev are not reported; the check uses the host's, the chain sums are compared below
            check_f64(prm, o, kp, reach, base, stable, ref, A, FK, np.where(base["status"] == 0, 0, 1), base["nfev"],
                      (leg, n_chain, n_frame, schedule))
            s2 = stable.reshape(n_chain, n_frame).all(axis=1)
            host_sum = base["nfev"].reshape(n_chain, n_frame).sum(axis=1)
            assert (nf[s2] == host_sum[s2]).all(), (leg, schedule, np.where(s2 & (nf != host_sum))[0])
            n_stable += int(stable.sum())
            n_chain_eq += int(s2.sum())
        else:
            t64 = C.formed_target(o, kp, np.float64)
            ref = C.reference(C.host(prm, t64), prm, t64, reach)
            t = C.formed_target(o, kp, np.float32)
            assert np.isfinite(A).all() and C.feasible(A, prm.astype(np.float32), np.float32).all()
            fails, _ = C.check(A, FK, np.full(len(prm), C.UNKNOWN), prm.astype(np.float32).astype(np.float64), o, t, reach, ref,
                               np.float32)
            for key, bad in fails.items():
                assert not bad.any(), (leg, schedule, key, np.where(bad)[0])
        assert (st == 1).all()
        n_all += n_chain * n_frame
    if dtype == np.float64:
        print(f"schedule {schedule}: {n_stable}/{n_all} replayed frames stable, {n_chain_eq} chains with every frame stable")


# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def maxfev_case(work):
    """A stable MAXFEV solve (float64): (prm row, claw target with the ThC at 0)."""
    prm, o, kp, reach, base, stable, ref = work["RF", "maxfev"]
    k = int(np.where(stable & (base["status"] == 0))[0][0])
    return prm[k], kp[k]


def status_batch(grooming_leg, maxfev_case, n_frame=5, n_chain=12):
    """Chains of RF grooming frames.  Chain 0: a NaN claw in frame 0, then the MAXFEV frame (seeded, after the skip, from
    the same seed as the stable MAXFEV solve), then normal frames.  Chain 1: the MAXFEV frame, then normal frames.  Chain
    2: the MAXFEV frame, a normal frame, an inf origin in frame 2, normal frames.  Every other chain is normal."""
    _, seg, lb, ub, seed = consts("RF")
    row = params_row(seg, lb, ub, seed)
    p = grooming_leg["pose"][0]
    pose = np.stack([p[37 * k:37 * k + n_frame] for k in range(n_chain)]).astype(np.float64)
    rows = np.tile(row, (n_chain, 1))
    mrow, mt = maxfev_case
    for c, f in ((0, 1), (1, 0), (2, 0)):
        rows[c] = mrow
        pose[c, f] = 0.0
        pose[c, f, 4] = mt
    pose[0, 0, 4, 0] = np.nan
    pose[2, 2, 0, 1] = np.inf
    return pose, rows


@pytest.mark.parametrize("schedule", SCHEDULES)
def test_status_aggregation_and_skipped_frames(api, grooming_leg, maxfev_case, schedule):
    """Per-chain status: -1 when a frame was skipped (non-finite key point), whether the MAXFEV frame comes after or
    before it; 0 when a frame hit the evaluation limit and none was skipped; 1 otherwise.  A skipped frame costs one
    evaluation, returns the angles it was seeded with (the seed for frame 0, else the previous frame's), its FK rows are
    those angles placed at its own origin (not finite when the origin is not), and the next frame starts from the same
    angles, as if the skipped frame were absent.  Chains without a bad frame are bit-identical to a run without the bad
    chains."""
    torch, engine = api
    pose, rows = status_batch(grooming_leg, maxfev_case)
    T = lambda x: torch.tensor(x, dtype=torch.float64, device="cuda")
    a, fk, st, nf = (x.cpu().numpy() for x in engine.leg_solve_generic(T(pose), T(rows), schedule=schedule))
    assert st[0] == -1 and st[1] == 0 and st[2] == -1 and (st[3:] == 1).all(), st
    good = engine.leg_solve_generic(T(pose[3:]), T(rows[3:]), schedule=schedule)
    assert np.array_equal(a[3:], good[0].cpu().numpy()) and np.array_equal(fk[3:], good[1].cpu().numpy())
    assert np.array_equal(nf[3:], good[3].cpu().numpy())
    # chain 0: frame 0 skipped -> the seed; frames 1.. = the chain without frame 0, which ends at the evaluation limit
    assert np.array_equal(a[0, 0], rows[0, 18:25])
    assert np.isfinite(fk[0, 0]).all() and (fk[0, 0, :4] == pose[0, 0, 0]).all()       # NaN claw, finite origin
    drop = engine.leg_solve_generic(T(pose[0:1, 1:]), T(rows[0:1]), schedule=schedule)
    assert drop[2].item() == 0
    assert np.array_equal(a[0, 1:], drop[0].cpu().numpy()[0]) and np.array_equal(a[0, 1], a[1, 0])
    assert nf[0] == drop[3].item() + 1
    # chain 2: frame 2 skipped (inf origin) after the MAXFEV frame
    assert np.array_equal(a[2, 2], a[2, 1]) and not np.isfinite(fk[2, 2]).all()
    drop2 = engine.leg_solve_generic(T(np.delete(pose[2:3], 2, axis=1)), T(rows[2:3]), schedule=schedule)
    assert drop2[2].item() == 0
    assert np.array_equal(a[2, [0, 1, 3, 4]], drop2[0].cpu().numpy()[0]) and nf[2] == drop2[3].item() + 1
    assert np.isfinite(a[1]).all() and np.isfinite(fk[1]).all()


def mixed_batch(grooming_leg, maxfev_case, n_chain=37, n_frame=3):
    """n_chain (not a multiple of any chains-per-warp tried) RF chains; every fifth starts with a MAXFEV-bound frame."""
    _, seg, lb, ub, seed = consts("RF")
    rows = np.tile(params_row(seg, lb, ub, seed), (n_chain, 1))
    p = grooming_leg["pose"][0]
    pose = np.stack([p[41 * k:41 * k + n_frame] for k in range(n_chain)]).astype(np.float64)
    mrow, mt = maxfev_case
    for c in range(0, n_chain, 5):
        rows[c] = mrow
        pose[c, 0] = 0.0
        pose[c, 0, 4] = mt
    return pose, rows


@pytest.mark.parametrize("dtype", ["float64", "float32"])
def test_chains_per_warp_bit_identical(api, grooming_leg, maxfev_case, dtype):
    """schedule 1 with 1, 5 and 32 chains per warp, schedule 2 with 1-4 chains per warp: the same bits within a mapping,
    with MAXFEV-bound and easy chains sharing warps."""
    torch, engine = api
    td = getattr(torch, dtype)
    pose, rows = mixed_batch(grooming_leg, maxfev_case)
    d_pose, d_rows = torch.tensor(pose, dtype=td, device="cuda"), torch.tensor(rows, dtype=td, device="cuda")
    for schedule, cpws in ((1, (1, 5, 32)), (2, (1, 2, 3, 4))):
        ref = [x.cpu() for x in engine.leg_solve_generic(d_pose, d_rows, schedule=schedule, chains_per_warp=cpws[0])]
        if dtype == "float64":
            assert (ref[2].numpy()[::5] == 0).all()
        for cpw in cpws[1:]:
            out = [x.cpu() for x in engine.leg_solve_generic(d_pose, d_rows, schedule=schedule, chains_per_warp=cpw)]
            for r, o in zip(ref, out):
                assert torch.equal(r, o), (schedule, cpw)


@pytest.mark.parametrize("dtype,small,large", [("float32", 2000, 20000), ("float64", 3000, 30000)])
def test_automatic_schedule(api, work, dtype, small, large):
    """The automatic choice: eight lanes per chain at `small` chains, a lane per chain at `large` (sizes on either side
    of the launcher's threshold for every register count its clamp allows), bit for bit."""
    torch, engine = api
    td = getattr(torch, dtype)
    prm, o, kp, reach, *_ = work["RF", "grooming"]
    for n, forced in ((small, 2), (large, 1)):
        idx = np.arange(n) % len(prm)
        pose = np.stack([o[idx], kp[idx]], axis=1)[:, None]
        d_pose, d_rows = torch.tensor(pose, dtype=td, device="cuda"), torch.tensor(prm[idx], dtype=td, device="cuda")
        auto = engine.leg_solve_generic(d_pose, d_rows)
        want = engine.leg_solve_generic(d_pose, d_rows, schedule=forced)
        other = engine.leg_solve_generic(d_pose, d_rows, schedule=3 - forced)
        for x, y in zip(auto, want):
            assert torch.equal(x, y), (dtype, n, forced)
        assert not torch.equal(auto[0], other[0]), (dtype, n)        # the two mappings do differ in the last bits somewhere


@pytest.mark.parametrize("schedule", SCHEDULES)
def test_warm_target_row_and_stride(api, work, schedule):
    """warm= in place of the params seeds, the claw in another row, and a pose with unread rows (a frame stride larger
    than the rows read) give the same bits as the plain call, on the seeds-at-the-box workload."""
    torch, engine = api
    prm, o, kp, *_ = work["LF", "seed_bound"]
    for td in (torch.float32, torch.float64):
        T = lambda x: torch.tensor(x, dtype=td, device="cuda")
        plain = engine.leg_solve_generic(T(np.stack([o, kp], axis=1)[:, None]), T(prm), schedule=schedule)
        junk = prm.copy()
        junk[:, 18:25] = 0.5 * (prm[:, 4:11] + prm[:, 11:18])
        warm = engine.leg_solve_generic(T(np.stack([o, kp], axis=1)[:, None]), T(junk), warm=T(prm[:, 18:25]), schedule=schedule)
        wide = np.full((len(o), 1, 5, 3), np.nan)
        wide[:, 0, 0], wide[:, 0, 2] = o, kp
        row = engine.leg_solve_generic(T(wide), T(prm), target_row=2, schedule=schedule)
        for out in (warm, row):
            for x, y in zip(plain, out):
                assert torch.equal(x, y), (schedule, td)
