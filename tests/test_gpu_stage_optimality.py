"""Every stage solve of the leg solver on the B200 against its float64 stage minimiser (tests/model_stage.py): teacher-forced
on the kernel's own angles, cost and angles within the error bound stated there, every angle inside its limits with no
slack.  On every kernel path -- schedule 3 with the lean and the robust kernel, schedules 2 and 1 with the default flags,
schedule 2 with the reference-iterates flags; the first frame of every call is the first-frame kernel's fresh solve -- and
on the synthetic workload, both grooming legs, the locomotion recording, ragged lengths, a warm-started range off the
32-frame grid, stage 1 frozen, the alignment map applied on load and a chain with 1.0-1.25 rad moves between frames.
Run with -s for the largest ratio to each bound per workload."""
import numpy as np
import pytest

import model_stage as MS

pytestmark = pytest.mark.gpu

PATHS = (("schedule 3 lean", dict(schedule=3, block_variant=1)), ("schedule 3 robust", dict(schedule=3, block_variant=2)),
         ("schedule 2", dict(schedule=2)), ("schedule 1", dict(schedule=1)),
         ("schedule 2 reference iterates", dict(schedule=2, flags="FLAG_REFERENCE_ITERATES")))


@pytest.fixture(scope="module")
def env():
    import torch
    from seqikpy_b200 import _native as N, data as D, engine, synthetic as S
    from seqikpy_b200.batch import chain_param_table
    from seqikpy_b200.kinematic_chain import KinematicChainSeq
    N.load_library()
    size, bounds, init = S.chain_constants()
    chain = KinematicChainSeq(bounds, list(S.LEGS), size)

    class E:
        pass
    e = E()
    e.torch, e.N, e.D, e.engine, e.S = torch, N, D, engine, S
    e.pose = S.to_chains(torch.from_numpy(S.make_trials(range(8), 1000)).cuda())            # 48 chains x 1000 frames
    e.params = torch.from_numpy(chain_param_table(chain, init, S.LEGS, 8)).cuda()
    return e


def solve(env, pose, params, path, **kw):
    kw = dict(kw, **path)
    if isinstance(kw.get("flags"), str):
        kw["flags"] = getattr(env.N, kw["flags"])
    ang, _, st, _ = env.engine.leg_solve(pose, params, **kw)
    env.torch.cuda.synchronize()
    return ang.cpu().numpy(), st.cpu().numpy()


def check(pose, ang, status, params, label, stages=(1, 2, 3, 4), frames=None):
    """All bounds on every chain but those with non-finite key points (status -1); returns the worst ratios."""
    pose, params = np.asarray(pose), np.asarray(params)
    lo, hi = (0, pose.shape[1]) if frames is None else frames
    res = []
    for c in range(pose.shape[0]):
        if status[c] == -1:
            continue
        r = MS.check_chain(pose[c, lo:hi], ang[c, lo:hi], params[c], stages=stages)
        res.append(MS.assert_within(r, (label, c)))
    w = MS.merge(res)
    print("\n  " + MS.report(label, w))
    return w


def all_paths(env, pose, params, label, **kw):
    p_np, prm_np = pose.cpu().numpy(), params.cpu().numpy()
    for name, path in PATHS:
        ang, st = solve(env, pose, params, path, **kw)
        check(p_np, ang, st, prm_np, f"{label}, {name}")


def grooming(env, grooming_leg):
    from seqikpy_b200.kinematic_chain import KinematicChainSeq
    chain = KinematicChainSeq(env.D.BOUNDS, ["RF", "LF"], None)
    params = np.stack([chain.pack_chain_params(leg, env.D.INITIAL_ANGLES[leg]) for leg in ("RF", "LF")]).astype(np.float32)
    return (env.torch.from_numpy(np.ascontiguousarray(grooming_leg["pose"], dtype=np.float32)).cuda(),
            env.torch.from_numpy(params).cuda())


def test_synthetic_workload(env):
    all_paths(env, env.pose, env.params, "synthetic 48 x 1000")


def test_grooming_legs(env, grooming_leg):
    pose, params = grooming(env, grooming_leg)
    all_paths(env, pose, params, "grooming 2 x 6000")


def test_locomotion_recording(env, locomotion):
    from seqikpy_b200.kinematic_chain import KinematicChainSeq
    from seqikpy_b200.utils import calculate_body_size
    legs = list(locomotion["legs"])
    chain = KinematicChainSeq(env.D.BOUNDS_LOCOMOTION, legs, calculate_body_size(env.D.TEMPLATE_NMF_LOCOMOTION, legs))
    params = np.stack([chain.pack_chain_params(l, env.D.INITIAL_ANGLES_LOCOMOTION[l]) for l in legs]).astype(np.float32)
    pose = env.torch.from_numpy(np.ascontiguousarray(locomotion["aligned"], dtype=np.float32)).cuda()
    all_paths(env, pose, env.torch.from_numpy(params).cuda(), "locomotion 6 x 100")


@pytest.mark.parametrize("n_frame", [1, 31, 33])
def test_ragged_lengths(env, n_frame):
    all_paths(env, env.pose[:, :n_frame].contiguous(), env.params, f"synthetic, {n_frame} frames")


def test_warm_started_range_off_the_grid(env, grooming_leg):
    """frames=(333, 777) solved in place, warm-started from frame 332 of a full call: the range's first frame is a fresh
    solve from a carried angle that is not on the 32-frame grid."""
    for label, (pose, params) in (("synthetic", (env.pose, env.params)), ("grooming", grooming(env, grooming_leg))):
        for name, path in PATHS:
            kw = dict(path)
            if isinstance(kw.get("flags"), str):
                kw["flags"] = getattr(env.N, kw["flags"])
            ang, _, _, _ = env.engine.leg_solve(pose, params, **kw)
            ang[:, 333:777] = 0.0
            _, _, st, _ = env.engine.leg_solve(pose, params, angles=ang, frames=(333, 777), **kw)
            env.torch.cuda.synchronize()
            check(pose.cpu().numpy(), ang.cpu().numpy(), st.cpu().numpy(), params.cpu().numpy(),
                  f"{label} frames (333, 777), {name}", frames=(333, 777))


def test_stage_one_frozen(env, grooming_leg):
    """stages=(2, 3, 4): stage 1 is read from the angles tensor (here a full solve's, perturbed by 0.02 rad inside its
    limits) and frozen; stages 2-4 solve against it."""
    for label, (pose, params) in (("synthetic", (env.pose, env.params)), ("grooming", grooming(env, grooming_leg))):
        full, _, _, _ = env.engine.leg_solve(pose, params)
        lb, ub = params[:, None, 4:6], params[:, None, 11:13]
        seed = full.clone()
        seed[..., 0:2] = env.torch.minimum(env.torch.maximum(full[..., 0:2] + 0.02, lb), ub)
        for name, path in PATHS[2:4]:                              # schedules 2 and 1 take partial stage sets
            ang = seed.clone()
            _, _, st, _ = env.engine.leg_solve(pose, params, angles=ang, stages=(2, 3, 4), **path)
            env.torch.cuda.synchronize()
            assert env.torch.equal(ang[..., 0:2], seed[..., 0:2])
            check(pose.cpu().numpy(), ang.cpu().numpy(), st.cpu().numpy(), params.cpu().numpy(),
                  f"{label} stages (2, 3, 4), {name}", stages=(2, 3, 4))


def test_alignment_map_on_load(env):
    """The affine map applied on load: the kernels see align_apply's float32 pose -- first asserted bit for bit -- and
    every stage is checked against that pose."""
    torch = env.torch
    n = 12
    aff = torch.tensor([[0.1, -0.2, 0.3, 1.05, 0.0, 0.0, 0.0, 0.0]], device="cuda").repeat(n, 1)
    aff[:, 4:7] = env.pose[:n, 0, 0]
    raw = ((env.pose[:n, :300] - env.pose[:n, :1, :1]) / 1.05 + env.pose[:n, :1, :1] + 0.0).contiguous()
    aligned = env.engine.align_apply(raw, aff)
    for name, path in PATHS:
        a1, s1 = solve(env, raw, env.params[:n], path, affine=aff)
        a2, s2 = solve(env, aligned, env.params[:n], path)
        assert np.array_equal(a1, a2) and np.array_equal(s1, s2), name
        check(aligned.cpu().numpy(), a1, s1, env.params[:n].cpu().numpy(), f"alignment map on load, {name}")


def large_move_chain(n_frame=200):
    """One synthetic leg whose target jumps between two poses 1.0-1.25 rad apart in ThC_yaw/pitch, ThC_roll, CTr_roll and
    TiTa_pitch every frame: closed-form warm steps of half-angle sine 0.48-0.59, beyond the arcsine series' admission
    limit of 0.44 -- these frames must iterate."""
    from seqikpy_b200 import synthetic as S
    from seqikpy_b200.kinematic_chain import DOF_ORDER, SEGMENTS
    size, bounds, init = S.chain_constants()
    leg = "RF"
    rng = np.random.default_rng(7)
    lb = np.array([bounds[f"{leg}_{d}"][0] for d in DOF_ORDER]) + 0.02
    ub = np.array([bounds[f"{leg}_{d}"][1] for d in DOF_ORDER]) - 0.02
    mid = 0.5 * (lb + ub)
    d = rng.uniform(1.0, 1.25, (n_frame, 7)) * np.where(np.arange(n_frame) % 2 == 0, 0.5, -0.5)[:, None]
    theta = np.clip(mid + d, lb, ub)
    seg = np.array([size[f"{leg}_{s}"] for s in SEGMENTS])
    pose = np.zeros((n_frame, 5, 3))
    pose[:, 0] = (0.3, -0.2, 1.0)
    pose[:, 1:] = pose[:, None, 0] + S.leg_key_points(theta, seg) + rng.normal(0, 0.005, (n_frame, 4, 3))
    from seqikpy_b200.kinematic_chain import KinematicChainSeq
    row = KinematicChainSeq(bounds, [leg], size).pack_chain_params(leg, init[leg]).astype(np.float32)
    return pose.astype(np.float32), row


def test_large_moves(env):
    pose, row = large_move_chain()
    torch = env.torch
    all_paths(env, torch.from_numpy(pose[None]).cuda(), torch.from_numpy(row[None]).cuda(), "large moves 1 x 200")


def test_device_against_the_host_build(env, grooming_leg):
    """The schedule-3 kernels against the float32 host build of the same source (tests/hostsim) on both grooming legs: the
    device takes reciprocals and square roots from the SFU approximations (<= 2 ulp), the host build from IEEE division
    and sqrtf, so the two are not bit-identical; the share of identical frames and the largest difference are reported,
    and both sides stay within the stage bound (above and test_stage_model_cpu.py).  Outside the reference's own singular
    episodes (helpers.singular_windows), where the two may settle on different branches, they agree to 1e-3 rad."""
    import hostsim_build as H
    from helpers import singular_windows
    pose, params = grooming(env, grooming_leg)
    ang, _ = solve(env, pose, params, dict(schedule=3))
    for li, leg in enumerate(("RF", "LF")):
        host = H.run_block_f32(pose[li].cpu().numpy(), params[li].cpu().numpy(), 0xFF)[0]
        same = (ang[li] == host).all(1)
        d = np.abs(ang[li].astype(np.float64) - host).max(1)
        off = np.setdiff1d(np.arange(len(d)), sorted(singular_windows(grooming_leg["ref_angles"][li])))
        print(f"\n  device vs host build, grooming {leg}: {same.mean():.4f} of the frames bit-identical, largest angle "
              f"difference {d.max():.3g} rad, {d[off].max():.3g} rad outside the singular episodes")
        assert d[off].max() < 1e-3
