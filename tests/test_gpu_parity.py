"""GPU parity tests: the CUDA path (through the reference-compatible classes -> ctypes C ABI) against
the reference's shipped outputs and the CPU oracle's outputs held in tests/golden/.

Tolerances (BASELINE.json north_star): joint angles within 1e-3 rad; FK residual not worse than the
reference's by more than 1e-4 mm per joint.  SURVEY.md finding 4 documents the one place where the
reference itself is irreproducible (LF frames ~280-304 of the grooming trial: a noise-driven
bound-to-bound flip at the CTr_pitch = 0 singularity); those frames are bounded, not skipped.
"""
import numpy as np
import pytest

from helpers import (ANGLE_TOL, F32_FK_NOISE, FK_TOL, angles_dict_to_array, bad_frames, fk_residual, residual_of_angles,
                     singular_windows)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def api():
    import torch
    assert torch.cuda.is_available(), "these tests need the B200"
    from seqikpy_b200 import _native, data, engine, synthetic
    from seqikpy_b200.alignment import AlignPose
    from seqikpy_b200.head_inverse_kinematics import HeadInverseKinematics
    from seqikpy_b200.kinematic_chain import KinematicChainSeq
    from seqikpy_b200.leg_inverse_kinematics import LegInvKinSeq
    _native.load_library()

    class A:
        pass
    a = A()
    a.torch, a.native, a.data, a.engine, a.synthetic = torch, _native, data, engine, synthetic
    a.AlignPose, a.Head, a.Chain, a.Leg = AlignPose, HeadInverseKinematics, KinematicChainSeq, LegInvKinSeq
    return a


def seg_of(size, leg):
    return [size[f"{leg}_{s}"] for s in ("Coxa", "Femur", "Tibia", "Tarsus")]


# ------------------------------------------------------------------------------------------ grooming trial (config 2)
@pytest.fixture(scope="module")
def grooming_run(api, grooming_leg):
    pose = {"RF_leg": grooming_leg["pose"][0], "LF_leg": grooming_leg["pose"][1]}
    chain = api.Chain(api.data.BOUNDS, ["RF", "LF"])
    ik = api.Leg(pose, chain, api.data.INITIAL_ANGLES, log_level="ERROR")
    angles, fk = ik.run_ik_and_fk(hide_progress_bar=True)
    return pose, chain, ik, angles, fk


def test_grooming_layout(grooming_run, grooming_leg):
    pose, chain, ik, angles, fk = grooming_run
    assert list(angles.keys()) == list(grooming_leg["angle_keys"])          # insertion order of the reference pickle
    assert list(fk.keys()) == ["RF_leg", "LF_leg"]
    for v in angles.values():
        assert v.shape == (6000,) and v.dtype == np.float64
    for v in fk.values():
        assert v.shape == (6000, 9, 3) and v.dtype == np.float64
    assert ik.solver_stats["RF"]["status"] == 1 and ik.solver_stats["LF"]["status"] == 1


def test_grooming_rf_angles_all_frames(grooming_run, grooming_leg):
    _, _, _, angles, _ = grooming_run
    ours = angles_dict_to_array(angles, "RF")
    assert len(bad_frames(ours, grooming_leg["ref_angles"][0])) == 0          # vs the reference's shipped angles
    assert len(bad_frames(ours, grooming_leg["oracle_angles"][0])) == 0       # vs the CPU oracle
    assert np.median(np.abs(ours - grooming_leg["ref_angles"][0])) < 5e-6


def test_grooming_lf_angles(grooming_run, grooming_leg):
    _, _, _, angles, _ = grooming_run
    ours = angles_dict_to_array(angles, "LF")
    bad = bad_frames(ours, grooming_leg["ref_angles"][1])
    # mismatches only around the frames where the reference itself sits on the CTr_pitch = 0 singularity (two episodes
    # in this trial, see helpers.singular_windows); everywhere else -- 5900+ frames -- every DOF is within 1e-3 rad
    allowed = singular_windows(grooming_leg["ref_angles"][1])
    assert 0 < len(allowed) < 120
    assert len(bad) <= 30 and set(bad) <= allowed, bad
    good = np.setdiff1d(np.arange(6000), sorted(allowed))
    assert np.abs(ours[good] - grooming_leg["ref_angles"][1][good]).max() < ANGLE_TOL
    assert len(singular_windows(grooming_leg["ref_angles"][0])) == 0          # RF: no singular episode, no exception


def test_grooming_bounds_respected(grooming_run, api):
    _, _, _, angles, _ = grooming_run
    for key, v in angles.items():
        lb, ub = api.data.BOUNDS[key.replace("Angle_", "")]
        assert v.min() >= lb - 1e-6 and v.max() <= ub + 1e-6, key


def test_grooming_fk_consistent_and_residual(grooming_run, grooming_leg):
    pose, chain, _, angles, fk = grooming_run
    for li, leg in enumerate(("RF", "LF")):
        ours = angles_dict_to_array(angles, leg)
        seg = seg_of(chain.body_size, leg)
        # the FK the kernel returns is the FK of the angles it returns
        from oracle import seqik_oracle as O
        fk64 = O.fk_closed_form(ours, seg, pose[f"{leg}_leg"][:, 0])
        assert np.abs(fk64 - fk[f"{leg}_leg"]).max() < 1e-5
        assert np.abs(fk[f"{leg}_leg"][:600] - grooming_leg["ref_fk"][li]).max() < (1e-3 if leg == "RF" else 2.0)
        # FK residual vs the reference's residual, per (frame, joint)
        r_ours = fk_residual(fk[f"{leg}_leg"], pose[f"{leg}_leg"])
        r_ref = residual_of_angles(grooming_leg["ref_angles"][li], seg, pose[f"{leg}_leg"])
        worse = (r_ours - r_ref) > FK_TOL + F32_FK_NOISE
        allowed = singular_windows(grooming_leg["ref_angles"][li])
        frames = np.where(worse.any(axis=1))[0]
        assert len(frames) <= 30 and set(frames) <= allowed, frames           # RF: allowed is empty
        assert r_ours.mean() < r_ref.mean() + 1e-4                             # never worse on average


def test_stagewise_calls_equal_one_shot(grooming_run, api):
    """calculate_ik_stage stage by stage (frozen earlier DOFs read back from joint_angles_dict) == run_ik_and_fk."""
    pose, chain, _, angles, fk = grooming_run
    n = 400
    arr = pose["RF_leg"][:n]
    ik = api.Leg({"RF_leg": arr}, chain, api.data.INITIAL_ANGLES, log_level="ERROR")
    for stage in (1, 2, 3, 4):
        out = ik.calculate_ik_stage(arr[:, stage], arr[:, 0], api.data.INITIAL_ANGLES["RF"][f"stage_{stage}"], "RF",
                                    stage=stage, hide_progress_bar=True)
        assert out.shape == (n, (4, 6, 8, 9)[stage - 1], 3)
    # (not bit-identical: a frozen stage rebuilds its rotation from the stored angle, the one-shot run carries the
    #  solver's own sin/cos; the difference is float32 rounding -- 5e-5 rad is 1/20 of the parity bar)
    for k in ik.joint_angles_dict:
        assert np.abs(ik.joint_angles_dict[k] - angles[k][:n]).max() < 5e-5, k
    assert np.allclose(out, fk["RF_leg"][:n], atol=5e-5)
    # stages=[1,2] then [3,4]
    ik2 = api.Leg({"RF_leg": arr}, chain, api.data.INITIAL_ANGLES, log_level="ERROR")
    a12, fk12 = ik2.run_ik_and_fk(stages=[1, 2], hide_progress_bar=True)
    assert list(a12.keys()) == [f"Angle_RF_{d}" for d in ("ThC_yaw", "ThC_pitch", "ThC_roll", "CTr_pitch")]
    assert fk12["RF_leg"].shape == (n, 6, 3)
    a, f = ik2.run_ik_and_fk(stages=[3, 4], hide_progress_bar=True)
    assert len(a) == 7 and f["RF_leg"].shape == (n, 9, 3)
    for k in a:
        assert np.abs(a[k] - angles[k][:n]).max() < 5e-5, k


def test_entire_pipeline_from_raw_like_the_reference_example(api, grooming_align, grooming_leg, grooming_head, tmp_path):
    """examples/example_entire_pipeline.py:60-101 on the bundled trial: raw key points -> AlignPose -> LegInvKinSeq (+ head)
    -> pickles, against the reference's shipped aligned pose and joint angles."""
    raw = {"RF_leg": grooming_align["raw_full_RF"], "LF_leg": grooming_align["raw_full_LF"]}
    aligned = api.AlignPose(raw, legs_list=["RF", "LF"], include_claw=False, body_template=api.data.NMF_TEMPLATE,
                            log_level="ERROR").align_pose(export_path=tmp_path)
    assert list(aligned.keys()) == ["RF_leg", "LF_leg", "Neck"] and aligned["Neck"].shape == (1, 1, 3)
    for li, leg in enumerate(("RF", "LF")):
        assert np.allclose(aligned[f"{leg}_leg"], grooming_leg["pose"][li], rtol=1e-5, atol=2e-6)
    aligned["R_head"], aligned["L_head"] = grooming_head["r_head"], grooming_head["l_head"]
    head = api.Head(aligned, api.data.NMF_TEMPLATE, log_level="ERROR").compute_head_angles(export_path=tmp_path)
    ik = api.Leg(aligned, api.Chain(api.data.BOUNDS, ["RF", "LF"], body_size=None), api.data.INITIAL_ANGLES, log_level="ERROR")
    angles, fk = ik.run_ik_and_fk(export_path=tmp_path, hide_progress_bar=True)
    body = {**head, **angles}
    assert len(body) == 21 and list(body.keys())[:3] == ["Angle_head_roll", "Angle_head_pitch", "Angle_head_yaw"]
    from seqikpy_b200.utils import load_file, save_file
    save_file(tmp_path / "body_joint_angles.pkl", body)
    for name in ("pose3d_aligned.pkl", "head_joint_angles.pkl", "leg_joint_angles.pkl", "forward_kinematics.pkl", "body_joint_angles.pkl"):
        assert (tmp_path / name).exists(), name
    assert list(load_file(tmp_path / "leg_joint_angles.pkl").keys()) == list(grooming_leg["angle_keys"])
    assert load_file(tmp_path / "forward_kinematics.pkl")["LF_leg"].shape == (6000, 9, 3)
    rf = angles_dict_to_array(angles, "RF")
    assert len(bad_frames(rf, grooming_leg["ref_angles"][0])) == 0
    lf = angles_dict_to_array(angles, "LF")
    assert set(bad_frames(lf, grooming_leg["ref_angles"][1])) <= singular_windows(grooming_leg["ref_angles"][1])


# ------------------------------------------------------------------------------------------ locomotion (config 1)
def test_locomotion_pipeline(api, locomotion):
    legs = list(locomotion["legs"])
    raw = {f"{leg}_leg": locomotion["raw"][i] for i, leg in enumerate(legs)}
    al = api.AlignPose(raw, legs_list=legs, include_claw=False, body_template=api.data.TEMPLATE_NMF_LOCOMOTION,
                       log_level="ERROR").align_pose()
    assert list(al.keys()) == [f"{leg}_leg" for leg in legs]
    for i, leg in enumerate(legs):
        assert al[f"{leg}_leg"].dtype == np.float64
        assert np.abs(al[f"{leg}_leg"] - locomotion["aligned"][i]).max() < 2e-6
    from seqikpy_b200.utils import calculate_body_size
    chain = api.Chain(api.data.BOUNDS_LOCOMOTION, legs, calculate_body_size(api.data.TEMPLATE_NMF_LOCOMOTION, legs))
    aligned = {f"{leg}_leg": locomotion["aligned"][i] for i, leg in enumerate(legs)}
    angles, fk = api.Leg(aligned, chain, api.data.INITIAL_ANGLES_LOCOMOTION, log_level="ERROR").run_ik_and_fk()
    for i, leg in enumerate(legs):
        ours = angles_dict_to_array(angles, leg)
        assert np.abs(ours - locomotion["oracle_angles"][i]).max() < ANGLE_TOL, leg
        r_ours = fk_residual(fk[f"{leg}_leg"], aligned[f"{leg}_leg"])
        r_ref = fk_residual(locomotion["oracle_fk"][i], aligned[f"{leg}_leg"])
        assert (r_ours - r_ref).max() < FK_TOL + F32_FK_NOISE, leg
    # the fused path: raw pose + affine applied inside the solver load == align then solve
    t = api.torch
    d_raw = t.from_numpy(np.ascontiguousarray(locomotion["raw"], dtype=np.float32)).cuda()
    consts = np.array([list(api.data.TEMPLATE_NMF_LOCOMOTION[f"{leg}_Coxa"])
                       + [chain.body_size[leg] - chain.body_size[f"{leg}_Tarsus"]] for leg in legs], dtype=np.float32)
    aff = api.engine.leg_affine(d_raw, t.from_numpy(consts).cuda())
    params = t.from_numpy(np.stack([chain.pack_chain_params(leg, api.data.INITIAL_ANGLES_LOCOMOTION[leg])
                                    for leg in legs]).astype(np.float32)).cuda()
    a_fused, fk_fused, _, _ = api.engine.leg_solve(d_raw, params, affine=aff)
    a_two, fk_two, _, _ = api.engine.leg_solve(api.engine.align_apply(d_raw, aff), params)
    assert t.equal(a_fused, a_two) and t.equal(fk_fused, fk_two)
    assert np.abs(a_fused.cpu().numpy() - locomotion["oracle_angles"]).max() < ANGLE_TOL


# ------------------------------------------------------------------------------------------ synthetic (configs 3-5)
def test_synthetic_vs_oracle_and_shard_invariance(api, synthetic_gold):
    S, t = api.synthetic, api.torch
    n_frame = synthetic_gold["pose"].shape[1]
    pose = S.make_trials([0, 1, 2, 3], 1000)[:, :n_frame]
    assert np.abs(pose[:2] - synthetic_gold["pose"]).max() < 1e-6            # the generator is pinned by the fixture
    size, bounds, init = S.chain_constants()
    chain = api.Chain(bounds, list(S.LEGS), size)
    row = np.stack([chain.pack_chain_params(leg, init[leg]) for leg in S.LEGS]).astype(np.float32)
    params = t.from_numpy(np.tile(row, (4, 1))).cuda()
    chains = S.to_chains(t.from_numpy(np.ascontiguousarray(pose)).cuda())
    ang, fk, status, nfev = api.engine.leg_solve(chains, params)
    a = ang.cpu().numpy().reshape(4, 6, n_frame, 7)
    assert np.abs(a[:2] - synthetic_gold["oracle_angles"]).max() < ANGLE_TOL
    f = fk.cpu().numpy().reshape(4, 6, n_frame, 9, 3)
    pose_c = pose.transpose(0, 2, 1, 3, 4)
    for tr in range(2):
        for li in range(6):
            r_ours = fk_residual(f[tr, li], pose_c[tr, li])
            r_ref = fk_residual(synthetic_gold["oracle_fk"][tr, li], pose_c[tr, li])
            assert (r_ours - r_ref).max() < FK_TOL + F32_FK_NOISE
    assert int(status.min()) == 1
    # chains are independent: any shard gives bit-identical results (what the multi-GPU split relies on)
    for lo, hi in ((0, 6), (6, 24), (5, 7)):
        a_s, f_s, _, _ = api.engine.leg_solve(chains[lo:hi].contiguous(), params[lo:hi].contiguous())
        assert t.equal(a_s, ang[lo:hi]) and t.equal(f_s, fk[lo:hi])
    # results do not depend on how chains are packed into warps (bit-identical).  The one-lane-per-chain schedule starts
    # every solve afresh from the warm start (no carried state, hence no closed-form warm step): it iterates to the
    # same minimisers and stops where the ftol test says, up to a few 1e-4 rad from them on flat (bound-active) solves
    for cpw, gate in ((1, 0), (2, 1), (3, 2), (8, 3), (8, 1), (4, 7), (8, 15)):
        a2, f2, s2, n2 = api.engine.leg_solve(chains, params, schedule=api.native.SCHED_STAGE_PIPELINE, chains_per_warp=cpw, gate=gate)
        assert t.equal(ang, a2) and t.equal(fk, f2) and t.equal(nfev, n2) and t.equal(status, s2), (cpw, gate)
    a1, f1, s1, n1 = api.engine.leg_solve(chains, params, schedule=api.native.SCHED_LANE_PER_CHAIN)
    assert (a1 - ang).abs().max() < 5e-4 and (f1 - fk).abs().max() < 1e-4 and int(s1.min()) == 1
    # with the reference's iterates in both schedules the agreement is float32 rounding
    ref_it = api.native.FLAG_REFERENCE_ITERATES
    a3, f3, _, _ = api.engine.leg_solve(chains, params, flags=ref_it)
    a4, f4, _, _ = api.engine.leg_solve(chains, params, flags=ref_it, schedule=api.native.SCHED_LANE_PER_CHAIN)
    assert (a3 - a4).abs().max() < 2e-4 and (f3 - f4).abs().max() < 1e-4
    assert (a3 - ang).abs().max() < 5e-4 and (f3 - fk).abs().max() < 1e-4


def test_synthetic_trials_2_to_7_all_frames_vs_oracle(api, synthetic_wide):
    """SURVEY.md 8d parity run, second half: trials 2-7 x 6 legs x all 1000 frames (36 000 leg-frames) against the
    oracle: angles within 1e-3 rad, FK residual per joint never worse than the oracle's by more than 1e-4 mm, and the
    same mean FK error."""
    S, t = api.synthetic, api.torch
    trials = [int(x) for x in synthetic_wide["trials"]]
    n_frame = int(synthetic_wide["n_frame"])
    pose = S.make_trials(trials, n_frame)
    size, bounds, init = S.chain_constants()
    chain = api.Chain(bounds, list(S.LEGS), size)
    row = np.stack([chain.pack_chain_params(leg, init[leg]) for leg in S.LEGS]).astype(np.float32)
    params = t.from_numpy(np.tile(row, (len(trials), 1))).cuda()
    chains = S.to_chains(t.from_numpy(np.ascontiguousarray(pose)).cuda())
    ang, fk, status, nfev = api.engine.leg_solve(chains, params)
    a = ang.cpu().numpy().reshape(len(trials), 6, n_frame, 7)
    dev = np.abs(a - synthetic_wide["oracle_angles"])
    assert dev.max() < ANGLE_TOL and np.median(dev) < 5e-6
    f = fk.cpu().numpy().reshape(len(trials), 6, n_frame, 9, 3)
    pose_c = pose.transpose(0, 2, 1, 3, 4)
    r_ours = np.linalg.norm(f[:, :, :, [5, 6, 7, 8]] - pose_c[:, :, :, 1:5], axis=-1)
    assert (r_ours - synthetic_wide["oracle_fk_residual"]).max() < FK_TOL + F32_FK_NOISE
    assert abs(r_ours.mean() - synthetic_wide["oracle_fk_residual"].mean()) < 1e-5
    assert int(status.min()) == 1 and int(status.max()) == 1


def test_full_size_properties(api):
    """BASELINE config 3 at full size (1000 trials x 1000 frames x 6 legs = 6e6 leg-frames), through size-independent
    properties: every chain converges, every angle is inside its limits, the FK rows the solver carries equal the
    standalone FK kernel applied to the angles it returns, rows 0-3 repeat the origin and row 4 = row 5, the mean FK
    error equals the oracle's on this workload (0.0264 mm), trials that hold the same data give bit-identical
    results wherever they sit in the batch, and the result does not depend on the launch's frame chunking."""
    S, t = api.synthetic, api.torch
    from seqikpy_b200.batch import BatchedLegIK
    n_trial, n_frame, n_unique = 1000, 1000, 20
    size, bounds, init = S.chain_constants()
    chain = api.Chain(bounds, list(S.LEGS), size)
    uniq = t.from_numpy(np.ascontiguousarray(S.make_trials(range(n_unique), n_frame).transpose(0, 2, 1, 3, 4))).cuda()
    sess = BatchedLegIK(chain, init, S.LEGS, n_trial, n_frame)
    sess.d_pose.copy_(uniq.repeat(n_trial // n_unique, 1, 1, 1, 1).reshape(sess.n_chain, n_frame, 5, 3))
    ang, fk = sess.solve_device()
    assert int(sess.status.min()) == 1 and int(sess.status.max()) == 1
    lb, ub = sess.params[:, None, 4:11], sess.params[:, None, 11:18]
    assert bool(((ang >= lb - 1e-6) & (ang <= ub + 1e-6)).all())
    fk2 = api.engine.forward_kinematics(ang, sess.d_pose[:, :, 0].contiguous(), sess.params)
    assert float((fk2 - fk).abs().max()) < 1e-5
    assert t.equal(fk[:, :, :4], sess.d_pose[:, :, :1].expand(-1, -1, 4, -1)) and t.equal(fk[:, :, 4], fk[:, :, 5])
    err = (fk[:, :, 5:9] - sess.d_pose[:, :, 1:5]).norm(dim=-1).mean().item()
    assert abs(err - 0.0264) < 5e-4, err
    a5 = ang.view(n_trial // n_unique, n_unique * 6, n_frame, 7)
    assert t.equal(a5[0], a5[-1]) and t.equal(a5[0], a5[17])
    ref = ang.clone()
    api.engine.leg_solve(sess.d_pose, sess.params, angles=sess.d_angles, fk=sess.d_fk, frames=(0, 512))
    api.engine.leg_solve(sess.d_pose, sess.params, angles=sess.d_angles, fk=sess.d_fk, frames=(512, 1000))
    assert t.equal(sess.d_angles, ref)


def test_long_warm_start_chain_vs_oracle(api, synthetic_long):
    """2000 serially warm-started frames (62 of the kernel's 32-frame resync periods) against the oracle: the carried
    solver state does not drift."""
    S, t = api.synthetic, api.torch
    size, bounds, init = S.chain_constants()
    chain = api.Chain(bounds, list(S.LEGS), size)
    n_frame = int(synthetic_long["n_frame"])
    pose = S.make_trial(int(synthetic_long["trial"]), n_frame)
    legs = [str(l) for l in synthetic_long["legs"]]
    d_pose = t.from_numpy(np.ascontiguousarray(np.stack([pose[:, S.LEGS.index(l)] for l in legs]), dtype=np.float32)).cuda()
    params = t.from_numpy(np.stack([chain.pack_chain_params(l, init[l]) for l in legs]).astype(np.float32)).cuda()
    ang, fk, status, _ = api.engine.leg_solve(d_pose, params)
    assert np.abs(ang.cpu().numpy() - synthetic_long["oracle_angles"]).max() < ANGLE_TOL and status.tolist() == [1, 1]
    from oracle import seqik_oracle as O
    for i, l in enumerate(legs):          # FK the kernel carries vs float64 FK of the angles it returns
        seg = [size[f"{l}_{s}"] for s in O.SEGMENTS]
        fk64 = O.fk_closed_form(ang[i].cpu().numpy().astype(np.float64), seg, pose[:, S.LEGS.index(l), 0])
        assert np.abs(fk64 - fk[i].cpu().numpy()).max() < 1e-5


def test_frame_chunks_and_host_pipeline_equal_one_launch(api):
    """Frames solved in chunks (warm start from the previous chunk's last frame) and the pipelined host call
    (2-D async copies on side streams) are bit-identical to one launch over all frames."""
    S, t = api.synthetic, api.torch
    from seqikpy_b200.batch import BatchedLegIK
    n_trial, n_frame = 3, 197
    size, bounds, init = S.chain_constants()
    chain = api.Chain(bounds, list(S.LEGS), size)
    pose = S.make_trials(range(n_trial), 1000)[:, :n_frame]
    host = t.from_numpy(np.ascontiguousarray(pose.transpose(0, 2, 1, 3, 4))).pin_memory()
    sess = BatchedLegIK(chain, init, S.LEGS, n_trial, n_frame)
    sess.d_pose.copy_(host.reshape(sess.n_chain, n_frame, 5, 3))
    a_ref, f_ref = (x.clone() for x in sess.solve_device())
    ang = t.zeros_like(a_ref)
    fk = t.zeros_like(f_ref)
    for lo, hi in ((0, 64), (64, 128), (128, 192), (192, 197)):          # chunk starts on the 32-frame resync grid
        api.engine.leg_solve(sess.d_pose, sess.params, angles=ang, fk=fk, frames=(lo, hi))
    assert t.equal(ang, a_ref) and t.equal(fk, f_ref)
    for lo, hi in ((0, 1), (1, 40), (40, 41), (41, 197)):                # any other split: equal to float32 rounding
        api.engine.leg_solve(sess.d_pose, sess.params, angles=ang, fk=fk, frames=(lo, hi))
    assert (ang - a_ref).abs().max() < 2e-4 and (fk - f_ref).abs().max() < 1e-4
    for chunks in (1, 2, 3, 200):
        sess.d_angles.zero_(); sess.d_fk.zero_()
        h_a, h_f = sess.solve_host(host, n_chunks=chunks)
        assert t.equal(h_a, a_ref.cpu()) and t.equal(h_f, f_ref.cpu()), chunks
    with pytest.raises(ValueError):
        api.engine.leg_solve(sess.d_pose, sess.params, angles=ang, fk=fk, frames=(5, 200))


def test_joints_only_fk_layout(api):
    """fk_layout="joints" returns exactly rows 5..8 of the full layout (bitwise), through the tensor API, both kernel
    schedules, frame chunks and the pipelined host call; angles are unaffected."""
    S, t = api.synthetic, api.torch
    from seqikpy_b200.batch import BatchedLegIK
    n_trial, n_frame = 3, 160
    size, bounds, init = S.chain_constants()
    chain = api.Chain(bounds, list(S.LEGS), size)
    pose = S.make_trials(range(n_trial), 1000)[:, :n_frame]
    host = t.from_numpy(np.ascontiguousarray(pose.transpose(0, 2, 1, 3, 4))).pin_memory()
    full = BatchedLegIK(chain, init, S.LEGS, n_trial, n_frame)
    full.d_pose.copy_(host.reshape(full.n_chain, n_frame, 5, 3))
    a_ref, f_ref = (x.clone() for x in full.solve_device())
    slim = BatchedLegIK(chain, init, S.LEGS, n_trial, n_frame, fk_layout="joints")
    slim.d_pose.copy_(full.d_pose)
    a_j, f_j = slim.solve_device()
    assert tuple(f_j.shape) == (slim.n_chain, n_frame, 4, 3)
    assert t.equal(a_j, a_ref) and t.equal(f_j, f_ref[:, :, 5:9])
    assert abs(slim.mean_fk_error() - full.mean_fk_error()) < 1e-9
    h_a, h_f = slim.solve_host(host, n_chunks=3)
    assert t.equal(h_a, a_ref.cpu()) and t.equal(h_f, f_ref[:, :, 5:9].cpu())
    _, f_lane, _, _ = api.engine.leg_solve(full.d_pose, full.params, schedule=api.native.SCHED_LANE_PER_CHAIN, fk_layout="joints")
    _, f_lane_full, _, _ = api.engine.leg_solve(full.d_pose, full.params, schedule=api.native.SCHED_LANE_PER_CHAIN)
    assert t.equal(f_lane, f_lane_full[:, :, 5:9])
    with pytest.raises(ValueError):
        api.engine.leg_solve(full.d_pose, full.params, fk=f_ref, fk_layout="joints")        # a 9-row buffer for the 4-row layout
    with pytest.raises(ValueError):
        api.engine.leg_solve(full.d_pose, full.params, fk_layout="rows")


def test_fk_kernel_matches_solver_and_oracle(api, synthetic_gold):
    S, t = api.synthetic, api.torch
    size, bounds, init = S.chain_constants()
    chain = api.Chain(bounds, list(S.LEGS), size)
    ang = t.from_numpy(synthetic_gold["oracle_angles"][0].astype(np.float32)).cuda()          # (6, F, 7)
    origin = t.from_numpy(np.ascontiguousarray(synthetic_gold["pose"][0][:, :, 0].transpose(1, 0, 2), dtype=np.float32)).cuda()
    params = t.from_numpy(np.stack([chain.pack_chain_params(leg, init[leg]) for leg in S.LEGS]).astype(np.float32)).cuda()
    fk = api.engine.forward_kinematics(ang, origin, params).cpu().numpy()
    assert np.abs(fk - synthetic_gold["oracle_fk"][0]).max() < 3e-6
    fk0 = api.engine.forward_kinematics(ang, origin[:, 0].contiguous(), params).cpu().numpy()   # constant origin per chain
    assert np.abs(fk0 - fk).max() < 1e-6


def test_fused_pipeline_equals_the_three_classes(api):
    """Config-5 style pass (alignment statistics + align-on-load solver + head alignment + head angles, all on the
    device) against AlignPose -> LegInvKinSeq / HeadInverseKinematics run one after the other through the dict API."""
    S, t = api.synthetic, api.torch
    from seqikpy_b200.batch import FusedPipeline
    from seqikpy_b200.utils import calculate_body_size
    n_trial, n_frame = 2, 300
    legs = ["RF", "LF"]
    tmpl, size = api.data.NMF_TEMPLATE, calculate_body_size(api.data.NMF_TEMPLATE, legs)
    chain = api.Chain(api.data.BOUNDS, legs, size)
    # leg key points from the grooming-like ranges of the default seeds, head key points from the synthetic generator
    rng = np.random.default_rng(5)
    raw_legs = np.zeros((n_trial, 2, n_frame, 5, 3))
    heads = []
    for tr in range(n_trial):
        for li, leg in enumerate(legs):
            th0 = np.array(api.data.INITIAL_ANGLES[leg]["stage_4"][1:8], dtype=float)
            th0[6] = -0.6
            theta = th0 + 0.2 * np.sin(2 * np.pi * rng.uniform(1, 3, 7) * np.arange(n_frame)[:, None] / 300.0 + rng.uniform(0, 6, 7))
            lb = np.array([api.data.BOUNDS[f"{leg}_{d}"][0] for d in S.DOF_ORDER]) + 0.05
            ub = np.array([api.data.BOUNDS[f"{leg}_{d}"][1] for d in S.DOF_ORDER]) - 0.05
            pts = S.leg_key_points(np.clip(theta, lb, ub), np.array([size[f"{leg}_{s}"] for s in S.SEGMENTS]))
            coxa = np.asarray(tmpl[f"{leg}_Coxa"]) + rng.normal(0, 0.003, (n_frame, 3))
            raw_legs[tr, li, :, 0] = coxa
            raw_legs[tr, li, :, 1:] = pts + coxa[:, None] + rng.normal(0, 0.01, (n_frame, 4, 3))
        heads.append(S.make_head_trial(tr, n_frame))
    raw_legs = S.to_raw(raw_legs)
    r_head = S.to_raw(np.stack([h[0] for h in heads])); l_head = S.to_raw(np.stack([h[1] for h in heads]))
    thorax = S.to_raw(np.stack([h[2] for h in heads]))
    f32 = lambda a: t.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()
    pipe = FusedPipeline(chain, api.data.INITIAL_ANGLES, legs, tmpl, size, n_trial, n_frame)
    out = pipe.run(f32(raw_legs), f32(r_head), f32(l_head), f32(thorax))
    t.cuda.synchronize()
    for tr in range(n_trial):
        raw = {"RF_leg": raw_legs[tr, 0].astype(np.float32).astype(np.float64), "LF_leg": raw_legs[tr, 1].astype(np.float32).astype(np.float64),
               "R_head": r_head[tr].astype(np.float32).astype(np.float64), "L_head": l_head[tr].astype(np.float32).astype(np.float64),
               "Thorax": thorax[tr].astype(np.float32).astype(np.float64)}
        al = api.AlignPose(raw, legs_list=legs, include_claw=False, body_template=tmpl, log_level="ERROR").align_pose()
        ang, fk = api.Leg(al, chain, api.data.INITIAL_ANGLES, log_level="ERROR").run_ik_and_fk()
        head = api.Head(al, tmpl, log_level="ERROR").compute_head_angles()
        for li, leg in enumerate(legs):
            ours = out["angles"][tr, li].cpu().numpy()
            assert np.abs(ours - angles_dict_to_array(ang, leg)).max() < 2e-4, (tr, leg)          # float32 pose rounding
            assert np.abs(out["fk"][tr, li].cpu().numpy() - fk[f"{leg}_leg"]).max() < 1e-4
        for i, k in enumerate(head):
            assert np.abs(out["head_angles"][tr, i].cpu().numpy() - head[k]).max() < 2e-4, (tr, k)


# ------------------------------------------------------------------------------------------ head
def test_head_angles_vs_reference(api, grooming_head):
    pos = {"R_head": grooming_head["r_head"], "L_head": grooming_head["l_head"], "Neck": grooming_head["neck"]}
    hk = api.Head(pos, api.data.NMF_TEMPLATE, log_level="ERROR")
    assert abs(hk.rest_head_pitch[0] - grooming_head["rest"][0]) < 1e-12
    assert abs(hk.rest_antenna_pitch[0] - grooming_head["rest"][1]) < 1e-12
    out = hk.compute_head_angles()
    assert list(out.keys()) == list(grooming_head["keys"])
    for i, k in enumerate(out):
        assert out[k].shape == (6000,) and out[k].dtype == np.float64
        assert np.abs(out[k] - grooming_head["ref_angles"][i]).max() < 2e-5, k     # FP32 atan2 of ~0.1 mm vectors
    assert list(hk.compute_head_angles(compute_ant_angles=False).keys()) == list(grooming_head["keys"][:3])
    # per-frame neck (N,1,3) gives the same result as the broadcast template neck
    pos2 = dict(pos, Neck=np.tile(grooming_head["neck"], (6000, 1, 1)))
    out2 = api.Head(pos2, api.data.NMF_TEMPLATE, log_level="ERROR").compute_head_angles()
    for k in out:
        assert np.array_equal(out[k], out2[k])
    with pytest.raises(ValueError):
        api.Head({"R_head": pos["R_head"]}, api.data.NMF_TEMPLATE)


# ------------------------------------------------------------------------------------------ alignment
def test_alignment_vs_reference(api, grooming_align):
    raw = {k: grooming_align[f"raw_{k}"] for k in grooming_align["raw_keys"]}
    al = api.AlignPose(raw, legs_list=["RF", "LF"], include_claw=False, log_level="ERROR")
    out = al.align_pose()
    assert list(out.keys()) == list(grooming_align["ref_keys"])
    for k in out:
        ref = grooming_align[f"ref_{k}"]
        assert out[k].shape == ref.shape and out[k].dtype == np.float64
        assert np.allclose(out[k], ref, rtol=1e-5, atol=2e-6), (k, np.abs(out[k] - ref).max())   # cf. reference tests/test_alignment.py:93
    # known answers of reference tests/test_alignment.py:54-78 on the full trial
    for leg in ("RF", "LF"):
        ml = al.get_mean_length(grooming_align[f"raw_full_{leg}"], segment_is_leg=True)
        got = np.array([ml[s] for s in ("coxa", "femur", "tibia", "tarsus")])
        assert np.allclose(got, grooming_align[f"{leg}_lengths"], rtol=2e-7, atol=0)
        assert np.isclose(al.find_scale_leg(leg, ml), float(grooming_align[f"{leg}_scale"]), rtol=1e-6)
    assert np.allclose(api.AlignPose.get_fixed_pos(grooming_align["raw_full_RF"][:, 0]), grooming_align["full_RF_coxa_fixed"], rtol=2e-7)
    no_thorax = {k: v for k, v in raw.items() if k != "Thorax"}
    with pytest.raises(AssertionError):
        api.AlignPose(no_thorax, legs_list=["RF", "LF"], log_level="ERROR").align_pose()


def test_mid_quantile_matches_numpy(api):
    t = api.torch
    rng = np.random.default_rng(7)
    for n in (1, 2, 3, 10, 11, 100, 1000, 4097, 8192, 8193, 30011):   # up to 8192 the series is cached in shared memory
        x = rng.normal(size=(5, n)).astype(np.float32)
        x[1] = np.round(x[1], 1)                       # many ties
        x[2] = -np.abs(x[2])                           # all negative
        x[3, : n // 2] = 0.0                           # zeros and signs
        got = api.engine.mid_quantile(t.from_numpy(x).cuda()).cpu().numpy()
        ref = 0.5 * (np.quantile(x.astype(np.float64), 0.45, axis=1) + np.quantile(x.astype(np.float64), 0.55, axis=1))
        assert np.allclose(got, ref, rtol=3e-7, atol=1e-7), n
    with pytest.raises(ValueError):
        api.engine.mid_quantile(t.zeros((3, 0), device="cuda"))


def test_mid_quantile_narrow_ranges_ties_and_counts(api):
    """The warp select starts at the first bit in which the keys of a series differ and compacts the candidates after every
    pass: series that live in a sliver of an octave (segment lengths with 1e-3 noise), constants, two-valued series, series
    that straddle zero, +inf padding with `counts` (the head series), lengths around the 32-key direct finish."""
    t = api.torch
    rng = np.random.default_rng(11)
    for n in (1, 2, 31, 32, 33, 64, 65, 500, 1000, 1023, 1024, 1025, 4096, 4097, 20000, 100003):
        # (beyond 4096 samples: the sampled-range kernel; the constant, two-valued and four-valued series span fewer than
        #  4096 keys and are read off its first sweep's histogram (shift 0); tests/test_gpu_quantile.py covers every route)
        rows = [0.7312 + 1e-3 * rng.normal(size=n), np.full(n, -3.25), rng.choice([1.5, 1.5000001], size=n),
                1e-3 * rng.normal(size=n), np.where(rng.random(n) < 0.5, 0.0, -0.0), 1e30 * rng.normal(size=n),
                np.sort(rng.normal(size=n)), 0.4 + 1e-6 * rng.integers(0, 4, size=n),
                0.5 + 2e-3 * rng.normal(size=n), np.linspace(-1.0, 3.0, n) + 0.05 * rng.normal(size=n)]
        x = np.stack(rows).astype(np.float32)
        got = api.engine.mid_quantile(t.from_numpy(x).cuda()).cpu().numpy()
        ref = 0.5 * (np.quantile(x.astype(np.float64), 0.45, axis=1) + np.quantile(x.astype(np.float64), 0.55, axis=1))
        scale = np.abs(x).max(axis=1).astype(np.float64)               # float32 interpolation between two order statistics
        assert (np.abs(got - ref) <= 3e-7 * scale).all(), (n, got, ref)
        # only the m smallest take part (the rest is +inf padding)
        m = rng.integers(1, n + 1, size=x.shape[0]).astype(np.int32)
        y = x.copy()
        for r in range(y.shape[0]):
            y[r] = np.sort(y[r])
            y[r, m[r]:] = np.inf
            y[r] = rng.permutation(y[r])
        got = api.engine.mid_quantile(t.from_numpy(y).cuda(), t.from_numpy(m).cuda()).cpu().numpy()
        ref = np.array([0.5 * (np.quantile(np.sort(y[r].astype(np.float64))[:m[r]], 0.45) + np.quantile(np.sort(y[r].astype(np.float64))[:m[r]], 0.55))
                        for r in range(y.shape[0])])
        assert (np.abs(got - ref) <= 3e-7 * scale).all(), (n, "counts", got, ref)


@pytest.mark.parametrize("n_frame", [1, 7, 224, 225, 1000, 1024, 1025, 3000])
def test_fused_leg_affine_equals_the_three_kernels(api, n_frame):
    """seqik_leg_affine_from_pose_f32 (one kernel per chain up to 1024 frames, series never written) against the series /
    select / affine kernels, bit for bit, and against numpy on the same key points."""
    t = api.torch
    rng = np.random.default_rng(n_frame)
    n_chain = 13
    pose = (rng.normal(size=(n_chain, 1, 5, 3)) + 0.02 * rng.normal(size=(n_chain, n_frame, 5, 3))).astype(np.float32)
    consts = (1.0 + rng.random((n_chain, 4))).astype(np.float32)
    d_pose, d_consts = t.from_numpy(pose).cuda(), t.from_numpy(consts).cuda()
    for claw in (False, True):
        fused = api.engine.leg_affine(d_pose, d_consts, include_claw=claw)
        three = api.engine.leg_affine_unfused(d_pose, d_consts, include_claw=claw)
        assert t.equal(fused, three)
    p64 = pose.astype(np.float64)
    mid = lambda a: 0.5 * (np.quantile(a, 0.45, axis=1) + np.quantile(a, 0.55, axis=1))
    seg = np.linalg.norm(np.diff(pose, axis=2).astype(np.float32), axis=-1)          # (chain, frame, 4)
    ref_len = mid(seg.astype(np.float64))[:, :3].sum(1)
    got = fused.cpu().numpy() if not claw else api.engine.leg_affine(d_pose, d_consts).cpu().numpy()
    got = api.engine.leg_affine(d_pose, d_consts).cpu().numpy()
    assert np.allclose(got[:, :3], mid(p64[:, :, 0]), rtol=1e-6, atol=1e-7)
    assert np.allclose(got[:, 3], consts[:, 3] / ref_len, rtol=2e-6)
    assert np.array_equal(got[:, 4:7], consts[:, :3]) and (got[:, 7] == 0).all()


# ------------------------------------------------------------------------------------------ edge cases and errors
def test_edge_cases(api):
    chain = api.Chain(api.data.BOUNDS, ["RF", "LF"])
    empty = api.Leg({"RF_leg": np.zeros((0, 5, 3))}, chain, log_level="ERROR").run_ik_and_fk()
    assert empty[0]["Angle_RF_ThC_yaw"].shape == (0,) and empty[1]["RF_leg"].shape == (0, 9, 3)
    rng = np.random.default_rng(3)
    one = rng.normal(scale=0.5, size=(1, 5, 3))
    a, f = api.Leg({"RF_leg": one, "Neck": np.zeros((1, 1, 3)), "XX_leg": one}, chain, log_level="ERROR").run_ik_and_fk()
    assert len(a) == 7 and list(f.keys()) == ["RF_leg"] and np.isfinite(f["RF_leg"]).all()     # XX skipped (not in body_size)
    with pytest.raises(ValueError):
        api.Leg({"RF_leg": one}, chain, log_level="ERROR").run_ik_and_fk(stages=[1, 3])
    with pytest.raises(ValueError):
        api.Leg({"RF_leg": one}, chain, log_level="ERROR").run_ik_and_fk(stages=[3, 4, 5])
    bad_seed = {"RF": {k: v.copy() for k, v in api.data.INITIAL_ANGLES["RF"].items()}}
    bad_seed["RF"]["stage_3"][7] = 0.5                                                           # inert slot, TiTa ub = 0
    with pytest.raises(ValueError, match="Initial guess is outside of provided bounds"):
        api.Leg({"RF_leg": one}, chain, bad_seed, log_level="ERROR").run_ik_and_fk()
    ik = api.Leg({"RF_leg": one}, chain, log_level="ERROR")
    with pytest.raises(ValueError):
        ik.calculate_ik_stage(one[:, 1], one[:, 0], api.data.INITIAL_ANGLES["RF"]["stage_1"], "XX", stage=1)
    with pytest.raises(ValueError):
        ik.calculate_ik_stage(one[:, 1], one[:, 0], api.data.INITIAL_ANGLES["RF"]["stage_1"], "RF", stage=5)
    # NaN key points: the reference (scipy) raises; the batched API flags the chain (-1) and keeps going
    nan_pose = rng.normal(scale=0.5, size=(6, 5, 3))
    nan_pose[3, 2] = np.nan
    with pytest.raises(ValueError, match="not finite"):
        api.Leg({"RF_leg": nan_pose}, chain, log_level="ERROR").run_ik_and_fk()
    t = api.torch
    params = t.from_numpy(np.stack([chain.pack_chain_params(l, api.data.INITIAL_ANGLES[l]) for l in ("RF", "LF")]).astype(np.float32)).cuda()
    both = t.from_numpy(np.stack([nan_pose, rng.normal(scale=0.5, size=(6, 5, 3))]).astype(np.float32)).cuda()
    ang, _, status, _ = api.engine.leg_solve(both, params)
    assert status.tolist() == [-1, 1] and bool(t.isfinite(ang).all())
    # unreachable / degenerate targets still terminate with finite angles inside the bounds
    wild = np.zeros((4, 5, 3))
    wild[1, 1:] = 100.0
    wild[2, 1:] = 1e-30
    wild[3, 1:] = -50.0
    a, f = api.Leg({"LF_leg": wild}, chain, log_level="ERROR").run_ik_and_fk()
    for k, v in a.items():
        lb, ub = api.data.BOUNDS[k.replace("Angle_", "")]
        assert np.isfinite(v).all() and v.min() >= lb - 1e-6 and v.max() <= ub + 1e-6
