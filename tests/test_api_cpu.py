"""Host-side logic of the drop-in layer (no GPU): chain definitions, constants, packing, validation, sharding."""
import numpy as np
import pytest

from seqikpy_b200 import data as D
from seqikpy_b200 import synthetic as S
from seqikpy_b200.batch import chain_param_table, shard_range
from seqikpy_b200.engine import stages_to_mask
from seqikpy_b200.kinematic_chain import DOF_ORDER, KinematicChainSeq
from seqikpy_b200.utils import calculate_body_size, load_file, save_file


@pytest.fixture(scope="module")
def chain():
    return KinematicChainSeq(bounds_dof=D.BOUNDS, legs_list=["RF", "LF"], body_size=None)


@pytest.mark.parametrize("leg", ["RF", "LF"])
def test_link_names_per_stage(chain, leg, grooming_leg):
    """Mirror of reference tests/test_kin_chain.py:24-85 (same attributes, link-name sets and exceptions)."""
    for attr in ("bounds_dof", "body_size", "create_leg_chain_stage_1", "create_leg_chain_stage_2",
                 "create_leg_chain_stage_3", "create_leg_chain_stage_4"):
        assert hasattr(chain, attr)
    li = 0 if leg == "RF" else 1
    angles = {f"Angle_{leg}_{d}": grooming_leg["ref_angles"][li][:, i] for i, d in enumerate(DOF_ORDER)}
    s1 = chain.create_leg_chain(leg_name=leg, stage=1)
    assert {l.name for l in s1.links} == {"Base link", f"{leg}_ThC_yaw", f"{leg}_ThC_pitch", f"{leg}_CTr_pitch"}
    s2 = chain.create_leg_chain(leg_name=leg, stage=2, angles=angles, t=0)
    assert {l.name for l in s2.links} == {"Base link", f"{leg}_ThC_yaw", f"{leg}_ThC_pitch", f"{leg}_ThC_roll",
                                         f"{leg}_CTr_pitch", f"{leg}_FTi_pitch"}
    s3 = chain.create_leg_chain(leg_name=leg, stage=3, angles=angles, t=0)
    assert len(s3.links) == 8 and f"{leg}_CTr_roll" in {l.name for l in s3.links}
    s4 = chain.create_leg_chain(leg_name=leg, stage=4, angles=angles, t=5)
    assert [l.name for l in s4.links] == ["Base link"] + [f"{leg}_{d}" for d in DOF_ORDER] + [f"{leg}_Claw"]
    # frozen links carry the angle of frame t in the matching rpy slot; the free link keeps its bounds
    assert s4.links[1].joint_type == "fixed" and s4.links[1].origin_orientation[0] == angles[f"Angle_{leg}_ThC_yaw"][5]
    assert s4.links[4].origin_orientation[1] == angles[f"Angle_{leg}_CTr_pitch"][5]
    assert s4.links[7].joint_type == "revolute" and tuple(s4.links[7].bounds) == tuple(D.BOUNDS[f"{leg}_TiTa_pitch"])
    assert np.allclose(s4.links[4].origin_translation, [0, 0, -chain.body_size[f"{leg}_Coxa"]])
    assert tuple(s4.links[8].bounds) == (-np.pi, np.pi)


def test_chain_errors(chain):
    with pytest.raises(ValueError):
        chain.create_leg_chain(leg_name="XX", stage=1)
    with pytest.raises(ValueError):
        chain.create_leg_chain(leg_name="RF", stage=5)


def test_body_size_and_pickle_io(tmp_path):
    size = calculate_body_size(D.NMF_TEMPLATE, ["RF", "LF"])
    assert list(size.keys())[:4] == ["RF_Coxa", "LF_Coxa", "RF_Femur", "LF_Femur"]          # reference key order
    for k in ("RF_Coxa", "RF_Femur", "RF_Tibia", "RF_Tarsus", "RF", "Antenna", "Antenna_mid_thorax"):
        assert np.isclose(size[k], D.NMF_SIZE[k]), k
    with pytest.raises(NameError):
        calculate_body_size(D.NMF_TEMPLATE, ["XX"])
    save_file(tmp_path / "x.pkl", {"a": np.arange(3.0)})
    assert np.array_equal(load_file(tmp_path / "x.pkl")["a"], np.arange(3.0))


def test_pack_chain_params_layout(chain):
    row = chain.pack_chain_params("RF", D.INITIAL_ANGLES["RF"])
    assert row.shape == (32,)
    assert np.allclose(row[0:4], [0.4, 0.69, 0.54, 0.63])
    assert np.allclose(row[4:11], [D.BOUNDS[f"RF_{d}"][0] for d in DOF_ORDER])
    assert np.allclose(row[11:18], [D.BOUNDS[f"RF_{d}"][1] for d in DOF_ORDER])
    assert np.allclose(row[18:25], [0.45, -0.07, -0.32, -2.14, -1.25, 1.48, 0.0])
    # squared norms of the inert slots (SURVEY.md 3.3): 2.14, 1.472, 2.211, 2.940
    assert np.allclose(np.sqrt(row[25:29]), [2.14, 1.4722, 2.2112, 2.9398], atol=1e-3)
    assert np.all(row[29:] == 0)


def test_seed_validation_matches_scipy_semantics(chain):
    ok = {k: v.copy() for k, v in D.INITIAL_ANGLES["RF"].items()}
    chain.pack_chain_params("RF", ok)                                     # TiTa seed 0.0 == ub is legal (on the bound)
    bad = {k: v.copy() for k, v in ok.items()}
    bad["stage_2"][5] = -0.1                                              # inert last slot FTi_pitch below lb = 0
    with pytest.raises(ValueError, match="Initial guess is outside of provided bounds"):
        chain.pack_chain_params("RF", bad)
    chain.pack_chain_params("RF", bad, stages=(1,))                       # only the stages that run are checked
    short = {k: v.copy() for k, v in ok.items()}
    short["stage_3"] = short["stage_3"][:7]
    with pytest.raises(ValueError, match="Inconsistent shapes"):
        chain.pack_chain_params("RF", short)


def test_stage_list_validation():
    assert stages_to_mask([1, 2, 3, 4]) == 0xF and stages_to_mask([2, 3]) == 0b0110 and stages_to_mask([4]) == 0b1000
    for bad in ([1, 3], [0, 1], [3, 4, 5], [2, 1], []):
        with pytest.raises(ValueError):
            stages_to_mask(bad)


def test_shard_range_partitions_trials():
    for n, w in ((10000, 8), (1000, 3), (7, 8), (0, 2), (5, 1)):
        spans = [shard_range(n, r, w) for r in range(w)]
        assert spans[0][0] == 0 and spans[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        sizes = [hi - lo for lo, hi in spans]
        assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        shard_range(10, 2, 2)


def test_synthetic_workload_is_reproducible_and_feasible(synthetic_gold):
    pose = S.make_trial(1, 1000)
    assert pose.shape == (1000, 6, 5, 3)
    assert np.array_equal(pose, S.make_trial(1, 1000))
    assert np.abs(pose[:250] - synthetic_gold["pose"][1]).max() == 0.0       # fixture == generator
    assert not np.array_equal(pose, S.make_trial(2, 1000))
    size, bounds, init = S.chain_constants()
    chain6 = KinematicChainSeq(bounds, list(S.LEGS), size)
    table = chain_param_table(chain6, init, S.LEGS, 3)
    assert table.shape == (18, 32) and table.dtype == np.float32 and np.array_equal(table[:6], table[12:])
    # segment lengths of the noise-free key points equal the template's
    p, truth = S.make_trial(0, 50, return_truth=True)
    for li, leg in enumerate(S.LEGS):
        clean = S.leg_key_points(truth[:, li], np.array([size[f"{leg}_{s}"] for s in ("Coxa", "Femur", "Tibia", "Tarsus")]))
        assert np.allclose(np.linalg.norm(clean[:, 0], axis=1), size[f"{leg}_Coxa"])
        assert np.allclose(np.linalg.norm(clean[:, 3] - clean[:, 2], axis=1), size[f"{leg}_Tarsus"])
    chains = S.to_chains(S.make_trials([0, 1], 20))
    assert chains.shape == (12, 20, 5, 3) and np.array_equal(chains[7, 3], S.make_trial(1, 20)[3, 1].astype(np.float32))


def test_constants_equal_reference():
    """The public constants equal the reference's seqikpy/data.py, stored in tests/golden/reference_constants.json
    (oracle/make_golden.py --constants-only); its key-point names also travel in loader.npz."""
    import json
    import conftest
    ref_all = json.loads((conftest.GOLDEN / "reference_constants.json").read_text())
    loader = np.load(conftest.GOLDEN / "loader.npz")
    for seg in loader["anipose_segments"]:
        assert D.PTS2ALIGN[str(seg)] == [str(k) for k in loader[f"anipose_kps_{seg}"]], seg
    for name in ("INITIAL_ANGLES", "BOUNDS", "NMF_SIZE", "PTS2ALIGN", "NMF_TEMPLATE"):
        ours, ref = getattr(D, name), ref_all[name]
        assert list(ours.keys()) == list(ref.keys()), name
        for k in ours:
            if isinstance(ours[k], dict):
                assert all(np.array_equal(ours[k][kk], ref[k][kk]) for kk in ref[k]), (name, k)
            else:
                assert np.array_equal(np.asarray(ours[k]), np.asarray(ref[k])), (name, k)


def test_raw_format_converters(locomotion, tmp_path):
    """Converters feeding AlignPose (reference alignment.py:103-226): shapes, values, and agreement with the reference's
    own functions on the inputs and outputs of them stored in tests/golden/loader.npz."""
    import pickle
    import conftest
    from seqikpy_b200.alignment import (AlignPose, convert_from_anipose_to_dict, convert_from_df3d_to_dict,
                                        convert_from_df3dpp_to_dict)
    rng = np.random.default_rng(0)
    n = 17
    table = {f"{kp}_{ax}": rng.normal(size=n) for kps in D.PTS2ALIGN.values() for kp in kps for ax in "xyz"}
    conv = convert_from_anipose_to_dict(table, D.PTS2ALIGN)
    assert list(conv.keys()) == list(D.PTS2ALIGN.keys())
    assert conv["RF_leg"].shape == (n, 5, 3) and conv["Thorax"].shape == (n, 3, 3) and conv["R_head"].shape == (n, 2, 3)
    assert np.array_equal(conv["LF_leg"][:, 2, 1], table["femur_tibia_L_y"])
    arr = rng.normal(size=(n, 38, 3))
    idx = {"RF_leg": np.arange(0, 5), "LH_leg": np.arange(29, 34)}
    d3 = convert_from_df3d_to_dict(arr, idx)
    assert np.array_equal(d3["LH_leg"], arr[:, 29:34]) and d3["RF_leg"].base is None
    pp = {f"{leg}_leg": {kp: {"raw_pos_aligned": locomotion["raw"][i][:, j]} for j, kp in enumerate(("Coxa", "Femur", "Tibia", "Tarsus", "Claw"))}
          for i, leg in enumerate(locomotion["legs"])}
    dpp = convert_from_df3dpp_to_dict(pp, ["RF_leg", "LM_leg"])
    assert list(dpp.keys()) == ["RF_leg", "LM_leg"] and np.array_equal(dpp["LM_leg"], locomotion["raw"][4])
    # from_file_path: newest match, optional conversion, FileNotFoundError (reference tests/test_alignment.py:22-27)
    with open(tmp_path / "pose3d.h5", "wb") as f:
        pickle.dump(table, f)
    al = AlignPose.from_file_path(main_dir=tmp_path, file_name="pose3d.*", legs_list=["RF", "LF"],
                                  convert_func=convert_from_anipose_to_dict, pts2align=D.PTS2ALIGN, log_level="ERROR")
    assert al.pose_data_dict["RF_leg"].shape == (n, 5, 3) and al.include_claw is False
    with pytest.raises(FileNotFoundError):
        AlignPose.from_file_path(main_dir=tmp_path, file_name="nothing.*", legs_list=["RF"])
    gold = np.load(conftest.GOLDEN / "loader.npz")
    table_r = {str(k): gold["anipose_table"][i] for i, k in enumerate(gold["anipose_columns"])}
    pts_r = {str(s): [str(k) for k in gold[f"anipose_kps_{s}"]] for s in gold["anipose_segments"]}
    conv_r = convert_from_anipose_to_dict(table_r, pts_r)
    assert list(conv_r.keys()) == list(pts_r.keys()) and all(np.array_equal(v, gold[f"anipose_ref_{k}"]) for k, v in conv_r.items())
    segs = [f"{leg}_leg" for leg in ("RF", "RM", "RH", "LF", "LM", "LH")]
    d3_r = convert_from_df3d_to_dict(gold["df3d_array"], {s: gold[f"df3d_idx_{s}"] for s in segs})
    assert all(np.array_equal(d3_r[s], gold[f"df3d_ref_{s}"]) for s in segs)
    pp_r = {s: {kp: {"raw_pos_aligned": gold[f"df3dpp_raw_{s}"][j]} for j, kp in enumerate(("Coxa", "Femur", "Tibia", "Tarsus", "Claw"))}
            for s in segs}
    dpp_r = convert_from_df3dpp_to_dict(pp_r, segs)
    assert list(dpp_r.keys()) == segs and all(np.array_equal(dpp_r[s], gold[f"df3dpp_ref_{s}"]) for s in segs)


def test_interpolate_joint_angles_needs_the_device():
    """utils.interpolate_* run the pchip kernel (tests/test_gpu_resample.py holds the parity checks against scipy and the
    reference's function); without a CUDA device they raise like every other compute path."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    from seqikpy_b200._native import SeqIKNativeError
    from seqikpy_b200.utils import interpolate_joint_angles, interpolate_signal
    with pytest.raises(SeqIKNativeError):
        interpolate_signal(np.arange(5.0), 1.0, 0.5)
    with pytest.raises(SeqIKNativeError):
        interpolate_joint_angles({"Angle_RF_ThC_yaw": np.arange(5.0)}, original_ts=0.01, new_ts=0.001)



def test_missing_stage_seed_raises_keyerror(chain):
    """A stage that is solved needs its seed vector: the reference indexes initial_angles[leg]["stage_k"] (KeyError,
    leg_inverse_kinematics.py:376); only stages that are NOT solved may be absent."""
    seeds = dict(D.INITIAL_ANGLES["RF"])
    del seeds["stage_3"]
    with pytest.raises(KeyError):
        chain.pack_chain_params("RF", seeds)
    row = chain.pack_chain_params("RF", seeds, stages=(1, 2))          # stage 3 not solved: allowed
    assert row[18 + 4] == 0.0 and row[18 + 2] == D.INITIAL_ANGLES["RF"]["stage_2"][3]


def test_leg_ik_class_exposes_the_solver_mode():
    """LegInvKinSeq(reference_iterates=True) / flags= select the validated flag sets of include/seqik.h."""
    from seqikpy_b200 import _native as N
    from seqikpy_b200.leg_inverse_kinematics import LegInvKinSeq
    ch = KinematicChainSeq(bounds_dof=D.BOUNDS, legs_list=["RF"], body_size=None)
    pose = {"RF_leg": np.zeros((2, 5, 3))}
    assert LegInvKinSeq(pose, ch, D.INITIAL_ANGLES, log_level="ERROR").flags == N.FLAG_DEFAULT
    assert LegInvKinSeq(pose, ch, D.INITIAL_ANGLES, log_level="ERROR", reference_iterates=True).flags == N.FLAG_REFERENCE_ITERATES
    assert LegInvKinSeq(pose, ch, D.INITIAL_ANGLES, log_level="ERROR", flags=0x7F).flags == 0x7F

