"""Generates tests/golden/*.npz.  TEST INFRASTRUCTURE; run in the build container only.

    python oracle/make_golden.py [--reuse-cache DIR]

Reads /root/reference (the read-only reference checkout): its shipped outputs are copied into
compact fixtures, its importable classes (AlignPose, HeadInverseKinematics) are RUN here to
produce outputs for sub-sampled inputs, and the CPU oracle (oracle/seqik_oracle.py = restated
ikpy glue + the installed scipy TRF) is run where the reference ships no output.  The GPU box has
no /root/reference, so everything the parity tests need travels inside these files.

Fixtures
  grooming_leg.npz   bundled data/anipose_220525_aJO_Fly001_001: aligned RF/LF pose (6000,5,3) f64, the reference's
                     shipped leg_joint_angles.pkl (2,6000,7) and forward_kinematics.pkl (first 600 frames), and
                     the oracle's own angles for the same input (2,6000,7)
  grooming_head.npz  same trial: aligned R/L_head, Neck, shipped head_joint_angles.pkl (7,6000)
  grooming_align.npz raw converted_dict.pkl, first 2000 frames, and the output of the reference AlignPose
                     class run on them; plus the known answers of reference tests/test_alignment.py:54-78
                     recomputed on the full trial
  locomotion.npz     bundled data/df3d_pose_result__210902_PR_Fly1 (BASELINE config 1): raw frames 300:400 of the
                     6 legs, reference AlignPose output (== shipped pose3d_aligned.pkl), oracle angles + FK
  synthetic.npz      trials 0-1 x 6 legs x first 250 frames of the synthetic workload: pose, oracle angles + FK
  synthetic_wide.npz trials 2-7 x 6 legs x all 1000 frames of the synthetic workload: oracle angles (float32) and the
                     oracle's FK residual per joint (float32) -- with synthetic.npz the "trials 0-7" parity run of SURVEY.md 8d
  generic_leg.npz    generic 7-DOF IK (LegInvKinGeneric) of the oracle on the first 500 frames of the grooming RF/LF legs:
                     the free-running angles (2,500,9) with status/nfev/cost, and -- because that problem is under-determined and
                     its free-running answer depends on rounding noise -- the SAME solves repeated with the target
                     perturbed by 1e-12 mm from the same seeds (the oracle's own reproducibility, frame by frame)
  loader.npz         the reference's OWN raw-format converters (seqikpy.alignment.convert_from_anipose_to_dict / _df3d_to_dict /
                     _df3dpp_to_dict, imported from /root/reference) run on small inputs in the three formats: an anipose table
                     rebuilt from the bundled converted_dict.pkl with data.PTS2ALIGN's key-point names (40 frames), a
                     DeepFly3D array (30 frames x 38 key points) and the bundled df3dPP dictionary (frames 300:330) --
                     inputs and converter outputs, for the batched loader's key-order semantics
  synthetic_long.npz trial 5, legs RM and LH, 2000 frames: oracle angles (float32) -- a long warm-start chain that spans
                     many of the kernel's 64-frame resync periods
  reference_constants.json
                     INITIAL_ANGLES, BOUNDS, NMF_SIZE, PTS2ALIGN and NMF_TEMPLATE of the reference's seqikpy/data.py
                     (`--constants-only`): key order kept, floats written exactly
"""
import argparse
import os
import pickle
import sys
import time
from multiprocessing import Pool
from pathlib import Path

os.environ.setdefault("OMP_NUM_THREADS", "1")
import numpy as np

ROOT = Path(__file__).resolve().parent.parent
REF = Path("/root/reference")
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(REF))

from oracle import seqik_oracle as O            # noqa: E402
from seqikpy_b200 import data as D             # noqa: E402  (constants only; verified equal to the reference's)
from seqikpy_b200 import synthetic as S        # noqa: E402

GOLD = ROOT / "tests" / "golden"
GROOM = REF / "data/anipose_220525_aJO_Fly001_001/pose-3d"
LOCO = REF / "data/df3d_pose_result__210902_PR_Fly1"
LOCO_LEGS = ["RF", "RM", "RH", "LF", "LM", "LH"]


def load(p):
    with open(p, "rb") as f:
        return pickle.load(f)


def stack7(ang, leg):
    return np.stack([ang[f"Angle_{leg}_{d}"] for d in O.DOF_ORDER], 1)


def _oracle_leg(args):
    key, arr, size, bounds, init = args
    ang, fk = O.run_ik_and_fk({key: arr}, size, bounds, init)
    leg = key.split("_")[0]
    return key, stack7(ang, leg), fk[key]


def _generic_leg(args):
    """Free-running generic oracle + the same solves (same seeds) with the target perturbed by 1e-12 mm."""
    leg, arr, size, bounds, init = args
    stats = []
    ja, fk = O.run_generic_leg(leg, arr[:, -1], arr[:, 0], init, size, bounds, stats=stats)
    teacher = np.vstack([np.asarray(init, dtype=float)[None], ja[:-1]])
    noise = 1e-12 * np.random.default_rng(7).normal(size=(arr.shape[0], 3))
    ja2, _ = O.run_generic_leg(leg, arr[:, -1] + noise, arr[:, 0], init, size, bounds, teacher=teacher)
    st = np.array([(s[2], s[3], s[4]) for s in stats], dtype=float)
    return ja, fk[:, 8], st, ja2


def oracle_legs(pose_dict, size, bounds, init, procs=8):
    """Oracle over several legs in parallel processes (legs are independent)."""
    jobs = [(k, v, size, bounds, init) for k, v in pose_dict.items()]
    with Pool(min(procs, len(jobs))) as pool:
        res = pool.map(_oracle_leg, jobs)
    return {k: (a, f) for k, a, f in res}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reuse-cache", default=None, help="directory with oracle_full_{RF,LF}.pkl from a previous run")
    ap.add_argument("--only", default="", help="comma-separated subset: leg,head,align,loco,synth,wide,long,generic")
    args = ap.parse_args()
    only = set(filter(None, args.only.split(",")))
    GOLD.mkdir(parents=True, exist_ok=True)
    import seqikpy.data as RD
    from seqikpy.alignment import AlignPose, convert_from_df3dpp_to_dict
    from seqikpy.head_inverse_kinematics import HeadInverseKinematics

    aligned = load(GROOM / "pose3d_aligned.pkl")
    # ---------------------------------------------------------------- grooming: legs
    if not only or "leg" in only:
        gold_ang = load(GROOM / "leg_joint_angles.pkl")
        assert gold_ang.keys() == load(REF / "tests/leg_joint_angles.pkl").keys()
        gold_fk = load(GROOM / "forward_kinematics.pkl")
        size = O.calculate_body_size(RD.NMF_TEMPLATE, ["RF", "LF"])
        pose = {k: aligned[k] for k in ("RF_leg", "LF_leg")}
        t0 = time.time()
        if args.reuse_cache:
            orc = {}
            for leg in ("RF", "LF"):
                a, f, _ = load(Path(args.reuse_cache) / f"oracle_full_{leg}.pkl")
                orc[f"{leg}_leg"] = (stack7(a, leg), f[f"{leg}_leg"])
        else:
            orc = oracle_legs(pose, size, RD.BOUNDS, RD.INITIAL_ANGLES)
        print(f"grooming oracle: {time.time() - t0:.1f} s")
        np.savez_compressed(
            GOLD / "grooming_leg.npz",
            pose=np.stack([pose["RF_leg"], pose["LF_leg"]]),
            ref_angles=np.stack([stack7(gold_ang, "RF"), stack7(gold_ang, "LF")]),
            ref_fk=np.stack([gold_fk["RF_leg"][:600], gold_fk["LF_leg"][:600]]),
            oracle_angles=np.stack([orc["RF_leg"][0], orc["LF_leg"][0]]),
            legs=np.array(["RF", "LF"]), angle_keys=np.array(list(gold_ang.keys())))
    # ---------------------------------------------------------------- grooming: head
    if not only or "head" in only:
        gold_head = load(GROOM / "head_joint_angles.pkl")
        # the reference class itself, with the scipy>=1.12 shim for Rotation.from_euler on an (N,) angle array
        def derotate(self, roll, vec):
            c, s = np.cos(-roll), np.sin(-roll)
            out = np.array(vec, dtype=float)
            out[..., 1] = c * vec[..., 1] - s * vec[..., 2]
            out[..., 2] = s * vec[..., 1] + c * vec[..., 2]
            return out
        HeadInverseKinematics.derotate_vector = derotate
        run = HeadInverseKinematics(aligned, RD.NMF_TEMPLATE, log_level="ERROR")
        try:
            ref_run = run.compute_head_angles()
            dev = max(np.abs(ref_run[k] - gold_head[k]).max() for k in gold_head)
            print("reference head class (shimmed) vs shipped pickle:", dev)
        except Exception as e:   # the shim is only a cross-check; the shipped pickle is the golden
            print("reference head class could not be run here:", type(e).__name__, e)
        np.savez_compressed(
            GOLD / "grooming_head.npz",
            r_head=aligned["R_head"], l_head=aligned["L_head"], neck=aligned["Neck"],
            ref_angles=np.stack([gold_head[k] for k in gold_head]), keys=np.array(list(gold_head.keys())),
            rest=np.array([float(run.rest_head_pitch[0]), float(run.rest_antenna_pitch[0])]))
    # ---------------------------------------------------------------- grooming: alignment
    if not only or "align" in only:
        raw = load(GROOM / "converted_dict.pkl")
        n_sub = 2000
        sub = {k: v[:n_sub].copy() for k, v in raw.items()}
        ref_sub = AlignPose(sub, legs_list=["RF", "LF"], include_claw=False, log_level="ERROR").align_pose()
        full_cls = AlignPose(raw, legs_list=["RF", "LF"], include_claw=False, log_level="ERROR")
        full = full_cls.align_pose()
        for k in full:
            assert np.array_equal(full[k], aligned[k]), k            # reference class reproduces its shipped output
        ant = np.load(REF / "tests/antenna.npy")
        assert np.array_equal(ant[:, :2], full["R_head"]) and np.array_equal(ant[:, 2:], full["L_head"])
        known = {}
        for leg in ("RF", "LF"):
            ml = full_cls.get_mean_length(raw[f"{leg}_leg"], segment_is_leg=True)
            known[f"{leg}_lengths"] = np.array([ml[s] for s in ("coxa", "femur", "tibia", "tarsus")])
            known[f"{leg}_scale"] = np.array(full_cls.find_scale_leg(leg, ml))
        # literals of reference tests/test_alignment.py:54-78 (a test the reference's own suite shadows and never runs)
        assert known["RF_lengths"].tolist() == [0.33463473686922274, 0.6652300069548103, 0.5083878473974696, 0.5542674489903121]
        assert known["LF_lengths"].tolist() == [0.3042863816867363, 0.6616840367058072, 0.5101094810133566, 0.5423598868556229]
        assert np.isclose(known["RF_scale"], 1.0807208351486381) and np.isclose(known["LF_scale"], 1.1042762662482228)
        np.savez_compressed(
            GOLD / "grooming_align.npz",
            **{f"raw_{k}": v for k, v in sub.items()}, **{f"ref_{k}": v for k, v in ref_sub.items()},
            raw_keys=np.array(list(sub.keys())), ref_keys=np.array(list(ref_sub.keys())),
            full_RF_coxa_fixed=np.array(AlignPose.get_fixed_pos(raw["RF_leg"][:, 0])), **known,
            full_first_frames=np.stack([full["RF_leg"][:5], full["LF_leg"][:5]]),
            raw_full_RF=raw["RF_leg"].astype(np.float64), raw_full_LF=raw["LF_leg"].astype(np.float64))
    # ---------------------------------------------------------------- locomotion (config 1)
    if not only or "loco" in only:
        rawl = convert_from_df3dpp_to_dict(load(LOCO / "pose_result__210902_PR_Fly1_aligned.pkl"), None)
        subl = {k: v[300:400].copy() for k, v in rawl.items()}       # examples/seqikpy_locomotion.ipynb uses frames 300:400
        al = AlignPose(subl, legs_list=LOCO_LEGS, include_claw=False, body_template=D.TEMPLATE_NMF_LOCOMOTION,
                       log_level="ERROR").align_pose()
        ship = load(LOCO / "pose3d_aligned.pkl")
        for k in ship:
            assert np.array_equal(al[k], ship[k]), k
        size = O.calculate_body_size(D.TEMPLATE_NMF_LOCOMOTION, LOCO_LEGS)
        t0 = time.time()
        orc = oracle_legs({k: al[k] for k in al if "leg" in k}, size, D.BOUNDS_LOCOMOTION, D.INITIAL_ANGLES_LOCOMOTION)
        print(f"locomotion oracle: {time.time() - t0:.1f} s")
        keys = [f"{leg}_leg" for leg in LOCO_LEGS]
        np.savez_compressed(
            GOLD / "locomotion.npz", legs=np.array(LOCO_LEGS),
            raw=np.stack([subl[k] for k in keys]), aligned=np.stack([al[k] for k in keys]),
            oracle_angles=np.stack([orc[k][0] for k in keys]), oracle_fk=np.stack([orc[k][1] for k in keys]))
    # ---------------------------------------------------------------- synthetic (configs 3-5)
    if not only or "synth" in only:
        n_frame, trials = 250, (0, 1)
        size, bounds, init = S.chain_constants()
        poses, angs, fks = [], [], []
        t0 = time.time()
        for tr in trials:
            pose = S.make_trial(tr, 1000)[:n_frame]                  # first frames of the 1000-frame trial
            d = {f"{leg}_leg": np.ascontiguousarray(pose[:, li]) for li, leg in enumerate(S.LEGS)}
            orc = oracle_legs(d, size, bounds, init)
            poses.append(pose)
            angs.append(np.stack([orc[f"{leg}_leg"][0] for leg in S.LEGS]))
            fks.append(np.stack([orc[f"{leg}_leg"][1] for leg in S.LEGS]))
        print(f"synthetic oracle: {time.time() - t0:.1f} s")
        np.savez_compressed(GOLD / "synthetic.npz", trials=np.array(trials), legs=np.array(S.LEGS),
                            pose=np.stack(poses), oracle_angles=np.stack(angs), oracle_fk=np.stack(fks))
    # ---------------------------------------------------------------- synthetic trials 2-7, all 1000 frames (SURVEY.md 8d parity run)
    if not only or "wide" in only:
        trials, n_frame = [2, 3, 4, 5, 6, 7], 1000
        size, bounds, init = S.chain_constants()
        t0 = time.time()
        jobs = {}
        for tr in trials:
            pose = S.make_trial(tr, n_frame)
            for li, leg in enumerate(S.LEGS):
                jobs[(tr, leg)] = (f"{leg}_leg", np.ascontiguousarray(pose[:, li]), size, bounds, init)
        with Pool(8) as pool:
            res = pool.map(_oracle_leg, list(jobs.values()))
        ang = np.stack([r[1] for r in res]).reshape(len(trials), 6, n_frame, 7)
        fk = np.stack([r[2] for r in res]).reshape(len(trials), 6, n_frame, 9, 3)
        poses = np.stack([S.make_trial(tr, n_frame) for tr in trials]).transpose(0, 2, 1, 3, 4)      # (trial, leg, frame, 5, 3)
        resid = np.linalg.norm(fk[:, :, :, [5, 6, 7, 8]] - poses[:, :, :, 1:5], axis=-1)
        print(f"wide synthetic oracle: {time.time() - t0:.1f} s, mean FK error {resid.mean():.5f} mm")
        np.savez_compressed(GOLD / "synthetic_wide.npz", trials=np.array(trials), legs=np.array(S.LEGS), n_frame=np.array(n_frame),
                            oracle_angles=ang.astype(np.float32), oracle_fk_residual=resid.astype(np.float32))
    # ---------------------------------------------------------------- generic 7-DOF IK (LegInvKinGeneric)
    if not only or "generic" in only:
        n_frame = 500
        size = O.calculate_body_size(RD.NMF_TEMPLATE, ["RF", "LF"])
        t0 = time.time()
        with Pool(2) as pool:
            res = pool.map(_generic_leg, [(leg, aligned[f"{leg}_leg"][:n_frame], size, RD.BOUNDS, RD.INITIAL_ANGLES[leg]["stage_4"])
                                          for leg in ("RF", "LF")])
        print(f"generic oracle: {time.time() - t0:.1f} s")
        np.savez_compressed(GOLD / "generic_leg.npz", legs=np.array(["RF", "LF"]), n_frame=np.array(n_frame),
                            oracle_angles=np.stack([r[0] for r in res]), oracle_fk_claw=np.stack([r[1] for r in res]),
                            oracle_stats=np.stack([r[2] for r in res]), perturbed_angles=np.stack([r[3] for r in res]))
    # ---------------------------------------------------------------- long warm-start chain (drift check)
    if not only or "long" in only:
        n_frame, trial, legs = 2000, 5, ("RM", "LH")
        size, bounds, init = S.chain_constants()
        pose = S.make_trial(trial, n_frame)
        t0 = time.time()
        d = {f"{leg}_leg": np.ascontiguousarray(pose[:, S.LEGS.index(leg)]) for leg in legs}
        orc = oracle_legs(d, size, bounds, init)
        print(f"long-chain oracle: {time.time() - t0:.1f} s")
        np.savez_compressed(GOLD / "synthetic_long.npz", trial=np.array(trial), legs=np.array(legs), n_frame=np.array(n_frame),
                            oracle_angles=np.stack([orc[f"{leg}_leg"][0] for leg in legs]).astype(np.float32))
    for f in sorted(GOLD.glob("*.npz")):
        print(f.name, f.stat().st_size // 1024, "KiB")


def make_loader_fixture():
    """Inputs in the three raw formats + what the reference's converters make of them."""
    from seqikpy import alignment as RA                       # the reference's module (imports without ikpy)
    from seqikpy.data import PTS2ALIGN as REF_PTS
    out = {}
    # anipose: a table rebuilt from the bundled converted dictionary
    conv = load(GROOM / "converted_dict.pkl")
    n = 40
    table = {}
    for seg, kps in REF_PTS.items():
        if seg not in conv:
            continue
        for i, kp in enumerate(kps):
            for a, ax in enumerate("xyz"):
                table[f"{kp}_{ax}"] = np.asarray(conv[seg][:n, i, a], dtype=np.float64)
    pts = {seg: kps for seg, kps in REF_PTS.items() if seg in conv}
    ref = RA.convert_from_anipose_to_dict(table, pts)
    out["anipose_columns"] = np.array(sorted(table.keys()))
    out["anipose_table"] = np.stack([table[k] for k in sorted(table.keys())])
    out["anipose_segments"] = np.array(list(pts.keys()))
    for seg in pts:
        out[f"anipose_ref_{seg}"] = ref[seg]
        out[f"anipose_kps_{seg}"] = np.array(pts[seg])
        assert np.array_equal(ref[seg], conv[seg][:n])
    # df3d: an array of 38 key points and the index map of the reference's docstring (alignment.py:172-179)
    rng = np.random.default_rng(7)
    arr = rng.normal(size=(30, 38, 3))
    idx = {"RF_leg": np.arange(0, 5), "RM_leg": np.arange(5, 10), "RH_leg": np.arange(10, 15),
           "LF_leg": np.arange(19, 24), "LM_leg": np.arange(24, 29), "LH_leg": np.arange(29, 34)}
    ref = RA.convert_from_df3d_to_dict(arr, idx)
    out["df3d_array"] = arr
    for seg, ix in idx.items():
        out[f"df3d_idx_{seg}"] = ix
        out[f"df3d_ref_{seg}"] = ref[seg]
    # df3dPP: the bundled dictionary
    pp = load(LOCO / "pose_result__210902_PR_Fly1_aligned.pkl")
    segs = [f"{leg}_leg" for leg in LOCO_LEGS]
    cut = {seg: {kp: {"raw_pos_aligned": np.asarray(pp[seg][kp]["raw_pos_aligned"])[300:330]} for kp in ("Coxa", "Femur", "Tibia", "Tarsus", "Claw")}
           for seg in segs}
    ref = RA.convert_from_df3dpp_to_dict(cut, segs)
    for seg in segs:
        out[f"df3dpp_raw_{seg}"] = np.stack([cut[seg][kp]["raw_pos_aligned"] for kp in ("Coxa", "Femur", "Tibia", "Tarsus", "Claw")])
        out[f"df3dpp_ref_{seg}"] = ref[seg]
    np.savez_compressed(GOLD / "loader.npz", **out)
    print("loader.npz", {k: v.shape for k, v in out.items() if k.endswith(("_table", "_array")) or "_ref_RF" in k})


REFERENCE_CONSTANTS = ("INITIAL_ANGLES", "BOUNDS", "NMF_SIZE", "PTS2ALIGN", "NMF_TEMPLATE")


def make_constants_fixture(data_module):
    """The public constants of `data_module` (the reference's seqikpy.data) as JSON; json writes floats by repr, so the
    values read back bit for bit."""
    import json

    def plain(v):
        if isinstance(v, dict):
            return {str(k): plain(x) for k, x in v.items()}
        return np.asarray(v).tolist()
    out = {name: plain(getattr(data_module, name)) for name in REFERENCE_CONSTANTS}
    (GOLD / "reference_constants.json").write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    if "--constants-only" in sys.argv:
        import seqikpy.data as RD
        make_constants_fixture(RD)
    elif "--loader-only" in sys.argv:
        make_loader_fixture()
    else:
        main()
