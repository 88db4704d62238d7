"""Builds and loads tests/hostsim (the g++ build of csrc/seqik_core.cuh).  TEST INFRASTRUCTURE."""
import ctypes
import os
import subprocess
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
CSRC = ROOT / "sequential-inverse-kinematics_b200" / "csrc"
SRC = Path(__file__).resolve().parent / "hostsim" / "hostsim.cpp"
OUT = Path(__file__).resolve().parent / "hostsim" / "libhostsim.so"

_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    deps = [SRC, CSRC / "seqik_core.cuh", CSRC / "seqik_generic.cuh", CSRC / "seqik_block.cuh"]
    if not OUT.exists() or any(d.stat().st_mtime > OUT.stat().st_mtime for d in deps):
        # -ffp-contract=off: no FMA contraction, so the f64 build tracks the Python model closely
        cmd = ["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-std=c++17", "-x", "c++", str(SRC),
               "-I", str(CSRC), "-o", str(OUT)]
        subprocess.run(cmd, check=True)
    _lib = ctypes.CDLL(os.fspath(OUT))
    return _lib


def solve_chain(pose, seg, lb, ub, null_sq, seed, dtype=np.float32, stage_mask=0xF, gn_mask=0):
    """pose (N,5,3) -> angles (N,7), fk (N,9,3), nfev (N,4), status (N,4) computed by the host build."""
    lib = load()
    fn = lib.hostsim_chain_f32 if dtype == np.float32 else lib.hostsim_chain_f64
    pose = np.ascontiguousarray(pose, dtype=dtype)
    n = pose.shape[0]
    args = [np.ascontiguousarray(a, dtype=dtype) for a in (seg, lb, ub, null_sq, seed)]
    angles = np.zeros((n, 7), dtype=dtype)
    fk = np.zeros((n, 9, 3), dtype=dtype)
    nfev = np.zeros((n, 4), dtype=np.int32)
    status = np.zeros((n, 4), dtype=np.int32)
    P = ctypes.c_void_p
    fn.argtypes = [P, ctypes.c_int64, P, P, P, P, P, P, P, P, P, ctypes.c_int, ctypes.c_int]
    fn.restype = None
    fn(pose.ctypes.data, n, *(a.ctypes.data for a in args), angles.ctypes.data, fk.ctypes.data,
       nfev.ctypes.data, status.ctypes.data, stage_mask, gn_mask)
    return angles, fk, nfev, status


def chain_iterates_f32(pose, seg, lb, ub, null_sq, seed, gn_mask=0):
    """solve_chain (float32, all stages) -> angles (N,7) and the final iterates before the output clamp (N,7) float64."""
    lib = load()
    pose = np.ascontiguousarray(pose, dtype=np.float32)
    n = pose.shape[0]
    args = [np.ascontiguousarray(a, dtype=np.float32) for a in (seg, lb, ub, null_sq, seed)]
    angles = np.zeros((n, 7), dtype=np.float32)
    it = np.zeros((n, 7), dtype=np.float64)
    P = ctypes.c_void_p
    fn = lib.hostsim_chain_iterates_f32
    fn.argtypes = [P, ctypes.c_int64, P, P, P, P, P, P, P, ctypes.c_int]
    fn.restype = None
    fn(pose.ctypes.data, n, *(a.ctypes.data for a in args), angles.ctypes.data, it.ctypes.data, gn_mask)
    return angles, it


def run_runner_f32(pose, seg, lb, ub, null_sq, seed, stage_mask=0xF, gn_mask=0):
    """Same chain through ChainRunner::step() (the kernels' per-lane state machine)."""
    lib = load()
    dtype = np.float32
    pose = np.ascontiguousarray(pose, dtype=dtype)
    n = pose.shape[0]
    args = [np.ascontiguousarray(a, dtype=dtype) for a in (seg, lb, ub, null_sq, seed)]
    angles = np.zeros((n, 7), dtype=dtype)
    fk = np.zeros((n, 9, 3), dtype=dtype)
    nfev_sum = np.zeros(4, dtype=np.uint32)
    P = ctypes.c_void_p
    fn = lib.hostsim_runner_f32
    fn.argtypes = [P, ctypes.c_int64, P, P, P, P, P, P, P, P, ctypes.c_int, ctypes.c_int]
    fn.restype = ctypes.c_int64
    steps = fn(pose.ctypes.data, n, *(a.ctypes.data for a in args), angles.ctypes.data, fk.ctypes.data,
               nfev_sum.ctypes.data, stage_mask, gn_mask)
    return angles, fk, nfev_sum, steps


def run_carried_f32(pose, prm, gn_mask=0xFF):
    """The stage-pipeline kernel's per-lane arithmetic (solves carried frame to frame by StageSolve::restart, re-derived
    every SEQIK_RESYNC frames), run serially on the host build: pose (N,5,3), prm (32,) -> angles (N,7), fk (N,9,3),
    nfev (N,4)."""
    lib = load()
    pose = np.ascontiguousarray(pose, dtype=np.float32)
    prm = np.ascontiguousarray(prm, dtype=np.float32)
    n = pose.shape[0]
    angles = np.zeros((n, 7), dtype=np.float32)
    fk = np.zeros((n, 9, 3), dtype=np.float32)
    nfev = np.zeros((n, 4), dtype=np.int32)
    P = ctypes.c_void_p
    fn = lib.hostsim_carried_f32
    fn.argtypes = [P, ctypes.c_int64, P, P, P, P, ctypes.c_int]
    fn.restype = None
    fn(pose.ctypes.data, n, prm.ctypes.data, angles.ctypes.data, fk.ctypes.data, nfev.ctypes.data, gn_mask)
    return angles, fk, nfev


def run_block_f32(pose, prm, gn_mask=0xFF, warm=None):
    """The frame-parallel block schedule (csrc/seqik_block.cuh; leg_solve_block_kernel) emulated lane by lane on the host
    build: pose (N,5,3), prm (32,) -> angles (N,7), fk (N,9,3), nfev (N,4), stats (blocks, passes, serial frames, of which
    first frames, of which not admitted).  Must equal run_carried_f32 bit for bit."""
    lib = load()
    pose = np.ascontiguousarray(pose, dtype=np.float32)
    prm = np.ascontiguousarray(prm, dtype=np.float32)
    n = pose.shape[0]
    angles = np.zeros((n, 7), dtype=np.float32)
    fk = np.zeros((n, 9, 3), dtype=np.float32)
    nfev = np.zeros((n, 4), dtype=np.int32)
    stats = np.zeros(5, dtype=np.int64)
    w = None if warm is None else np.ascontiguousarray(warm, dtype=np.float32)
    P = ctypes.c_void_p
    fn = lib.hostsim_block_f32
    fn.argtypes = [P, ctypes.c_int64, P, P, P, P, P, ctypes.c_int, P]
    fn.restype = None
    fn(pose.ctypes.data, n, prm.ctypes.data, None if w is None else w.ctypes.data, angles.ctypes.data, fk.ctypes.data,
       nfev.ctypes.data, gn_mask, stats.ctypes.data)
    return angles, fk, nfev, stats


def solve_generic(pose2, prm, teacher=None, dtype=np.float32, want_fk=True):
    """Generic 7-DOF chain on the host build: pose2 (N,2,3) = ThC origin + claw, prm (32,) generic constants row,
    teacher (N,7) optional per-frame seeds -> angles (N,7) in generic chain order, fk (N,9,3), nfev (N,), status (N,)."""
    lib = load()
    fn = lib.hostsim_generic_f32 if dtype == np.float32 else lib.hostsim_generic_f64
    pose2 = np.ascontiguousarray(pose2, dtype=dtype)
    n = pose2.shape[0]
    prm = np.ascontiguousarray(prm, dtype=dtype)
    teacher = None if teacher is None else np.ascontiguousarray(teacher, dtype=dtype)
    angles = np.zeros((n, 7), dtype=dtype)
    fk = np.zeros((n, 9, 3), dtype=dtype)
    nfev = np.zeros(n, dtype=np.int32)
    status = np.zeros(n, dtype=np.int32)
    P = ctypes.c_void_p
    fn.argtypes = [P, ctypes.c_int64, P, P, P, P, P, P]
    fn.restype = None
    fn(pose2.ctypes.data, n, prm.ctypes.data, None if teacher is None else teacher.ctypes.data, angles.ctypes.data,
       fk.ctypes.data if want_fk else None, nfev.ctypes.data, status.ctypes.data)
    return angles, fk, nfev, status


def solve_generic_many(prm, target, dtype=np.float64):
    """n independent generic solves on the host build: prm (n,32) constants rows (seed in 18..24, null_sq in 25), target
    (n,3) claw minus origin as the kernel forms it -> angles (n,7), fk rows relative to the origin (n,9,3), nfev (n,),
    status (n,)."""
    lib = load()
    fn = lib.hostsim_generic_solves_f32 if dtype == np.float32 else lib.hostsim_generic_solves_f64
    prm = np.ascontiguousarray(prm, dtype=dtype).reshape(-1, 32)
    target = np.ascontiguousarray(target, dtype=dtype).reshape(-1, 3)
    n = prm.shape[0]
    assert target.shape[0] == n
    angles = np.zeros((n, 7), dtype=dtype)
    fk = np.zeros((n, 9, 3), dtype=dtype)
    nfev = np.zeros(n, dtype=np.int32)
    status = np.zeros(n, dtype=np.int32)
    P = ctypes.c_void_p
    fn.argtypes = [ctypes.c_int64, P, P, P, P, P, P]
    fn.restype = None
    fn(n, prm.ctypes.data, target.ctypes.data, angles.ctypes.data, fk.ctypes.data, nfev.ctypes.data, status.ctypes.data)
    return angles, fk, nfev, status
