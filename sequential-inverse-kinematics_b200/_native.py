"""ctypes binding of ``libseqik_sm100.so`` (C ABI: include/seqik.h).

There is NO fallback: if the library is missing or no CUDA device is present every entry
point raises.  Device memory and streams come from torch (plumbing only).
"""
import ctypes
import os
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "csrc" / "libseqik_sm100.so"

ABI_VERSION = 13
CHAIN_PARAM_FLOATS = 32
FLAG_ESCAPE = 1 << 4
FLAG_SKIP_CONFIRM = 1 << 5
FLAG_NEWTON = 1 << 6
FLAG_REFERENCE_ITERATES = 0x3F          # SEQIK_FLAG_REFERENCE_ITERATES: Gauss-Newton mode in all four stages + escape + skip-confirm
FLAG_CLOSED_FORM = 1 << 7
FLAG_DEFAULT = 0xFF                     # SEQIK_FLAG_DEFAULT: the above + Newton steps + closed-form warm step
FLAG_FK_JOINTS = 1 << 20
FLAG_SCHED_SHIFT = 8
SCHED_AUTO, SCHED_LANE_PER_CHAIN, SCHED_STAGE_PIPELINE, SCHED_FRAME_BLOCKS = 0, 1, 2, 3

_lib = None

_vp, _i64, _u32, _f32, _int = ctypes.c_void_p, ctypes.c_int64, ctypes.c_uint32, ctypes.c_float, ctypes.c_int

# name -> (restype, argtypes): one entry per prototype of include/seqik.h
_SIGNATURES = {
    "seqik_abi_version": (_int, []),
    "seqik_last_error": (ctypes.c_char_p, []),
    "seqik_leg_solve_f32": (_int, [_vp, _i64, _i64, _vp, _vp, _vp, _i64, _i64, _vp, _i64, _i64, _vp, _i64, _vp, _vp,
                                   _i64, _i64, _u32, _u32, _vp]),
    "seqik_leg_solve_generic_f32": (_int, [_vp, _i64, _i64, ctypes.c_int32, _vp, _vp, _i64, _i64, _vp, _i64, _i64, _vp, _i64,
                                           _vp, _vp, _i64, _i64, _u32, _vp]),
    "seqik_leg_solve_generic_f64": (_int, [_vp, _i64, _i64, ctypes.c_int32, _vp, _vp, _i64, _i64, _vp, _i64, _i64, _vp, _i64,
                                           _vp, _vp, _i64, _i64, _u32, _vp]),
    "seqik_pchip_resample_f32": (_int, [_vp, _vp, _i64, _i64, _i64, _i64, ctypes.c_double, ctypes.c_double, _vp]),
    "seqik_pchip_resample_f64": (_int, [_vp, _vp, _i64, _i64, _i64, _i64, ctypes.c_double, ctypes.c_double, _vp]),
    "seqik_pchip_resample_backward_f32": (_int, [_vp, _vp, _vp, _i64, _i64, _i64, _i64, ctypes.c_double, ctypes.c_double, _vp]),
    "seqik_pchip_resample_backward_f64": (_int, [_vp, _vp, _vp, _i64, _i64, _i64, _i64, ctypes.c_double, ctypes.c_double, _vp]),
    "seqik_memcpy2d_async": (_int, [_vp, _i64, _vp, _i64, _i64, _i64, _int, _vp]),
    "seqik_fk_expand_host_f32": (_int, [_vp, _i64, _i64, _vp, _i64, _i64, _vp, _i64, _i64, _i64, _i64, _i64, _int]),
    "seqik_fk_f32": (_int, [_vp, _vp, _i64, _vp, _vp, _i64, _i64, _vp]),
    "seqik_fk_backward_f32": (_int, [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "seqik_head_angles_f32": (_int, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "seqik_head_angles_backward_f32": (_int, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "seqik_mid_quantile_f32": (_int, [_vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "seqik_leg_series_f32": (_int, [_vp, _i64, _i64, _vp, _i64, _i64, _vp]),
    "seqik_leg_affine_f32": (_int, [_vp, _vp, _int, _vp, _i64, _vp]),
    "seqik_origin_rows_f32": (_int, [_vp, _i64, _i64, _vp, _i64, _i64, _i64, _i64, _vp]),
    "seqik_leg_affine_from_pose_f32": (_int, [_vp, _i64, _i64, _vp, _int, _vp, _vp, _i64, _i64, _vp]),
    "seqik_align_apply_f32": (_int, [_vp, _i64, _i64, _vp, _vp, _i64, _i64, _vp]),
    "seqik_align_apply_backward_f32": (_int, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "seqik_leg_affine_backward_f32": (_int, [_vp, _i64, _i64, _vp, _int, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "seqik_head_series_f32": (_int, [_vp, _vp, _i64, _f32, _vp, _vp, _i64, _i64, _vp]),
    "seqik_head_series_f64": (_int, [_vp, _vp, _i64, ctypes.c_double, _vp, _vp, _i64, _i64, _vp]),
    "seqik_head_affine_f32": (_int, [_vp, _vp, _vp, _i64, _vp]),
    "seqik_head_apply_f32": (_int, [_vp, _vp, _vp, _i64, _i64, _vp]),
    "seqik_head_apply_backward_f32": (_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "seqik_head_affine_backward_f32": (_int, [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "seqik_head_affine_backward_f64": (_int, [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)


class SeqIKNativeError(RuntimeError):
    """The CUDA library is missing, stale, or a call failed."""


def load_library():
    """Load (once) and return the ctypes handle; raises SeqIKNativeError if it cannot."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise SeqIKNativeError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no CPU fallback.")
    lib = ctypes.CDLL(os.fspath(LIB_PATH))
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)        # AttributeError -> stale library
        fn.restype, fn.argtypes = res, args
    if lib.seqik_abi_version() != ABI_VERSION:
        raise SeqIKNativeError(f"ABI mismatch: library {lib.seqik_abi_version()} != binding {ABI_VERSION}; rebuild")
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load_library().seqik_last_error().decode(errors="replace")
        if rc == -1:
            raise ValueError(f"{what}: {msg}")
        raise SeqIKNativeError(f"{what} failed ({rc}): {msg}")


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise SeqIKNativeError("a CUDA device (B200, sm_100a) is required; there is no CPU fallback")
    return torch


def ptr(t):
    return 0 if t is None else t.data_ptr()


def stream_ptr(torch, device):
    return torch.cuda.current_stream(device).cuda_stream
