"""CPU tests of the streaming-kernel references and of the host half of the joints-only FK wire format.

* ``model_head`` (the float64 restatement of the head angles that tests/test_gpu_stream.py compares the kernel with) against
  the reference's own output on the grooming trial.
* ``seqik_fk_expand_host_f32`` (host code in the library: no GPU needed) on numpy buffers: unaligned outputs, frame ranges
  that do not start on a multiple of four (the SSE path streams four frames at a time), padded strides, more threads than
  chains.  Bitwise against numpy; nothing outside the frame range or inside the padding is written.
"""
import ctypes

import numpy as np
import pytest

import model_head


def test_model_head_equals_reference_output(grooming_head):
    """The model reproduces the reference's head_joint_angles of the grooming trial (6000 frames, template neck) to
    1e-15 rad (measured: 6.7e-16): it is a faithful float64 statement of what the kernel has to compute."""
    g = grooming_head
    out = model_head.head_angles(g["r_head"], g["l_head"], g["neck"].reshape(3), g["rest"][0], g["rest"][1])
    assert out.shape == g["ref_angles"].shape == (7, 6000)
    assert np.abs(out - g["ref_angles"]).max() < 1e-15


def test_model_head_sign_convention():
    """angle_between_segments: det = 0 counts as negative, so antiparallel vectors give -pi (the reference's arccos * -1)."""
    v1 = np.array([[0.0, 1.0, 0.0], [0.0, 1.0, 0.0], [0.0, 1.0, 0.0]])
    v2 = np.array([[0.0, -2.0, 0.0], [0.0, 0.0, 3.0], [0.0, 0.0, -3.0]])
    got = model_head.angle_between_segments(v1, v2, 0)
    assert got[0] == -np.pi and np.isclose(got[1], np.pi / 2) and np.isclose(got[2], -np.pi / 2)


def _p(a, offset=0):
    return ctypes.c_void_p(a.ctypes.data + 4 * offset)


def _expand_case(lib, rng, n_chain, n_frame, t0, t1, out_off, f_fs, j_fs, p_fs, n_threads):
    pad = int(rng.integers(0, 5))
    j_cs, p_cs, f_cs = n_frame * j_fs + pad, n_frame * p_fs + pad, n_frame * f_fs + pad
    joints = rng.normal(size=n_chain * j_cs).astype(np.float32)
    pose = rng.normal(size=n_chain * p_cs).astype(np.float32)
    sentinel = np.float32(-7777.25)
    fk = np.full(out_off + n_chain * f_cs + 8, sentinel, dtype=np.float32)
    exp = fk.copy()
    for c in range(n_chain):
        for t in range(t0, t1):
            o = out_off + c * f_cs + t * f_fs
            j = joints[c * j_cs + t * j_fs: c * j_cs + t * j_fs + 12]
            p = pose[c * p_cs + t * p_fs: c * p_cs + t * p_fs + 3]
            exp[o: o + 12] = np.tile(p, 4)                    # rows 0-3: origin
            exp[o + 12: o + 15] = j[:3]                       # row 4 = row 5: first joint
            exp[o + 15: o + 27] = j                           # rows 5-8
    rc = lib.seqik_fk_expand_host_f32(_p(joints), j_cs, j_fs, _p(pose), p_cs, p_fs, _p(fk, out_off), f_cs, f_fs,
                                      n_chain, t0, t1, n_threads)
    assert rc == 0
    assert np.array_equal(fk.view(np.uint32), exp.view(np.uint32)), (n_chain, n_frame, t0, t1, out_off, f_fs, n_threads)


def test_fk_expand_host_bitwise_and_bounded():
    from seqikpy_b200 import _native as N
    lib = N.load_library()
    rng = np.random.default_rng(23)
    n_cases = 0
    for f_fs in (27, 30):
        for out_off in (0, 1, 2, 3):
            for t0 in (0, 1, 2, 3, 5, 8):
                for length in (0, 1, 3, 4, 5, 9, 17):
                    n_chain = int(rng.integers(1, 5))
                    n_frame = t0 + length + int(rng.integers(0, 3))
                    n_threads = int(rng.choice([1, 2, n_chain + 3]))   # more threads than chains: capped
                    _expand_case(lib, rng, n_chain, n_frame, t0, t0 + length, out_off, f_fs,
                                 int(rng.choice([12, 13])), int(rng.choice([3, 15])), n_threads)
                    n_cases += 1
    assert n_cases == 2 * 4 * 6 * 7


def test_fk_expand_host_argument_checks():
    from seqikpy_b200 import _native as N
    lib = N.load_library()
    buf = np.zeros(64, dtype=np.float32)
    assert lib.seqik_fk_expand_host_f32(_p(buf), 12, 12, _p(buf), 3, 3, _p(buf), 27, 27, 1, 2, 1, 1) == -1    # t1 < t0
    assert lib.seqik_fk_expand_host_f32(_p(buf), 12, 12, _p(buf), 3, 3, _p(buf), 26, 26, 1, 0, 1, 1) == -1    # stride < 27
    assert lib.seqik_fk_expand_host_f32(_p(buf), 12, 12, _p(buf), 3, 3, None, 27, 27, 1, 0, 1, 1) == -1       # NULL
    assert lib.seqik_fk_expand_host_f32(None, 12, 12, None, 3, 3, None, 27, 27, 1, 3, 3, 1) == 0              # empty range
    with pytest.raises(ValueError):
        N.check(-1, "seqik_fk_expand_host_f32")
