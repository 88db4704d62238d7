"""CPU side of the differentiable FK: the float64 gradient model against the reference's closed-form FK, and the argument
checks of seqik_fk_backward_f32 (they run before any CUDA call)."""
import numpy as np
import torch

import model_fk
from oracle import seqik_oracle as O


def test_model_equals_the_closed_form_fk():
    rng = np.random.default_rng(7)
    n = 500
    ang = rng.uniform(-2 * np.pi, 2 * np.pi, (n, 7))
    org = rng.uniform(-2.0, 2.0, (n, 3))
    for _ in range(3):
        seg = rng.uniform(0.1, 1.0, 4)
        ref = O.fk_closed_form(ang, seg, org)
        got = model_fk.fk(torch.from_numpy(ang), torch.from_numpy(org), torch.from_numpy(seg)).numpy()
        assert np.abs(got - ref).max() <= 1e-12


def test_model_broadcasts_a_per_chain_origin_and_lengths():
    rng = np.random.default_rng(8)
    ang = torch.from_numpy(rng.uniform(-3, 3, (4, 6, 7)))
    org, seg = torch.from_numpy(rng.normal(size=(4, 1, 3))), torch.from_numpy(rng.uniform(0.1, 1, (4, 1, 4)))
    got = model_fk.fk(ang, org, seg)
    assert got.shape == (4, 6, 9, 3)
    for c in range(4):
        ref = O.fk_closed_form(ang[c].numpy(), seg[c, 0].numpy(), org[c].numpy())
        assert np.abs(got[c].numpy() - ref).max() <= 1e-12


def test_backward_argument_validation_without_gpu():
    from seqikpy_b200 import _native as N
    lib = N.load_library()
    f = lib.seqik_fk_backward_f32
    #      angles origin stride params grad_fk g_ang g_org g_len n_chain n_frame stream
    assert f(8, 8, 3, 8, 8, 8, 0, 0, -1, 10, 0) == -1                             # negative size
    assert b"negative" in lib.seqik_last_error()
    assert f(8, 8, 3, 8, 8, 8, 0, 0, 4, -1, 0) == -1
    assert f(0, 0, 3, 0, 0, 0, 0, 0, 0, 10, 0) == 0                               # empty batch: ok, nothing read
    assert f(0, 0, 3, 0, 0, 0, 0, 0, 4, 0, 0) == 0
    for k in range(5):                                                            # each required pointer NULL
        args = [8, 8, 3, 8, 8, 8, 0, 0, 4, 10, 0]
        args[(0, 1, 3, 4, 5)[k]] = 0
        assert f(*args) == -1, k
        assert b"NULL" in lib.seqik_last_error()
    assert f(8, 8, 1, 8, 8, 8, 8, 8, 4, 10, 0) == -1                              # origin stride neither 0 nor 3
    assert b"origin_frame_stride" in lib.seqik_last_error()
    assert f(8, 8, 6, 8, 8, 8, 0, 0, 4, 10, 0) == -1
