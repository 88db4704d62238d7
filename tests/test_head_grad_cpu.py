"""CPU side of the differentiable head angles: the float64 torch model against the reference-form numpy model, its
autograd against finite differences, and the argument checks of seqik_head_angles_backward_f32 (they run before any CUDA
call)."""
import numpy as np
import torch

import model_head
import model_head_torch
from seqikpy_b200 import synthetic as S


def wrap(a):
    return (a + np.pi) % (2 * np.pi) - np.pi


def close_to_reference_form(got, ref, rest):
    """|got - ref| (mod 2 pi) <= 1e-12 + 1e-15 / |sin theta|: the reference form's arccos has derivative 1 / sin theta, so
    the few float64 roundings of its cosine turn into that much angle near 0 and pi (1.7e-6 rad: 7e-11)."""
    raw = ref - np.array([0.0, rest[0], 0.0, 0.0, -rest[1], 0.0, -rest[1]])[:, None]
    err = np.abs(wrap(got - ref))
    return (err <= 1e-12 + 1e-15 / np.abs(np.sin(raw))).all(), err.max()


def model_t(r, l, neck, rest):
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64))
    return model_head_torch.head_angles_torch(t(r), t(l), t(neck), float(rest[0]), float(rest[1])).numpy()


def synthetic_trials(n_trial, n_frame):
    out = []
    for tr in range(n_trial):
        r, l, _, neck = S.make_head_trial(tr, n_frame)
        out.append((r, l, neck))
    return out


def test_torch_model_equals_reference_form_on_grooming_golden(grooming_head):
    d = grooming_head
    neck = d["neck"].reshape(3)
    ref = model_head.head_angles(d["r_head"], d["l_head"], neck, d["rest"][0], d["rest"][1])
    got = model_t(d["r_head"], d["l_head"], neck, d["rest"])
    ok, worst = close_to_reference_form(got, ref, d["rest"])
    assert ok, worst
    assert np.abs(got - d["ref_angles"]).max() <= 1e-9        # and the reference's own angles


def test_torch_model_equals_reference_form_on_synthetic_trials():
    rng = np.random.default_rng(3)
    for r, l, neck in synthetic_trials(4, 500):
        rest = rng.uniform(-0.3, 0.3, 2)
        for nk in (neck, neck + rng.normal(0, 0.01, (500, 3))):            # one neck, a neck per frame
            ref = model_head.head_angles(r, l, nk, rest[0], rest[1])
            got = model_t(r, l, nk, rest)
            ok, worst = close_to_reference_form(got, ref, rest)
            assert ok, worst


def test_torch_model_autograd_equals_finite_differences():
    """Central differences of the numpy reference-form model (step 1e-6 mm on points ~0.1-1 mm apart) against the torch
    model's autograd, for a random weighting of the seven angles, per point and coordinate."""
    rng = np.random.default_rng(4)
    (r, l, neck), = synthetic_trials(1, 64)
    neck = neck + rng.normal(0, 0.01, (64, 3))
    rest = (0.2, -0.1)
    w = rng.normal(size=(7, 64))
    x = np.concatenate([r.reshape(64, 6), l.reshape(64, 6), neck], 1)        # (frame, 15)

    def loss_np(x):
        ang = model_head.head_angles(x[:, :6].reshape(-1, 2, 3), x[:, 6:12].reshape(-1, 2, 3), x[:, 12:], *rest)
        return (ang * w).sum(axis=0)                                             # per frame: frames are independent

    xt = torch.from_numpy(x.copy()).requires_grad_()
    ang = model_head_torch.head_angles_torch(xt[:, :6].reshape(-1, 2, 3), xt[:, 6:12].reshape(-1, 2, 3), xt[:, 12:], *rest)
    (ang * torch.from_numpy(w)).sum().backward()
    grad = xt.grad.numpy()
    h = 1e-6
    fd = np.empty_like(x)
    for k in range(15):
        e = np.zeros_like(x)
        e[:, k] = h
        fd[:, k] = (loss_np(x + e) - loss_np(x - e)) / (2 * h)
    rel = np.abs(grad - fd).max(axis=1) / np.abs(grad).max(axis=1)
    assert rel.max() <= 1e-7, rel.max()


def test_torch_model_degenerate_vectors_give_zero_terms():
    """A zero projected vector contributes torch.atan2's zero gradient: hor along x (roll undefined), tip = base."""
    r = torch.tensor([[[0.0, 0.0, 0.0], [0.1, -0.3, 0.2]]], dtype=torch.float64, requires_grad=True)
    l = torch.tensor([[[0.4, 0.0, 0.0], [0.4, 0.0, 0.0]]], dtype=torch.float64, requires_grad=True)
    neck = torch.tensor([[-0.5, 0.0, -0.3]], dtype=torch.float64, requires_grad=True)
    ang = model_head_torch.head_angles_torch(r, l, neck, 0.0, 0.0)
    gr, gl, gn = torch.autograd.grad(ang.sum(), [r, l, neck])
    assert all(torch.isfinite(g).all() for g in (gr, gl, gn))
    assert (gl[0, 1] == 0).all()                          # the left tip enters only through the zero antenna vector


def test_backward_argument_validation_without_gpu():
    from seqikpy_b200 import _native as N
    lib = N.load_library()
    f = lib.seqik_head_angles_backward_f32
    #      r  l  neck stride aff_r aff_l grad_out g_r g_l g_neck n_trial n_frame stream
    assert f(8, 8, 8, 3, 0, 0, 8, 8, 8, 0, -1, 10, 0) == -1                      # negative size
    assert b"negative" in lib.seqik_last_error()
    assert f(8, 8, 8, 3, 0, 0, 8, 8, 8, 0, 4, -1, 0) == -1
    assert f(0, 0, 0, 3, 0, 0, 0, 0, 0, 0, 0, 10, 0) == 0                        # empty batch: ok, nothing read
    assert f(0, 0, 0, 3, 0, 0, 0, 0, 0, 0, 4, 0, 0) == 0
    for k in (0, 1, 2, 6, 7, 8):                                                 # each required pointer NULL
        args = [8, 8, 8, 3, 0, 0, 8, 8, 8, 0, 4, 10, 0]
        args[k] = 0
        assert f(*args) == -1, k
        assert b"NULL" in lib.seqik_last_error()
    for stride in (1, 6, -3):                                                    # neck stride neither 0 nor 3
        assert f(8, 8, 8, stride, 0, 0, 8, 8, 8, 8, 4, 10, 0) == -1
        assert b"neck_stride" in lib.seqik_last_error()
    assert f(8, 8, 8, 0, 8, 0, 8, 8, 8, 8, 4, 10, 0) == -1                       # one affine row pointer only
    assert b"both" in lib.seqik_last_error()
    assert f(8, 8, 8, 0, 0, 8, 8, 8, 8, 8, 4, 10, 0) == -1
