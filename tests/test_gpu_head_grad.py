"""Differentiable head angles: seqik_head_angles_backward_f32 on both load paths, its affine contract, against the float64
model's autograd (tests/model_head_torch.py), on degenerate frames, through torch.autograd, and in a fit of
per-frame head rotations to measured angles.

Shapes and inputs are those of tests/test_gpu_stream.py (HEAD_SHAPES: trial boundaries inside and across blocks, one case
of 2.4 million frames; the synthetic head motion of ``realistic_heads``; the grooming golden).

Bound against the float64 model, per frame, with u the float32 unit roundoff, G = sum over the seven angles of |g_k|
(g = dL/dangles), P the largest input coordinate of the frame and V the shortest projected plane vector that enters its
angles (hor|x=0, mid|y=0, hor|z=0, and per antenna a|x=0, ad|y=0 and gd|y=0):  64 u G P / V^2.
Every gradient term is g_k (e x v) / |v|^2, of size |g_k| / |v| <= |g_k| P / V^2 up to a constant (|v| <= 2 sqrt(3) P).  The
coordinates of v are float32 differences of coordinates up to P, off by a few u P, which moves (e x v) / |v|^2 by a few
u P / |v|^2; the roll carries a few u of absolute error (atan2_pos, sincosv_) that turns the de-rotated vectors and so the
terms by that, a few u / V <= a few u 2 sqrt(3) P / V^2; products and sums add roundings of the same size.  A float32
transcription of the kernel's arithmetic reaches 0.6 of 1 u G P / V^2 on the synthetic motion, which leaves 64 a wide
margin.  Frames with V < 1e-3 P are reported and only checked for finiteness.
"""
import itertools

import numpy as np
import pytest
import torch

import model_head_torch
from test_gpu_stream import HEAD_SHAPES, U, dev, offset_view, realistic_heads, head_point_f32, head_apply_ref

pytestmark = pytest.mark.gpu

C_BOUND = 64


@pytest.fixture(scope="module")
def eng():
    assert torch.cuda.is_available(), "these tests need the B200"
    from seqikpy_b200 import _native as N, engine
    N.load_library()
    return engine, N


def bits(t):
    return t.contiguous().view(torch.int32)


def head_inputs(rng, n_trial, n_frame, neck_per_frame=True):
    r, l, neck = realistic_heads(n_trial, n_frame)
    if neck_per_frame:
        neck = neck[:, None] + rng.normal(0, 0.01, (n_trial, n_frame, 3)).astype(np.float32)
    g = rng.normal(size=(n_trial, 7, n_frame)).astype(np.float32)
    return r, l, neck, g


def head_affine_rows(rng, n_trial):
    rows = []
    for _ in range(2):
        a = np.zeros((n_trial, 8), np.float32)
        a[:, 0:3] = rng.normal(0, 0.1, (n_trial, 3))
        a[:, 3], a[:, 7] = rng.uniform(0.9, 1.1, n_trial), rng.uniform(2.5, 4.0, n_trial)     # scale_tip far from scale_base
        a[:, 4:7] = rng.normal(0, 0.1, (n_trial, 3))
        rows.append(a)
    return rows


def call_abi(N, r, l, neck, stride, ar, al, g, gr, gl, gn, n_trial, n_frame):
    lib = N.load_library()
    N.check(lib.seqik_head_angles_backward_f32(r.data_ptr(), l.data_ptr(), neck.data_ptr(), stride, N.ptr(ar), N.ptr(al),
                                               g.data_ptr(), gr.data_ptr(), gl.data_ptr(), N.ptr(gn), n_trial, n_frame,
                                               torch.cuda.current_stream().cuda_stream), "seqik_head_angles_backward_f32")


def shortest_plane_vector(r, l, neck):
    """V per frame (float64): the shortest projected plane vector entering the seven angles, the roll from the model."""
    r, l, neck = (np.asarray(a, np.float64) for a in (r, l, neck))
    h = l[..., 0, :] - r[..., 0, :]
    m = 0.5 * (r[..., 0, :] + l[..., 0, :]) - neck
    roll = np.arctan2(h[..., 2], h[..., 1])
    c, s = np.cos(roll), np.sin(roll)
    vs = [np.hypot(h[..., 1], h[..., 2]), np.hypot(m[..., 0], m[..., 2]), np.hypot(h[..., 0], h[..., 1])]
    for side in (r, l):
        a = side[..., 1, :] - side[..., 0, :]
        gd = neck - side[..., 0, :]
        vs += [np.hypot(a[..., 1], a[..., 2]), np.hypot(a[..., 0], -a[..., 1] * s + a[..., 2] * c),
               np.hypot(gd[..., 0], -gd[..., 1] * s + gd[..., 2] * c)]
    return np.stack(vs)


def model_grads(r, l, neck, g, device="cuda"):
    """The float64 model's autograd at the given (float32) points: (grad_r, grad_l, grad_neck per frame), numpy float64."""
    n_trial, n_frame = r.shape[:2]
    neck = np.broadcast_to(np.asarray(neck).reshape(n_trial, -1, 3), (n_trial, n_frame, 3))
    t = lambda a: torch.tensor(np.asarray(a, np.float64), device=device, requires_grad=True)
    tr, tl, tn = t(r), t(l), t(neck)
    ang = model_head_torch.head_angles_torch(tr, tl, tn, 0.0, 0.0)                 # (7, n_trial, n_frame)
    (ang * torch.tensor(np.asarray(g, np.float64), device=device).permute(1, 0, 2)).sum().backward()
    return tr.grad.cpu().numpy(), tl.grad.cpu().numpy(), tn.grad.cpu().numpy()


def check_vs_model(got, r, l, neck, g, scales=None, label=""):
    """got = (grad_r, grad_l, grad_neck per frame) of the kernel at the aligned float32 points r, l; scales = the affine
    scales (sr_base, sr_tip, sl_base, sl_tip), each (n_trial,), or None.  Returns the worst ratio to the bound."""
    n_trial, n_frame = r.shape[:2]
    neck_f = np.broadcast_to(np.asarray(neck, np.float64).reshape(n_trial, -1, 3), (n_trial, n_frame, 3))
    ref = list(model_grads(r, l, neck_f, g))
    smax = np.ones(n_trial)
    if scales is not None:
        sc = np.stack([np.asarray(s, np.float64) for s in scales], 1)         # (n_trial, 4)
        ref[0] = ref[0] * sc[:, None, 0:2, None]
        ref[1] = ref[1] * sc[:, None, 2:4, None]
        smax = sc.max(1)
    pts = np.concatenate([r.reshape(n_trial, n_frame, 6), l.reshape(n_trial, n_frame, 6), neck_f], -1)
    P = np.abs(pts).max(-1)
    V = shortest_plane_vector(r, l, neck_f).min(0)
    G = np.abs(np.asarray(g, np.float64)).sum(1)
    bound = C_BOUND * U * G * P / V ** 2 * np.maximum(smax, 1.0)[:, None]
    ok = V >= 1e-3 * P
    err = np.zeros((n_trial, n_frame))
    for a, b in zip(got, ref):
        a = np.asarray(a, np.float64)
        assert np.isfinite(a).all(), label
        err = np.maximum(err, np.abs(a - b).reshape(n_trial, n_frame, -1).max(-1))
    ratio = np.where(ok, err / bound, 0.0)
    if (~ok).any():
        print(f"{label}: {(~ok).sum()} frames with V < 1e-3 P checked for finiteness only")
    worst = float(ratio.max())
    assert worst <= 1.0, (label, worst, np.unravel_index(np.argmax(ratio), ratio.shape))
    return worst


@pytest.mark.parametrize("n_trial,n_frame", HEAD_SHAPES)
def test_head_backward_paths_bitwise_and_vs_float64(eng, n_trial, n_frame):
    E, N = eng
    rng = np.random.default_rng(7000 + n_frame)
    r, l, neck, g = head_inputs(rng, n_trial, n_frame)
    d_r, d_l, d_n, d_g = (dev(torch, a) for a in (r, l, neck, g))
    ref = E.head_angles_backward(d_r, d_l, d_n, d_g)                           # 64-bit loads and stores
    ref_bits = [bits(t) for t in ref]

    def same(out, which=(0, 1, 2)):
        return all(torch.equal(bits(out[i]), ref_bits[i]) for i in which)

    assert same(E.head_angles_backward(d_r, d_l, d_n, d_g))                    # repeatable
    for k in (1, 3):                                                           # odd float offsets: the 32-bit instantiation
        assert same(E.head_angles_backward(offset_view(torch, d_r, k), d_l, d_n, d_g)), ("r_head", k)
        assert same(E.head_angles_backward(d_r, offset_view(torch, d_l, k), d_n, d_g)), ("l_head", k)
        assert same(E.head_angles_backward(d_r, d_l, d_n, offset_view(torch, d_g, k))), ("grad_out", k)
        # an output record at an odd float offset (through the C ABI: the engine allocates aligned outputs)
        out = [torch.empty_like(t) for t in ref]
        out[0] = offset_view(torch, out[0], k)
        call_abi(N, d_r, d_l, d_n, 3, None, None, d_g, *out, n_trial, n_frame)
        assert same(out), ("grad_r_head", k)
    gr, gl, gn = E.head_angles_backward(d_r, d_l, d_n, d_g, want_neck=False)  # NULL grad_neck changes nothing else
    assert gn is None and same((gr, gl, None), (0, 1))
    # one neck per trial (stride 0) equal to the same neck repeated per frame: the same bits
    n0 = np.ascontiguousarray(neck[:, 0])
    per_trial = E.head_angles_backward(d_r, d_l, dev(torch, n0), d_g)
    per_frame = E.head_angles_backward(d_r, d_l, dev(torch, np.repeat(n0[:, None], n_frame, 1)), d_g)
    assert all(torch.equal(bits(a), bits(b)) for a, b in zip(per_trial, per_frame))

    worst = check_vs_model([t.cpu().numpy() for t in ref], r, l, neck, g, label=f"{n_trial}x{n_frame}")
    print(f"{n_trial}x{n_frame}: worst ratio to the bound {worst:.4f}")


@pytest.mark.parametrize("n_trial,n_frame", [(9, 257), (500, 7)])
def test_affine_contract_bitwise(eng, n_trial, n_frame):
    """backward(raw, affine) = float32(scale x backward(head_apply(raw, affine))): the aligned points' gradient times the
    row's scale (aff[3] for a base, aff[7] for a tip), one float32 multiplication; the neck is not aligned."""
    E, _ = eng
    rng = np.random.default_rng(7100 + n_frame)
    r, l, neck, g = head_inputs(rng, n_trial, n_frame)
    ar, al = head_affine_rows(rng, n_trial)
    d_r, d_l, d_n, d_g, d_ar, d_al = (dev(torch, a) for a in (r, l, neck, g, ar, al))
    got = E.head_angles_backward(d_r, d_l, d_n, d_g, d_ar, d_al)
    aligned_r, aligned_l = E.head_apply(d_r, d_ar), E.head_apply(d_l, d_al)
    assert np.array_equal(aligned_r.cpu().numpy(), head_apply_ref(r, ar))       # head_apply rounds like head_point
    plain = [t.cpu().numpy() for t in E.head_angles_backward(aligned_r, aligned_l, d_n, d_g)]
    for k, (p, a) in enumerate(((plain[0], ar), (plain[1], al))):
        want = np.empty_like(p)
        want[:, :, 0] = p[:, :, 0] * a[:, None, 3:4]
        want[:, :, 1] = p[:, :, 1] * a[:, None, 7:8]
        assert np.array_equal(got[k].cpu().numpy().view(np.int32), want.view(np.int32)), k
    assert np.array_equal(got[2].cpu().numpy().view(np.int32), plain[2].view(np.int32))


@pytest.mark.parametrize("neck_per_frame", [False, True])
@pytest.mark.parametrize("with_affine", [False, True])
def test_head_backward_vs_float64_model(eng, neck_per_frame, with_affine):
    """The synthetic motion (3 trials x 1001 frames) and the grooming golden, against the float64 model's autograd at the
    float32 points the kernel sees (the affine rows applied in float32 first), within the bound of the module docstring."""
    E, _ = eng
    rng = np.random.default_rng(7200 + 2 * neck_per_frame + with_affine)
    r, l, neck, g = head_inputs(rng, 3, 1001, neck_per_frame)
    cases = [(r, l, neck, g, "synthetic")]
    gold = np.load(__import__("pathlib").Path(__file__).parent / "golden" / "grooming_head.npz")
    gn = gold["neck"].reshape(1, 3).astype(np.float32)
    gr_, gl_ = gold["r_head"][None].astype(np.float32), gold["l_head"][None].astype(np.float32)
    n_g = gr_.shape[1]
    if neck_per_frame:
        gn = np.ascontiguousarray(gn[:, None] + rng.normal(0, 0.01, (1, n_g, 3)).astype(np.float32))
    cases.append((gr_, gl_, gn, rng.normal(size=(1, 7, n_g)).astype(np.float32), "grooming"))
    for r, l, neck, g, label in cases:
        n_trial = r.shape[0]
        aff = head_affine_rows(rng, n_trial) if with_affine else None
        got = E.head_angles_backward(*(dev(torch, a) for a in (r, l, neck, g)), *(dev(torch, a) for a in (aff or [])))
        scales = None
        if with_affine:
            ar, al = aff
            r = np.stack([head_point_f32(r[:, :, 0], ar, False), head_point_f32(r[:, :, 1], ar, True)], 2)
            l = np.stack([head_point_f32(l[:, :, 0], al, False), head_point_f32(l[:, :, 1], al, True)], 2)
            scales = (ar[:, 3], ar[:, 7], al[:, 3], al[:, 7])
        worst = check_vs_model([t.cpu().numpy() for t in got], r, l, neck, g, scales, label)
        print(f"{label} (neck per frame {neck_per_frame}, affine {with_affine}): worst ratio to the bound {worst:.4f}")


def degenerate_frames():
    """Frames (all coordinates dyadic, so the float32 and float64 differences are exact) with a zero projected vector:
    0 hor along x (roll undefined), 1 right tip = base, 2 left tip = base, 3 mid - neck along y, 4 neck - left base along y
    (with hor|z = 0 so that the roll is exactly 0), 5 all of 1-3 at once."""
    base_r = np.array([[0.0, -0.25, 0.125], [0.125, -0.5, 0.375]])
    base_l = np.array([[0.0, 0.25, 0.125], [0.25, 0.5, 0.5]])
    neck = np.array([-0.5, 0.0, -0.25])
    r, l, n = [], [], []
    for k in range(6):
        rr, ll, nk = base_r.copy(), base_l.copy(), neck.copy()
        if k == 0:
            ll[0] = rr[0] + [0.5, 0.0, 0.0]
        if k in (1, 5):
            rr[1] = rr[0]
        if k in (2, 5):
            ll[1] = ll[0]
        if k in (3, 5):
            nk = 0.5 * (rr[0] + ll[0]) + [0.0, -0.375, 0.0]
        if k == 4:
            nk = ll[0] + [0.0, -0.75, 0.0]
        r.append(rr); l.append(ll); n.append(nk)
    return np.array(r, np.float32)[None], np.array(l, np.float32)[None], np.array(n, np.float32)[None]


def test_degenerate_frames(eng):
    """Zero projected vectors give finite gradients, exactly 0 where the model's (torch.atan2's convention at (0, 0)) is
    exactly 0, and within the bound elsewhere, V taken over the non-zero vectors."""
    E, _ = eng
    r, l, neck = degenerate_frames()
    g = np.random.default_rng(73).normal(size=(1, 7, r.shape[1])).astype(np.float32)
    got = [t.cpu().numpy() for t in E.head_angles_backward(*(dev(torch, a) for a in (r, l, neck, g)))]
    ref = model_grads(r, l, neck, g)
    vs = shortest_plane_vector(r, l, neck)
    assert (vs == 0).any(axis=0).all()                                          # every frame has a zero vector
    V = np.where(vs > 0, vs, np.inf).min(0)
    P = np.abs(np.concatenate([r.reshape(1, -1, 6), l.reshape(1, -1, 6), neck], -1)).max(-1)
    bound = C_BOUND * U * np.abs(g).sum(1) * P / V ** 2
    for a, b in zip(got, ref):
        assert np.isfinite(a).all()
        assert (a[b == 0] == 0).all()
        assert (np.abs(a - b).reshape(1, r.shape[1], -1).max(-1) <= bound).all(), np.abs(a - b).max()
    assert (got[0][0, 1, 1] == 0).all() and (got[1][0, 2, 1] == 0).all()      # the tips that equal their base


@pytest.mark.parametrize("per_frame_neck", [True, False])
@pytest.mark.parametrize("with_affine", [False, True])
def test_autograd_equals_the_direct_backward(eng, per_frame_neck, with_affine):
    """Every subset of {r_head, l_head, neck, rest} that requires grad: torch.autograd.grad through head_angles equals
    head_angles_backward (+ the frame sums of a shared neck, + the rest sums) bit for bit."""
    E, _ = eng
    rng = np.random.default_rng(7300 + per_frame_neck)
    n_trial, n_frame = 5, 257
    r, l, neck, g = head_inputs(rng, n_trial, n_frame, per_frame_neck)
    rest = rng.uniform(-0.3, 0.3, (n_trial, 2)).astype(np.float32)
    d_r, d_l, d_n, d_rest, d_g = (dev(torch, a) for a in (r, l, neck, rest, g))
    aff = [dev(torch, a) for a in head_affine_rows(rng, n_trial)] if with_affine else []
    gr, gl, gn = E.head_angles_backward(d_r, d_l, d_n, d_g, *aff)
    want = {"r_head": gr, "l_head": gl, "neck": gn if per_frame_neck else gn.sum(dim=1),
            "rest": torch.stack([d_g[:, 1].sum(-1), -(d_g[:, 4] + d_g[:, 6]).sum(-1)], dim=1)}
    plain = E.head_angles(d_r, d_l, d_n, d_rest, *aff)
    assert plain.grad_fn is None
    names = ("r_head", "l_head", "neck", "rest")
    for k in range(1, 5):
        for subset in itertools.combinations(names, k):
            x = {n: t.clone().requires_grad_(n in subset) for n, t in zip(names, (d_r, d_l, d_n, d_rest))}
            out = E.head_angles(x["r_head"], x["l_head"], x["neck"], x["rest"], *aff)
            assert torch.equal(bits(out), bits(plain)), subset                 # grad mode does not change the result
            grads = torch.autograd.grad((out * d_g).sum(), [x[n] for n in subset])
            for n, gr_ in zip(subset, grads):
                assert gr_.shape == x[n].shape and torch.equal(bits(gr_), bits(want[n])), (subset, n)
            with torch.no_grad():
                assert E.head_angles(x["r_head"], x["l_head"], x["neck"], x["rest"], *aff).grad_fn is None


def test_autograd_noncontiguous_gradient_affine_rows_and_first_order_only(eng):
    E, _ = eng
    rng = np.random.default_rng(74)
    r, l, neck, _ = head_inputs(rng, 3, 301)
    d_r = dev(torch, r).requires_grad_()
    d_l, d_n = dev(torch, l), dev(torch, neck)
    rest = torch.zeros((3, 2), device="cuda")
    # a non-contiguous incoming gradient (a transposed view's backward) is made contiguous
    w = dev(torch, rng.normal(size=(301, 7, 3)).astype(np.float32))
    out = E.head_angles(d_r, d_l, d_n, rest)
    (gr,) = torch.autograd.grad((out.permute(2, 1, 0) * w).sum(), [d_r])
    g = w.permute(2, 1, 0).contiguous()
    assert torch.equal(bits(gr), bits(E.head_angles_backward(d_r.detach(), d_l, d_n, g, want_neck=False)[0]))
    # affine rows that require grad raise: the rows are constants of the backward
    ar, al = (dev(torch, a) for a in head_affine_rows(rng, 3))
    with pytest.raises(ValueError, match="affine"):
        E.head_angles(d_r, d_l, d_n, rest, ar.requires_grad_(), al)
    with pytest.raises(ValueError, match="affine"):
        E.head_angles(d_r.detach(), d_l, d_n, rest, ar.detach(), al.requires_grad_())
    with torch.no_grad():                                                      # no graph, no gradient asked for
        E.head_angles(d_r, d_l, d_n, rest, ar, al)
    # second derivatives are not supported
    (gr,) = torch.autograd.grad(E.head_angles(d_r, d_l, d_n, rest).pow(2).sum(), [d_r], create_graph=True)
    with pytest.raises(RuntimeError, match="once_differentiable"):
        gr.sum().backward()


def rotated_heads(rot, base0, stalk0, neck):
    """Template antenna points rotated about the neck by Rz(yaw) Ry(pitch) Rx(roll), per frame (torch ops, as
    synthetic.make_head_trial): rot (F, 3) -> r_head, l_head (1, F, 2, 3)."""
    c, s = torch.cos(rot), torch.sin(rot)
    one, zero = torch.ones_like(c[:, 0]), torch.zeros_like(c[:, 0])
    rx = torch.stack([one, zero, zero, zero, c[:, 0], -s[:, 0], zero, s[:, 0], c[:, 0]], 1).view(-1, 3, 3)
    ry = torch.stack([c[:, 1], zero, s[:, 1], zero, one, zero, -s[:, 1], zero, c[:, 1]], 1).view(-1, 3, 3)
    rz = torch.stack([c[:, 2], -s[:, 2], zero, s[:, 2], c[:, 2], zero, zero, zero, one], 1).view(-1, 3, 3)
    R = rz @ ry @ rx
    sides = []
    for k in range(2):
        b = R @ base0[k] + neck
        t = b + R @ stalk0[k]
        sides.append(torch.stack([b, t], 1)[None])
    return sides[0], sides[1]


def test_lbfgs_fit_recovers_head_rotation(eng):
    """200 frames of measured head and antenna angles (from the synthetic motion's rotations); the antenna points are the
    template's rotated about the neck by a per-frame head rotation (3 parameters per frame).  Starting 0.1 rad off the true
    rotation in every parameter, a float32 LBFGS fit of the seven angles through head_angles recovers the rotation to
    1e-4 rad and the seven angles to 1e-5 rad."""
    E, _ = eng
    from seqikpy_b200.data import NMF_TEMPLATE as T
    n_frame = 200
    neck = torch.tensor(T["Neck"], dtype=torch.float32, device="cuda")
    base0 = torch.tensor(np.array([np.subtract(T[f"{s}_Antenna_base"], T["Neck"]) for s in "RL"]), dtype=torch.float32, device="cuda")
    stalk0 = torch.tensor(np.array([np.subtract(T[f"{s}_Antenna_edge"], T[f"{s}_Antenna_base"]) for s in "RL"]),
                          dtype=torch.float32, device="cuda")
    t = np.arange(n_frame)
    rng = np.random.default_rng(75)
    true = np.stack([0.2 * np.sin(2 * np.pi * rng.uniform(0.5, 3) * t / 1000 + rng.uniform(0, 2 * np.pi)) for _ in range(3)], 1)
    true_t = torch.tensor(true, dtype=torch.float32, device="cuda")
    rest = torch.zeros((1, 2), device="cuda")
    with torch.no_grad():
        target = E.head_angles(*rotated_heads(true_t, base0, stalk0, neck), neck[None], rest)
    rot = (true_t + torch.tensor(rng.choice([-0.1, 0.1], true.shape), dtype=torch.float32, device="cuda")).requires_grad_()
    opt = torch.optim.LBFGS([rot], lr=1, max_iter=200, history_size=50, tolerance_grad=0, tolerance_change=0,
                            line_search_fn="strong_wolfe")

    def closure():
        opt.zero_grad()
        loss = (E.head_angles(*rotated_heads(rot, base0, stalk0, neck), neck[None], rest) - target).pow(2).sum()
        loss.backward()
        return loss

    for _ in range(5):
        opt.step(closure)
        with torch.no_grad():
            ang_err = float((E.head_angles(*rotated_heads(rot, base0, stalk0, neck), neck[None], rest) - target).abs().max())
        rot_err = float((rot.detach() - true_t).abs().max())
        if rot_err < 1e-4 and ang_err < 1e-5:
            break
    evals = opt.state[opt._params[0]]["func_evals"]
    print(f"LBFGS: {evals} evaluations, worst rotation error {rot_err:.3e} rad, worst angle error {ang_err:.3e} rad")
    assert rot_err < 1e-4 and ang_err < 1e-5, (evals, rot_err, ang_err)
