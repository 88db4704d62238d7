"""Differentiable FK: seqik_fk_backward_f32 on every launch path, against the float64 model's autograd, through
torch.autograd, and in a fit of angles and segment lengths to key points.

Shapes and inputs are those of tests/test_gpu_stream.py (angles over [-2 pi, 2 pi] with the branch points of sincosv_, chain
boundaries inside tiles and tails, one case where every persistent CTA walks at least four tiles).

Bounds per leg-frame, with G = sum over the nine rows of |g_r| (g = dL/dfk) and u the float32 unit roundoff:
* grad_angles: 64 u (sum of the segment lengths) G.  dL/dangle = u . T_k with |T_k| <= sum_j l_j |S_j| <= (sum l) G; the frames
  carry the few-u errors of the forward (tests/test_gpu_stream.py fk_bound) and each cross product, sum and dot adds a
  rounding of at most that magnitude.
* grad_lengths: 64 u G (-A_k.c2 . S_k, |A_k.c2| = 1 + O(u), |S_k| <= G).
* grad_origin: the float32 sums of include/seqik.h in that order, bit for bit.
"""
import itertools

import numpy as np
import pytest
import torch

import model_fk
from test_gpu_stream import LEG_SHAPES, TILE, U, dev, fk_inputs, fk_sample, offset_view, same_bits

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    assert torch.cuda.is_available(), "these tests need the B200"
    from seqikpy_b200 import _native as N, engine
    N.load_library()
    return engine, N


def grad_inputs(rng, n_chain, n_frame):
    ang, org, params = fk_inputs(rng, n_chain, n_frame)
    g = rng.normal(size=(n_chain, n_frame, 9, 3)).astype(np.float32)
    return ang, org, params, g


def bits(t):
    return t.contiguous().view(torch.int32)


def origin_order_f32(g):
    """grad_origin in the header's float32 summation order (numpy float32, one rounding per addition)."""
    g = g.astype(np.float32)
    s = g[..., 8, :]
    s = g[..., 7, :] + s
    s = g[..., 6, :] + s
    s = (g[..., 4, :] + g[..., 5, :]) + s
    return (((g[..., 0, :] + g[..., 1, :]) + g[..., 2, :]) + g[..., 3, :]) + s


def call_abi(N, ang, org, org_stride, prm, g, ga, go, gl, n_chain, n_frame):
    lib = N.load_library()
    N.check(lib.seqik_fk_backward_f32(ang.data_ptr(), org.data_ptr(), org_stride, prm.data_ptr(), g.data_ptr(), ga.data_ptr(),
                                      N.ptr(go), N.ptr(gl), n_chain, n_frame, torch.cuda.current_stream().cuda_stream),
            "seqik_fk_backward_f32")


@pytest.mark.parametrize("n_chain,n_frame", LEG_SHAPES)
def test_fk_backward_paths_bitwise_and_vs_float64(eng, n_chain, n_frame):
    E, N = eng
    rng = np.random.default_rng(5000 + n_frame)
    ang, org, params, g = grad_inputs(rng, n_chain, n_frame)
    d_ang, d_org, d_prm, d_g = (dev(torch, a) for a in (ang, org, params, g))
    ref = E.forward_kinematics_backward(d_ang, d_org, d_prm, d_g, want_origin=True, want_lengths=True)   # tiles + tail
    ref_bits = [bits(t) for t in ref]

    def same(out, which=(0, 1, 2)):
        return all(torch.equal(bits(out[i]), ref_bits[i]) for i in which)

    assert same(E.forward_kinematics_backward(d_ang, d_org, d_prm, d_g, want_origin=True, want_lengths=True))   # repeatable
    for k in (1, 2, 3):                                                                 # plain kernel: inputs unaligned
        assert same(E.forward_kinematics_backward(offset_view(torch, d_ang, k), d_org, d_prm, d_g, True, True)), ("angles", k)
        assert same(E.forward_kinematics_backward(d_ang, d_org, d_prm, offset_view(torch, d_g, k), True, True)), ("grad_fk", k)
    # plain kernel: one output unaligned (through the C ABI, the engine allocates aligned outputs)
    for k in (1, 2, 3):
        for j in range(3):
            out = [torch.empty_like(t) for t in ref]
            out[j] = offset_view(torch, out[j], k)
            call_abi(N, d_ang, d_org, 3, d_prm, d_g, *out, n_chain, n_frame)
            assert same(out), ("output", j, k)
    # outputs left out (NULL) change nothing in the others
    ga, go, gl = E.forward_kinematics_backward(d_ang, d_org, d_prm, d_g, want_origin=False, want_lengths=False)
    assert go is None and gl is None and torch.equal(bits(ga), ref_bits[0])
    ga, go, gl = E.forward_kinematics_backward(d_ang, d_org, d_prm, d_g, want_origin=False, want_lengths=True)
    assert go is None and same((ga, None, gl), (0, 2))
    # origin per chain (stride 0) equal to the per-frame origins: the same bits
    org0 = np.repeat(org[:, :1], n_frame, axis=1)
    per_frame = E.forward_kinematics_backward(d_ang, dev(torch, org0), d_prm, d_g, True, True)
    per_chain = E.forward_kinematics_backward(d_ang, dev(torch, org[:, 0].copy()), d_prm, d_g, True, True)
    assert all(torch.equal(bits(a), bits(b)) for a, b in zip(per_frame, per_chain))

    ga, go, gl = (t.cpu().numpy() for t in ref)
    assert same_bits(go, origin_order_f32(g))
    # float64 model's autograd on a sample of leg-frames (every tile's first and last, chain boundaries, the tail, random)
    sample = fk_sample(rng, n_chain, n_frame)
    c, t = sample // n_frame, sample % n_frame
    q64 = torch.from_numpy(ang[c, t].astype(np.float64)).requires_grad_()
    l64 = torch.from_numpy(params[c, :4].astype(np.float64)).requires_grad_()
    o64 = torch.from_numpy(org[c, t].astype(np.float64)).requires_grad_()
    g64 = torch.from_numpy(g[c, t].astype(np.float64))
    (model_fk.fk(q64, o64, l64) * g64).sum().backward()
    G = np.linalg.norm(g[c, t].astype(np.float64), axis=-1).sum(axis=-1)
    b_ang = 64 * U * params[c, :4].astype(np.float64).sum(axis=1) * G
    b_len = 64 * U * G
    e_ang = np.abs(ga[c, t] - q64.grad.numpy()).max(axis=1)
    e_len = np.abs(gl[c, t] - l64.grad.numpy()).max(axis=1)
    assert (e_ang <= b_ang).all(), (e_ang.max(), sample[np.argmax(e_ang / b_ang)])
    assert (e_len <= b_len).all(), (e_len.max(), sample[np.argmax(e_len / b_len)])
    assert np.abs(go[c, t] - o64.grad.numpy()).max() <= 16 * U * G.max()                # and the sum order is a float32 one
    print(f"{n_chain}x{n_frame}: worst ratio to bound: grad_angles {(e_ang / b_ang).max():.4f}, "
          f"grad_lengths {(e_len / b_len).max():.4f}")


@pytest.mark.parametrize("per_frame_origin", [True, False])
@pytest.mark.parametrize("n_chain,n_frame", [(5, 257), (100, 7)])
def test_autograd_equals_the_direct_backward(eng, n_chain, n_frame, per_frame_origin):
    """Every subset of {angles, origin, params} that requires grad: torch.autograd.grad through forward_kinematics equals
    forward_kinematics_backward (+ the frame sums) bit for bit; inputs that do not require grad get None."""
    E, _ = eng
    rng = np.random.default_rng(6000 + n_frame)
    ang, org, params, g = grad_inputs(rng, n_chain, n_frame)
    if not per_frame_origin:
        org = org[:, 0].copy()
    d_ang, d_org, d_prm, d_g = (dev(torch, a) for a in (ang, org, params, g))
    ga, go, gl = E.forward_kinematics_backward(d_ang, d_org, d_prm, d_g, want_origin=True, want_lengths=True)
    want = {"angles": ga, "origin": go if per_frame_origin else go.sum(dim=1),
            "params": torch.cat([gl.sum(dim=1), torch.zeros((n_chain, 28), device="cuda")], 1)}
    fk_plain = E.forward_kinematics(d_ang, d_org, d_prm)
    assert fk_plain.grad_fn is None
    names = ("angles", "origin", "params")
    for r in range(1, 4):
        for subset in itertools.combinations(names, r):
            x = {n: t.clone().requires_grad_(n in subset) for n, t in zip(names, (d_ang, d_org, d_prm))}
            fk = E.forward_kinematics(x["angles"], x["origin"], x["params"])
            assert torch.equal(bits(fk), bits(fk_plain)), subset                   # grad mode does not change the result
            grads = torch.autograd.grad((fk * d_g).sum(), [x[n] for n in subset])
            for n, gr in zip(subset, grads):
                assert gr.shape == x[n].shape and torch.equal(bits(gr), bits(want[n])), (subset, n)
            with torch.no_grad():
                assert E.forward_kinematics(x["angles"], x["origin"], x["params"]).grad_fn is None


def test_autograd_sliced_loss_and_first_order_only(eng):
    E, _ = eng
    rng = np.random.default_rng(61)
    ang, org, params, _ = grad_inputs(rng, 7, 301)
    d_ang = dev(torch, ang).requires_grad_()
    d_org, d_prm = dev(torch, org), dev(torch, params)
    fk = E.forward_kinematics(d_ang, d_org, d_prm)
    loss = fk[:, :, 5:9].pow(2).sum()                     # the incoming gradient is zero outside rows 5-8
    (gr,) = torch.autograd.grad(loss, [d_ang])
    g = torch.zeros_like(fk)
    g[:, :, 5:9] = 2 * fk.detach()[:, :, 5:9]
    assert torch.equal(bits(gr), bits(E.forward_kinematics_backward(d_ang.detach(), d_org, d_prm, g, want_origin=False)[0]))
    # a non-contiguous incoming gradient (a transposed view's backward) is made contiguous
    w = dev(torch, rng.normal(size=(3, 9, 301, 7)).astype(np.float32))
    fk = E.forward_kinematics(d_ang, d_org, d_prm)
    (gr,) = torch.autograd.grad((fk.permute(3, 2, 1, 0) * w).sum(), [d_ang])
    g = w.permute(3, 2, 1, 0).contiguous()
    assert torch.equal(bits(gr), bits(E.forward_kinematics_backward(d_ang.detach(), d_org, d_prm, g, want_origin=False)[0]))
    # second derivatives are not supported
    (gr,) = torch.autograd.grad(E.forward_kinematics(d_ang, d_org, d_prm).pow(2).sum(), [d_ang], create_graph=True)
    with pytest.raises(RuntimeError, match="once_differentiable"):
        gr.sum().backward()


def synthetic_legs(n_trial, n_frame, seed):
    """Noise-free leg key points of the synthetic workload: (angles (C, T, 7), lengths (C, 4), origins (C, 3), joints (C, T, 4, 3))."""
    from seqikpy_b200 import synthetic as S
    size, _, init = S.chain_constants()
    rng = np.random.default_rng(seed)
    t = np.arange(n_frame, dtype=float)
    th, seg, org = [], [], []
    for _ in range(n_trial):
        for leg in S.LEGS:
            theta0 = np.array(init[leg]["stage_4"][1:8], dtype=float)
            theta0[6] = -0.6
            th.append(theta0 + 0.3 * np.sin(2 * np.pi * rng.uniform(1, 4, 7) * t[:, None] / 1000 + rng.uniform(0, 2 * np.pi, 7)))
            seg.append([size[f"{leg}_{s}"] for s in S.SEGMENTS])
            org.append(S.TEMPLATE_NMF_LOCOMOTION[f"{leg}_Coxa"])
    th, seg, org = np.array(th), np.array(seg), np.array(org, dtype=float)
    joints = np.stack([S.leg_key_points(th[c], seg[c]) for c in range(len(seg))]) + org[:, None, None]
    return th, seg, org, joints


def test_lbfgs_fit_recovers_segment_lengths(eng):
    """12 chains x 200 frames of noise-free key points; start with every segment length 3-5 % off and every angle 0.05 rad
    off; a float32 LBFGS fit of angles and lengths through forward_kinematics recovers the lengths to 1e-3 relative and
    the joints to 1e-3 mm."""
    E, _ = eng
    th, seg, org, joints = synthetic_legs(2, 200, 11)
    rng = np.random.default_rng(12)
    n_chain = seg.shape[0]
    l0 = seg * (1 + rng.choice([-1.0, 1.0], seg.shape) * rng.uniform(0.03, 0.05, seg.shape))
    q = torch.tensor(th + rng.choice([-0.05, 0.05], th.shape), dtype=torch.float32, device="cuda", requires_grad=True)
    lengths = torch.tensor(l0, dtype=torch.float32, device="cuda", requires_grad=True)
    rest = torch.zeros((n_chain, 28), dtype=torch.float32, device="cuda")
    origin = torch.tensor(org, dtype=torch.float32, device="cuda")
    target = torch.tensor(joints, dtype=torch.float32, device="cuda")
    opt = torch.optim.LBFGS([q, lengths], lr=1, max_iter=250, history_size=50, tolerance_grad=0, tolerance_change=0,
                            line_search_fn="strong_wolfe")

    def closure():
        opt.zero_grad()
        fk = E.forward_kinematics(q, origin, torch.cat([lengths, rest], 1))
        loss = (fk[:, :, 5:9] - target).pow(2).sum()
        loss.backward()
        return loss

    for _ in range(12):
        opt.step(closure)
        with torch.no_grad():
            resid = float((E.forward_kinematics(q, origin, torch.cat([lengths, rest], 1))[:, :, 5:9] - target).norm(dim=-1).max())
        rel = float(np.abs(lengths.detach().cpu().numpy() / seg - 1).max())
        if resid < 1e-3 and rel < 1e-3:
            break
    evals = opt.state[opt._params[0]]["func_evals"]
    print(f"LBFGS: {evals} evaluations, worst joint residual {resid:.3e} mm, worst length error {rel:.3e} (relative)")
    assert rel < 1e-3 and resid < 1e-3, (evals, rel, resid)
