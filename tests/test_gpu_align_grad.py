"""The differentiable leg alignment on the device: seqik_align_apply_backward_f32 and seqik_leg_affine_backward_f32 against
the float64 model (tests/model_align.py) and against each other on every launch path, the frames of the order statistics
under the tie rule, the composite's invariances, autograd through engine.leg_affine -> engine.align_apply, and an LBFGS fit of
per-chain rotations through it."""
import numpy as np
import pytest
import torch

import model_align as A
import model_quantile as Q

pytestmark = pytest.mark.gpu
U = 2.0 ** -24
RATIOS = {}                          # largest observed |kernel - model| / bound, per check


def _E():
    from seqikpy_b200 import engine
    return engine


def _lib():
    from seqikpy_b200 import _native as N
    return N, N.load_library()


def _cuda(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _note(name, ratio):
    RATIOS[name] = max(RATIOS.get(name, 0.0), float(ratio))


# ------------------------------------------------------------------------------------------------------------ workloads
KINDS = ("synthetic", "normal", "integer", "constant", "duplicated", "signed_zero", "zero_segment")


def _chain(kind, n, rng):
    from seqikpy_b200 import synthetic as S
    if kind == "synthetic":
        return S.make_trials([int(rng.integers(0, 1000))], n)[0, :, int(rng.integers(0, 6))]
    base = rng.normal(size=(1, 5, 3)).cumsum(axis=1)
    if kind == "normal":
        return rng.normal(size=(n, 5, 3))
    if kind == "integer":
        steps = rng.integers(1, 3, (1, 5, 3)).cumsum(axis=1)
        return steps + rng.integers(-1, 2, (n, 5, 3)) * (rng.random((n, 5, 3)) < 0.3)
    if kind == "constant":
        return np.repeat(base, n, axis=0)
    if kind == "duplicated":
        q = base + 0.1 * rng.normal(size=(n // 2 + 1, 5, 3))
        return q[np.arange(n) // 2]
    if kind == "signed_zero":
        p = base + 0.1 * rng.normal(size=(n, 5, 3))
        z = rng.random((n, 5, 3)) < 0.3
        return np.where(z, np.where(rng.random((n, 5, 3)) < 0.5, -0.0, 0.0), p)
    p = base + 0.1 * rng.normal(size=(n, 5, 3))                                     # zero_segment
    p[::2, 2] = p[::2, 1]
    return p


def _batch(n, seed, kinds=KINDS):
    rng = np.random.default_rng(seed)
    pose = np.stack([_chain(k, n, rng) for k in kinds]).astype(np.float32)
    consts = np.concatenate([rng.normal(size=(len(kinds), 3)), rng.uniform(1.0, 3.0, (len(kinds), 1))], axis=1).astype(np.float32)
    return pose, consts


# ------------------------------------------------------------------------------------------------------------ apply backward
def _apply_bw(pose_t, cs, fs, aff, g_out, n_chain, n_frame, want_pose=True, want_part=True):
    N, lib = _lib()
    gp = torch.full((n_chain, n_frame, 5, 3), 7.0, device="cuda") if want_pose else None
    part = torch.full((n_chain, n_frame, 8), 7.0, device="cuda") if want_part else None
    rc = lib.seqik_align_apply_backward_f32(pose_t.data_ptr(), cs, fs, aff.data_ptr(), g_out.data_ptr(), N.ptr(gp), N.ptr(part),
                                            n_chain, n_frame, N.stream_ptr(torch, pose_t.device))
    N.check(rc, "seqik_align_apply_backward_f32")
    torch.cuda.synchronize()
    return gp, part


@pytest.mark.parametrize("n_chain,n_frame", [(3, 1000), (2, 128), (1, 100), (7, 333)])
def test_apply_backward_paths_agree_bit_for_bit(n_chain, n_frame):
    rng = np.random.default_rng(n_chain * 1000 + n_frame)
    pose = _cuda(rng.normal(size=(n_chain, n_frame, 5, 3)).astype(np.float32))
    aff = _E().leg_affine(pose, _cuda(rng.uniform(0.5, 2.0, (n_chain, 4)).astype(np.float32)))
    g = _cuda(rng.normal(size=(n_chain, n_frame, 5, 3)).astype(np.float32))
    gp, part = _apply_bw(pose, n_frame * 15, 15, aff, g, n_chain, n_frame)           # tile path (+ tail) where there are tiles
    ref = aff[:, 3, None, None, None] * g
    ref[:, :, 0] = 0.0
    assert torch.equal(gp, ref) and not torch.signbit(gp[:, :, 0]).any()
    for off in (1, 2, 3):                                                            # unaligned pose: the plain kernel
        buf = torch.empty(pose.numel() + off, device="cuda")
        buf[off:] = pose.flatten()
        gq, pq = _apply_bw(buf[off:], n_frame * 15, 15, aff, g, n_chain, n_frame)
        assert torch.equal(gq, gp) and torch.equal(pq, part), off
    wide = torch.zeros((n_chain, n_frame, 19), device="cuda")                       # frame stride 19 > 15
    wide[..., :15] = pose.reshape(n_chain, n_frame, 15)
    gq, pq = _apply_bw(wide, n_frame * 19, 19, aff, g, n_chain, n_frame)
    assert torch.equal(gq, gp) and torch.equal(pq, part)
    gq, _ = _apply_bw(pose, n_frame * 15, 15, aff, g, n_chain, n_frame, want_part=False)
    _, pq = _apply_bw(pose, n_frame * 15, 15, aff, g, n_chain, n_frame, want_pose=False)
    assert torch.equal(gq, gp) and torch.equal(pq, part)
    gq, pq = _apply_bw(pose, n_frame * 15, 15, aff, g, n_chain, n_frame)            # repeated call
    assert torch.equal(gq, gp) and torch.equal(pq, part)
    # values: the partial rows summed against the float64 VJP
    p64 = pose.double().requires_grad_()
    a64 = aff.double().requires_grad_()
    gp64, ga64 = torch.autograd.grad(A.align_apply(p64, a64), [p64, a64], g.double())
    _, ga = _E().align_apply_backward(pose, aff, g)
    pa, absg = pose.double().abs(), g.double().abs()
    terms = torch.cat([absg[:, :, 1:].sum((1, 2)) * aff[:, 3:4].double().abs(),
                       ((pa[:, :, 1:] + aff[:, None, None, :3].double().abs()) * absg[:, :, 1:]).sum((1, 2, 3))[:, None],
                       absg.sum((1, 2)), torch.zeros((n_chain, 1), device="cuda", dtype=torch.float64)], dim=1)
    bound = 4 * U * (15 * n_frame) * terms
    err = (ga.double() - ga64).abs()
    assert torch.all(err <= bound), (err / bound).max()
    _note("align_apply_backward grad_affine", (err / bound.clamp_min(1e-300)).max())
    assert torch.equal(gp, gp64.float())                                             # fl(a3 g): one rounding of the exact product


# ------------------------------------------------------------------------------------------------------------ statistics backward
N_FRAMES = (1, 2, 3, 4, 5, 6, 8, 10, 31, 32, 33, 1000, 1024, 1025, 6000, 30011, 100000)


def _coxa_expected(frames, f45, f55, n_frame):
    """float32 dL/dp[t, 0, c] for H = e_c: the four weights added in the kernel's order (sorted rank position)."""
    ranks, _, _ = Q.mid_quantile_ranks(np.array([n_frame]))
    swap = ranks[1, 0] > ranks[2, 0]
    f32 = np.float32
    w = [f32(0.5) * (f32(1) - f32(f45)), f32(0.5) * f32(f45), f32(0.5) * (f32(1) - f32(f55)), f32(0.5) * f32(f55)]
    out = np.zeros(n_frame, dtype=np.float32)
    for i in ((0, 2, 1, 3) if swap else (0, 1, 2, 3)):
        out[frames[i]] = out[frames[i]] + w[i]
    return out


@pytest.mark.parametrize("include_claw", [False, True])
@pytest.mark.parametrize("n_frame", N_FRAMES)
def test_statistics_frames_and_values(n_frame, include_claw):
    E = _E()
    pose, consts = _batch(n_frame, 11 * n_frame + include_claw)
    n_chain = pose.shape[0]
    pose_t, consts_t = _cuda(pose), _cuda(consts)
    aff = E.leg_affine(pose_t, consts_t, include_claw)
    aff_np = aff.cpu().numpy()
    frames, f45, f55 = A.stat_frames(pose)
    # the float32 statistics at the model's frames are the forward's row, bit for bit
    d = pose[:, :, 1:] - pose[:, :, :-1]
    sq = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
    series = np.concatenate([pose[:, :, 0].transpose(0, 2, 1), np.sqrt(sq).transpose(0, 2, 1)], axis=1)
    v = np.take_along_axis(series, frames, axis=2)
    m = Q.mid_quantile_value(v[..., 0], v[..., 1], v[..., 2], v[..., 3], f45, f55)
    length = (m[:, 3] + m[:, 4]) + m[:, 5]
    if include_claw:
        length = length + m[:, 6]
    assert np.array_equal(m[:, :3], aff_np[:, :3])
    assert np.array_equal(consts[:, 3] / length, aff_np[:, 3])
    zero_pose = torch.zeros_like(pose_t)
    # H = e_c on a coxa statistic: the nonzero pattern and values are the weights at the model's frames
    for c in range(3):
        h = torch.zeros((n_chain, 8), device="cuda")
        h[:, c] = 1.0
        gp, gk = E.leg_affine_backward(pose_t, consts_t, aff, h, include_claw)
        gp = gp.cpu().numpy()
        for ch in range(n_chain):
            want = np.zeros((n_frame, 5, 3), dtype=np.float32)
            want[:, 0, c] = _coxa_expected(frames[ch, c], f45, f55, n_frame)
            assert np.array_equal(gp[ch], want), (ch, c)
        assert not gk.cpu().numpy().any()
    # H = e_3 (scale): dL/dconsts[3] = 1 / len bit for bit; the length statistics within the bound (zeros exact)
    rng = np.random.default_rng(n_frame)
    for h_np in (np.tile(np.eye(8, dtype=np.float32)[3], (n_chain, 1)), rng.normal(size=(n_chain, 8)).astype(np.float32)):
        gp, gk = E.leg_affine_backward(pose_t, consts_t, aff, _cuda(h_np), include_claw, grad_pose=zero_pose.clone())
        gp, gk = gp.cpu().numpy().astype(np.float64), gk.cpu().numpy()
        if h_np[0, 3] == 1 and not h_np[0, :3].any():
            assert np.array_equal(gk[:, 3], np.float32(1) / length)
        gp64, gk64, (cnt, acc) = A.stats_vjp(pose, consts, h_np, include_claw)
        bound = 64 * U * cnt * acc
        err = np.abs(gp - gp64)
        assert np.all(err <= bound), (err / np.where(bound > 0, bound, 1)).max()
        _note("leg_affine_backward grad_pose", (err / np.where(bound > 0, bound, np.inf)).max())
        kb = 16 * U * np.abs(gk64)
        assert np.all(np.abs(gk - gk64) <= kb)
        _note("leg_affine_backward grad_consts", (np.abs(gk - gk64) / np.where(kb > 0, kb, np.inf)).max())


@pytest.mark.parametrize("n_frame", [2, 4, 6, 8, 10, 33, 1025])
def test_scale_gradient_uses_the_forward_length(n_frame):
    """dL/dconsts[3] = H3 / len with the forward's len bit for bit: the mid-quantiles are recomputed from the selected keys with
    the forward's float32 operations, the middle two keys put back for m = 2, 4, 6, 8, 10 (256 chains: the plain average of
    the neighbours rounds differently on a few percent of them)."""
    E = _E()
    rng = np.random.default_rng(n_frame)
    pose = rng.normal(size=(256, n_frame, 5, 3)).astype(np.float32)
    consts = rng.uniform(1.0, 3.0, (256, 4)).astype(np.float32)
    pose_t, consts_t = _cuda(pose), _cuda(consts)
    aff = E.leg_affine(pose_t, consts_t)
    h = torch.zeros((256, 8), device="cuda")
    h[:, 3] = 1.0
    _, gk = E.leg_affine_backward(pose_t, consts_t, aff, h)
    _, stats, _ = Q.leg_stats_exact(pose, consts, False)
    length = (stats[:, 3] + stats[:, 4]) + stats[:, 5]
    assert np.array_equal(gk[:, 3].cpu().numpy(), np.float32(1) / length)


def test_statistics_backward_repeatable_and_adds_into_grad_pose():
    E = _E()
    pose, consts = _batch(2000, 5)
    pose_t, consts_t = _cuda(pose), _cuda(consts)
    for n in (700, 2000):                                                          # fused and long paths
        p = pose_t[:, :n].contiguous()
        aff = E.leg_affine(p, consts_t, True)
        h = torch.randn((p.shape[0], 8), device="cuda")
        g1, k1 = E.leg_affine_backward(p, consts_t, aff, h, True)
        g2, k2 = E.leg_affine_backward(p, consts_t, aff, h, True)
        assert torch.equal(g1, g2) and torch.equal(k1, k2)
        base = torch.randn_like(p)
        g3, _ = E.leg_affine_backward(p, consts_t, aff, h, True, grad_pose=base.clone())
        touched = g1 != 0
        assert torch.equal(g3[~touched], base[~touched])
        # strided pose (frame stride 19) through the C entry point: the same bits
        N, lib = _lib()
        wide = torch.zeros((p.shape[0], n, 19), device="cuda")
        wide[..., :15] = p.reshape(p.shape[0], n, 15)
        gw = torch.zeros_like(p)
        kw = torch.empty((p.shape[0], 4), device="cuda")
        scratch = torch.empty((p.shape[0] * 7 * (n + 12),), dtype=torch.int32, device="cuda")
        N.check(lib.seqik_leg_affine_backward_f32(wide.data_ptr(), n * 19, 19, consts_t.data_ptr(), 1, aff.data_ptr(), h.data_ptr(),
                                                  gw.data_ptr(), kw.data_ptr(), scratch.data_ptr(), p.shape[0], n,
                                                  N.stream_ptr(torch, p.device)), "seqik_leg_affine_backward_f32")
        assert torch.equal(gw, g1) and torch.equal(kw, k1)


# ------------------------------------------------------------------------------------------------------------ composite
@pytest.mark.parametrize("include_claw", [False, True])
@pytest.mark.parametrize("n_frame", [2, 6, 33, 1000, 1500])
def test_composite_invariances(n_frame, include_claw):
    """sum_{t,k} dL/dp = 0 per chain and coordinate, and sum p . dL/dp = 0 per chain (alignment is invariant under
    p -> a p + b), within the float32 bound 4 u (15 n) sum |terms|."""
    E = _E()
    pose, consts = _batch(n_frame, 3 * n_frame + include_claw)
    pose_t, consts_t = _cuda(pose), _cuda(consts)
    g = torch.randn(pose_t.shape, device="cuda")
    aff = E.leg_affine(pose_t, consts_t, include_claw)
    gp_apply, ga = E.align_apply_backward(pose_t, aff, g)
    gp_stats, _ = E.leg_affine_backward(pose_t, consts_t, aff, ga, include_claw)
    gp = (gp_apply + gp_stats).double()
    absterm = gp_apply.double().abs() + gp_stats.double().abs()
    p = pose_t.double()
    s1 = gp.sum(dim=(1, 2)).abs()
    b1 = 4 * U * 15 * n_frame * (absterm.sum(dim=(1, 2)) + aff[:, 3, None].double().abs() * g.double().abs().sum(dim=(1, 2)))
    assert torch.all(s1 <= b1), (s1 / b1).max()
    s2 = (gp * p).sum(dim=(1, 2, 3)).abs()
    b2 = 4 * U * 15 * n_frame * ((absterm * p.abs()).sum(dim=(1, 2, 3))
                                 + (aff[:, 3, None, None, None].double().abs() * g.double().abs() * p.abs()).sum(dim=(1, 2, 3))
                                 + (aff[:, None, None, :3].double().abs() * absterm).sum(dim=(1, 2, 3)))
    assert torch.all(s2 <= b2), (s2 / b2).max()
    _note("invariance sum dL/dp", (s1 / b1).max())
    _note("invariance sum p dL/dp", (s2 / b2).max())


@pytest.mark.parametrize("n_frame", [300, 1500])
def test_autograd_equals_the_direct_calls(n_frame):
    E = _E()
    pose, consts = _batch(n_frame, 23)
    pose0, consts0 = _cuda(pose), _cuda(consts)
    n_chain = pose0.shape[0]
    aff0 = E.leg_affine(pose0, consts0, True)
    out0 = E.align_apply(pose0, aff0)
    g = torch.randn((n_chain, n_frame, 3, 5), device="cuda").transpose(-1, -2)        # non-contiguous incoming gradients
    h = torch.randn((8, n_chain), device="cuda").T
    names = ("pose", "consts", "affine")
    for mask in range(1, 8):
        req = {nm: bool(mask >> i & 1) for i, nm in enumerate(names)}
        p = pose0.clone().requires_grad_(req["pose"])
        k = consts0.clone().requires_grad_(req["consts"])
        if req["affine"]:
            a = aff0.clone().requires_grad_()
            outs = [E.align_apply(p, a), E.leg_affine(p, k, True)]
        else:
            a = E.leg_affine(p, k, True)
            outs = [E.align_apply(p, a), a]
        assert torch.equal(outs[0].detach(), out0) and torch.equal(outs[1].detach(), aff0)
        assert outs[1].requires_grad == (req["pose"] or req["consts"])
        inputs = [t for t, nm in zip((p, k, a), names) if req[nm]]
        used = [(o, go) for o, go in zip(outs, (g, h)) if o.requires_grad]
        got = torch.autograd.grad([o for o, _ in used], inputs, [go for _, go in used])
        gp1, ga = E.align_apply_backward(pose0, aff0, g.contiguous())
        if req["affine"]:
            want_a = ga
            gps, gk = E.leg_affine_backward(pose0, consts0, aff0, h.contiguous(), True)
        else:
            gps, gk = E.leg_affine_backward(pose0, consts0, aff0, ga + h.contiguous(), True)
            want_a = None
        want = {"pose": gp1 + gps, "consts": gk, "affine": want_a}
        for t, nm in zip(got, [nm for nm in names if req[nm]]):
            assert torch.equal(t, want[nm]), (mask, nm)
    p = pose0.clone().requires_grad_()
    gx, = torch.autograd.grad(E.align_apply(p, E.leg_affine(p, consts0)).pow(2).sum(), p, create_graph=True)
    with pytest.raises(RuntimeError, match="once_differentiable"):
        gx.sum().backward()
    with torch.no_grad():                                                              # without grad: plain launches, same bits
        assert torch.equal(E.align_apply(p, E.leg_affine(p, consts0, True)), out0)


def _rotation(w):
    """(n, 3) rotation vectors -> (n, 3, 3) rotation matrices."""
    z = torch.zeros_like(w[:, 0])
    k = torch.stack([z, -w[:, 2], w[:, 1], w[:, 2], z, -w[:, 0], -w[:, 1], w[:, 0], z], dim=1).reshape(-1, 3, 3)
    return torch.linalg.matrix_exp(k)


def test_lbfgs_recovers_per_chain_rotations():
    """Raw key points of 12 chains x 200 frames seen through an unknown per-chain rotation; the rotation is fitted against the
    aligned pose of the true one, through leg_affine -> align_apply, from 0.1 rad off about each axis."""
    from seqikpy_b200 import synthetic as S
    E = _E()
    raw = torch.from_numpy(np.ascontiguousarray(S.to_chains(S.make_trials(range(2), 200)))).cuda()            # (12, 200, 5, 3)
    consts = torch.cat([torch.randn((12, 3), device="cuda", generator=torch.Generator("cuda").manual_seed(0)),
                        torch.full((12, 1), 2.0, device="cuda")], dim=1)
    w_true = 0.3 * torch.randn((12, 3), device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    rot = lambda w: torch.einsum("cij,cfkj->cfki", _rotation(w), raw).contiguous()
    with torch.no_grad():
        target = E.align_apply(rot(w_true), E.leg_affine(rot(w_true), consts))
    w = (w_true + 0.1).clone().requires_grad_()
    opt = torch.optim.LBFGS([w], lr=1, max_iter=500, tolerance_grad=1e-12, tolerance_change=1e-15, line_search_fn="strong_wolfe")

    def closure():
        opt.zero_grad()
        posed = rot(w)
        loss = (E.align_apply(posed, E.leg_affine(posed, consts)) - target).double().pow(2).sum()
        loss.backward()
        return loss

    loss0 = float(closure())
    opt.step(closure)
    loss1 = float(closure())
    err = float((w.detach() - w_true).abs().max())
    print(f"LBFGS rotation fit: loss {loss0:.3e} -> {loss1:.3e}, max |w - w_true| = {err:.2e} rad")
    _note("lbfgs max rotation error (rad)", err)
    assert err < 1e-5 and loss1 < 1e-10 * loss0                                    # measured: 2.7e-7 rad, 8.7e-13


def test_report_ratios():
    """Prints the largest observed ratio of every bounded check of this module (run with -s)."""
    for k, v in sorted(RATIOS.items()):
        print(f"largest ratio {k}: {v:.3g}")
