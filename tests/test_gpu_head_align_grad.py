"""The differentiable head alignment on the device: seqik_head_apply_backward_f32 and seqik_head_affine_backward_f32/_f64
against the float64 model (tests/model_head_align.py) and against each other on every launch path, the frames of the order
statistics over the stationary set under the tie rule, the composite's invariances, the composition with
head_angles_backward, autograd through engine.head_affine -> engine.head_apply, and an LBFGS fit of per-trial rotations
through it."""
from pathlib import Path

import numpy as np
import pytest
import torch

import model_head as H
import model_head_align as M
import model_quantile as Q

pytestmark = pytest.mark.gpu
U = 2.0 ** -24
RATIOS = {}                          # largest observed |kernel - model| / bound, per check
GOLDEN = Path(__file__).resolve().parent / "golden" / "grooming_align.npz"


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
def _recording(n_frame, dtype=np.float64, seed=0):
    """Three trials of the real grooming recording (raw_R_head, raw_L_head with raw_Thorax, and raw_R_head with every frame
    shown twice: ties), n_frame frames: the recording's first frames, played back and forth beyond its 2000 frames with
    1e-6 noise."""
    d = np.load(GOLDEN)
    t = np.arange(n_frame)
    idx = np.abs((t + 1999) % 3998 - 1999) if n_frame > 2000 else t
    r, l, th = d["raw_R_head"][idx], d["raw_L_head"][idx], d["raw_Thorax"][idx]
    if n_frame > 2000:
        rng = np.random.default_rng(seed)
        r, l, th = (x + 1e-6 * rng.normal(size=x.shape) for x in (r, l, th))
    head = np.stack([r, l, r[t // 2]])
    thorax = np.stack([th, th, th[t // 2]])
    consts = np.array([[0.1, -0.2, 0.3, 0.6, 0.35], [-0.1, -0.2, 0.3, 0.6, 0.35], [0.2, 0.1, 0.0, 0.5, 0.3]], dtype=np.float32)
    return head.astype(dtype), thorax.astype(dtype), consts


FRACTIONS = ("none", "few", "half", "all")


def _threshold(head, thorax, fraction):
    """A float32-representable threshold that makes about that fraction of trial 0's frames stationary."""
    dd = np.diff(np.diff(H.base_to_thorax_mid(head[0], thorax[0])))
    if fraction == "none":
        return -1e30
    if fraction == "all":
        return 1e30
    if dd.size == 0:
        return 0.0
    return float(np.float32(np.quantile(dd, 0.03 if fraction == "few" else 0.5)))


def _stats_bw(head_t, thorax_t, consts_t, aff, h, thr):
    return _E().head_affine_backward(head_t, thorax_t, consts_t, aff, h, threshold=thr)


# ------------------------------------------------------------------------------------------------------------ apply backward
def _apply_bw(head_t, aff, g_out, want_head=True, want_part=True):
    N, lib = _lib()
    n_trial, n_frame = aff.shape[0], g_out.numel() // (6 * aff.shape[0])
    gh = torch.full((n_trial, n_frame, 2, 3), 7.0, device="cuda") if want_head else None
    part = torch.full((n_trial, n_frame, 8), 7.0, device="cuda") if want_part else None
    rc = lib.seqik_head_apply_backward_f32(head_t.data_ptr(), aff.data_ptr(), g_out.data_ptr(), N.ptr(gh), N.ptr(part),
                                           n_trial, n_frame, N.stream_ptr(torch, head_t.device))
    N.check(rc, "seqik_head_apply_backward_f32")
    torch.cuda.synchronize()
    return gh, part


@pytest.mark.parametrize("n_trial,n_frame", [(3, 1000), (2, 128), (1, 100), (7, 333), (1, 70001)])
def test_apply_backward_paths_agree_bit_for_bit(n_trial, n_frame):
    rng = np.random.default_rng(n_trial * 1000 + n_frame)
    head = _cuda(rng.normal(size=(n_trial, n_frame, 2, 3)).astype(np.float32))
    aff = _cuda(np.concatenate([rng.normal(size=(n_trial, 3)), rng.uniform(0.5, 2, (n_trial, 1)), rng.normal(size=(n_trial, 3)),
                                rng.uniform(2, 4, (n_trial, 1))], axis=1).astype(np.float32))
    g = _cuda(rng.normal(size=(n_trial, n_frame, 2, 3)).astype(np.float32))
    gh, part = _apply_bw(head, aff, g)                                              # tile path (+ tail) where there are tiles
    ref = torch.stack([aff[:, 3, None, None] * g[:, :, 0], aff[:, 7, None, None] * g[:, :, 1]], dim=2)
    assert torch.equal(gh, ref)                                                     # base a3 G_b, tip a7 G_t
    for off in (1, 2, 3):                                                           # unaligned head / grad_out: the plain kernel
        buf = torch.empty(head.numel() + off, device="cuda")
        buf[off:] = head.flatten()
        gq, pq = _apply_bw(buf[off:], aff, g)
        assert torch.equal(gq, gh) and torch.equal(pq, part), off
        gbuf = torch.empty(g.numel() + off, device="cuda")
        gbuf[off:] = g.flatten()
        gq, pq = _apply_bw(head, aff, gbuf[off:])
        assert torch.equal(gq, gh) and torch.equal(pq, part), off
    gq, _ = _apply_bw(head, aff, g, want_part=False)
    _, pq = _apply_bw(head, aff, g, want_head=False)
    assert torch.equal(gq, gh) and torch.equal(pq, part)
    gq, pq = _apply_bw(head, aff, g)                                                # repeated call
    assert torch.equal(gq, gh) and torch.equal(pq, part)
    # the rows in the header's float order, and their frame sum against the float64 VJP
    o = aff[:, None, :3]
    pb, pt = head[:, :, 0] - o, head[:, :, 1] - o
    dot = lambda p, q: (p[..., 0] * q[..., 0] + p[..., 1] * q[..., 1]) + p[..., 2] * q[..., 2]
    want = torch.cat([-(ref[:, :, 0] + ref[:, :, 1]), dot(pb, g[:, :, 0])[..., None], g[:, :, 0] + g[:, :, 1],
                      dot(pt, g[:, :, 1])[..., None]], dim=-1)
    assert torch.equal(part, want)
    h64, a64 = head.double().requires_grad_(), aff.double().requires_grad_()
    _, ga64 = torch.autograd.grad(M.head_apply(h64, a64), [h64, a64], g.double())
    _, ga = _E().head_apply_backward(head, aff, g)
    ah, ag = head.double().abs(), g.double().abs()
    ao = aff[:, None, :3].double().abs()
    terms = torch.cat([(aff[:, None, 3:4].double().abs() * ag[:, :, 0] + aff[:, None, 7:8].double().abs() * ag[:, :, 1]).sum(1),
                       ((ah[:, :, 0] + ao) * ag[:, :, 0]).sum((1, 2))[:, None], ag.sum((1, 2)),
                       ((ah[:, :, 1] + ao) * ag[:, :, 1]).sum((1, 2))[:, None]], dim=1)
    bound = 4 * U * (6 * n_frame) * terms
    err = (ga.double() - ga64).abs()
    assert torch.all(err <= bound), (err / bound).max()
    _note("head_apply_backward grad_affine", (err / bound.clamp_min(1e-300)).max())


# ------------------------------------------------------------------------------------------------------------ statistics backward
N_FRAMES = (1, 2, 3, 4, 5, 10, 33, 1000, 1024, 1025, 2000, 6000, 100000)


def _coordinate_expected(frames, f45, f55, m, n_frame, dtype):
    """dL/dbase[t][c] for H = e_c: the four float32 weights added in the kernel's order (sorted rank position), in dtype."""
    out = np.zeros(n_frame, dtype=dtype)
    if m == 0:
        return out
    ranks, _, _ = Q.mid_quantile_ranks(np.array([m]))
    swap = ranks[1, 0] > ranks[2, 0]
    f32 = np.float32
    w = [f32(0.5) * (f32(1) - f32(f45)), f32(0.5) * f32(f45), f32(0.5) * (f32(1) - f32(f55)), f32(0.5) * f32(f55)]
    for i in ((0, 2, 1, 3) if swap else (0, 1, 2, 3)):
        out[frames[i]] = out[frames[i]] + dtype(w[i])
    return out


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("fraction", FRACTIONS)
@pytest.mark.parametrize("n_frame", N_FRAMES)
def test_statistics_frames_and_values(n_frame, fraction, dtype):
    E = _E()
    head, thorax, consts = _recording(n_frame, dtype, seed=n_frame)
    thr = _threshold(head, thorax, fraction)
    dthr = M.device_threshold(thr, dtype)
    n_trial = head.shape[0]
    head_t, thorax_t, consts_t = _cuda(head), _cuda(thorax), _cuda(consts)
    aff, counts = E.head_affine(head_t, thorax_t, consts_t, threshold=thr)
    frames, m_counts, f45, f55 = M.stat_frames(head, thorax, dthr)
    assert np.array_equal(counts.cpu().numpy(), m_counts)
    if fraction == "none" or n_frame < 3:
        assert not m_counts[:, :4].any()
    if fraction == "all" and n_frame >= 3:
        assert (m_counts[:, :4] == n_frame - 2).all()
    # H = e_c on a base coordinate: the gradient is the weights at the model's frames, bit for bit
    for c in range(3):
        h = torch.zeros((n_trial, 8), device="cuda")
        h[:, c] = 1.0
        gh, gt, gk = _stats_bw(head_t, thorax_t, consts_t, aff, h, thr)
        gh = gh.cpu().numpy()
        for tr in range(n_trial):
            want = np.zeros((n_frame, 2, 3), dtype=dtype)
            want[:, 0, c] = _coordinate_expected(frames[tr, c], f45[tr, c], f55[tr, c], m_counts[tr, c], n_frame, dtype)
            assert np.array_equal(gh[tr], want), (tr, c)
        assert not gt.cpu().numpy().any()
    # H = e_3 / e_7: the frames that receive the distance's / the tip length's gradient are the model's
    for col, j in ((3, 3), (7, 4)):
        h = torch.zeros((n_trial, 8), device="cuda")
        h[:, col] = 1.0
        gh, gt, _ = _stats_bw(head_t, thorax_t, consts_t, aff, h, thr)
        hit = (gh.cpu().numpy() != 0).any(axis=(2, 3))
        for tr in range(n_trial):
            want = np.zeros(n_frame, dtype=bool)
            if m_counts[tr, j]:
                want[frames[tr, j]] = True
            assert np.array_equal(hit[tr], want), (tr, j)
        assert (gt.cpu().numpy() != 0).any() == (j == 3 and m_counts[:, 3].any())
    # random H: against the float64 VJP within 64 u N A (16 u for dL/dconsts); repeated calls bit for bit
    h_np = np.random.default_rng(n_frame).normal(size=(n_trial, 8)).astype(np.float32)
    gh, gt, gk = _stats_bw(head_t, thorax_t, consts_t, aff, _cuda(h_np), thr)
    gh2, gt2, gk2 = _stats_bw(head_t, thorax_t, consts_t, aff, _cuda(h_np), thr)
    assert torch.equal(gh, gh2) and torch.equal(gt, gt2) and torch.equal(gk.view(torch.int32), gk2.view(torch.int32))
    gh, gt, gk = (x.cpu().numpy().astype(np.float64) for x in (gh, gt, gk))
    gh64, gt64, gk64, (cnt_h, acc_h, cnt_t, acc_t) = M.stats_vjp(head, thorax, consts, h_np, dthr)
    for name, got, ref, cnt, acc in (("grad_head", gh, gh64, cnt_h, acc_h), ("grad_thorax", gt, gt64, cnt_t, acc_t)):
        bound = 64 * U * cnt * acc
        err = np.abs(got - ref)
        assert np.all(err <= bound), (name, (err / np.where(bound > 0, bound, 1)).max())
        _note(f"head_affine_backward {name} ({np.dtype(dtype).name})", (err / np.where(bound > 0, bound, np.inf)).max())
    assert np.array_equal(np.isnan(gk), np.isnan(gk64))
    ok = ~np.isnan(gk64)
    kb = 16 * U * np.abs(gk64[ok])
    assert np.all(np.abs(gk[ok] - gk64[ok]) <= kb)
    _note("head_affine_backward grad_consts", (np.abs(gk[ok] - gk64[ok]) / np.where(kb > 0, kb, np.inf)).max())


@pytest.mark.parametrize("n_frame", [700, 2000])
def test_float32_and_float64_statistics_select_the_same_frames(n_frame):
    """float64 tensors holding float32 values give the float32 series bit for bit, so both entry points select the same
    frames: the coordinate gradients agree exactly and the others within rounding, on both paths; grad_thorax = NULL skips
    only the thorax."""
    E = _E()
    head32, thorax32, consts = _recording(n_frame, np.float32)
    thr = float(np.float32(5e-5))                                                  # the same threshold for both entry points
    h_np = np.random.default_rng(2).normal(size=(3, 8)).astype(np.float32)
    out = {}
    for dt in (np.float32, np.float64):
        ht, tt, kt = _cuda(head32.astype(dt)), _cuda(thorax32.astype(dt)), _cuda(consts)
        aff, counts = E.head_affine(ht, tt, kt, threshold=thr)
        out[dt] = (aff, counts) + E.head_affine_backward(ht, tt, kt, aff, _cuda(h_np), threshold=thr)
        # the C entry point with grad_thorax NULL: the same grad_head and grad_consts
        N, lib = _lib()
        series = torch.empty((15, n_frame), device="cuda")
        cnt = torch.empty((15,), dtype=torch.int32, device="cuda")
        fn = lib.seqik_head_series_f32 if dt == np.float32 else lib.seqik_head_series_f64
        N.check(fn(ht.data_ptr(), tt.data_ptr(), 3, thr, series.data_ptr(), cnt.data_ptr(), 3, n_frame, 0), "series")
        gh = torch.zeros_like(ht)
        gk = torch.empty((3, 5), device="cuda")
        scratch = torch.empty((15 * (n_frame + 12),), dtype=torch.int32, device="cuda")
        bw = lib.seqik_head_affine_backward_f32 if dt == np.float32 else lib.seqik_head_affine_backward_f64
        N.check(bw(ht.data_ptr(), tt.data_ptr(), 3, series.data_ptr(), cnt.data_ptr(), kt.data_ptr(), aff.data_ptr(),
                   _cuda(h_np).data_ptr(), gh.data_ptr(), 0, gk.data_ptr(), scratch.data_ptr(), 3, n_frame, 0), "backward")
        torch.cuda.synchronize()
        assert torch.equal(gh, out[dt][2]) and torch.equal(gk, out[dt][4])
    a32, c32, gh32, gt32, gk32 = out[np.float32]
    a64, c64, gh64, gt64, gk64 = out[np.float64]
    assert torch.equal(c32, c64) and torch.equal(a32, a64)
    assert torch.equal(gk32, gk64)
    assert torch.equal((gh32 != 0), (gh64 != 0)) and torch.equal((gt32 != 0), (gt64 != 0))
    assert torch.allclose(gh64, gh32.double(), rtol=1e-5, atol=1e-6 * float(gh64.abs().max()))
    # the coordinate series alone: exact
    h = torch.zeros((3, 8), device="cuda")
    h[:, :3] = _cuda(h_np[:, :3])
    g32 = E.head_affine_backward(_cuda(head32), _cuda(thorax32), _cuda(consts), a32, h, threshold=thr)[0]
    g64 = E.head_affine_backward(_cuda(head32.astype(np.float64)), _cuda(thorax32.astype(np.float64)), _cuda(consts), a64, h,
                                 threshold=thr)[0]
    assert torch.equal(g64, g32.double())


# ------------------------------------------------------------------------------------------------------------ composite
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("n_frame", [5, 33, 1000, 2000])
def test_composite_invariances(n_frame, dtype):
    """sum dL/dhead + sum dL/dthorax = 0 per trial and coordinate, and sum p . dL/dp over head and thorax = 0 per trial (the
    aligned head is invariant under p -> a p + b with the stationary set fixed), within 4 u (6 n) sum |terms|."""
    E = _E()
    head, thorax, consts = _recording(n_frame, dtype)
    head_t, thorax_t, consts_t = _cuda(head), _cuda(thorax), _cuda(consts)
    g = torch.randn((3, n_frame, 2, 3), device="cuda", generator=torch.Generator("cuda").manual_seed(n_frame))
    aff, _ = E.head_affine(head_t, thorax_t, consts_t)
    gh_apply, ga = E.head_apply_backward(head_t.float(), aff, g)
    gh_stats, gt, _ = E.head_affine_backward(head_t, thorax_t, consts_t, aff, ga)
    gh = gh_apply.double() + gh_stats.double()
    gt = gt.double()
    absh = gh_apply.double().abs() + gh_stats.double().abs()
    ph, pt = head_t.double(), thorax_t.double()
    s1 = (gh.sum(dim=(1, 2)) + gt.sum(dim=(1, 2))).abs()
    b1 = 4 * U * 6 * n_frame * (absh.sum(dim=(1, 2)) + gt.abs().sum(dim=(1, 2)))
    assert torch.all(s1 <= b1), (s1 / b1).max()
    s2 = ((gh * ph).sum(dim=(1, 2, 3)) + (gt * pt).sum(dim=(1, 2, 3))).abs()
    o = aff[:, None, None, :3].double().abs()
    b2 = 4 * U * 6 * n_frame * ((absh * (ph.abs() + o)).sum(dim=(1, 2, 3)) + (gt.abs() * (pt.abs() + o)).sum(dim=(1, 2, 3)))
    assert torch.all(s2 <= b2), (s2 / b2).max()
    _note("invariance sum dL/dp", (s1 / b1).max())
    _note("invariance sum p dL/dp", (s2 / b2).max())


def test_composition_with_head_angles_backward_bit_for_bit():
    """head_apply_backward of the aligned points' head_angles_backward gradient is head_angles_backward with the affine
    rows, for the raw points' gradient."""
    E = _E()
    head, thorax, consts = _recording(1000, np.float32)
    head_t, thorax_t, consts_t = _cuda(head), _cuda(thorax), _cuda(consts)
    aff, _ = E.head_affine(head_t, thorax_t, consts_t)
    r, l = head_t[:2], head_t[[1, 0]].contiguous()
    ar, al = aff[:2].contiguous(), aff[[1, 0]].contiguous()
    neck = torch.tensor([[0.0, 0.0, -0.3]] * 2, device="cuda")
    g = torch.randn((2, 7, 1000), device="cuda", generator=torch.Generator("cuda").manual_seed(5))
    gr_al, gl_al, _ = E.head_angles_backward(E.head_apply(r, ar), E.head_apply(l, al), neck, g)
    gr_raw, gl_raw, _ = E.head_angles_backward(r, l, neck, g, ar, al)
    assert torch.equal(E.head_apply_backward(r, ar, gr_al)[0], gr_raw)
    assert torch.equal(E.head_apply_backward(l, al, gl_al)[0], gl_raw)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("n_frame", [300, 1500])
def test_autograd_equals_the_direct_calls(n_frame, dtype):
    E = _E()
    head, thorax, consts = _recording(n_frame, dtype)
    head0, thorax0, consts0 = _cuda(head), _cuda(thorax), _cuda(consts)
    aff0, counts0 = E.head_affine(head0, thorax0, consts0)
    out0 = E.head_apply(head0.float(), aff0)
    g = torch.randn((3, n_frame, 3, 2), device="cuda").transpose(-1, -2)               # non-contiguous incoming gradients
    hh = torch.randn((8, 3), device="cuda").T
    names = ("head", "thorax", "consts", "affine")
    for mask in range(1, 16):
        req = {nm: bool(mask >> i & 1) for i, nm in enumerate(names)}
        h = head0.clone().requires_grad_(req["head"])
        t = thorax0.clone().requires_grad_(req["thorax"])
        k = consts0.clone().requires_grad_(req["consts"])
        if req["affine"]:
            a = aff0.clone().requires_grad_()
            a_stats, counts = E.head_affine(h, t, k)
            outs = [E.head_apply(h.float(), a), a_stats]
        else:
            a, counts = E.head_affine(h, t, k)
            outs = [E.head_apply(h.float(), a), a]
        assert torch.equal(outs[0].detach(), out0) and torch.equal(outs[1].detach(), aff0) and torch.equal(counts, counts0)
        assert outs[1].requires_grad == (req["head"] or req["thorax"] or req["consts"]) and not counts.requires_grad
        inputs = [x for x, nm in zip((h, t, k, a), names) if req[nm]]
        used = [(o, go) for o, go in zip(outs, (g, hh)) if o.requires_grad]
        got = torch.autograd.grad([o for o, _ in used], inputs, [go for _, go in used])
        gh1, ga = E.head_apply_backward(head0.float(), aff0, g.contiguous())
        gh_s, gt_s, gk = E.head_affine_backward(head0, thorax0, consts0, aff0, hh.contiguous() if req["affine"] else ga + hh.contiguous())
        want = {"head": gh1.to(gh_s.dtype) + gh_s, "thorax": gt_s, "consts": gk, "affine": ga if req["affine"] else None}
        for x, nm in zip(got, [nm for nm in names if req[nm]]):
            assert x.dtype == want[nm].dtype and torch.equal(x, want[nm]), (mask, nm)
    h = head0.clone().requires_grad_()
    gx, = torch.autograd.grad(E.head_apply(h.float(), E.head_affine(h, thorax0, consts0)[0]).pow(2).sum(), h, create_graph=True)
    with pytest.raises(RuntimeError, match="once_differentiable"):
        gx.sum().backward()
    with torch.no_grad():                                                              # without grad: plain launches, same bits
        assert torch.equal(E.head_apply(h.float(), E.head_affine(h, thorax0, consts0)[0]), out0)


def _rotation(w):
    """(n, 3) rotation vectors -> (n, 3, 3) rotation matrices."""
    z = torch.zeros_like(w[:, 0])
    k = torch.stack([z, -w[:, 2], w[:, 1], w[:, 2], z, -w[:, 0], -w[:, 1], w[:, 0], z], dim=1).reshape(-1, 3, 3)
    return torch.linalg.matrix_exp(k)


def test_lbfgs_recovers_per_trial_rotations():
    """The raw antenna and thorax points of 3 trials x 1000 frames of the grooming recording seen through an unknown per-trial
    rotation; the rotation is fitted against the aligned head of the true one, through head_affine -> head_apply, from 0.1
    rad off about each axis.  Rotating head and thorax together leaves d, and so the stationary set, unchanged."""
    E = _E()
    head, thorax, consts = _recording(1000, np.float64)
    head_t, thorax_t, consts_t = _cuda(head), _cuda(thorax), _cuda(consts)
    w_true = 0.3 * torch.randn((3, 3), device="cuda", dtype=torch.float64, generator=torch.Generator("cuda").manual_seed(1))
    rot = lambda w, p: torch.einsum("cij,cfkj->cfki", _rotation(w), p).contiguous()

    def aligned(w):
        h = rot(w, head_t)
        return E.head_apply(h.float(), E.head_affine(h, rot(w, thorax_t), consts_t)[0])

    with torch.no_grad():
        target = aligned(w_true)
        counts_true = E.head_affine(rot(w_true, head_t), rot(w_true, thorax_t), consts_t)[1]
    w = (w_true + 0.1).clone().requires_grad_()
    opt = torch.optim.LBFGS([w], lr=1, max_iter=500, tolerance_grad=1e-12, tolerance_change=1e-15, line_search_fn="strong_wolfe")

    def closure():
        opt.zero_grad()
        loss = (aligned(w) - target).double().pow(2).sum()
        loss.backward()
        return loss

    loss0 = float(closure())
    opt.step(closure)
    loss1 = float(closure())
    err = float((w.detach() - w_true).abs().max())
    with torch.no_grad():
        counts = E.head_affine(rot(w, head_t), rot(w, thorax_t), consts_t)[1]
    print(f"LBFGS rotation fit: loss {loss0:.3e} -> {loss1:.3e}, max |w - w_true| = {err:.2e} rad, "
          f"stationary frames {counts[:, 0].tolist()}")
    _note("lbfgs max rotation error (rad)", err)
    assert torch.equal(counts, counts_true)
    assert err < 1e-5 and loss1 < 1e-8 * loss0


def test_report_ratios():
    """Prints the largest observed ratio of every bounded check of this module (run with -s)."""
    for k, v in sorted(RATIOS.items()):
        print(f"largest ratio {k}: {v:.3g}")
