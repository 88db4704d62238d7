"""HBM-bound satellite kernels against the measured copy bandwidth (GPU box).  Prints one JSON line per kernel.

Algorithmic bytes per unit (DESIGN.md 5.3): fk 28+12+108 B/leg-frame (origin per frame), fk backward 28+108 in and 28+12
(+16 with the lengths) out, head 48+28 B/frame (+12 with a
per-frame neck), head backward 48+28 in and 48+12 out, head_apply backward 24+24 in and 24+32 out, pchip n+m values per block row and channel, pchip backward n+m in
and n out, align_apply 60+60 B/leg-frame, align_apply backward 60+60 in and 60+32 out, leg_affine backward 60 B read twice
(fused path; the long path writes 28 B of keys and reads them in the select's four passes and the frame sweep), leg_series 60 in + 28 out, mid_quantile 4 B/element read (4 ranks x
4 radix passes re-read the series: from L2 when it fits)."""
import json, sys
from pathlib import Path
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import numpy as np, torch
from seqikpy_b200 import engine, synthetic as S
from seqikpy_b200.batch import chain_param_table
from seqikpy_b200.kinematic_chain import KinematicChainSeq

peak = json.loads((ROOT / "MEASURED_PEAKS.json").read_text()).get("hbm_gbs", 6650.0) if (ROOT / "MEASURED_PEAKS.json").exists() else 6650.0
size, bounds, init = S.chain_constants()
chain = KinematicChainSeq(bounds, list(S.LEGS), size)


def timeit(fn, reps=10):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def report(name, ms, nbytes, units, unit_name):
    gbs = nbytes / ms / 1e6
    print(json.dumps({"kernel": name, "ms": round(ms, 4), "GB/s": round(gbs, 1), "frac_of_measured_hbm": round(gbs / peak, 3),
                      "algorithmic_bytes": nbytes, unit_name + "/s": units / ms * 1e3}), flush=True)


n_trial, n_frame = 1000, 1000
n_chain = n_trial * 6
g = torch.Generator(device="cuda").manual_seed(1)
params = torch.from_numpy(chain_param_table(chain, init, S.LEGS, n_trial)).cuda()
lb, ub = params[:, 4:11], params[:, 11:18]
angles = (lb + (ub - lb).clamp(max=6.0) * torch.rand((n_chain, 7), device="cuda", generator=g))[:, None, :].expand(n_chain, n_frame, 7).contiguous()
angles += 0.01 * torch.randn(angles.shape, device="cuda", generator=g)
origin = torch.randn((n_chain, n_frame, 3), device="cuda", generator=g)
lf = n_chain * n_frame
report("fk_kernel", timeit(lambda: engine.forward_kinematics(angles, origin, params)), lf * (28 + 12 + 108), lf, "leg-frames")
# FK backward: angles + grad_fk in (the origin is not read: FK is a translation by it), grad_angles + grad_origin out (+ grad_lengths)
grad_fk = torch.randn((n_chain, n_frame, 9, 3), device="cuda", generator=g)
report("fk_backward_kernel", timeit(lambda: engine.forward_kinematics_backward(angles, origin, params, grad_fk)),
       lf * (28 + 108 + 28 + 12), lf, "leg-frames")
report("fk_backward_kernel, with grad_lengths", timeit(lambda: engine.forward_kinematics_backward(angles, origin, params, grad_fk, want_lengths=True)),
       lf * (28 + 108 + 28 + 12 + 16), lf, "leg-frames")
# forward + VJP (angles, origin): through engine.forward_kinematics' autograd, and through torch autograd of the same FK in
# float32 torch ops (tests/model_fk.py: what a user writes without the kernel).  Bytes: those of the two kernels.
sys.path.insert(0, str(ROOT / "tests"))
import model_fk
a_req, o_req = angles.clone().requires_grad_(), origin.clone().requires_grad_()
lengths = params[:, None, :4]
report("forward_kinematics + backward through autograd (kernels)",
       timeit(lambda: torch.autograd.grad(engine.forward_kinematics(a_req, o_req, params), [a_req, o_req], grad_fk)),
       lf * (28 + 12 + 108 + 28 + 108 + 28 + 12), lf, "leg-frames")
report("float32 torch-ops FK + torch autograd VJP (reference point)",
       timeit(lambda: torch.autograd.grad(model_fk.fk(a_req, o_req, lengths), [a_req, o_req], grad_fk), reps=3),
       lf * (28 + 12 + 108 + 28 + 108 + 28 + 12), lf, "leg-frames")
del grad_fk, a_req, o_req
pose = torch.randn((n_chain, n_frame, 5, 3), device="cuda", generator=g)
aff = torch.rand((n_chain, 8), device="cuda", generator=g) + 0.5
report("align_apply_kernel", timeit(lambda: engine.align_apply(pose, aff)), lf * 120, lf, "leg-frames")
consts = torch.rand((n_chain, 4), device="cuda", generator=g) + 1.0
base = S.to_chains(torch.from_numpy(S.make_trials(range(32), n_frame)).cuda())
rec = base.repeat((n_chain + base.shape[0] - 1) // base.shape[0], 1, 1, 1)[:n_chain].contiguous()       # key points as a recording has them
report("leg_affine fused, recording-like key points", timeit(lambda: engine.leg_affine(rec, consts)), lf * 60 + n_chain * 32, lf, "leg-frames")
report("leg_affine fused, normal-random key points (wide-range series)", timeit(lambda: engine.leg_affine(pose, consts)), lf * 60 + n_chain * 32, lf, "leg-frames")
report("leg_affine three-kernel path (series + select + affine), recording-like", timeit(lambda: engine.leg_affine_unfused(rec, consts)), lf * (60 + 28 + 28), lf, "leg-frames")
# alignment backward: apply backward (pose + dL/dout in, dL/dpose + per-leg-frame dL/daffine rows out, + the frame sum), the
# statistics backward on the fused path (key points read twice, 28 scattered contributions per chain), forward + backward
# through autograd, and the same VJP through torch autograd of the alignment in float32 torch ops with torch.quantile
aff_rec = engine.leg_affine(rec, consts)
g_al = torch.randn(rec.shape, device="cuda", generator=g)
h_al = torch.randn((n_chain, 8), device="cuda", generator=g)
gp_buf = torch.zeros_like(rec)
report("align_apply_backward (tile kernel + frame sum)", timeit(lambda: engine.align_apply_backward(rec, aff_rec, g_al)), lf * (60 + 60 + 60 + 32), lf, "leg-frames")
report("leg_affine_backward fused, recording-like", timeit(lambda: engine.leg_affine_backward(rec, consts, aff_rec, h_al, grad_pose=gp_buf)),
       lf * 120 + n_chain * 32, lf, "leg-frames")
rec_req = rec.clone().requires_grad_()
report("align_apply(leg_affine) + backward through autograd (kernels)",
       timeit(lambda: torch.autograd.grad(engine.align_apply(rec_req, engine.leg_affine(rec_req, consts)), [rec_req], g_al)),
       lf * (60 + 60 + 60 + 60 + 60 + 32 + 120 + 60), lf, "leg-frames")


def torch_align(p, k):
    seg = p[:, :, 1:] - p[:, :, :-1]
    series = torch.cat([p[:, :, 0], torch.linalg.vector_norm(seg, dim=-1)], dim=-1)                     # (chain, frame, 7)
    m = torch.quantile(series, torch.tensor([0.45, 0.55], device=p.device), dim=1).mean(0)
    scale = k[:, 3] / ((m[:, 3] + m[:, 4]) + m[:, 5])
    moved = (p[:, :, 1:] - m[:, None, None, :3]) * scale[:, None, None, None] + k[:, None, None, :3]
    return torch.cat([k[:, None, None, :3].expand(-1, p.shape[1], 1, 3), moved], dim=2)


def torch_align_vjp():                                             # torch.quantile takes at most 2^24 values per call
    for c0 in range(0, n_chain, 1000):
        torch.autograd.grad(torch_align(rec_req[c0:c0 + 1000], consts[c0:c0 + 1000]), [rec_req], g_al[c0:c0 + 1000])


report("float32 torch-ops alignment (torch.quantile) + torch autograd VJP (reference point)", timeit(torch_align_vjp, reps=3),
       lf * (60 + 60 + 60 + 60 + 60 + 32 + 120 + 60), lf, "leg-frames")
del g_al, gp_buf, rec_req, aff_rec
# the long path: 600 chains x 100 000 frames (series through scratch): the recording-like chains repeated, with 1 um noise
lp = rec[:600].repeat(1, 100, 1, 1) + 1e-3 * torch.randn((600, 100 * n_frame, 5, 3), device="cuda", generator=g)
lc = consts[:lp.shape[0]].contiguous()
lf_long = lp.shape[0] * lp.shape[1]
aff_long = engine.leg_affine(lp, lc)
h_long = torch.randn((lp.shape[0], 8), device="cuda", generator=g)
gp_long = torch.zeros_like(lp)
report("leg_affine long path (600 x 100 000)", timeit(lambda: engine.leg_affine(lp, lc), reps=5), lf_long * (60 + 28 + 28), lf_long, "leg-frames")
report("leg_affine_backward long path (600 x 100 000): keys + select + frames + scatter", timeit(lambda: engine.leg_affine_backward(lp, lc, aff_long, h_long, grad_pose=gp_long), reps=5),
       lf_long * (60 + 28 + 4 * 28 + 28), lf_long, "leg-frames")
del lp, gp_long
del base
nf = n_trial * n_frame * 6
r = torch.randn((n_trial, 6 * n_frame, 2, 3), device="cuda", generator=g); l = torch.randn((n_trial, 6 * n_frame, 2, 3), device="cuda", generator=g)
neck = torch.randn((n_trial, 3), device="cuda", generator=g); rest = torch.zeros((n_trial, 2), device="cuda")
report("head_kernel", timeit(lambda: engine.head_angles(r, l, neck, rest)), nf * (48 + 28), nf, "frames")
# head-angle backward: r_head, l_head + grad_out in, grad_r_head, grad_l_head + grad_neck (per frame) out
g_head = torch.randn((n_trial, 7, 6 * n_frame), device="cuda", generator=g)
report("head_backward_kernel", timeit(lambda: engine.head_angles_backward(r, l, neck, g_head)), nf * (48 + 28 + 48 + 12), nf, "frames")
# forward + VJP (r_head, l_head): through engine.head_angles' autograd, and through torch autograd of the same angles in
# float64 torch ops (tests/model_head_torch.py).  Bytes: those of the two kernels.
r_req, l_req = r.clone().requires_grad_(), l.clone().requires_grad_()
report("head_angles + backward through autograd (kernels)",
       timeit(lambda: torch.autograd.grad(engine.head_angles(r_req, l_req, neck, rest), [r_req, l_req], g_head)),
       nf * (48 + 28 + 48 + 28 + 48), nf, "frames")
import model_head_torch
r64, l64, n64 = r.double().requires_grad_(), l.double().requires_grad_(), neck.double()[:, None]
g64 = g_head.double().permute(1, 0, 2)
report("float64 torch-ops head angles + torch autograd VJP (reference point)",
       timeit(lambda: torch.autograd.grad(model_head_torch.head_angles_torch(r64, l64, n64, 0.0, 0.0), [r64, l64], g64), reps=3),
       nf * (48 + 28 + 48 + 28 + 48), nf, "frames")
del g_head, r_req, l_req, r64, l64, n64, g64
th = torch.randn((n_trial, 6 * n_frame, 3, 3), device="cuda", generator=g); hc = torch.rand((n_trial, 5), device="cuda", generator=g) + 0.5
report("head_affine (series fp64 + radix select + affine)", timeit(lambda: engine.head_affine(r, th, hc)), nf * (24 + 36 + 20 + 20), nf, "frames")
report("head_apply_kernel", timeit(lambda: engine.head_apply(r, torch.rand((n_trial, 8), device="cuda") + 0.5)), nf * 48, nf, "frames")
# head alignment backward: apply backward (head + dL/dout in, dL/dhead + per-frame dL/daffine rows out, + the frame sum); the
# statistics backward alone (the forward's series and counts kept, as autograd keeps them): 20 B of series read per frame
# (twice on the long path, which writes and re-reads 20 B of keys), the scattered contributions per trial; forward + backward
# through autograd; and the same VJP through torch autograd of the head alignment in float32 torch ops with torch.nanquantile
aff_h, _, series_h = engine._head_affine(torch, r, th, hc, 5e-5)
counts_h = engine.head_affine(r, th, hc)[1].flatten()
g_ha = torch.randn(r.shape, device="cuda", generator=g)
h_ha = torch.randn((n_trial, 8), device="cuda", generator=g)
report("head_apply_backward (tile kernel + frame sum)", timeit(lambda: engine.head_apply_backward(r, aff_h, g_ha)), nf * (24 + 24 + 24 + 32), nf, "frames")
gh_buf, gt_buf = torch.zeros_like(r), torch.zeros_like(th)
vjp = lambda hd, t, k, a, s, c, gh, gt: engine._head_affine_vjp(torch, hd, t, k, a, h_ha[:hd.shape[0]].contiguous(), s, c, gh, gt, True, True)
report(f"head_affine_backward statistics ({n_trial} x {6 * n_frame}: long path)",
       timeit(lambda: vjp(r, th, hc, aff_h, series_h, counts_h, gh_buf, gt_buf)), nf * (20 + 20 + 20), nf, "frames")
r_f, th_f = r.view(6 * n_trial, n_frame, 2, 3), th.view(6 * n_trial, n_frame, 3, 3)       # the same frames as 1000-frame trials
hc_f = hc.repeat(6, 1)
aff_f, _, series_f = engine._head_affine(torch, r_f, th_f, hc_f, 5e-5)
counts_f = engine.head_affine(r_f, th_f, hc_f)[1].flatten()
h_ha = torch.randn((6 * n_trial, 8), device="cuda", generator=g)
report("head_affine (series fp64 + radix select + affine), 6000 x 1000", timeit(lambda: engine.head_affine(r_f, th_f, hc_f)), nf * (24 + 36 + 20 + 20), nf, "frames")
report(f"head_affine_backward statistics ({6 * n_trial} x {n_frame}: fused path)",
       timeit(lambda: vjp(r_f, th_f, hc_f, aff_f, series_f, counts_f, gh_buf.view(r_f.shape), gt_buf.view(th_f.shape))), nf * 20, nf, "frames")
r_req, th_req = r_f.clone().requires_grad_(), th_f.clone().requires_grad_()
report("head_apply(head_affine) + backward through autograd (kernels, 6000 x 1000)",
       timeit(lambda: torch.autograd.grad(engine.head_apply(r_req, engine.head_affine(r_req, th_req, hc_f)[0]), [r_req, th_req],
                                          g_ha.view(r_f.shape))),
       nf * (24 + 36 + 20 + 20 + 24 + 24 + 24 + 24 + 32 + 20 + 24 + 36), nf, "frames")


def torch_head_align(hd, t, k, thr=5e-5):
    base, tip = hd[:, :, 0], hd[:, :, 1]
    d = torch.linalg.vector_norm(base - 0.5 * (t[:, :, 0] + t[:, :, -1]), dim=-1)
    with torch.no_grad():
        dd = (d[:, 2:] - d[:, 1:-1]) - (d[:, 1:-1] - d[:, :-2])
        still = torch.cat([dd < thr, torch.zeros_like(dd[:, :2], dtype=torch.bool)], dim=1)
    nan = torch.full_like(d, float("nan"))
    series = torch.stack([torch.where(still, base[..., c], nan) for c in range(3)]
                         + [torch.where(still, d, nan), torch.linalg.vector_norm(tip - base, dim=-1)], dim=1)
    q = torch.nanquantile(series, torch.tensor([0.45, 0.55], device=hd.device), dim=2).mean(0)           # (trial, 5)
    o = q[:, None, :3]
    b = (base - o) * (k[:, 3:4] / q[:, 3:4])[:, None] + k[:, None, :3]
    tp = (tip - o) * (k[:, 4:5] / q[:, 4:5])[:, None] + k[:, None, :3]
    return torch.stack([b, tp], dim=2)


def torch_head_vjp():                                             # torch.nanquantile takes at most 2^24 values per call
    for c0 in range(0, 6 * n_trial, 3000):
        sl = slice(c0, c0 + 3000)
        torch.autograd.grad(torch_head_align(r_req[sl], th_req[sl], hc_f[sl]), [r_req, th_req], g_ha.view(r_f.shape)[sl])


report("float32 torch-ops head alignment (torch.nanquantile) + torch autograd VJP (reference point, 6000 x 1000)", timeit(torch_head_vjp, reps=3),
       nf * (24 + 36 + 20 + 20 + 24 + 24 + 24 + 24 + 32 + 20 + 24 + 36), nf, "frames")
del g_ha, gh_buf, gt_buf, r_req, th_req, series_h, series_f
# the long path: 600 trials x 100 000 frames (series and keys through scratch), normal-random key points
lh = torch.randn((600, 100000, 2, 3), device="cuda", generator=g)
lt = torch.randn((600, 100000, 3, 3), device="cuda", generator=g)
lk = hc[:600].contiguous()
nf_long = 600 * 100000
aff_l, _, series_l = engine._head_affine(torch, lh, lt, lk, 5e-5)
counts_l = engine.head_affine(lh, lt, lk)[1].flatten()
h_ha = torch.randn((600, 8), device="cuda", generator=g)
gl_h, gl_t = torch.zeros_like(lh), torch.zeros_like(lt)
report("head_affine long path (600 x 100 000)", timeit(lambda: engine.head_affine(lh, lt, lk), reps=5), nf_long * (24 + 36 + 20 + 20), nf_long, "frames")
report("head_affine_backward long path (600 x 100 000): keys + select + frames + scatter",
       timeit(lambda: vjp(lh, lt, lk, aff_l, series_l, counts_l, gl_h, gl_t), reps=5),
       nf_long * (20 + 20 + 4 * 20 + 20), nf_long, "frames")
del lh, lt, series_l, gl_h, gl_t
# pchip resampler: the 6000 x 1000 x 7 angles of this workload from 100 Hz onto a 1 kHz grid (42e6 in, 420e6 out)
for dt, nb in ((torch.float32, 4), (torch.float64, 8)):
    a = angles.to(dt)
    n_out = n_chain * 10 * n_frame * 7
    report(f"pchip_kernel ({str(dt).split('.')[1]}, x10 upsampling of the angles tensor)", timeit(lambda: engine.pchip_resample(a, 0.01, 0.001), reps=5),
           (angles.numel() + n_out) * nb, n_out, "samples")
    # backward: series + grad_out in, grad_in out ((m + 2 n) width values per block row)
    g_out = torch.randn((n_chain, 10 * n_frame, 7), device="cuda", generator=g).to(dt)
    report(f"pchip_backward_kernel ({str(dt).split('.')[1]})", timeit(lambda: engine.pchip_resample_backward(a, g_out, 0.01, 0.001), reps=5),
           (2 * angles.numel() + n_out) * nb, n_out, "samples")
    a_req = a.clone().requires_grad_()
    report(f"pchip_resample + backward through autograd ({str(dt).split('.')[1]}, kernels)",
           timeit(lambda: torch.autograd.grad(engine.pchip_resample(a_req, 0.01, 0.001), [a_req], g_out), reps=5),
           (3 * angles.numel() + 2 * n_out) * nb, n_out, "samples")
    del g_out, a_req, a
# what a user would write without the kernels: the float32 torch-ops model (tests/model_pchip.py) + torch autograd VJP,
# on the (series, sample) layout; bytes: those of the two kernels
sys.path.insert(0, str(ROOT / "tests"))
import model_pchip
a_t = angles.permute(0, 2, 1).reshape(-1, n_frame).contiguous().requires_grad_()
g_t = torch.randn((a_t.shape[0], 10 * n_frame), device="cuda", generator=g)
report("float32 torch-ops pchip + torch autograd VJP (reference point)",
       timeit(lambda: torch.autograd.grad(model_pchip.resample(a_t, 0.01, 0.001), [a_t], g_t), reps=3),
       (3 * angles.numel() + 2 * n_chain * 10 * n_frame * 7) * 4, n_chain * 10 * n_frame * 7, "samples")
del a_t, g_t
x = torch.empty(1 << 28, device="cuda"); y = torch.empty_like(x)
report("torch copy (reference point)", timeit(lambda: y.copy_(x)), 2 * x.numel() * 4, x.numel(), "elements")
