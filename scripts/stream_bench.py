"""HBM-bound satellite kernels against the measured copy bandwidth (GPU box).  Prints one JSON line per kernel.

Algorithmic bytes per unit (DESIGN.md 5.3): fk 28+12+108 B/leg-frame (origin per frame), fk backward 28+108 in and 28+12
(+16 with the lengths) out, head 48+28 B/frame (+12 with a
per-frame neck), head backward 48+28 in and 48+12 out, align_apply 60+60 B/leg-frame, leg_series 60 in + 28 out, mid_quantile 4 B/element read (4 ranks x
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
# pchip resampler: the 6000 x 1000 x 7 angles of this workload from 100 Hz onto a 1 kHz grid (42e6 in, 420e6 out)
for dt, nb in ((torch.float32, 4), (torch.float64, 8)):
    a = angles.to(dt)
    n_out = n_chain * 10 * n_frame * 7
    report(f"pchip_kernel ({str(dt).split('.')[1]}, x10 upsampling of the angles tensor)", timeit(lambda: engine.pchip_resample(a, 0.01, 0.001), reps=5),
           (angles.numel() + n_out) * nb, n_out, "samples")
    del a
x = torch.empty(1 << 28, device="cuda"); y = torch.empty_like(x)
report("torch copy (reference point)", timeit(lambda: y.copy_(x)), 2 * x.numel() * 4, x.numel(), "elements")
