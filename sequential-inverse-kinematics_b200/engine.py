"""Tensor-level entry points: torch CUDA tensors in, torch CUDA tensors out.

This is the batched face of the hot path -- ``(trial, leg)`` chains by frames -- that the
reference-compatible classes (``LegInvKinSeq`` & co.) and ``bench.py`` both sit on.  Every
function enqueues hand-written sm_100a kernels from ``libseqik_sm100.so`` (C ABI:
include/seqik.h) on the CURRENT torch stream of the tensors' device and returns without
synchronising.  torch supplies device memory and streams only; there is no CPU fallback.

Shapes (float32, contiguous):
  pose    (n_chain, n_frame, 5, 3)   key points: ThC origin, then the targets of stages 1-4
  params  (n_chain, 32)              per-chain constants, see ``KinematicChainSeq.pack_chain_params``
  angles  (n_chain, n_frame, 7)      DOF order ThC_yaw, ThC_pitch, ThC_roll, CTr_pitch, CTr_roll, FTi_pitch, TiTa_pitch
  fk      (n_chain, n_frame, 9, 3)   joint positions of the stage-4 chain
"""
from typing import Optional, Sequence, Tuple

from . import _native as N


def _check(t, name, shape_tail, dtype=None):
    torch = N.require_cuda()
    dtype = torch.float32 if dtype is None else dtype
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise N.SeqIKNativeError(f"{name} must be a CUDA tensor (there is no CPU path)")
    if t.dtype != dtype:
        raise ValueError(f"{name} must be {dtype}, got {t.dtype}")
    if tuple(t.shape[-len(shape_tail):]) != tuple(shape_tail):
        raise ValueError(f"{name} must end in shape {tuple(shape_tail)}, got {tuple(t.shape)}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")
    return t


def stages_to_mask(stages: Sequence[int]) -> int:
    """[a..b] -> bit mask; ValueError like leg_inverse_kinematics.py:350-353."""
    stages = [int(s) for s in stages]
    if len(stages) == 0 or max(stages) > 4 or min(stages) < 1 or any(b - a != 1 for a, b in zip(stages, stages[1:])):
        raise ValueError("Maximum stage number is 4 and the list should be strictly incremental.")
    mask = 0
    for s in stages:
        mask |= 1 << (s - 1)
    return mask


def leg_solve(pose, params, affine=None, stages: Sequence[int] = (1, 2, 3, 4), want_fk: bool = True,
              angles=None, fk=None, flags: int = N.FLAG_DEFAULT, schedule: int = N.SCHED_AUTO,
              want_stats: bool = True, chains_per_warp: int = 0, frames=None, gate: int = 0, fk_layout: str = "full", trip_period: int = 0,
              block_variant: int = 0):
    """4-stage sequential IK (+FK) of every chain.  Returns (angles, fk|None, status|None, nfev|None).

    ``angles`` must be given (and is updated in place) when ``stages`` does not start at 1:
    the DOFs of the earlier stages are then read from it and frozen.  ``schedule`` / ``chains_per_warp``
    override the automatic kernel schedule (tuning and tests); results do not depend on them.
    ``frames=(t0, t1)`` solves only that frame range IN PLACE of the full-size pose/angles/fk tensors, warm-started
    from frame t0-1 of ``angles`` (t0 > 0).  Chunked calls over consecutive ranges are bit-identical to one call over
    all frames when every t0 is a multiple of 32 (the kernel re-derives sin/cos from the angles every 32 frames and at
    the first frame of a call); otherwise they agree to float32 rounding.
    ``block_variant`` (schedule 3): 0 automatic, 1 lean kernel, 2 robust kernel (replay-heavy recordings); same results.
    ``fk_layout="joints"``: ``fk`` is (n_chain, n_frame, 4, 3), the joint rows 5..8 of the full layout only (rows 0-3
    repeat the origin, row 4 repeats row 5) -- 76 instead of 136 result bytes per leg-frame.
    """
    torch = N.require_cuda()
    lib = N.load_library()
    pose = _check(pose, "pose", (5, 3))
    if pose.dim() != 4:
        raise ValueError(f"pose must be (n_chain, n_frame, 5, 3), got {tuple(pose.shape)}")
    n_chain, n_frame = int(pose.shape[0]), int(pose.shape[1])
    params = _check(params, "params", (N.CHAIN_PARAM_FLOATS,))
    if params.shape[0] != n_chain:
        raise ValueError("params must have one row per chain")
    mask = stages_to_mask(stages)
    dev = pose.device
    if angles is None:
        if not mask & 1:
            raise ValueError("stages do not start at 1: pass the angles tensor holding the earlier stages' DOFs")
        if frames is not None and int(frames[0]) > 0:
            raise ValueError("a frame range that does not start at 0 is warm-started from frame t0-1 of `angles`: "
                             "pass the angles tensor that already holds that frame")
        angles = torch.empty((n_chain, n_frame, 7), dtype=torch.float32, device=dev)
    else:
        _check(angles, "angles", (7,))
        if tuple(angles.shape) != (n_chain, n_frame, 7):
            raise ValueError("angles must be (n_chain, n_frame, 7)")
    if fk_layout not in ("full", "joints"):
        raise ValueError(f"fk_layout must be 'full' or 'joints', got {fk_layout!r}")
    fk_rows = 9 if fk_layout == "full" else 4
    if want_fk and fk is None:
        fk = torch.empty((n_chain, n_frame, fk_rows, 3), dtype=torch.float32, device=dev)
    if fk is not None:
        _check(fk, "fk", (fk_rows, 3))
        if tuple(fk.shape[:2]) != (n_chain, n_frame):
            raise ValueError(f"fk must be (n_chain, n_frame, {fk_rows}, 3)")
    if affine is not None:
        _check(affine, "affine", (8,))
    status = torch.empty((n_chain,), dtype=torch.int32, device=dev) if want_stats else None
    nfev = torch.empty((n_chain, 4), dtype=torch.int32, device=dev) if want_stats else None
    t0, t1 = (0, n_frame) if frames is None else (int(frames[0]), int(frames[1]))
    if not 0 <= t0 <= t1 <= n_frame:
        raise ValueError(f"frames {frames} outside [0, {n_frame}]")
    if t0 > 0 and not mask & 1:
        raise ValueError("a frame range that does not start at 0 needs stages starting at 1")
    fk_floats = 3 * fk_rows
    p_fk = 0 if fk is None else fk.data_ptr() + 4 * fk_floats * t0
    warm = 0 if t0 == 0 else angles.data_ptr() + 4 * 7 * (t0 - 1)
    with torch.cuda.device(dev):
        rc = lib.seqik_leg_solve_f32(
            pose.data_ptr() + 4 * 15 * t0, n_frame * 15, 15, N.ptr(affine), N.ptr(params),
            angles.data_ptr() + 4 * 7 * t0, n_frame * 7, 7, p_fk, n_frame * fk_floats, fk_floats,
            warm, n_frame * 7,
            N.ptr(status), N.ptr(nfev), n_chain, t1 - t0, mask,
            (flags & 0xFF) | ((schedule & 0xF) << N.FLAG_SCHED_SHIFT) | ((chains_per_warp & 0x3F) << 12) | ((gate & 0xF) << 21) | ((trip_period & 7) << 25)
            | (N.FLAG_FK_JOINTS if fk_layout == "joints" else 0) | ((block_variant & 3) << 28),
            N.stream_ptr(torch, dev))
    N.check(rc, "seqik_leg_solve_f32")
    return angles, fk, status, nfev


def leg_solve_generic(pose, params, target_row: int = -1, want_fk: bool = True, warm=None, want_stats: bool = True,
                      chains_per_warp: int = 0, schedule: int = 0):
    """Generic single-target leg IK (LegInvKinGeneric): pose (n_chain, n_frame, k, 3) with the ThC at row 0 and the end
    effector at ``target_row`` (default: the last row, like the reference); params (n_chain, 32) from
    ``KinematicChainGeneric.pack_chain_params``.  float32 tensors run the FP32 kernel, float64 tensors the FP64 one
    (data and device arithmetic; see include/seqik.h).  Returns (angles (n_chain, n_frame, 7) in GENERIC chain order --
    ThC_roll, ThC_yaw, ThC_pitch, CTr_pitch, CTr_roll, FTi_pitch, TiTa_pitch --, fk (n_chain, n_frame, 9, 3) | None,
    status | None, nfev | None).  ``warm`` (n_chain, 7) replaces the seeds of ``params``.
    ``schedule``: 0 automatic (2 while the batch is resident at once, else 1), 1 one lane per chain (the host-buildable form), 2 eight lanes per chain (a joint per
    lane, sums by butterfly shuffles: same iteration, different summation order).  ``chains_per_warp``: tuning / tests
    (1..32 for schedule 1, capped at 4 for schedule 2); results do not depend on it."""
    torch = N.require_cuda()
    lib = N.load_library()
    if not isinstance(pose, torch.Tensor) or pose.dim() != 4 or pose.shape[-1] != 3:
        raise ValueError("pose must be a (n_chain, n_frame, k, 3) tensor")
    dtype = pose.dtype
    if dtype not in (torch.float32, torch.float64):
        raise ValueError(f"pose must be float32 or float64, got {dtype}")
    k = int(pose.shape[2])
    pose = _check(pose, "pose", (k, 3), dtype)
    row = target_row if target_row >= 0 else k + target_row
    if not 1 <= row < k:
        raise ValueError(f"target_row {target_row} outside the {k} key points (row 0 is the origin)")
    n_chain, n_frame = int(pose.shape[0]), int(pose.shape[1])
    params = _check(params, "params", (N.CHAIN_PARAM_FLOATS,), dtype)
    if params.shape[0] != n_chain:
        raise ValueError("params must have one row per chain")
    dev = pose.device
    if warm is not None:
        warm = _check(warm, "warm", (7,), dtype)
        if warm.shape[0] != n_chain:
            raise ValueError("warm must be (n_chain, 7)")
    angles = torch.empty((n_chain, n_frame, 7), dtype=dtype, device=dev)
    fk = torch.empty((n_chain, n_frame, 9, 3), dtype=dtype, device=dev) if want_fk else None
    status = torch.empty((n_chain,), dtype=torch.int32, device=dev) if want_stats else None
    nfev = torch.empty((n_chain,), dtype=torch.int32, device=dev) if want_stats else None
    fn = lib.seqik_leg_solve_generic_f32 if dtype == torch.float32 else lib.seqik_leg_solve_generic_f64
    with torch.cuda.device(dev):
        rc = fn(pose.data_ptr(), n_frame * k * 3, k * 3, row, N.ptr(params),
                angles.data_ptr(), n_frame * 7, 7, N.ptr(fk), n_frame * 27, 27,
                N.ptr(warm), 7, N.ptr(status), N.ptr(nfev), n_chain, n_frame, ((chains_per_warp & 0x3F) << 12) | ((schedule & 0xF) << N.FLAG_SCHED_SHIFT),
                N.stream_ptr(torch, dev))
    N.check(rc, "seqik_leg_solve_generic")
    return angles, fk, status, nfev


def _fk_inputs(angles, origin, params):
    """Checks of the FK inputs -> (n_chain, n_frame, origin frame stride)."""
    angles = _check(angles, "angles", (7,))
    n_chain, n_frame = int(angles.shape[0]), int(angles.shape[1])
    origin = _check(origin, "origin", (3,))
    params = _check(params, "params", (N.CHAIN_PARAM_FLOATS,))
    if origin.dim() == 3 and tuple(origin.shape[:2]) == (n_chain, n_frame):
        return n_chain, n_frame, 3
    if origin.dim() == 2 and origin.shape[0] == n_chain:
        return n_chain, n_frame, 0
    raise ValueError("origin must be (n_chain, n_frame, 3) or (n_chain, 3)")


def forward_kinematics(angles, origin, params):
    """angles (n_chain, n_frame, 7) + origin (n_chain, n_frame, 3) or (n_chain, 3) -> fk (n_chain, n_frame, 9, 3).

    Differentiable: when grad mode is on and any input requires grad, the result carries a ``grad_fn`` whose backward is
    the ``seqik_fk_backward_f32`` kernel (see ``forward_kinematics_backward``).  ``params`` then gets an (n_chain, 32)
    gradient with the segment lengths' gradients in columns 0-3 and zeros elsewhere (no other entry enters FK); an
    (n_chain, 3) origin gets the sum over frames.  First derivatives only: a second backward raises.  Without inputs that
    require grad the call is the plain kernel launch."""
    torch = N.require_cuda()
    if torch.is_grad_enabled() and any(isinstance(t, torch.Tensor) and t.requires_grad for t in (angles, origin, params)):
        return _fk_function().apply(angles, origin, params)
    return _forward_kinematics(torch, angles, origin, params)


def _forward_kinematics(torch, angles, origin, params):
    lib = N.load_library()
    n_chain, n_frame, stride = _fk_inputs(angles, origin, params)
    fk = torch.empty((n_chain, n_frame, 9, 3), dtype=torch.float32, device=angles.device)
    with torch.cuda.device(angles.device):
        rc = lib.seqik_fk_f32(N.ptr(angles), N.ptr(origin), stride, N.ptr(params), N.ptr(fk), n_chain, n_frame,
                              N.stream_ptr(torch, angles.device))
    N.check(rc, "seqik_fk_f32")
    return fk


def forward_kinematics_backward(angles, origin, params, grad_fk, want_origin: bool = True, want_lengths: bool = False):
    """Vector-Jacobian product of ``forward_kinematics``: grad_fk (n_chain, n_frame, 9, 3) = dL/dfk ->
    (grad_angles (n_chain, n_frame, 7), grad_origin (n_chain, n_frame, 3) | None, grad_lengths (n_chain, n_frame, 4) | None),
    all per leg-frame: grad_origin is per frame also for an (n_chain, 3) origin, and grad_lengths holds each frame's
    contribution to dL/dparams[:, 0:4].  Sum over frames where the input is shared.  The summation order of grad_origin is
    that of include/seqik.h."""
    torch = N.require_cuda()
    lib = N.load_library()
    n_chain, n_frame, stride = _fk_inputs(angles, origin, params)
    grad_fk = _check(grad_fk, "grad_fk", (9, 3))
    if tuple(grad_fk.shape) != (n_chain, n_frame, 9, 3):
        raise ValueError(f"grad_fk must be ({n_chain}, {n_frame}, 9, 3), got {tuple(grad_fk.shape)}")
    dev = angles.device
    grad_angles = torch.empty((n_chain, n_frame, 7), dtype=torch.float32, device=dev)
    grad_origin = torch.empty((n_chain, n_frame, 3), dtype=torch.float32, device=dev) if want_origin else None
    grad_lengths = torch.empty((n_chain, n_frame, 4), dtype=torch.float32, device=dev) if want_lengths else None
    with torch.cuda.device(dev):
        rc = lib.seqik_fk_backward_f32(N.ptr(angles), N.ptr(origin), stride, N.ptr(params), N.ptr(grad_fk), N.ptr(grad_angles),
                                       N.ptr(grad_origin), N.ptr(grad_lengths), n_chain, n_frame, N.stream_ptr(torch, dev))
    N.check(rc, "seqik_fk_backward_f32")
    return grad_angles, grad_origin, grad_lengths


_FK_FUNCTION = None


def _fk_function():
    """The torch.autograd.Function of forward_kinematics (built on first use: torch is imported lazily)."""
    global _FK_FUNCTION
    if _FK_FUNCTION is not None:
        return _FK_FUNCTION
    import torch
    from torch.autograd.function import once_differentiable

    class ForwardKinematics(torch.autograd.Function):
        @staticmethod
        def forward(ctx, angles, origin, params):
            ctx.save_for_backward(angles, origin, params)
            return _forward_kinematics(torch, angles, origin, params)

        @staticmethod
        @once_differentiable
        def backward(ctx, grad_fk):
            angles, origin, params = ctx.saved_tensors
            need_angles, need_origin, need_params = ctx.needs_input_grad
            ga, go, gl = forward_kinematics_backward(angles, origin, params, grad_fk.contiguous(),
                                                     want_origin=need_origin, want_lengths=need_params)
            if need_origin and origin.dim() == 2:
                go = go.sum(dim=1)
            g_params = None
            if need_params:
                g_params = torch.zeros_like(params)
                g_params[:, :4] = gl.sum(dim=1)
            return (ga if need_angles else None), go, g_params

    _FK_FUNCTION = ForwardKinematics
    return _FK_FUNCTION


def _head_inputs(r_head, l_head, neck, affine_r, affine_l):
    """Checks of the head-angle inputs -> (n_trial, n_frame, neck stride)."""
    r_head = _check(r_head, "r_head", (2, 3))
    l_head = _check(l_head, "l_head", (2, 3))
    if r_head.dim() != 4 or r_head.shape != l_head.shape:
        raise ValueError("r_head and l_head must both be (n_trial, n_frame, 2, 3)")
    n_trial, n_frame = int(r_head.shape[0]), int(r_head.shape[1])
    neck = _check(neck, "neck", (3,))
    if neck.dim() == 3 and tuple(neck.shape[:2]) == (n_trial, n_frame):
        stride = 3
    elif neck.dim() == 2 and neck.shape[0] == n_trial:
        stride = 0
    else:
        raise ValueError("neck must be (n_trial, n_frame, 3) or (n_trial, 3)")
    if affine_r is not None:
        _check(affine_r, "affine_r", (8,))
        _check(affine_l, "affine_l", (8,))
    return n_trial, n_frame, stride


def head_angles(r_head, l_head, neck, rest, affine_r=None, affine_l=None):
    """r_head, l_head (n_trial, n_frame, 2, 3); neck (n_trial, n_frame, 3) or (n_trial, 3); rest (n_trial, 2)
    -> (n_trial, 7, n_frame): head roll, pitch, yaw, antenna yaw L, pitch L, yaw R, pitch R.

    Differentiable: when grad mode is on and ``r_head``, ``l_head``, ``neck`` or ``rest`` requires grad, the result
    carries a ``grad_fn`` whose backward is the ``seqik_head_angles_backward_f32`` kernel (see ``head_angles_backward``).
    An (n_trial, 3) neck gets the sum over frames; ``rest`` gets dL/drest[:, 0] = the sum of dL/dhead_pitch and
    dL/drest[:, 1] = minus the sums of dL/dantenna_pitch L and R.  The affine rows are constants of the backward: one
    that requires grad raises ValueError.  To differentiate through the head alignment, align first and pass no rows:
    ``head_angles(head_apply(raw, head_affine(raw, thorax, consts)[0]), ...)``.  First derivatives only: a second backward
    raises.  Without inputs that require grad the call is the plain kernel launch."""
    torch = N.require_cuda()
    if torch.is_grad_enabled():
        if any(isinstance(t, torch.Tensor) and t.requires_grad for t in (affine_r, affine_l)):
            raise ValueError("head_angles: the affine rows have no gradient; pass them detached")
        if any(isinstance(t, torch.Tensor) and t.requires_grad for t in (r_head, l_head, neck, rest)):
            return _head_function().apply(r_head, l_head, neck, rest, affine_r, affine_l)
    return _head_angles(torch, r_head, l_head, neck, rest, affine_r, affine_l)


def _head_angles(torch, r_head, l_head, neck, rest, affine_r, affine_l):
    lib = N.load_library()
    n_trial, n_frame, stride = _head_inputs(r_head, l_head, neck, affine_r, affine_l)
    rest = _check(rest, "rest", (2,))
    out = torch.empty((n_trial, 7, n_frame), dtype=torch.float32, device=r_head.device)
    with torch.cuda.device(r_head.device):
        rc = lib.seqik_head_angles_f32(N.ptr(r_head), N.ptr(l_head), N.ptr(neck), stride, N.ptr(affine_r), N.ptr(affine_l),
                                       N.ptr(rest), N.ptr(out), n_trial, n_frame, N.stream_ptr(torch, r_head.device))
    N.check(rc, "seqik_head_angles_f32")
    return out


def head_angles_backward(r_head, l_head, neck, grad_out, affine_r=None, affine_l=None, want_neck: bool = True):
    """Vector-Jacobian product of ``head_angles``: grad_out (n_trial, 7, n_frame) = dL/dangles ->
    (grad_r_head (n_trial, n_frame, 2, 3), grad_l_head (n_trial, n_frame, 2, 3), grad_neck (n_trial, n_frame, 3) | None).
    grad_neck is per frame also for an (n_trial, 3) neck: sum over frames there.  The gradients are those of the points
    as passed: with affine rows, the aligned points' gradients times the rows' scales (include/seqik.h).  The rest angles
    are additive constants and the affine rows get no gradient."""
    torch = N.require_cuda()
    lib = N.load_library()
    n_trial, n_frame, stride = _head_inputs(r_head, l_head, neck, affine_r, affine_l)
    grad_out = _check(grad_out, "grad_out", (n_frame,))
    if tuple(grad_out.shape) != (n_trial, 7, n_frame):
        raise ValueError(f"grad_out must be ({n_trial}, 7, {n_frame}), got {tuple(grad_out.shape)}")
    dev = r_head.device
    grad_r = torch.empty((n_trial, n_frame, 2, 3), dtype=torch.float32, device=dev)
    grad_l = torch.empty((n_trial, n_frame, 2, 3), dtype=torch.float32, device=dev)
    grad_neck = torch.empty((n_trial, n_frame, 3), dtype=torch.float32, device=dev) if want_neck else None
    with torch.cuda.device(dev):
        rc = lib.seqik_head_angles_backward_f32(N.ptr(r_head), N.ptr(l_head), N.ptr(neck), stride, N.ptr(affine_r),
                                                N.ptr(affine_l), N.ptr(grad_out), N.ptr(grad_r), N.ptr(grad_l),
                                                N.ptr(grad_neck), n_trial, n_frame, N.stream_ptr(torch, dev))
    N.check(rc, "seqik_head_angles_backward_f32")
    return grad_r, grad_l, grad_neck


_HEAD_FUNCTION = None


def _head_function():
    """The torch.autograd.Function of head_angles (built on first use: torch is imported lazily)."""
    global _HEAD_FUNCTION
    if _HEAD_FUNCTION is not None:
        return _HEAD_FUNCTION
    import torch
    from torch.autograd.function import once_differentiable

    class HeadAngles(torch.autograd.Function):
        @staticmethod
        def forward(ctx, r_head, l_head, neck, rest, affine_r, affine_l):
            ctx.save_for_backward(r_head, l_head, neck, affine_r, affine_l)
            return _head_angles(torch, r_head, l_head, neck, rest, affine_r, affine_l)

        @staticmethod
        @once_differentiable
        def backward(ctx, grad_out):
            r_head, l_head, neck, affine_r, affine_l = ctx.saved_tensors
            need_r, need_l, need_neck, need_rest = ctx.needs_input_grad[:4]
            grad_out = grad_out.contiguous()
            gr = gl = gn = g_rest = None
            if need_r or need_l or need_neck:
                gr, gl, gn = head_angles_backward(r_head, l_head, neck, grad_out, affine_r, affine_l, want_neck=need_neck)
                if need_neck and neck.dim() == 2:
                    gn = gn.sum(dim=1)
            if need_rest:
                g_rest = torch.stack([grad_out[:, 1].sum(-1), -(grad_out[:, 4] + grad_out[:, 6]).sum(-1)], dim=1)
            return (gr if need_r else None), (gl if need_l else None), gn, g_rest, None, None

    _HEAD_FUNCTION = HeadAngles
    return _HEAD_FUNCTION


def mid_quantile(series, counts=None):
    """Mean of the 0.45 and 0.55 quantiles of each row of ``series`` (n_series, n) -> (n_series,)."""
    torch = N.require_cuda()
    lib = N.load_library()
    if series.dim() != 2:
        raise ValueError("series must be (n_series, n)")
    series = _check(series, "series", (series.shape[-1],))
    n_series, n = int(series.shape[0]), int(series.shape[1])
    if counts is not None:
        counts = _check(counts, "counts", (n_series,), torch.int32)
    out = torch.empty((n_series,), dtype=torch.float32, device=series.device)
    with torch.cuda.device(series.device):
        rc = lib.seqik_mid_quantile_f32(N.ptr(series), N.ptr(counts), 0, N.ptr(out), n_series, n,
                                        N.stream_ptr(torch, series.device))
    N.check(rc, "seqik_mid_quantile_f32")
    return out


def leg_affine(pose, consts, include_claw: bool = False):
    """AlignPose.align_leg statistics: pose (n_chain, n_frame, 5, 3), consts (n_chain, 4) = template coxa xyz + model
    length -> affine (n_chain, 8) = (fixed_coxa xyz, scale, template xyz, 0).

    Differentiable: when grad mode is on and ``pose`` or ``consts`` requires grad, the result carries a ``grad_fn`` whose
    backward is the ``seqik_leg_affine_backward_f32`` kernel (see ``leg_affine_backward``): each mid-quantile passes its
    gradient to the key points of the frames that hold its four order statistics (ties: the first frames in frame order,
    include/seqik.h).  First derivatives only: a second backward raises.  Without inputs that require grad the call is the
    plain kernel launch."""
    torch = N.require_cuda()
    if torch.is_grad_enabled() and any(isinstance(t, torch.Tensor) and t.requires_grad for t in (pose, consts)):
        return _align_functions()[0].apply(pose, consts, bool(include_claw))
    return _leg_affine(torch, pose, consts, include_claw)


def _leg_affine_inputs(pose, consts):
    pose = _check(pose, "pose", (5, 3))
    if pose.dim() != 4:
        raise ValueError(f"pose must be (n_chain, n_frame, 5, 3), got {tuple(pose.shape)}")
    consts = _check(consts, "consts", (4,))
    if consts.dim() != 2 or consts.shape[0] != pose.shape[0]:
        raise ValueError("consts must have one row per chain")
    return int(pose.shape[0]), int(pose.shape[1])


def _leg_affine(torch, pose, consts, include_claw):
    lib = N.load_library()
    pose = _check(pose, "pose", (5, 3))
    n_chain, n_frame = int(pose.shape[0]), int(pose.shape[1])
    consts = _check(consts, "consts", (4,))
    dev = pose.device
    if consts.shape[0] != n_chain:
        raise ValueError("consts must have one row per chain")
    affine = torch.empty((n_chain, 8), dtype=torch.float32, device=dev)
    # recordings of up to 1024 frames: one fused kernel, the series never exist in global memory; longer ones need them
    scratch = None if n_frame <= 1024 else torch.empty((n_chain * 7 * (n_frame + 1),), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        N.check(lib.seqik_leg_affine_from_pose_f32(N.ptr(pose), n_frame * 15, 15, N.ptr(consts), int(bool(include_claw)),
                                                   N.ptr(scratch), N.ptr(affine), n_chain, n_frame, N.stream_ptr(torch, dev)),
                "seqik_leg_affine_from_pose_f32")
    return affine


def leg_affine_backward(pose, consts, affine, grad_affine, include_claw: bool = False, grad_pose=None):
    """Vector-Jacobian product of ``leg_affine``: grad_affine (n_chain, 8) = dL/daffine -> (grad_pose (n_chain, n_frame, 5, 3),
    grad_consts (n_chain, 4)).  ``affine`` is the forward's result.  The statistics' contributions are ADDED into
    ``grad_pose`` when it is given (e.g. the output of ``align_apply_backward``; updated in place), else into zeros.  The
    frames, the tie rule and the float summation order are those of include/seqik.h: the result is deterministic."""
    torch = N.require_cuda()
    lib = N.load_library()
    n_chain, n_frame = _leg_affine_inputs(pose, consts)
    _check(affine, "affine", (8,))
    grad_affine = _check(grad_affine, "grad_affine", (8,))
    if tuple(affine.shape) != (n_chain, 8) or tuple(grad_affine.shape) != (n_chain, 8):
        raise ValueError(f"affine and grad_affine must be ({n_chain}, 8)")
    dev = pose.device
    if grad_pose is None:
        grad_pose = torch.zeros_like(pose)
    else:
        _check(grad_pose, "grad_pose", (5, 3))
        if grad_pose.shape != pose.shape:
            raise ValueError(f"grad_pose must be {tuple(pose.shape)}")
    grad_consts = torch.empty((n_chain, 4), dtype=torch.float32, device=dev)
    scratch = None if n_frame <= 1024 else torch.empty((n_chain * 7 * (n_frame + 12),), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        rc = lib.seqik_leg_affine_backward_f32(N.ptr(pose), n_frame * 15, 15, N.ptr(consts), int(bool(include_claw)), N.ptr(affine),
                                               N.ptr(grad_affine), N.ptr(grad_pose), N.ptr(grad_consts), N.ptr(scratch),
                                               n_chain, n_frame, N.stream_ptr(torch, dev))
    N.check(rc, "seqik_leg_affine_backward_f32")
    return grad_pose, grad_consts


def leg_affine_unfused(pose, consts, include_claw: bool = False):
    """The same through the three separate entry points (series, mid-quantiles, affine rows): the path of recordings longer
    than 1024 frames, kept callable at any length for tests and measurements."""
    torch = N.require_cuda()
    lib = N.load_library()
    pose = _check(pose, "pose", (5, 3))
    n_chain, n_frame = int(pose.shape[0]), int(pose.shape[1])
    consts = _check(consts, "consts", (4,))
    dev = pose.device
    series = torch.empty((n_chain * 7, n_frame), dtype=torch.float32, device=dev)
    affine = torch.empty((n_chain, 8), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        st = N.stream_ptr(torch, dev)
        N.check(lib.seqik_leg_series_f32(N.ptr(pose), n_frame * 15, 15, N.ptr(series), n_chain, n_frame, st),
                "seqik_leg_series_f32")
        stats = mid_quantile(series)
        N.check(lib.seqik_leg_affine_f32(N.ptr(stats), N.ptr(consts), int(bool(include_claw)), N.ptr(affine), n_chain, st),
                "seqik_leg_affine_f32")
    return affine


def align_apply(pose, affine):
    """The affine map of align_leg as a standalone pass -> aligned pose (n_chain, n_frame, 5, 3).

    Differentiable: when grad mode is on and ``pose`` or ``affine`` requires grad, the result carries a ``grad_fn`` whose
    backward is the ``seqik_align_apply_backward_f32`` kernel (see ``align_apply_backward``).  Composed with ``leg_affine``
    under autograd, ``align_apply(pose, leg_affine(pose, consts))`` gives the full gradient with respect to the raw key
    points.  First derivatives only: a second backward raises.  Without inputs that require grad the call is the plain
    kernel launch."""
    torch = N.require_cuda()
    if torch.is_grad_enabled() and any(isinstance(t, torch.Tensor) and t.requires_grad for t in (pose, affine)):
        return _align_functions()[1].apply(pose, affine)
    return _align_apply(torch, pose, affine)


def _align_apply(torch, pose, affine):
    lib = N.load_library()
    pose = _check(pose, "pose", (5, 3))
    affine = _check(affine, "affine", (8,))
    n_chain, n_frame = int(pose.shape[0]), int(pose.shape[1])
    out = torch.empty_like(pose)
    with torch.cuda.device(pose.device):
        rc = lib.seqik_align_apply_f32(N.ptr(pose), n_frame * 15, 15, N.ptr(affine), N.ptr(out), n_chain, n_frame,
                                       N.stream_ptr(torch, pose.device))
    N.check(rc, "seqik_align_apply_f32")
    return out


def align_apply_backward(pose, affine, grad_out, want_pose: bool = True, want_affine: bool = True):
    """Vector-Jacobian product of ``align_apply``: grad_out (n_chain, n_frame, 5, 3) = dL/dout -> (grad_pose (n_chain,
    n_frame, 5, 3) | None, grad_affine (n_chain, 8) | None).  grad_pose is aff[3] * grad_out with key point 0 at 0; grad_affine
    is the sum over frames of the kernel's per-leg-frame rows (include/seqik.h)."""
    torch = N.require_cuda()
    lib = N.load_library()
    pose = _check(pose, "pose", (5, 3))
    affine = _check(affine, "affine", (8,))
    if pose.dim() != 4 or affine.dim() != 2 or affine.shape[0] != pose.shape[0]:
        raise ValueError("pose must be (n_chain, n_frame, 5, 3) and affine (n_chain, 8)")
    grad_out = _check(grad_out, "grad_out", (5, 3))
    if grad_out.shape != pose.shape:
        raise ValueError(f"grad_out must be {tuple(pose.shape)}, got {tuple(grad_out.shape)}")
    n_chain, n_frame = int(pose.shape[0]), int(pose.shape[1])
    dev = pose.device
    grad_pose = torch.empty_like(pose) if want_pose else None
    part = torch.empty((n_chain, n_frame, 8), dtype=torch.float32, device=dev) if want_affine else None
    with torch.cuda.device(dev):
        rc = lib.seqik_align_apply_backward_f32(N.ptr(pose), n_frame * 15, 15, N.ptr(affine), N.ptr(grad_out), N.ptr(grad_pose),
                                                N.ptr(part), n_chain, n_frame, N.stream_ptr(torch, dev))
    N.check(rc, "seqik_align_apply_backward_f32")
    return grad_pose, (part.sum(dim=1) if want_affine else None)


_ALIGN_FUNCTIONS = None


def _align_functions():
    """The torch.autograd.Functions of leg_affine and align_apply (built on first use: torch is imported lazily)."""
    global _ALIGN_FUNCTIONS
    if _ALIGN_FUNCTIONS is not None:
        return _ALIGN_FUNCTIONS
    import torch
    from torch.autograd.function import once_differentiable

    class LegAffine(torch.autograd.Function):
        @staticmethod
        def forward(ctx, pose, consts, include_claw):
            affine = _leg_affine(torch, pose, consts, include_claw)
            ctx.save_for_backward(pose, consts, affine)
            ctx.include_claw = include_claw
            return affine

        @staticmethod
        @once_differentiable
        def backward(ctx, grad_affine):
            pose, consts, affine = ctx.saved_tensors
            need_pose, need_consts = ctx.needs_input_grad[:2]
            gp, gk = leg_affine_backward(pose, consts, affine, grad_affine.contiguous(), ctx.include_claw)
            return (gp if need_pose else None), (gk if need_consts else None), None

    class AlignApply(torch.autograd.Function):
        @staticmethod
        def forward(ctx, pose, affine):
            ctx.save_for_backward(pose, affine)
            return _align_apply(torch, pose, affine)

        @staticmethod
        @once_differentiable
        def backward(ctx, grad_out):
            pose, affine = ctx.saved_tensors
            need_pose, need_affine = ctx.needs_input_grad
            return align_apply_backward(pose, affine, grad_out.contiguous(), want_pose=need_pose, want_affine=need_affine)

    _ALIGN_FUNCTIONS = (LegAffine, AlignApply)
    return _ALIGN_FUNCTIONS


def head_affine(head, thorax, consts, threshold: float = 5e-5):
    """AlignPose.align_head statistics: head (n_trial, n_frame, 2, 3), thorax (n_trial, n_frame, k, 3) -- both float32
    or both float64 --, consts (n_trial, 5) float32 = template antenna base xyz, Antenna_mid_thorax, Antenna
    -> affine (n_trial, 8) = (origin xyz, scale_base, template xyz, scale_tip), counts (n_trial, 5).

    Differentiable: when grad mode is on and ``head``, ``thorax`` or ``consts`` requires grad, ``affine`` carries a
    ``grad_fn`` whose backward is the ``seqik_head_affine_backward`` kernel (see ``head_affine_backward``); the gradients
    come back in the inputs' dtype and ``counts`` is not differentiable.  The stationary frames are held fixed as the
    forward chose them, and each mid-quantile passes its gradient to the frames that hold its four order statistics
    (ties: the first frames in frame order, include/seqik.h).  The differentiable route to the head angles is
    ``head_angles(head_apply(raw, head_affine(raw, thorax, consts)[0]), ...)``.  First derivatives only: a second
    backward raises.  Without inputs that require grad the call is the plain kernel launches."""
    torch = N.require_cuda()
    if torch.is_grad_enabled() and any(isinstance(t, torch.Tensor) and t.requires_grad for t in (head, thorax, consts)):
        return _head_align_functions()[0].apply(head, thorax, consts, float(threshold))
    affine, counts, _ = _head_affine(torch, head, thorax, consts, threshold)
    return affine, counts


def _head_affine_inputs(torch, head, thorax, consts):
    dtype = head.dtype
    if dtype not in (torch.float32, torch.float64) or thorax.dtype != dtype:
        raise ValueError("head and thorax must both be float32 or both float64")
    head = _check(head, "head", (2, 3), dtype)
    n_trial, n_frame = int(head.shape[0]), int(head.shape[1])
    if thorax.dim() != 4 or tuple(thorax.shape[:2]) != (n_trial, n_frame):
        raise ValueError("thorax must be (n_trial, n_frame, n_kp, 3)")
    thorax = _check(thorax, "thorax", (3,), dtype)
    _check(consts, "consts", (5,))
    return n_trial, n_frame


def _head_series(torch, lib, head, thorax, threshold, n_trial, n_frame):
    dev = head.device
    series = torch.empty((n_trial * 5, n_frame), dtype=torch.float32, device=dev)
    counts = torch.empty((n_trial * 5,), dtype=torch.int32, device=dev)
    fn = lib.seqik_head_series_f32 if head.dtype == torch.float32 else lib.seqik_head_series_f64
    with torch.cuda.device(dev):
        N.check(fn(N.ptr(head), N.ptr(thorax), int(thorax.shape[2]), float(threshold), N.ptr(series),
                   N.ptr(counts), n_trial, n_frame, N.stream_ptr(torch, dev)), "seqik_head_series")
    return series, counts


def _head_affine(torch, head, thorax, consts, threshold):
    """-> (affine (n_trial, 8), counts (n_trial, 5), series (n_trial * 5, n_frame)): the series and counts are what the
    backward needs."""
    lib = N.load_library()
    n_trial, n_frame = _head_affine_inputs(torch, head, thorax, consts)
    dev = head.device
    series, counts = _head_series(torch, lib, head, thorax, threshold, n_trial, n_frame)
    affine = torch.empty((n_trial, 8), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        stats = mid_quantile(series, counts)
        N.check(lib.seqik_head_affine_f32(N.ptr(stats), N.ptr(consts), N.ptr(affine), n_trial, N.stream_ptr(torch, dev)),
                "seqik_head_affine_f32")
    return affine, counts.view(n_trial, 5), series


def _head_affine_vjp(torch, head, thorax, consts, affine, grad_affine, series, counts, grad_head, grad_thorax,
                     want_thorax, want_consts):
    lib = N.load_library()
    n_trial, n_frame = _head_affine_inputs(torch, head, thorax, consts)
    _check(affine, "affine", (8,))
    grad_affine = _check(grad_affine, "grad_affine", (8,))
    if tuple(affine.shape) != (n_trial, 8) or tuple(grad_affine.shape) != (n_trial, 8):
        raise ValueError(f"affine and grad_affine must be ({n_trial}, 8)")
    dev, dtype = head.device, head.dtype
    if grad_head is None:
        grad_head = torch.zeros_like(head)
    elif grad_head.shape != head.shape:
        raise ValueError(f"grad_head must be {tuple(head.shape)}")
    else:
        _check(grad_head, "grad_head", (2, 3), dtype)
    if not want_thorax:
        grad_thorax = None
    elif grad_thorax is None:
        grad_thorax = torch.zeros_like(thorax)
    elif grad_thorax.shape != thorax.shape:
        raise ValueError(f"grad_thorax must be {tuple(thorax.shape)}")
    else:
        _check(grad_thorax, "grad_thorax", (3,), dtype)
    grad_consts = torch.empty((n_trial, 5), dtype=torch.float32, device=dev) if want_consts else None
    scratch = None if n_frame <= 1024 else torch.empty((n_trial * 5 * (n_frame + 12),), dtype=torch.int32, device=dev)
    fn = lib.seqik_head_affine_backward_f32 if dtype == torch.float32 else lib.seqik_head_affine_backward_f64
    with torch.cuda.device(dev):
        rc = fn(N.ptr(head), N.ptr(thorax), int(thorax.shape[2]), N.ptr(series), N.ptr(counts), N.ptr(consts), N.ptr(affine),
                N.ptr(grad_affine), N.ptr(grad_head), N.ptr(grad_thorax), N.ptr(grad_consts), N.ptr(scratch), n_trial, n_frame,
                N.stream_ptr(torch, dev))
    N.check(rc, "seqik_head_affine_backward")
    return grad_head, grad_thorax, grad_consts


def head_affine_backward(head, thorax, consts, affine, grad_affine, threshold: float = 5e-5, grad_head=None, grad_thorax=None):
    """Vector-Jacobian product of ``head_affine``: grad_affine (n_trial, 8) = dL/daffine -> (grad_head (n_trial, n_frame, 2, 3),
    grad_thorax (n_trial, n_frame, k, 3), grad_consts (n_trial, 5)), the first two in the inputs' dtype.  ``affine`` is the
    forward's result; the series and the stationary frames are recomputed with ``threshold``.  The statistics'
    contributions are ADDED into ``grad_head`` / ``grad_thorax`` when they are given (e.g. the output of
    ``head_apply_backward``; updated in place), else into zeros.  The frames, the tie rule and the float summation order
    are those of include/seqik.h: the result is deterministic."""
    torch = N.require_cuda()
    lib = N.load_library()
    n_trial, n_frame = _head_affine_inputs(torch, head, thorax, consts)
    series, counts = _head_series(torch, lib, head, thorax, threshold, n_trial, n_frame)
    return _head_affine_vjp(torch, head, thorax, consts, affine, grad_affine, series, counts, grad_head, grad_thorax, True, True)


def head_apply(head, affine):
    """The affine map of align_head (alignment.py:547-553) as a standalone pass: head (n_trial, n_frame, 2, 3) float32,
    affine (n_trial, 8) = (origin xyz, scale_base, template xyz, scale_tip) -> aligned head (n_trial, n_frame, 2, 3) with
    base' = (base - origin) * scale_base + template and tip' = (tip - origin) * scale_tip + template.

    Differentiable: when grad mode is on and ``head`` or ``affine`` requires grad, the result carries a ``grad_fn`` whose
    backward is the ``seqik_head_apply_backward_f32`` kernel (see ``head_apply_backward``).  Composed with ``head_affine``
    under autograd, ``head_apply(head, head_affine(head, thorax, consts)[0])`` gives the full gradient with respect to the
    raw antenna points, the thorax and the consts.  First derivatives only: a second backward raises.  Without inputs that
    require grad the call is the plain kernel launch."""
    torch = N.require_cuda()
    if torch.is_grad_enabled() and any(isinstance(t, torch.Tensor) and t.requires_grad for t in (head, affine)):
        return _head_align_functions()[1].apply(head, affine)
    return _head_apply(torch, head, affine)


def _head_apply(torch, head, affine):
    lib = N.load_library()
    head = _check(head, "head", (2, 3))
    affine = _check(affine, "affine", (8,))
    n_trial, n_frame = int(head.shape[0]), int(head.shape[1])
    out = torch.empty_like(head)
    with torch.cuda.device(head.device):
        rc = lib.seqik_head_apply_f32(N.ptr(head), N.ptr(affine), N.ptr(out), n_trial, n_frame, N.stream_ptr(torch, head.device))
    N.check(rc, "seqik_head_apply_f32")
    return out


def head_apply_backward(head, affine, grad_out, want_head: bool = True, want_affine: bool = True):
    """Vector-Jacobian product of ``head_apply``: grad_out (n_trial, n_frame, 2, 3) = dL/dout -> (grad_head (n_trial, n_frame,
    2, 3) | None, grad_affine (n_trial, 8) | None).  grad_head is scale_base * grad_out for the bases and scale_tip * grad_out
    for the tips; grad_affine is the sum over frames of the kernel's per-frame rows (include/seqik.h)."""
    torch = N.require_cuda()
    lib = N.load_library()
    head = _check(head, "head", (2, 3))
    affine = _check(affine, "affine", (8,))
    if head.dim() != 4 or affine.dim() != 2 or affine.shape[0] != head.shape[0]:
        raise ValueError("head must be (n_trial, n_frame, 2, 3) and affine (n_trial, 8)")
    grad_out = _check(grad_out, "grad_out", (2, 3))
    if grad_out.shape != head.shape:
        raise ValueError(f"grad_out must be {tuple(head.shape)}, got {tuple(grad_out.shape)}")
    n_trial, n_frame = int(head.shape[0]), int(head.shape[1])
    dev = head.device
    grad_head = torch.empty_like(head) if want_head else None
    part = torch.empty((n_trial, n_frame, 8), dtype=torch.float32, device=dev) if want_affine else None
    with torch.cuda.device(dev):
        rc = lib.seqik_head_apply_backward_f32(N.ptr(head), N.ptr(affine), N.ptr(grad_out), N.ptr(grad_head), N.ptr(part),
                                               n_trial, n_frame, N.stream_ptr(torch, dev))
    N.check(rc, "seqik_head_apply_backward_f32")
    return grad_head, (part.sum(dim=1) if want_affine else None)


_HEAD_ALIGN_FUNCTIONS = None


def _head_align_functions():
    """The torch.autograd.Functions of head_affine and head_apply (built on first use: torch is imported lazily)."""
    global _HEAD_ALIGN_FUNCTIONS
    if _HEAD_ALIGN_FUNCTIONS is not None:
        return _HEAD_ALIGN_FUNCTIONS
    import torch
    from torch.autograd.function import once_differentiable

    class HeadAffine(torch.autograd.Function):
        @staticmethod
        def forward(ctx, head, thorax, consts, threshold):
            affine, counts, series = _head_affine(torch, head, thorax, consts, threshold)
            ctx.save_for_backward(head, thorax, consts, affine, series, counts)
            ctx.mark_non_differentiable(counts)
            return affine, counts

        @staticmethod
        @once_differentiable
        def backward(ctx, grad_affine, _grad_counts):
            head, thorax, consts, affine, series, counts = ctx.saved_tensors
            need_head, need_thorax, need_consts = ctx.needs_input_grad[:3]
            gh, gt, gk = _head_affine_vjp(torch, head, thorax, consts, affine, grad_affine.contiguous(), series, counts,
                                          None, None, need_thorax, need_consts)
            return (gh if need_head else None), gt, gk, None

    class HeadApply(torch.autograd.Function):
        @staticmethod
        def forward(ctx, head, affine):
            ctx.save_for_backward(head, affine)
            return _head_apply(torch, head, affine)

        @staticmethod
        @once_differentiable
        def backward(ctx, grad_out):
            head, affine = ctx.saved_tensors
            need_head, need_affine = ctx.needs_input_grad
            return head_apply_backward(head, affine, grad_out.contiguous(), want_head=need_head, want_affine=need_affine)

    _HEAD_ALIGN_FUNCTIONS = (HeadAffine, HeadApply)
    return _HEAD_ALIGN_FUNCTIONS


def pchip_resample(series, original_ts: float, new_ts: float):
    """Shape-preserving cubic resampling (``utils.interpolate_signal``, reference utils.py:332-349) of uniformly sampled
    series on the device: ``series`` (n_block, n, width) -- e.g. an angles tensor (n_chain, n_frame, 7) -- or (n_series, n);
    float32 or float64.  Returns the same layout with ``m = len(np.arange(0, n * original_ts, new_ts))`` samples.
    Like the reference's retry (utils.py:343-347: ``signal[np.isinf(signal)] = 0; signal[-1] = 0`` on the WHOLE array of one
    call), +-inf samples are zeroed and, in every block that held one, the last sample of ALL its channels; NaN raises.

    Differentiable: when grad mode is on and ``series`` requires grad, the result carries a ``grad_fn`` whose backward is
    the ``seqik_pchip_resample_backward`` kernel (see ``pchip_resample_backward``); the samples the forward replaced by 0
    get gradient 0.  First derivatives only: a second backward raises.  Without grad the call is the plain kernel launch."""
    torch = N.require_cuda()
    if torch.is_grad_enabled() and isinstance(series, torch.Tensor) and series.requires_grad:
        return _pchip_function().apply(series, original_ts, new_ts)
    x, flat, m, _ = _pchip_inputs(torch, series, original_ts, new_ts)
    n_block, n, width = (int(v) for v in x.shape)
    lib = N.load_library()
    out = torch.empty((n_block, m, width), dtype=x.dtype, device=x.device)
    fn = lib.seqik_pchip_resample_f32 if x.dtype == torch.float32 else lib.seqik_pchip_resample_f64
    with torch.cuda.device(x.device):
        rc = fn(x.data_ptr(), out.data_ptr(), n_block, n, m, width, float(original_ts), float(new_ts),
                N.stream_ptr(torch, x.device))
    N.check(rc, "seqik_pchip_resample")
    return out.squeeze(-1) if flat else out


def _pchip_inputs(torch, series, original_ts, new_ts):
    """Checks of the resampler's input -> (the series as the kernel reads it (n_block, n, width), whether it was 2-D, m,
    the mask of the samples replaced by 0 or None)."""
    import numpy as np
    if not isinstance(series, torch.Tensor) or not series.is_cuda:
        raise N.SeqIKNativeError("series must be a CUDA tensor (there is no CPU path)")
    if series.dtype not in (torch.float32, torch.float64):
        raise ValueError(f"series must be float32 or float64, got {series.dtype}")
    if series.dim() not in (2, 3):
        raise ValueError("series must be (n_series, n) or (n_block, n, width)")
    flat = series.dim() == 2
    x = series.detach()
    x = x.unsqueeze(-1) if flat else x
    if not x.is_contiguous():
        raise ValueError("series must be contiguous")
    n = int(x.shape[1])
    if n < 2:
        raise ValueError("at least 2 samples are needed")
    if not (original_ts > 0 and new_ts > 0):
        raise ValueError("time steps must be positive")
    m = int(np.ceil((n * original_ts) / new_ts))                # length of np.arange(0, n * original_ts, new_ts)
    zeroed = None
    # one read-only pass; NaN propagates, +-inf shows up as an extreme (an empty batch has nothing to check)
    if x.numel() and not bool(torch.isfinite(torch.stack(torch.aminmax(x))).all()):
        finite = torch.isfinite(x)
        if bool(torch.isnan(x).any()):
            raise ValueError("`y` must contain only finite values.")
        x = torch.where(finite, x, torch.zeros_like(x))
        hit = (~finite).any(dim=1).any(dim=1, keepdim=True)       # (n_block, 1): blocks (= one reference call) that held an inf
        x[:, -1, :] = torch.where(hit, torch.zeros_like(x[:, -1, :]), x[:, -1, :])
        zeroed = ~finite
        zeroed[:, -1, :] |= hit
    return x, flat, m, zeroed


def pchip_resample_backward(series, grad_out, original_ts: float, new_ts: float):
    """Vector-Jacobian product of ``pchip_resample``: ``grad_out`` = dL/dout in the layout of the resampled series ->
    dL/dseries in the layout and dtype of ``series``, (n_series, n) or (n_block, n, width).  The gradient is taken at the
    values the forward resampled; the samples it replaced by 0 (+-inf, and the last sample of a block that held one) get
    gradient 0.  The float summation order is fixed (include/seqik.h), so the result is deterministic."""
    torch = N.require_cuda()
    x, flat, m, zeroed = _pchip_inputs(torch, series, original_ts, new_ts)
    n_block, n, width = (int(v) for v in x.shape)
    if not isinstance(grad_out, torch.Tensor) or grad_out.device != x.device or grad_out.dtype != x.dtype:
        raise ValueError(f"grad_out must be a {x.dtype} tensor on {x.device}")
    want = (n_block, m) if flat else (n_block, m, width)
    if tuple(grad_out.shape) != want:
        raise ValueError(f"grad_out must be {want}, got {tuple(grad_out.shape)}")
    g = grad_out.detach().reshape(n_block, m, width).contiguous()
    lib = N.load_library()
    grad = torch.empty_like(x)
    fn = lib.seqik_pchip_resample_backward_f32 if x.dtype == torch.float32 else lib.seqik_pchip_resample_backward_f64
    with torch.cuda.device(x.device):
        rc = fn(x.data_ptr(), g.data_ptr(), grad.data_ptr(), n_block, n, m, width, float(original_ts), float(new_ts),
                N.stream_ptr(torch, x.device))
    N.check(rc, "seqik_pchip_resample_backward")
    if zeroed is not None:
        grad.masked_fill_(zeroed, 0)
    return grad.squeeze(-1) if flat else grad


_PCHIP_FUNCTION = None


def _pchip_function():
    """The torch.autograd.Function of pchip_resample (built on first use: torch is imported lazily)."""
    global _PCHIP_FUNCTION
    if _PCHIP_FUNCTION is not None:
        return _PCHIP_FUNCTION
    import torch
    from torch.autograd.function import once_differentiable

    class PchipResample(torch.autograd.Function):
        @staticmethod
        def forward(ctx, series, original_ts, new_ts):
            ctx.save_for_backward(series)
            ctx.steps = (original_ts, new_ts)
            return pchip_resample(series, original_ts, new_ts)

        @staticmethod
        @once_differentiable
        def backward(ctx, grad_out):
            series, = ctx.saved_tensors
            return pchip_resample_backward(series, grad_out, *ctx.steps), None, None

    _PCHIP_FUNCTION = PchipResample
    return _PCHIP_FUNCTION
