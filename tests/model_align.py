"""A float64 torch model of the leg alignment -- ``leg_affine`` (the mid-quantile statistics of AlignPose.align_leg) followed
by ``align_apply`` (its affine map) -- for the gradients of ``seqik_align_apply_backward_f32`` and
``seqik_leg_affine_backward_f32``.  TEST/DEV TOOL.

It builds on ``model_quantile``: the same float32 order keys (coxa coordinates, and the float32 SQUARED segment lengths
(dx dx + dy dy) + dz dz), the same ranks and float32 weights, and the frames of the four order statistics of every series
from a stable argsort of the keys (the tie rule of include/seqik.h).  With those frames fixed the statistics are smooth
functions of the key points, so autograd in float64 gives the VJP the kernels approximate in float32.

The product never imports this file.
"""
import numpy as np
import torch

import model_quantile as Q


def series_keys(pose):
    """pose (n_chain, n_frame, 5, 3) float32 -> (n_chain, 7, n_frame) uint32: the keys the statistics kernels select on."""
    p = np.asarray(pose, dtype=np.float32)
    d = p[:, :, 1:] - p[:, :, :-1]
    sq = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
    return Q.order_key(np.concatenate([p[:, :, 0].transpose(0, 2, 1), sq.transpose(0, 2, 1)], axis=1))


def stat_frames(pose):
    """-> (frames (n_chain, 7, 4) int64 in rank order lo45, lo45 + 1, lo55, lo55 + 1; f45; f55): argsort(keys, stable)[r]."""
    keys = series_keys(pose)
    n_frame = keys.shape[-1]
    ranks, f45, f55 = Q.mid_quantile_ranks(np.array([n_frame]))
    order = np.argsort(keys, axis=-1, kind="stable")
    return order[..., ranks[:, 0]], float(f45[0]), float(f55[0])


def leg_affine(pose, consts, frames, f45, f55, include_claw):
    """float64 tensors pose (n_chain, n_frame, 5, 3), consts (n_chain, 4) -> affine (n_chain, 8), differentiable."""
    seg = pose[:, :, 1:] - pose[:, :, :-1]
    length = torch.linalg.vector_norm(seg, dim=-1)                                        # subgradient 0 at a zero segment
    series = torch.cat([pose[:, :, 0].transpose(1, 2), length.transpose(1, 2)], dim=1)   # (n_chain, 7, n_frame)
    v = torch.gather(series, 2, torch.as_tensor(frames, device=pose.device))
    m = 0.5 * ((v[..., 0] + (v[..., 1] - v[..., 0]) * f45) + (v[..., 2] + (v[..., 3] - v[..., 2]) * f55))
    length_sum = (m[:, 3] + m[:, 4]) + m[:, 5]
    if include_claw:
        length_sum = length_sum + m[:, 6]
    scale = consts[:, 3] / length_sum
    zero = torch.zeros_like(scale)
    return torch.cat([m[:, :3], scale[:, None], consts[:, :3], zero[:, None]], dim=1)


def align_apply(pose, affine):
    """out[:, :, 0] = template, out[:, :, i] = (pose[:, :, i] - fixed) * scale + template."""
    fixed, scale, tmpl = affine[:, None, None, 0:3], affine[:, None, None, 3:4], affine[:, None, None, 4:7]
    moved = (pose[:, :, 1:] - fixed) * scale + tmpl
    return torch.cat([tmpl.expand(-1, pose.shape[1], 1, 3), moved], dim=2)


def aligned(pose, consts, include_claw, frames=None):
    """The composite with the frames of ``pose`` (float32 numpy or tensor) unless given; float64 tensors in and out."""
    if frames is None:
        frames, f45, f55 = stat_frames(pose.detach().float().cpu().numpy())
    else:
        frames, f45, f55 = frames
    return align_apply(pose, leg_affine(pose, consts, frames, f45, f55, include_claw))


def stats_vjp(pose32, consts32, grad_affine, include_claw):
    """float64 VJP of leg_affine at the float32 inputs: grad_affine (n_chain, 8) -> (grad_pose, grad_consts, bound terms).

    The bound terms are, per float of grad_pose, (N, A): the number of contributions it receives and the sum of their
    absolute values, from the same chain rule with every factor replaced by its absolute value."""
    frames, f45, f55 = stat_frames(pose32)
    p = torch.from_numpy(np.asarray(pose32, dtype=np.float64)).requires_grad_()
    k = torch.from_numpy(np.asarray(consts32, dtype=np.float64)).requires_grad_()
    h = torch.from_numpy(np.asarray(grad_affine, dtype=np.float64))
    aff = leg_affine(p, k, frames, f45, f55, include_claw)
    gp, gk = torch.autograd.grad(aff, [p, k], h)
    # the absolute analogue: |dL/dm_s| * weight * |s_c| / |s| per contribution
    with torch.no_grad():
        scale = aff[:, 3]
        length = consts32[:, 3].astype(np.float64) / scale.numpy()
        dlen = np.abs(h[:, 3].numpy() * scale.numpy() / length)
        w = np.array([0.5 * (1 - f45), 0.5 * f45, 0.5 * (1 - f55), 0.5 * f55])
        n_chain = pose32.shape[0]
        cnt = np.zeros(pose32.shape, dtype=np.int64)
        acc = np.zeros(pose32.shape, dtype=np.float64)
        p64 = np.asarray(pose32, dtype=np.float64)
        for c in range(n_chain):
            for s in range(7 if include_claw else 6):
                gs = abs(float(h[c, s])) if s < 3 else float(dlen[c])
                for i in range(4):
                    t = frames[c, s, i]
                    if s < 3:
                        cnt[c, t, 0, s] += 1
                        acc[c, t, 0, s] += gs * w[i]
                        continue
                    j = s - 3
                    d = p64[c, t, j + 1] - p64[c, t, j]
                    nrm = np.linalg.norm(d)
                    if nrm == 0:
                        continue
                    for row in (j, j + 1):
                        cnt[c, t, row] += 1
                        acc[c, t, row] += gs * w[i] * np.abs(d) / nrm
    return gp.numpy(), gk.numpy(), (cnt, acc)
