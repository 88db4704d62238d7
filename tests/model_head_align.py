"""A float64 torch model of the head alignment -- ``head_affine`` (the antenna statistics of AlignPose.align_head) followed by
``head_apply`` (its scale-and-translate map) -- for the gradients of ``seqik_head_apply_backward_f32`` and
``seqik_head_affine_backward_f32/_f64``.  TEST/DEV TOOL.

The stationary frames are those ``model_head.head_stats`` finds (the float64 distances and second differences of
``seqik_head_series_*``).  Over them, the five float32 series values are turned into the kernels' order keys, and the
frame of each of the four order statistics of a series is ``argsort(keys, stable)[r]`` (the tie rule of include/seqik.h),
with the ranks and float32 weights of ``model_quantile``.  With those frames fixed the statistics are smooth functions of
the key points, so autograd in float64 gives the VJP the kernels approximate.

The product never imports this file.
"""
import numpy as np
import torch

import model_head as H
import model_quantile as Q


def device_threshold(threshold, dtype):
    """The threshold as seqik_head_series_f32 (a float32 argument) or _f64 receives it."""
    return float(np.float32(threshold)) if np.dtype(dtype) == np.float32 else float(threshold)


def stationary(head, thorax, threshold):
    """One trial: the stationary frames of model_head.head_stats (threshold as the device receives it)."""
    d = H.base_to_thorax_mid(head, thorax)
    return np.where(np.diff(np.diff(d)) < threshold)[0]


def series_values(head, thorax, threshold):
    """One trial: head (n_frame, 2, 3), thorax (n_frame, k, 3) -> the five float32 series over their frames, and those
    frames: (values, frames) lists (series 0-3 over the stationary frames, series 4 over every frame)."""
    idx = stationary(head, thorax, threshold)
    h = np.asarray(head, dtype=np.float64)
    d = H.base_to_thorax_mid(head, thorax)
    a = h[:, 1] - h[:, 0]
    tip = np.sqrt(a[:, 0] * a[:, 0] + a[:, 1] * a[:, 1] + a[:, 2] * a[:, 2])
    vals = [h[idx, 0, c].astype(np.float32) for c in range(3)] + [d[idx].astype(np.float32), tip.astype(np.float32)]
    return vals, [idx] * 4 + [np.arange(h.shape[0])]


def stat_frames(head, thorax, threshold):
    """head (n_trial, n_frame, 2, 3), thorax (n_trial, n_frame, k, 3) numpy, threshold as the device receives it ->
    (frames (n_trial, 5, 4) int64 in rank order lo45, lo45 + 1, lo55, lo55 + 1 (0 where the series is empty),
    counts (n_trial, 5), f45 (n_trial, 5), f55 (n_trial, 5))."""
    n_trial = head.shape[0]
    frames = np.zeros((n_trial, 5, 4), dtype=np.int64)
    counts = np.zeros((n_trial, 5), dtype=np.int64)
    f45 = np.zeros((n_trial, 5), dtype=np.float32)
    f55 = np.zeros((n_trial, 5), dtype=np.float32)
    for tr in range(n_trial):
        vals, where = series_values(head[tr], thorax[tr], threshold)
        for j in range(5):
            m = len(vals[j])
            counts[tr, j] = m
            if m == 0:
                continue
            ranks, a, b = Q.mid_quantile_ranks(np.array([m]))
            order = np.argsort(Q.order_key(vals[j]), kind="stable")
            frames[tr, j] = where[j][order[ranks[:, 0]]]
            f45[tr, j], f55[tr, j] = a[0], b[0]
    return frames, counts, f45, f55


def weights(f45, f55):
    """(..., 4) float64 weights of the ranks lo45, lo45 + 1, lo55, lo55 + 1 (the kernels' float32 weights)."""
    f32 = np.float32
    f45, f55 = np.asarray(f45, dtype=f32), np.asarray(f55, dtype=f32)
    return np.stack([f32(0.5) * (f32(1) - f45), f32(0.5) * f45, f32(0.5) * (f32(1) - f55), f32(0.5) * f55], -1).astype(np.float64)


def head_affine(head, thorax, consts, frames):
    """float64 tensors head (n_trial, n_frame, 2, 3), thorax (n_trial, n_frame, k, 3), consts (n_trial, 5) and the frames
    of stat_frames -> affine (n_trial, 8), differentiable (NaN where a series is empty)."""
    fr, counts, f45, f55 = frames
    base, tip = head[:, :, 0], head[:, :, 1]
    d = torch.linalg.vector_norm(base - 0.5 * (thorax[:, :, 0] + thorax[:, :, -1]), dim=-1)    # subgradient 0 at 0
    tl = torch.linalg.vector_norm(tip - base, dim=-1)
    series = torch.stack([base[..., 0], base[..., 1], base[..., 2], d, tl], dim=1)              # (n_trial, 5, n_frame)
    v = torch.gather(series, 2, torch.as_tensor(fr, device=head.device))
    a = torch.as_tensor(np.asarray(f45, dtype=np.float64), device=head.device)
    b = torch.as_tensor(np.asarray(f55, dtype=np.float64), device=head.device)
    s = 0.5 * ((v[..., 0] + (v[..., 1] - v[..., 0]) * a) + (v[..., 2] + (v[..., 3] - v[..., 2]) * b))
    s = torch.where(torch.as_tensor(counts, device=head.device) > 0, s, torch.full_like(s, float("nan")))
    return torch.cat([s[:, :3], consts[:, 3:4] / s[:, 3:4], consts[:, :3], consts[:, 4:5] / s[:, 4:5]], dim=1)


def head_apply(head, affine):
    """base' = (base - origin) * affine[3] + template, tip' = (tip - origin) * affine[7] + template."""
    o, t = affine[:, None, 0:3], affine[:, None, 4:7]
    base = (head[:, :, 0] - o) * affine[:, None, 3:4] + t
    tip = (head[:, :, 1] - o) * affine[:, None, 7:8] + t
    return torch.stack([base, tip], dim=2)


def aligned(head, thorax, consts, frames):
    return head_apply(head, head_affine(head, thorax, consts, frames))


def stats_vjp(head, thorax, consts, grad_affine, threshold):
    """float64 VJP of head_affine at the given (float32 or float64) numpy inputs: grad_affine (n_trial, 8) ->
    (grad_head, grad_thorax, grad_consts, (cnt_head, acc_head, cnt_thorax, acc_thorax)): per element, the number of
    contributions it receives and the sum of their absolute values, from the same chain rule with every factor replaced
    by its absolute value."""
    frames = stat_frames(head, thorax, threshold)
    fr, counts, f45, f55 = frames
    hd = torch.from_numpy(np.asarray(head, dtype=np.float64)).requires_grad_()
    th = torch.from_numpy(np.asarray(thorax, dtype=np.float64)).requires_grad_()
    k = torch.from_numpy(np.asarray(consts, dtype=np.float64)).requires_grad_()
    h = np.asarray(grad_affine, dtype=np.float64)
    aff = head_affine(hd, th, k, frames)
    gh, gt, gk = torch.autograd.grad(aff, [hd, th, k], torch.from_numpy(h), allow_unused=True)
    gt = torch.zeros_like(th) if gt is None else gt
    aff = aff.detach().numpy()
    w = weights(f45, f55)
    h64, t64 = hd.detach().numpy(), th.detach().numpy()
    cnt_h, acc_h = np.zeros(h64.shape, dtype=np.int64), np.zeros(h64.shape)
    cnt_t, acc_t = np.zeros(t64.shape, dtype=np.int64), np.zeros(t64.shape)
    n_kp = t64.shape[2]
    for tr in range(h64.shape[0]):
        s3, s4 = np.asarray(consts, dtype=np.float64)[tr, 3] / aff[tr, 3], np.asarray(consts, dtype=np.float64)[tr, 4] / aff[tr, 7]
        ds = [abs(h[tr, 0]), abs(h[tr, 1]), abs(h[tr, 2]), abs(h[tr, 3] * aff[tr, 3] / s3), abs(h[tr, 7] * aff[tr, 7] / s4)]
        for j in range(5):
            if counts[tr, j] == 0:
                continue
            for i in range(4):
                t, g = fr[tr, j, i], ds[j] * w[tr, j, i]
                if j < 3:
                    cnt_h[tr, t, 0, j] += 1
                    acc_h[tr, t, 0, j] += g
                    continue
                b = h64[tr, t, 0]
                vec = b - 0.5 * (t64[tr, t, 0] + t64[tr, t, -1]) if j == 3 else h64[tr, t, 1] - b
                nrm = np.linalg.norm(vec)
                if nrm == 0:
                    continue
                u = np.abs(vec) / nrm
                if j == 3:
                    cnt_h[tr, t, 0] += 1
                    acc_h[tr, t, 0] += g * u
                    for kp in (0, n_kp - 1):
                        cnt_t[tr, t, kp] += 1
                        acc_t[tr, t, kp] += 0.5 * g * u
                else:
                    for row in (1, 0):
                        cnt_h[tr, t, row] += 1
                        acc_h[tr, t, row] += g * u
    return gh.numpy(), gt.numpy(), gk.numpy(), (cnt_h, acc_h, cnt_t, acc_t)
