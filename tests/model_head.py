"""float64 models of the head kernels (``head_kernel``, ``head_series_kernel`` + ``head_affine_kernel``).  TEST/DEV TOOL.

``head_angles`` restates HeadInverseKinematics.compute_head_angles (reference head_inverse_kinematics.py:103-335) in
float64, in the reference's own form: every angle is ``angle_between_segments`` = arccos(v1.v2 / (|v1| |v2|)) times
(det > 0 ? 1 : -1), det = the rotation axis . (v1 x v2), of two vectors projected onto the plane normal to that axis; the
antenna vectors are first de-rotated by the head roll (``derotate_vector``: Rx(-roll) v).  It shares no code with the
kernel, which evaluates the same angles as atan2(|det|, dot) in float32 (csrc/seqik_kernels.cu, ``head_frame``).

``head_stats`` restates the antenna statistics of AlignPose.align_head (alignment.py:489-555) the way
``seqik_head_series_*`` evaluates them: distances in float64 as the square root of a sum of squares in the kernel's
order, so that a frame sitting on the stationarity threshold is classified the same way.  The product never imports
this file.
"""
import numpy as np


def angle_between_segments(v1, v2, axis):
    """(N, 3) x (N, 3) -> (N,): the reference's signed angle from v1 to v2 about ``axis`` (0 = X, 1 = Y, 2 = Z)."""
    v1 = np.asarray(v1, dtype=np.float64)
    v2 = np.asarray(v2, dtype=np.float64)
    cos = np.einsum("ij,ij->i", v1, v2) / (np.linalg.norm(v1, axis=1) * np.linalg.norm(v2, axis=1))
    det = np.cross(v1, v2)[:, axis]
    return np.arccos(np.clip(cos, -1.0, 1.0)) * np.where(det > 0, 1.0, -1.0)


def _drop(v, k):
    """Projection onto the plane normal to axis k."""
    v = np.array(v, dtype=np.float64)
    v[:, k] = 0.0
    return v


def derotate(v, roll):
    """Rx(-roll) v, row by row."""
    c, s = np.cos(roll), np.sin(roll)
    return np.stack([v[:, 0], c * v[:, 1] + s * v[:, 2], -s * v[:, 1] + c * v[:, 2]], axis=1)


def head_angles(r_head, l_head, neck, rest_head_pitch, rest_antenna_pitch):
    """r_head, l_head (N, 2, 3) (base, tip); neck (N, 3) or (3,) -> (7, N): head roll, pitch, yaw, antenna yaw L,
    antenna pitch L, antenna yaw R, antenna pitch R."""
    r = np.asarray(r_head, dtype=np.float64)
    l = np.asarray(l_head, dtype=np.float64)
    n = r.shape[0]
    neck = np.broadcast_to(np.asarray(neck, dtype=np.float64).reshape(-1, 3), (n, 3))
    x, y = np.tile([1.0, 0.0, 0.0], (n, 1)), np.tile([0.0, 1.0, 0.0], (n, 1))
    hor = l[:, 0] - r[:, 0]
    mid = 0.5 * (r[:, 0] + l[:, 0]) - neck
    roll = angle_between_segments(y, _drop(hor, 0), 0)
    pitch = angle_between_segments(x, _drop(mid, 1), 1) + rest_head_pitch
    yaw = angle_between_segments(y, _drop(hor, 2), 2)
    hor_d = derotate(hor, roll)
    out = [roll, pitch, yaw]
    for side in (l, r):
        ant = derotate(side[:, 1] - side[:, 0], roll)
        ant_yaw = angle_between_segments(_drop(ant, 0), _drop(hor_d, 0), 0)
        if side is r:
            ant_yaw = np.pi - ant_yaw
        ant_pitch = angle_between_segments(_drop(derotate(neck - side[:, 0], roll), 1), _drop(ant, 1), 1) - rest_antenna_pitch
        out += [ant_yaw, ant_pitch]
    return np.stack(out)


def base_to_thorax_mid(head, thorax):
    """(n_frame,) float64 |base - (thorax[0] + thorax[-1]) / 2|, in the order of ``base_to_thorax_mid`` (device)."""
    b = np.asarray(head, dtype=np.float64)[:, 0]
    t = np.asarray(thorax, dtype=np.float64)
    d = b - 0.5 * (t[:, 0] + t[:, -1])
    return np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2])


def mid_quantile(v):
    v = np.asarray(v, dtype=np.float64)
    return 0.5 * (np.quantile(v, 0.45) + np.quantile(v, 0.55)) if v.size else np.nan


def head_stats(head, thorax, consts, threshold):
    """One trial: head (n_frame, 2, 3), thorax (n_frame, k, 3), consts (5,) float32, threshold as the device receives it
    -> (count of stationary frames, affine row (8,) float64, the float32 values that enter each statistic).
    ``stationary = diff(diff(d)) < threshold``; base xyz and d are taken over the stationary frames, |tip - base| over
    all frames; the row is (base xyz, Antenna_mid_thorax / d, template xyz, Antenna / |tip - base|) with NaN where a
    statistic has no frame."""
    h = np.asarray(head, dtype=np.float64)
    d = base_to_thorax_mid(head, thorax)
    idx = np.where(np.diff(np.diff(d)) < threshold)[0]
    a = h[:, 1] - h[:, 0]
    tip = np.sqrt(a[:, 0] * a[:, 0] + a[:, 1] * a[:, 1] + a[:, 2] * a[:, 2])
    series = [h[idx, 0, k].astype(np.float32) for k in range(3)] + [d[idx].astype(np.float32), tip.astype(np.float32)]
    q = [mid_quantile(s) for s in series]
    k = np.asarray(consts, dtype=np.float64)
    row = np.array([q[0], q[1], q[2], k[3] / q[3], k[0], k[1], k[2], k[4] / q[4]])
    return len(idx), row, series
