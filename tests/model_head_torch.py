"""float64 torch model of the head angles, the reference for the gradients of ``seqik_head_angles_backward_f32``.  TEST/DEV
TOOL.

``head_angles_torch`` is the map of tests/model_head.py ``head_angles`` (the reference's HeadInverseKinematics
.compute_head_angles) in torch ops and in atan2 form: the signed angle from a to b about an axis is phi(b) - phi(a) wrapped
to [-pi, pi), phi the atan2 of a vector's two coordinates in the plane.  So its autograd is well conditioned at 0 and pi
(arccos' is not), and a zero projected vector contributes torch.atan2's gradient at (0, 0), which is 0.  The product never
imports this file.
"""
import math

import torch


def _phi_x(v):
    """Angle of v|x=0 about X, measured from Y."""
    return torch.atan2(v[..., 2], v[..., 1])


def _phi_y(v):
    """Angle of v|y=0 about Y, measured from X."""
    return torch.atan2(-v[..., 2], v[..., 0])


def _phi_z(v):
    """Angle of v|z=0 about Z, measured from Y."""
    return torch.atan2(-v[..., 0], v[..., 1])


def _wrap(a):
    return torch.remainder(a + math.pi, 2 * math.pi) - math.pi


def _derotate(v, c, s):
    """Rx(-roll) v, with c, s = cos / sin of the roll."""
    return torch.stack([v[..., 0], c * v[..., 1] + s * v[..., 2], -s * v[..., 1] + c * v[..., 2]], dim=-1)


def head_angles_torch(r_head, l_head, neck, rest_head_pitch, rest_antenna_pitch):
    """r_head, l_head (..., 2, 3) (base, tip); neck broadcastable to (..., 3); rest angles broadcastable to (...)
    -> (7, ...): head roll, pitch, yaw, antenna yaw L, antenna pitch L, antenna yaw R, antenna pitch R."""
    rb, rt, lb, lt = r_head[..., 0, :], r_head[..., 1, :], l_head[..., 0, :], l_head[..., 1, :]
    hor = lb - rb
    mid = 0.5 * (rb + lb) - neck
    roll = _phi_x(hor)
    pitch = _phi_y(mid) + rest_head_pitch
    yaw = _phi_z(hor)
    c, s = torch.cos(roll), torch.sin(roll)
    hor_d = _derotate(hor, c, s)
    out = [roll, pitch, yaw]
    for b, t, right in ((lb, lt, False), (rb, rt, True)):
        ant = _derotate(t - b, c, s)
        ant_yaw = _wrap(_phi_x(hor_d) - _phi_x(ant))
        if right:
            ant_yaw = math.pi - ant_yaw
        ant_pitch = _wrap(_phi_y(ant) - _phi_y(_derotate(neck - b, c, s))) - rest_antenna_pitch
        out += [ant_yaw, ant_pitch]
    return torch.stack(out)
