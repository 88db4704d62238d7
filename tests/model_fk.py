"""Float64 forward kinematics of the stage-4 leg chain in torch ops: the gradient reference of seqik_fk_backward_f32.

The rotation order is the kernel's (csrc/seqik_kernels.cu fk_rows): A = Rx(yaw) Ry(pitch) for stage 1, then A <- A Rz(roll) Ry(pitch)
for stages 2 and 3 and A <- A Ry(pitch) for stage 4; joint k = joint k-1 - l_k A[:, 2].  (The reference's order puts the
ThC roll before the first segment, which does not move it: the two agree, tests/test_fk_grad_cpu.py.)  torch autograd of
this function is the float64 gradient the kernel is compared with.
"""
import torch


def _rot(axis, a):
    """Rotation matrices (..., 3, 3) about a coordinate axis by angles a (...)."""
    c, s = torch.cos(a), torch.sin(a)
    o, z = torch.ones_like(a), torch.zeros_like(a)
    rows = {0: ((o, z, z), (z, c, -s), (z, s, c)),
            1: ((c, z, s), (z, o, z), (-s, z, c)),
            2: ((c, -s, z), (s, c, z), (z, z, o))}[axis]
    return torch.stack([torch.stack(r, -1) for r in rows], -2)


def fk(angles, origin, lengths):
    """angles (..., 7), origin (..., 3), lengths (..., 4) (broadcast against each other) -> (..., 9, 3): rows 0-3 the
    origin, 4-5 the Coxa-Femur joint, 6 Femur-Tibia, 7 Tibia-Tarsus, 8 the claw."""
    q = angles
    A = _rot(0, q[..., 0]) @ _rot(1, q[..., 1])
    frames = [A]
    A = A @ _rot(2, q[..., 2]) @ _rot(1, q[..., 3])
    frames.append(A)
    A = A @ _rot(2, q[..., 4]) @ _rot(1, q[..., 5])
    frames.append(A)
    A = A @ _rot(1, q[..., 6])
    frames.append(A)
    p = torch.broadcast_tensors(origin, A[..., :, 2])[0]
    rows = [p, p, p, p]
    for k, F in enumerate(frames):
        p = p - lengths[..., k:k + 1] * F[..., :, 2]
        rows.append(p)
        if k == 0:
            rows.append(p)
    return torch.stack(rows, -2)
