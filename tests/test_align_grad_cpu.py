"""CPU side of the differentiable leg alignment: the float64 model (tests/model_align.py) against the exact float32 statistics
of model_quantile and the align map, gradcheck, the two invariances of the composite, and the argument checks of
seqik_align_apply_backward_f32 / seqik_leg_affine_backward_f32 (they run before any CUDA call)."""
import numpy as np
import pytest
import torch

import model_align as A
import model_quantile as Q


def _pose(rng, n_chain, n_frame):
    base = rng.normal(size=(n_chain, 1, 5, 3)).cumsum(axis=2)
    return (base + 0.05 * rng.normal(size=(n_chain, n_frame, 5, 3))).astype(np.float32)


def _consts(rng, n_chain):
    return np.concatenate([rng.normal(size=(n_chain, 3)), rng.uniform(1.0, 3.0, (n_chain, 1))], axis=1).astype(np.float32)


@pytest.mark.parametrize("include_claw", [False, True])
@pytest.mark.parametrize("n_frame", [1, 2, 5, 6, 10, 31, 200])
def test_model_forward_equals_the_exact_statistics(n_frame, include_claw):
    rng = np.random.default_rng(n_frame)
    pose, consts = _pose(rng, 4, n_frame), _consts(rng, 4)
    _, stats, aff32 = Q.leg_stats_exact(pose, consts, include_claw)
    frames, f45, f55 = A.stat_frames(pose)
    p, k = torch.from_numpy(pose.astype(np.float64)), torch.from_numpy(consts.astype(np.float64))
    aff = A.leg_affine(p, k, frames, f45, f55, include_claw).numpy()
    # the order statistics are the same elements; float64 against float32 interpolation: a few ulp
    assert np.abs(aff[:, :3] - stats[:, :3]).max() <= 4 * 2.0 ** -24 * np.abs(stats[:, :3]).max()
    assert np.all(np.abs(aff[:, 3] - aff32[:, 3]) <= 8 * 2.0 ** -24 * np.abs(aff32[:, 3]))
    assert np.array_equal(aff[:, 4:], aff32[:, 4:].astype(np.float64))
    out = A.align_apply(p, torch.from_numpy(aff)).numpy()
    ref = (pose[:, :, 1:].astype(np.float64) - aff[:, None, None, :3]) * aff[:, None, None, 3:4] + aff[:, None, None, 4:7]
    assert np.abs(out[:, :, 1:] - ref).max() <= 1e-12
    assert np.array_equal(out[:, :, 0], np.broadcast_to(aff[:, None, 4:7], out[:, :, 0].shape))


def test_frames_follow_the_stable_argsort_and_the_square_keys():
    pose = np.zeros((1, 6, 5, 3), dtype=np.float32)
    pose[0, :, 0, 0] = [1.0, -0.0, 0.0, 1.0, -0.0, 2.0]            # -0 sorts below +0; ties keep frame order
    pose[0, :, 1:, 2] = np.arange(1, 5, dtype=np.float32)           # unit segments along z ...
    pose[0, 3, 2:, 2] += 1.0                                        # ... one longer segment in frame 3
    frames, _, _ = A.stat_frames(pose)
    keys = A.series_keys(pose)
    order = np.argsort(keys, axis=-1, kind="stable")
    assert list(order[0, 0]) == [1, 4, 2, 0, 3, 5]
    ranks, _, _ = Q.mid_quantile_ranks(np.array([6]))
    assert np.array_equal(frames[0], order[0][:, ranks[:, 0]])


@pytest.mark.parametrize("include_claw", [False, True])
def test_gradcheck_on_tie_free_inputs(include_claw):
    rng = np.random.default_rng(3)
    pose, consts = _pose(rng, 2, 7), _consts(rng, 2)
    frames = A.stat_frames(pose)
    p = torch.from_numpy(pose.astype(np.float64)).requires_grad_()
    k = torch.from_numpy(consts.astype(np.float64)).requires_grad_()
    assert torch.autograd.gradcheck(lambda p, k: A.aligned(p, k, include_claw, frames), (p, k), eps=1e-7, atol=1e-6)


@pytest.mark.parametrize("include_claw", [False, True])
@pytest.mark.parametrize("n_frame", [2, 6, 33, 300])
def test_composite_invariances(n_frame, include_claw):
    """Alignment is invariant under p -> a p + b (a > 0), so sum dL/dp = 0 per chain and coordinate and sum p . dL/dp = 0 per
    chain, for any loss and any tie choice.  Only a correct statistics term makes them hold."""
    rng = np.random.default_rng(n_frame + 17)
    pose, consts = _pose(rng, 3, n_frame), _consts(rng, 3)
    pose[:, :, :, 1] = np.round(pose[:, :, :, 1] * 4) / 4                          # ties in the y series
    p = torch.from_numpy(pose.astype(np.float64)).requires_grad_()
    k = torch.from_numpy(consts.astype(np.float64))
    g_out = torch.from_numpy(rng.normal(size=pose.shape))
    out = A.aligned(p, k, include_claw)
    gp, = torch.autograd.grad(out, [p], g_out)
    scale = gp.abs().sum(dim=(1, 2, 3)).max().item() * (1 + np.abs(pose).max())
    assert gp.sum(dim=(1, 2)).abs().max().item() <= 1e-12 * scale
    assert (gp * p.detach()).sum(dim=(1, 2, 3)).abs().max().item() <= 1e-12 * scale


def test_zero_length_segment_contributes_nothing():
    pose = np.zeros((1, 3, 5, 3), dtype=np.float32)
    pose[0, :, 1:, 0] = np.arange(1, 5, dtype=np.float32)
    pose[0, :, 2] = pose[0, :, 1]                                    # segment 1 has length 0 in every frame
    gp, gk, (cnt, _) = A.stats_vjp(pose, np.array([[0, 0, 0, 2]], dtype=np.float32), np.eye(8)[None, 3], False)
    assert np.isfinite(gp).all()
    assert cnt[0, :, 1].sum() == 12 and cnt[0, :, 2].sum() == 12                 # segments 0 and 2 only: 4 ranks x 3 coordinates


def test_backward_argument_validation_without_gpu():
    from seqikpy_b200 import _native as N
    lib = N.load_library()
    f = lib.seqik_align_apply_backward_f32
    #      pose cs fs aff g_out g_pose part n_chain n_frame stream
    assert f(8, 150, 15, 8, 8, 8, 8, -1, 10, 0) == -1
    assert b"negative" in lib.seqik_last_error()
    assert f(8, 150, 15, 8, 8, 8, 8, 4, -1, 0) == -1
    assert f(0, 0, 15, 0, 0, 0, 0, 0, 10, 0) == 0                                  # empty: ok, nothing read
    assert f(0, 0, 15, 0, 0, 0, 0, 4, 0, 0) == 0
    for k in (0, 3, 4):                                                            # pose, affine, grad_out NULL
        args = [8, 150, 15, 8, 8, 8, 8, 4, 10, 0]
        args[k] = 0
        assert f(*args) == -1, k
        assert b"NULL" in lib.seqik_last_error()
    assert f(8, 150, 14, 8, 8, 8, 8, 4, 10, 0) == -1                               # frame stride below the block
    assert b"stride" in lib.seqik_last_error()
    assert f(8, 150, 15, 8, 8, 0, 0, 4, 10, 0) == 0                                # both outputs NULL: nothing to do
    g = lib.seqik_leg_affine_backward_f32
    #      pose cs fs consts claw aff g_aff g_pose g_consts scratch n_chain n_frame stream
    ok = [8, 150, 15, 8, 0, 8, 8, 8, 0, 0, 4, 10, 0]
    bad = lambda i, v: [v if j == i else a for j, a in enumerate(ok)]
    assert g(*bad(10, -1)) == -1 and b"negative" in lib.seqik_last_error()
    assert g(*bad(11, -1)) == -1
    assert g(*bad(10, 0)) == 0                                                     # no chains: ok
    assert g(*bad(11, 0)) == -1 and b"empty recording" in lib.seqik_last_error()
    for i in (0, 3, 5, 6, 7):                                                      # pose, consts, affine, grad_affine, grad_pose
        assert g(*bad(i, 0)) == -1, i
        assert b"NULL" in lib.seqik_last_error()
    assert g(*bad(2, 12)) == -1 and b"stride" in lib.seqik_last_error()
    assert g(*bad(10, 1 << 31)) == -1 and b"too many chains" in lib.seqik_last_error()
    assert g(*bad(11, 1025)) == -1 and b"scratch" in lib.seqik_last_error()        # long recordings need scratch
