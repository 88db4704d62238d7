"""CPU side of the differentiable head alignment: the float64 model (tests/model_head_align.py) against model_head.head_stats,
gradcheck, the tie rule, the two invariances of the composite, and the argument checks of seqik_head_apply_backward_f32 /
seqik_head_affine_backward_f32/_f64 (they run before any CUDA call)."""
import numpy as np
import pytest
import torch

import model_head as H
import model_head_align as M
import model_quantile as Q


def _trial(rng, n_frame, k=3, still=0.5):
    """Antenna (n_frame, 2, 3) and thorax (n_frame, k, 3): a smooth walk with still stretches (second differences 0)."""
    thorax = rng.normal(size=(1, k, 3)) + 0.01 * rng.normal(size=(n_frame, k, 3))
    base = np.array([0.3, 0.5, 0.2]) + 0.02 * rng.normal(size=(n_frame, 3))
    hold = rng.random(n_frame) < still
    for t in range(1, n_frame):
        if hold[t]:
            base[t] = base[t - 1]
            thorax[t] = thorax[t - 1]
    tip = base + np.array([0.1, 0.2, 0.3]) + 0.02 * rng.normal(size=(n_frame, 3))
    return np.stack([base, tip], axis=1), thorax


def _batch(rng, n_trial, n_frame, k=3, dtype=np.float64):
    pairs = [_trial(rng, n_frame, k) for _ in range(n_trial)]
    head = np.stack([p[0] for p in pairs]).astype(dtype)
    thorax = np.stack([p[1] for p in pairs]).astype(dtype)
    consts = np.concatenate([rng.normal(size=(n_trial, 3)), rng.uniform(0.5, 2.0, (n_trial, 2))], axis=1).astype(np.float32)
    return head, thorax, consts


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("n_frame", [3, 4, 7, 12, 40, 300])
def test_model_forward_equals_head_stats(n_frame, dtype):
    rng = np.random.default_rng(n_frame)
    head, thorax, consts = _batch(rng, 3, n_frame, dtype=dtype)
    thr = M.device_threshold(5e-5, dtype)
    frames = M.stat_frames(head, thorax, thr)
    aff = M.head_affine(torch.from_numpy(head.astype(np.float64)), torch.from_numpy(thorax.astype(np.float64)),
                        torch.from_numpy(consts.astype(np.float64)), frames).numpy()
    for tr in range(3):
        count, row, _ = H.head_stats(head[tr], thorax[tr], consts[tr], thr)
        assert frames[1][tr, 0] == count and frames[1][tr, 4] == n_frame
        # the order statistics are the same elements; the float32 interpolation weights against numpy's float64 ones
        ok = np.isfinite(row)
        assert np.array_equal(ok, np.isfinite(aff[tr]))
        assert np.allclose(aff[tr][ok], row[ok], rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("k", [1, 3])
def test_gradcheck_on_tie_free_inputs(k):
    rng = np.random.default_rng(4 + k)
    head, thorax, consts = _batch(rng, 2, 12, k)
    head = head + 1e-3 * rng.normal(size=head.shape)                # no exact repeats: tie-free series
    thr = 1.0                                                        # every frame with a second difference is stationary
    frames = M.stat_frames(head, thorax, thr)
    assert (frames[1][:, :4] == 10).all()
    h = torch.from_numpy(head).requires_grad_()
    t = torch.from_numpy(thorax).requires_grad_()
    c = torch.from_numpy(consts.astype(np.float64)).requires_grad_()
    assert torch.autograd.gradcheck(lambda h, t, c: M.aligned(h, t, c, frames), (h, t, c), eps=1e-7, atol=1e-6)


def test_tie_rule_on_a_hand_built_case():
    """Keys are the float32 series values' order keys (-0 below +0), the frame of rank r is argsort(keys, stable)[r] over
    the stationary frames only, and equal float32 distances tie even where the float64 distances differ."""
    n = 10
    head = np.zeros((1, n, 2, 3))
    head[0, :, 1] = 1.0
    thorax = np.zeros((1, n, 2, 3))
    # base x over frames 0..7 (frames 8, 9 are never stationary: they have no second difference)
    head[0, :8, 0, 0] = [1.0, -0.0, 0.0, 1.0, -0.0, 2.0, 0.0, 1.0]
    # base y: distances |(0, y, 0)| with y and y + 1e-12 equal in float32
    head[0, :8, 0, 1] = [3.0, 3.0 + 1e-12, 2.0, 2.0, 3.0, 2.0 + 1e-12, 4.0, 3.0]
    thr = 1e30                                                       # frames 0..7 stationary
    frames, counts, _, _ = M.stat_frames(head, thorax, thr)
    assert counts[0, 0] == 8
    vals, where = M.series_values(head[0], thorax[0], thr)
    assert list(np.argsort(Q.order_key(vals[0]), kind="stable")) == [1, 4, 2, 6, 0, 3, 7, 5]
    ranks, _, _ = Q.mid_quantile_ranks(np.array([8]))               # 8 values: ranks 3, 4, 3, 4
    order_x = np.array([1, 4, 2, 6, 0, 3, 7, 5])
    assert np.array_equal(frames[0, 0], order_x[ranks[:, 0]])
    d = np.sqrt(head[0, :8, 0, 0] ** 2 + head[0, :8, 0, 1] ** 2)
    order_d = np.argsort(Q.order_key(d.astype(np.float32)), kind="stable")
    assert np.array_equal(frames[0, 3], order_d[ranks[:, 0]])
    # frames 2, 3 and 5 tie in float32 on y = 2 (5 is 1e-12 further in float64): the stable order keeps 2, 3, 5
    assert list(np.argsort(Q.order_key(vals[1]), kind="stable"))[:3] == [2, 3, 5]


@pytest.mark.parametrize("k", [1, 3])
@pytest.mark.parametrize("n_frame", [4, 9, 60, 400])
def test_composite_invariances(n_frame, k):
    """The aligned head does not change under (head, thorax) -> a (head, thorax) + b (a > 0) while the stationary set is held
    fixed, so sum dL/dhead + sum dL/dthorax = 0 per trial and coordinate and sum p . dL/dp over head and thorax = 0 per
    trial.  Without the thorax term of d, its 1/2, or the tip-length term into the base, they fail."""
    rng = np.random.default_rng(n_frame + 10 * k)
    head, thorax, consts = _batch(rng, 3, n_frame, k)
    head[:, :, :, 1] = np.round(head[:, :, :, 1] * 64) / 64                      # ties in the y series
    frames = M.stat_frames(head, thorax, 5e-5)
    h = torch.from_numpy(head).requires_grad_()
    t = torch.from_numpy(thorax).requires_grad_()
    c = torch.from_numpy(consts.astype(np.float64))
    g_out = torch.from_numpy(rng.normal(size=head.shape))
    gh, gt = torch.autograd.grad(M.aligned(h, t, c, frames), [h, t], g_out)
    scale = (gh.abs().sum(dim=(1, 2, 3)) + gt.abs().sum(dim=(1, 2, 3))).max().item() * (1 + np.abs(head).max() + np.abs(thorax).max())
    s1 = gh.sum(dim=(1, 2)) + gt.sum(dim=(1, 2))
    assert s1.abs().max().item() <= 1e-12 * scale
    s2 = (gh * h.detach()).sum(dim=(1, 2, 3)) + (gt * t.detach()).sum(dim=(1, 2, 3))
    assert s2.abs().max().item() <= 1e-12 * scale
    assert gt.abs().max().item() > 0                                             # the thorax does receive a gradient


def test_empty_stationary_set_gives_nan_statistics_and_no_scatter():
    rng = np.random.default_rng(1)
    head, thorax, consts = _batch(rng, 1, 20)
    gh, gt, gk, (cnt_h, _, cnt_t, _) = M.stats_vjp(head, thorax, consts, np.ones((1, 8)), -1e30)
    assert np.isnan(gk[0, 3]) and np.isfinite(gk[0, 4])
    assert cnt_t.sum() == 0 and cnt_h[0, :, 0].sum() == 4 * 3 and cnt_h[0, :, 1].sum() == 4 * 3   # series 4 only


def test_backward_argument_validation_without_gpu():
    from seqikpy_b200 import _native as N
    lib = N.load_library()
    f = lib.seqik_head_apply_backward_f32
    #      head aff g_out g_head part n_trial n_frame stream
    ok = [8, 8, 8, 8, 8, 4, 10, 0]
    bad = lambda args, i, v: [v if j == i else a for j, a in enumerate(args)]
    assert f(*bad(ok, 5, -1)) == -1 and b"negative" in lib.seqik_last_error()
    assert f(*bad(ok, 6, -1)) == -1
    assert f(0, 0, 0, 0, 0, 0, 10, 0) == 0 and f(0, 0, 0, 0, 0, 4, 0, 0) == 0    # empty: ok, nothing read
    for i in (0, 1, 2):                                                          # head, affine, grad_out NULL
        assert f(*bad(ok, i, 0)) == -1, i
        assert b"NULL" in lib.seqik_last_error()
    assert f(8, 8, 8, 0, 0, 4, 10, 0) == 0                                       # both outputs NULL: nothing to do
    for g in (lib.seqik_head_affine_backward_f32, lib.seqik_head_affine_backward_f64):
        #      head thorax kp series counts consts aff g_aff g_head g_thorax g_consts scratch n_trial n_frame stream
        ok = [8, 8, 3, 8, 8, 8, 8, 8, 8, 0, 0, 0, 4, 10, 0]
        assert g(*bad(ok, 12, -1)) == -1 and b"negative" in lib.seqik_last_error()
        assert g(*bad(ok, 13, -1)) == -1
        assert g(*bad(ok, 12, 0)) == 0                                           # no trials: ok
        assert g(*bad(ok, 13, 0)) == -1 and b"empty recording" in lib.seqik_last_error()
        for i in (0, 1, 3, 4, 5, 6, 7, 8):                                       # every required pointer
            assert g(*bad(ok, i, 0)) == -1, i
            assert b"NULL" in lib.seqik_last_error()
        assert g(*bad(ok, 2, 0)) == -1 and b"key point" in lib.seqik_last_error()
        assert g(*bad(ok, 13, 1 << 31)) == -1 and b"too many frames" in lib.seqik_last_error()
        assert g(*bad(ok, 13, 1025)) == -1 and b"scratch" in lib.seqik_last_error()   # long recordings need scratch
