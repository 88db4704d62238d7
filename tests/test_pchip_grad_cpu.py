"""CPU side of the differentiable pchip resampler: the float64 torch model against scipy's pchip_interpolate (called as the
reference calls it), its autograd against finite differences, the moment decomposition the backward kernel computes
against the model's autograd, and the argument checks of seqik_pchip_resample_backward_f32/_f64 (they run before any
CUDA call)."""
import numpy as np
import torch
from scipy.interpolate import pchip_interpolate

import model_pchip

GRIDS = [(0.01, 0.001), (1.0, 0.5), (0.005, 0.0007), (1 / 30, 1 / 100), (0.01, 0.025), (0.1, 0.3)]


def reference_resample(signal, original_ts, new_ts):                    # as tests/test_gpu_resample.py calls scipy
    total = signal.shape[0] * original_ts
    return np.array(pchip_interpolate(np.arange(0, total, original_ts), signal, np.arange(0, total, new_ts)))


def cases():
    """The resample test's series: random walks, plateaus, integer values, up- and down-sampling, n = 2, 3, 4."""
    rng = np.random.default_rng(3)
    out = []
    for case in range(42):
        n = [2, 3, 4][case % 3] if case >= 36 else int(rng.integers(2, 50))
        ts, new_ts = GRIDS[case % 6]
        y = rng.normal(size=(3, n)).cumsum(axis=1)
        if case % 3 == 0:
            y[:, n // 3:n // 2 + 1] = y[:, n // 3:n // 3 + 1]
        if case % 4 == 0:
            y = np.round(y)
        if len(np.arange(0, n * ts, ts)) != n:                           # numpy's arange over-ran: the reference raises there
            continue
        out.append((y, ts, new_ts))
    return out


def vjp_by_moments(y, g, ts, new_ts):
    """The backward kernel's decomposition (include/seqik.h), in float64 numpy: per-interval moments, then per knot."""
    n = len(y)
    h = ts
    k, s = model_pchip.grid(n, ts, new_ts)
    M = np.zeros((4, n - 1))
    for p in range(4):
        np.add.at(M[p], k, g * s ** p)
    A, B = M[2] / h, M[3] / h ** 2
    g_left, g_right, g_m = M[1] - 2 * A + B, B - A, 3 * A - 2 * B
    m = np.diff(y) / h
    lo, hi = np.zeros(n), np.zeros(n)                                    # dd_i/dm_{i-1}, dd_i/dm_i (knot 0: dd/dm1 in lo,
    if n == 2:                                                           # knot n-1: dd/dm_{n-3} in hi)
        hi[0], lo[1] = 1.0, 1.0
    else:
        def edge(m0, m1):
            d = (3 * m0 - m1) / 2
            if np.sign(d) != np.sign(m0):
                return 0.0, 0.0
            if np.sign(m0) != np.sign(m1) and abs(d) > 3 * abs(m0):
                return 3.0, 0.0
            return 1.5, -0.5
        hi[0], lo[0] = edge(m[0], m[1])
        lo[n - 1], hi[n - 1] = edge(m[n - 2], m[n - 3])
        for i in range(1, n - 1):
            a, b = m[i - 1], m[i]
            if np.sign(a) == np.sign(b) and a != 0 and b != 0:
                lo[i], hi[i] = 2 * b * b / (a + b) ** 2, 2 * a * a / (a + b) ** 2
    gd = np.zeros(n)
    gd[1:] += g_right
    gd[:-1] += g_left
    gm = g_m + (gd * hi)[:-1] + (gd * lo)[1:]
    if n > 2:
        gm[1] += gd[0] * lo[0]                                            # d_0 depends on m_1
        gm[n - 3] += gd[n - 1] * hi[n - 1]                                # d_{n-1} depends on m_{n-3}
    out = np.zeros(n)
    out[:-1] += M[0] - gm / h
    out[1:] += gm / h
    return out


def test_model_equals_scipy():
    for y, ts, new_ts in cases():
        got = model_pchip.resample(torch.from_numpy(y), ts, new_ts).numpy()
        for r in range(3):
            ref = reference_resample(y[r], ts, new_ts)
            assert got[r].shape == ref.shape
            assert np.abs(got[r] - ref).max() <= 1e-12 * max(1.0, np.abs(ref).max()), (len(y[r]), ts, new_ts)
    line = model_pchip.resample(torch.tensor([1.0, 3.0], dtype=torch.float64), 1.0, 0.25).numpy()
    assert np.allclose(line, 1.0 + 2.0 * np.arange(0, 2.0, 0.25), rtol=0, atol=1e-15)


def test_model_gradcheck_away_from_ties():
    rng = np.random.default_rng(5)
    for n, (ts, new_ts) in [(2, (1.0, 0.25)), (3, (0.01, 0.001)), (4, (0.1, 0.3)), (7, (0.01, 0.025)), (25, (1 / 30, 1 / 100))]:
        y = torch.from_numpy(rng.normal(size=(2, n)).cumsum(axis=1)).requires_grad_()
        assert torch.autograd.gradcheck(lambda v: model_pchip.resample(v, ts, new_ts), (y,), eps=1e-7, atol=1e-6, rtol=1e-5)


def test_moment_decomposition_equals_model_autograd():
    """Every resample case, plus clamped and zeroed end slopes: the decomposition equals autograd of the model."""
    rng = np.random.default_rng(6)
    extra = [(np.array([[0.0, 1.0, 4.0, 3.0, 5.0]] * 3), 1.0, 0.25),           # m0 = 1, m1 = 3: end slope zeroed
             (np.array([[0.0, 1.0, -4.0, -3.0, -1.0]] * 3), 1.0, 0.25)]        # m0 = 1, m1 = -5: end slope clamped to 3
    for y, ts, new_ts in cases() + extra:
        yt = torch.from_numpy(y).requires_grad_()
        out = model_pchip.resample(yt, ts, new_ts)
        g = rng.normal(size=out.shape)
        auto, = torch.autograd.grad(out, yt, torch.from_numpy(g))
        for r in range(3):
            mine = vjp_by_moments(y[r], g[r], ts, new_ts)
            scale = np.abs(g[r]).sum()
            assert np.abs(mine - auto[r].numpy()).max() <= 1e-13 * scale, (y.shape, ts, new_ts)


def test_float32_offsets_follow_the_kernel_recurrence():
    k, s = model_pchip.grid(40, 0.01, 0.001)
    s32 = model_pchip.float32_offsets(40, 0.01, 0.001)
    assert np.abs(s32 - s).max() <= 4 * np.finfo(np.float32).eps * 0.01 * 2      # the tail interval spans 2 steps
    assert (s32 == s32.astype(np.float32)).all()


def test_backward_argument_validation_without_gpu():
    from seqikpy_b200 import _native as N
    lib = N.load_library()
    for f in (lib.seqik_pchip_resample_backward_f32, lib.seqik_pchip_resample_backward_f64):
        #        in grad_out grad_in n_block n  m  width ts  new_ts stream
        assert f(8, 8, 8, -1, 5, 50, 1, 0.01, 0.001, 0) == -1                 # negative sizes
        assert b"negative" in lib.seqik_last_error()
        for args in ((8, 8, 8, 1, -5, 50, 1), (8, 8, 8, 1, 5, -50, 1), (8, 8, 8, 1, 5, 50, -1)):
            assert f(*args, 0.01, 0.001, 0) == -1
        assert f(8, 8, 8, 1, 1, 10, 1, 0.01, 0.001, 0) == -1                   # fewer than 2 samples
        assert b"at least 2" in lib.seqik_last_error()
        for k in range(3):                                                     # each pointer NULL
            args = [8, 8, 8, 1, 5, 50, 1, 0.01, 0.001, 0]
            args[k] = 0
            assert f(*args) == -1, k
            assert b"NULL" in lib.seqik_last_error()
        for ts, new_ts in ((0.0, 0.001), (0.01, 0.0), (-0.01, 0.001), (0.01, float("nan"))):
            assert f(8, 8, 8, 1, 5, 50, 1, ts, new_ts, 0) == -1                # non-positive steps
            assert b"positive" in lib.seqik_last_error()
        assert f(8, 8, 8, 1, 5, 50, 257, 0.01, 0.001, 0) == -1                 # more than 256 channels
        assert b"256" in lib.seqik_last_error()
        assert f(0, 0, 0, 0, 5, 50, 7, 0.01, 0.001, 0) == 0                    # empty batch: ok, nothing read
        assert f(0, 0, 0, 4, 5, 50, 0, 0.01, 0.001, 0) == 0
