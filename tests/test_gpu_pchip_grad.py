"""GPU tests of the pchip resampler's backward (seqik_pchip_resample_backward_f32/_f64, behind engine.pchip_resample's
autograd): the launch paths against each other bit for bit, the float64 model's autograd (tests/model_pchip.py) within
the per-knot bound of DESIGN.md 5.3, ties, down-sampling, +-inf inputs, autograd against the direct call, and an LBFGS fit
of capture-rate angles through pchip_resample -> forward_kinematics."""
import numpy as np
import pytest
import torch

import model_pchip
from test_pchip_grad_cpu import cases

pytestmark = pytest.mark.gpu
RATIOS = {}                        # largest observed |kernel - model| / bound, per dtype (printed by the last test)


@pytest.fixture(scope="module")
def E():
    assert torch.cuda.is_available()
    from seqikpy_b200 import engine
    return engine


def bits(t):
    return t.contiguous().view(torch.int64 if t.dtype == torch.float64 else torch.int32)


def model_grad(y, g, ts, new_ts, f32):
    """Autograd of the float64 model: y (rows, n), g (rows, m) float64 numpy -> (grad (rows, n), per-knot bound / u)."""
    n = y.shape[1]
    offs = model_pchip.float32_offsets(n, ts, new_ts) if f32 else None
    yt = torch.from_numpy(y).requires_grad_()
    out = model_pchip.resample(yt, ts, new_ts, offs)
    grad, = torch.autograd.grad(out, yt, torch.from_numpy(g))
    k, s = model_pchip.grid(n, ts, new_ts)
    q = np.bincount(k, minlength=n - 1).max()
    w = np.abs(g) * (1 + s / ts) ** 3                                   # (rows, m)
    per_iv = np.zeros((y.shape[0], n - 1))
    for r in range(y.shape[0]):
        np.add.at(per_iv[r], k, w[r])
    pad = np.pad(per_iv, ((0, 0), (2, 2)))                              # intervals i-2 .. i+1 of knot i
    near = pad[:, 0:n] + pad[:, 1:n + 1] + pad[:, 2:n + 2] + pad[:, 3:n + 3]
    return grad.numpy(), 64 * (q + 1) * near


def end_tie(y):
    """Rows whose float32 end-slope decisions lie within 1e-3 relative of a tie (excluded from the float32 comparison)."""
    out = np.zeros(y.shape[0], dtype=bool)
    if y.shape[1] < 3:
        return out
    m = np.diff(y, axis=1)
    for m0, m1 in ((m[:, 0], m[:, 1]), (m[:, -1], m[:, -2])):
        d = (3 * m0 - m1) / 2
        out |= np.abs(d) <= 1e-3 * (np.abs(3 * m0) + np.abs(m1))
        out |= (np.sign(m0) != np.sign(m1)) & (np.abs(np.abs(d) - 3 * np.abs(m0)) <= 1e-3 * (np.abs(d) + 3 * np.abs(m0)))
    return out


def check_against_model(E, y, g, ts, new_ts, dtype, tag=""):
    """y (rows, n), g (rows, m) in `dtype` on the device as width-1 series; kernel gradient within the bound."""
    f32 = dtype == torch.float32
    got = E.pchip_resample_backward(y, g, ts, new_ts).double().cpu().numpy()
    yd, gd = y.double().cpu().numpy(), g.double().cpu().numpy()
    ref, bound = model_grad(yd, gd, ts, new_ts, f32)
    u = 2.0 ** -24 if f32 else 2.0 ** -53
    keep = ~end_tie(yd) if f32 else np.ones(len(yd), dtype=bool)
    err = np.abs(got - ref)[keep]
    b = u * bound[keep] + 1e-300
    ratio = float((err / b).max()) if err.size else 0.0
    RATIOS[str(dtype)] = max(RATIOS.get(str(dtype), 0.0), ratio)
    assert ratio <= 1.0, (tag, ts, new_ts, ratio)
    return got


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_against_model_on_resample_cases(E, dtype):
    rng = np.random.default_rng(21)
    for y, ts, new_ts in cases():
        m = model_pchip.n_out(y.shape[1], ts, new_ts)
        yt = torch.tensor(y, dtype=dtype, device="cuda")
        g = torch.tensor(rng.normal(size=(3, m)), dtype=dtype, device="cuda")
        check_against_model(E, yt, g, ts, new_ts, dtype, tag=y.shape)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_against_model_on_grooming_angles(E, grooming_leg, dtype):
    """The shipped angles (2 x 6000 x 7), 100 Hz -> 1 kHz, through the width-7 path; every channel against the model."""
    ang = torch.tensor(grooming_leg["ref_angles"], dtype=dtype, device="cuda")
    g = torch.randn((2, 60000, 7), dtype=dtype, device="cuda", generator=torch.Generator("cuda").manual_seed(3))
    got = E.pchip_resample_backward(ang, g, 0.01, 0.001)
    rows = ang.permute(0, 2, 1).reshape(14, 6000)
    grows = g.permute(0, 2, 1).reshape(14, 60000).contiguous()
    one = check_against_model(E, rows.contiguous(), grows, 0.01, 0.001, dtype, tag="grooming")       # as width-1 series
    assert np.array_equal(got.permute(0, 2, 1).reshape(14, 6000).double().cpu().numpy(), one)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_launch_paths_bit_identical(E, dtype):
    """Width 1, inside width 7, inside run-time widths 5 and 200 (grad_out read directly: the range exceeds the buffer),
    extreme up-sampling (direct reads at width 1 and 7), block rows strided over by CTAs, and repeated calls."""
    rng = np.random.default_rng(22)
    for n, ts, new_ts in [(300, 0.01, 0.001), (57, 1 / 30, 1 / 100), (40, 0.1, 0.3), (12, 0.01, 1e-5)]:
        m = model_pchip.n_out(n, ts, new_ts)
        y = torch.tensor(rng.normal(size=(3, n)).cumsum(1), dtype=dtype, device="cuda")
        g = torch.tensor(rng.normal(size=(3, m)), dtype=dtype, device="cuda")
        ref = E.pchip_resample_backward(y, g, ts, new_ts)
        for width, ch in ((7, 3), (5, 2), (200, 131)):
            yw = torch.tensor(rng.normal(size=(3, n, width)), dtype=dtype, device="cuda")
            gw = torch.tensor(rng.normal(size=(3, m, width)), dtype=dtype, device="cuda")
            yw[:, :, ch] = y
            gw[:, :, ch] = g
            got = E.pchip_resample_backward(yw, gw, ts, new_ts)[:, :, ch]
            assert torch.equal(bits(got), bits(ref)), (n, ts, new_ts, width)
        assert torch.equal(bits(E.pchip_resample_backward(y, g, ts, new_ts)), bits(ref))
        if new_ts < 1e-4:
            check_against_model(E, y, g, ts, new_ts, dtype, tag="direct")
    # 5000 block rows of 50 knots at width 7: grid.y < n_block, each CTA strides over block rows
    yb = torch.tensor(rng.normal(size=(5000, 50, 7)).cumsum(1), dtype=dtype, device="cuda")
    gb = torch.tensor(rng.normal(size=(5000, 500, 7)), dtype=dtype, device="cuda")
    big = E.pchip_resample_backward(yb, gb, 0.01, 0.001)
    for b in (0, 1, 2047, 2048, 4999):
        assert torch.equal(bits(big[b]), bits(E.pchip_resample_backward(yb[b:b + 1], gb[b:b + 1], 0.01, 0.001)[0])), b


@pytest.mark.parametrize("ts", [1.0, 0.5, 0.25])
def test_ties_decided_identically(E, ts):
    """Dyadic steps and integer data (the float32 decisions are exact): plateaus, sign changes, an end slope zeroed
    (m0 = 1, m1 = 3) and one clamped to 3 m0 (m0 = 1, m1 = -5), at both ends; float32 against the model."""
    rows = np.array([[0, 1, 4, 3, 5, 5, 5, 2, 2, 7, 8, 8],               # left end zeroed (m0 = 1, m1 = 3); plateaus
                     [0, 1, -4, -3, -1, -1, 0, 3, 3, 1, 2, 3],           # left end clamped (m0 = 1, m1 = -5); sign changes
                     [8, 8, 3, 5, 4, 4, 6, 5, 2, 5, 4, 3],
                     [0, 0, 0, 1, 2, 3, 4, 4, 1, 9, 8, 4],
                     [5, 4, 4, 4, 3, 2, 2, 2, 2, 2, 2, 2]], dtype=float)
    rows = np.concatenate([rows, rows[:, ::-1], -rows])
    rng = np.random.default_rng(23)
    for new_ts in (ts / 4, ts * 2.5):
        m = model_pchip.n_out(rows.shape[1], ts, new_ts)
        for dtype in (torch.float32, torch.float64):
            y = torch.tensor(rows, dtype=dtype, device="cuda")
            g = torch.tensor(rng.integers(-3, 4, size=(len(rows), m)), dtype=dtype, device="cuda")
            f32 = dtype == torch.float32
            got = E.pchip_resample_backward(y, g, ts, new_ts).double().cpu().numpy()
            ref, bound = model_grad(rows, g.double().cpu().numpy(), ts, new_ts, f32)
            u = 2.0 ** -24 if f32 else 2.0 ** -53
            assert (np.abs(got - ref) <= u * bound).all(), (ts, new_ts, dtype, np.abs(got - ref).max())
    # the branches are taken: clamped (d0/dy = 3 (dm0/dy)) differs from the unclamped formula's gradient
    y = torch.tensor([[0.0, 1.0, -4.0, -3.0]], dtype=torch.float32, device="cuda")
    g = torch.zeros((1, model_pchip.n_out(4, ts, ts / 4)), dtype=torch.float32, device="cuda")
    g[0, 1] = 1.0                                                       # one sample at s = h / 4 of interval 0
    got = E.pchip_resample_backward(y, g, ts, ts / 4).double().cpu().numpy()
    ref, _ = model_grad(y.double().cpu().numpy(), g.double().cpu().numpy(), ts, ts / 4, True)
    assert np.abs(got - ref).max() <= 1e-6 and abs(ref[0, 1]) > 0.1


def raw_backward(E, y, g, ts, new_ts, width):
    """The C entry point with grad_in pre-filled with NaN: every knot must be written."""
    from seqikpy_b200 import _native as N
    lib = N.load_library()
    out = torch.full_like(y, float("nan"))
    fn = lib.seqik_pchip_resample_backward_f32 if y.dtype == torch.float32 else lib.seqik_pchip_resample_backward_f64
    n_block, n = y.shape[0], y.shape[1]
    m = g.shape[1]
    assert fn(y.data_ptr(), g.data_ptr(), out.data_ptr(), n_block, n, m, width, ts, new_ts, 0) == 0
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_downsampling_and_two_samples(E, dtype):
    """0.01 -> 0.025, 0.1 -> 0.3 and 0.01 -> 0.1 (whole CTAs without a sample at width 64): every knot written, the knots
    of intervals without samples get their slope terms, and the model agrees; n = 2 as well."""
    rng = np.random.default_rng(24)
    for n, ts, new_ts in [(200, 0.01, 0.025), (90, 0.1, 0.3), (300, 0.01, 0.1), (2, 0.01, 0.001), (2, 0.1, 0.3)]:
        m = model_pchip.n_out(n, ts, new_ts)
        for width in (1, 7, 64):
            y = torch.tensor(rng.normal(size=(2, n, width)).cumsum(1), dtype=dtype, device="cuda")
            g = torch.tensor(rng.normal(size=(2, m, width)), dtype=dtype, device="cuda")
            got = raw_backward(E, y, g, ts, new_ts, width)
            assert not torch.isnan(got).any(), (n, ts, new_ts, width)
            assert torch.equal(bits(got), bits(E.pchip_resample_backward(y, g, ts, new_ts)))
            rows = y.permute(0, 2, 1).reshape(-1, n).contiguous()
            grows = g.permute(0, 2, 1).reshape(-1, m).contiguous()
            check_against_model(E, rows, grows, ts, new_ts, dtype, tag=("down", n, width))
        if n > 10 and new_ts / ts > 2:
            k, _ = model_pchip.grid(n, ts, new_ts)
            empty = np.setdiff1d(np.arange(1, n - 2), k)                # intervals without a sample
            assert empty.size and (got[0, empty].abs() > 0).any()


def test_inf_inputs_get_zero_gradient(E):
    rng = np.random.default_rng(25)
    for dtype in (torch.float32, torch.float64):
        y = torch.tensor(rng.normal(size=(3, 30)), dtype=dtype, device="cuda")
        y[0, 7] = float("inf")
        y[2, 3] = -float("inf")
        m = model_pchip.n_out(30, 0.01, 0.002)
        g = torch.tensor(rng.normal(size=(3, m)), dtype=dtype, device="cuda")
        got = E.pchip_resample_backward(y, g, 0.01, 0.002)
        assert got[0, 7] == 0 and got[0, -1] == 0 and got[2, 3] == 0 and got[2, -1] == 0 and got[1, -1] != 0
        clean = y.clone()
        clean[0, 7] = 0; clean[0, -1] = 0; clean[2, 3] = 0; clean[2, -1] = 0
        ref = E.pchip_resample_backward(clean, g, 0.01, 0.002)
        ref[0, 7] = 0; ref[0, -1] = 0; ref[2, 3] = 0; ref[2, -1] = 0
        assert torch.equal(bits(got), bits(ref))
        x = y.clone().requires_grad_()
        E.pchip_resample(x, 0.01, 0.002).backward(g)
        assert torch.equal(bits(x.grad), bits(got))
        y[1, 4] = float("nan")
        with pytest.raises(ValueError):
            E.pchip_resample_backward(y, g, 0.01, 0.002)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_autograd_equals_direct_call(E, dtype):
    rng = np.random.default_rng(26)
    for shape in ((4, 120), (3, 120, 7)):
        y = torch.tensor(rng.normal(size=shape).cumsum(1), dtype=dtype, device="cuda")
        x = y.clone().requires_grad_()
        out = E.pchip_resample(x, 0.01, 0.001)
        assert out.requires_grad and torch.equal(bits(out.detach()), bits(E.pchip_resample(y, 0.01, 0.001)))
        with torch.no_grad():
            assert E.pchip_resample(x, 0.01, 0.001).grad_fn is None
        # a non-contiguous incoming gradient
        gt = torch.tensor(rng.normal(size=out.shape[::-1]), dtype=dtype, device="cuda")
        g = gt.permute(*range(out.dim() - 1, -1, -1))
        assert not g.is_contiguous()
        gx, = torch.autograd.grad(out, x, g)
        assert torch.equal(bits(gx), bits(E.pchip_resample_backward(y, g.contiguous(), 0.01, 0.001)))
        # a loss on a slice
        gx, = torch.autograd.grad(E.pchip_resample(x, 0.01, 0.001)[1:, 100:500].pow(2).sum(), x)
        full = torch.zeros_like(out)
        full[1:, 100:500] = 2 * out.detach()[1:, 100:500]
        assert torch.equal(bits(gx), bits(E.pchip_resample_backward(y, full, 0.01, 0.001)))
        # second derivatives are not supported
        gx, = torch.autograd.grad(E.pchip_resample(x, 0.01, 0.001).pow(2).sum(), x, create_graph=True)
        with pytest.raises(RuntimeError, match="once_differentiable"):
            gx.sum().backward()


def test_lbfgs_fit_of_capture_rate_angles(E):
    """12 chains x 200 frames of float32 angles at 100 Hz; the targets are forward_kinematics(pchip_resample(true angles,
    0.01, 0.001)); from angles 0.05 rad off, LBFGS through pchip_resample -> forward_kinematics recovers the angles."""
    from test_gpu_fk_grad import synthetic_legs
    th, seg, org, _ = synthetic_legs(2, 2000, 11)
    th = th[:, ::10]                                                    # 100 Hz
    rng = np.random.default_rng(27)
    n_chain = seg.shape[0]
    params = torch.tensor(np.concatenate([seg, np.zeros((n_chain, 28))], 1), dtype=torch.float32, device="cuda")
    origin = torch.tensor(org, dtype=torch.float32, device="cuda")
    true = torch.tensor(th, dtype=torch.float32, device="cuda")
    with torch.no_grad():
        target = E.forward_kinematics(E.pchip_resample(true, 0.01, 0.001), origin, params)
    q = (true + torch.tensor(rng.choice([-0.05, 0.05], th.shape), dtype=torch.float32, device="cuda")).requires_grad_()
    opt = torch.optim.LBFGS([q], lr=1, max_iter=200, history_size=50, tolerance_grad=0, tolerance_change=0,
                            line_search_fn="strong_wolfe")

    def closure():
        opt.zero_grad()
        # summed in float64: the line search compares losses that differ far below float32 resolution near the optimum
        loss = (E.forward_kinematics(E.pchip_resample(q, 0.01, 0.001), origin, params) - target).double().pow(2).sum()
        loss.backward()
        return loss

    for _ in range(30):
        opt.step(closure)
        with torch.no_grad():
            resid = float((E.forward_kinematics(E.pchip_resample(q, 0.01, 0.001), origin, params) - target).norm(dim=-1).max())
        worst = float((q.detach() - true).abs().max())
        if resid < 1e-4 and worst < 1e-4:
            break
    evals = opt.state[opt._params[0]]["func_evals"]
    err = (q.detach() - true).abs()
    rms, p99 = float(err.pow(2).mean().sqrt()), float(err.flatten().quantile(0.99))
    print(f"LBFGS: {evals} evaluations, worst angle error {worst:.3e} rad (rms {rms:.3e}, 99th percentile {p99:.3e}), "
          f"worst joint residual {resid:.3e} mm")
    # measured on a B200: rms 7.6e-4 rad, worst 2.8e-2 rad, residual 3.6e-2 mm; the worst angles sit where the key points
    # barely depend on them, so the fit is judged by the rms error and the residual, the worst error only has to improve
    assert rms < 2e-3 and resid < 0.1 and worst < 0.04, (evals, rms, worst, resid)


def test_report_bound_ratios():
    print("largest |kernel - model| / bound:", {k: f"{v:.3g}" for k, v in RATIOS.items()})
