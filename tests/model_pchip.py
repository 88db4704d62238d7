"""Float64 torch model of the pchip resampler (scipy.interpolate.pchip_interpolate on uniform grids, as the reference's
utils.interpolate_signal calls it): the specification that the backward kernel's gradients are checked against through
torch autograd.  Knot slopes follow scipy's PchipInterpolator (Fritsch-Carlson harmonic mean, _edge_case with its two
clamps); the gradient is taken on the branch each decision took, as the kernel's is."""
import numpy as np
import torch


def n_out(n, original_ts, new_ts):
    """Length of np.arange(0, n * original_ts, new_ts), as engine.pchip_resample computes it."""
    return int(np.ceil((n * original_ts) / new_ts))


def _edge(m0, m1):
    d = (3 * m0 - m1) / 2                                       # _edge_case with h0 = h1
    zero = torch.sign(d) != torch.sign(m0)
    clamp = ~zero & (torch.sign(m0) != torch.sign(m1)) & (d.abs() > 3 * m0.abs())
    return torch.where(zero, torch.zeros_like(d), torch.where(clamp, 3 * m0, d))


def slopes(y, h):
    """Knot derivatives d (..., n) of y (..., n) on a uniform grid of step h."""
    m = (y[..., 1:] - y[..., :-1]) / h
    if y.shape[-1] == 2:
        return torch.cat([m, m], dim=-1)
    a, b = m[..., :-1], m[..., 1:]
    ok = (torch.sign(a) == torch.sign(b)) & (a != 0) & (b != 0)
    den = torch.where(ok, a + b, torch.ones_like(a))           # a safe denominator off the branch keeps the gradient finite
    inner = torch.where(ok, 2 * a * b / den, torch.zeros_like(a))
    d0 = _edge(m[..., :1], m[..., 1:2])
    dn = _edge(m[..., -1:], m[..., -2:-1])
    return torch.cat([d0, inner, dn], dim=-1)


def grid(n, original_ts, new_ts):
    """(interval index, offset from its left knot) of every sample of the new grid, in float64 as the kernel computes
    them: k ts <= u new_ts < (k + 1) ts, the samples past the last knot in the last interval."""
    xs = np.arange(n) * float(original_ts)
    xn = np.arange(n_out(n, original_ts, new_ts)) * float(new_ts)
    k = np.clip(np.searchsorted(xs, xn, side="right") - 1, 0, n - 2)
    return k, xn - xs[k]


def resample(y, original_ts, new_ts, offsets=None):
    """y (..., n) float64 -> (..., m).  `offsets` replaces the sample offsets s (e.g. by the float32 kernel's)."""
    n = y.shape[-1]
    h = float(original_ts)
    k, s = grid(n, original_ts, new_ts)
    if offsets is not None:
        s = offsets
    k = torch.as_tensor(k, device=y.device)
    s = torch.as_tensor(s, dtype=y.dtype, device=y.device)
    d = slopes(y, h)
    m = (y[..., 1:] - y[..., :-1]) / h
    yk, dk, dk1, mk = y[..., :-1][..., k], d[..., :-1][..., k], d[..., 1:][..., k], m[..., k]
    t = (dk + dk1 - 2 * mk) / h
    c0, c1 = t / h, (mk - dk) / h - t
    return yk + dk * s + c1 * s ** 2 + c0 * s ** 3


def float32_offsets(n, original_ts, new_ts):
    """The float32 kernel's offsets: s0 = (float)(u_lo new_ts - k ts) in float64, then fmaf(u - u_lo, (float)new_ts, s0)
    (float32 fma is exact in float64 before its one rounding)."""
    k, _ = grid(n, original_ts, new_ts)
    m = len(k)
    u = np.arange(m)
    first = np.full(n - 1, m, dtype=np.int64)
    np.minimum.at(first, k, u)
    u_lo = first[k]
    s0 = (u_lo * float(new_ts) - k * float(original_ts)).astype(np.float32).astype(np.float64)
    dt = np.float64(np.float32(new_ts))
    return ((u - u_lo) * dt + s0).astype(np.float32).astype(np.float64)
