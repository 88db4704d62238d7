"""Exact models of the mid-quantile select (csrc/seqik_kernels.cu) and of the alignment statistics built on it.  TEST/DEV TOOL.

The four order statistics behind a mid-quantile are elements of the input, and the build has no fma contraction
(-fmad=false) and IEEE sqrtf / division, so the kernels' results can be computed exactly on the CPU:

* ``mid_quantile_exact`` -- what ``seqik_mid_quantile_f32`` returns, bit for bit: the order statistics of the m smallest
  keys (``order_key``: -0 < +0, a NaN with the sign bit clear above +inf, one with it set below -inf), the ranks and weights
  of ``quantile_pos`` (float64 position, float32 weight), and ``0.5f * ((a0 + (a1 - a0) f45) + (b0 + (b1 - b0) f55))`` in
  float32, one rounding per operation.
* ``route`` -- which kernel and which internal path a series takes (``mid_quantile_warp_kernel``, the sampled-range
  ``mid_quantile_long_kernel`` and its hand-off to ``mid_quantile_kernel``), and how ``warp_select4`` ends.  The constants
  are the source's.  It decides nothing about the values; it tells a test which code its cases reach.
* ``leg_stats_exact`` / ``head_rows_exact`` -- the affine rows of ``seqik_leg_affine_from_pose_f32`` (and of the three
  separate entry points) and of ``seqik_head_affine_f32``, in float32 with the kernels' operation order.

The product never imports this file.
"""
import numpy as np

WQ_N = 1024                 # mid_quantile_warp_kernel: series of up to this many samples
LQ_CAND = 4096              # mid_quantile_long_kernel: keys to shared memory directly up to this length; candidate cap
LQ_SAMPLE = 2048            # strided sample of the long kernel
LQ_BINS = 4096
SEL_CACHE = 8192            # mid_quantile_kernel caches the keys of series up to this length
KEY_INF = 0xFF800000        # order_key(+inf)
DIRECT = 64                 # warp_select4 reads the ranks off directly with at most this many candidates

ROUTES = ("warp", "long-small", "long-direct", "long-sweep", "retry-cached", "retry-global")
ENDS = ("constant", "gather", "compact", "passes")
RETRY_REASONS = ("empty-sample", "rank-outside-range", "too-many-candidates")


def order_key(x):
    """float32 array -> uint32 order keys (the kernels' ``order_key``)."""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)
    return np.where(u & np.uint32(0x80000000), ~u, u | np.uint32(0x80000000)).astype(np.uint32)


def key_value(k):
    """uint32 order keys -> float32 values (``key_value``)."""
    k = np.asarray(k, dtype=np.uint32)
    return np.where(k & np.uint32(0x80000000), k & np.uint32(0x7FFFFFFF), ~k).astype(np.uint32).view(np.float32)


def quantile_pos(q, m):
    """``quantile_pos``: m (int64 array, >= 1) -> (lo, frac) with the position q (m - 1) in float64 and a float32 weight."""
    m = np.asarray(m, dtype=np.int64)
    v = q * (m - 1).astype(np.float64)
    lo = np.minimum(np.floor(v).astype(np.int64), m - 1)
    return lo, (v - lo.astype(np.float64)).astype(np.float32)


def mid_quantile_ranks(m):
    """``mid_quantile_ranks``: (4, rows) int64 ranks among the m smallest, f45, f55."""
    m = np.asarray(m, dtype=np.int64)
    lo45, f45 = quantile_pos(0.45, m)
    lo55, f55 = quantile_pos(0.55, m)
    ranks = np.stack([lo45, lo45 + 1, lo55, lo55 + 1])
    return np.minimum(ranks, m - 1), f45, f55


def mid_quantile_value(a0, a1, b0, b1, f45, f55):
    """``mid_quantile_value`` in float32, one rounding per operation."""
    f32 = np.float32
    with np.errstate(all="ignore"):
        q0 = f32(a0) + (f32(a1) - f32(a0)) * f32(f45)
        q1 = f32(b0) + (f32(b1) - f32(b0)) * f32(f55)
        return (f32(0.5) * (q0 + q1)).astype(np.float32)


def _counts(x, counts):
    n = x.shape[1]
    if counts is None:
        return np.full(x.shape[0], n, dtype=np.int64)
    return np.asarray(counts, dtype=np.int64).reshape(x.shape[0])


def order_statistics(x, counts=None):
    """(4, rows) float32 order statistics a0, a1, b0, b1 of every row (rows with m <= 0: NaN) and f45, f55."""
    x = np.asarray(x, dtype=np.float32)
    m = _counts(x, counts)
    keys = np.sort(order_key(x), axis=1)
    ranks, f45, f55 = mid_quantile_ranks(np.maximum(m, 1))
    vals = key_value(np.take_along_axis(keys, ranks.T, axis=1)).T.copy()
    vals[:, m <= 0] = np.nan
    return vals, f45, f55


def mid_quantile_exact(x, counts=None):
    """x (rows, n) float32, counts (rows,) or None -> (rows,) float32: seqik_mid_quantile_f32's result on every row."""
    x = np.asarray(x, dtype=np.float32)
    vals, f45, f55 = order_statistics(x, counts)
    out = mid_quantile_value(vals[0], vals[1], vals[2], vals[3], f45, f55)
    out[_counts(x, counts) <= 0] = np.nan
    return out


# ------------------------------------------------------------------------------------------------------------ routes
def _bitlen(v):
    return int(v).bit_length()


def select_end(keys, ranks):
    """How ``warp_select4`` ends on ``keys`` (uint32) for the four ``ranks`` (non-decreasing): 'constant' (hi == 0),
    'gather' (first pass, at most 64 keys in the ranks' bins), 'compact' (at most 64 keys left after a compaction) or
    'passes' (the last 8-bit digit was resolved by a histogram: more than 64 keys share a prefix with a rank to the end)."""
    keys = np.asarray(keys, dtype=np.uint32).astype(np.int64)
    n = keys.size
    kmin = int(keys.min())
    hi = _bitlen(int(keys.max()) - kmin)
    if hi == 0:
        return "constant"
    cur = keys - kmin                                      # offsets (the kernel subtracts kmin on the fly until compaction)
    mask = ~((1 << hi) - 1) & 0xFFFFFFFF
    prefix = [0, 0, 0, 0]
    rank = [int(r) for r in ranks]
    cnt = n
    while hi > 0:
        lo = max(hi - 8, 0)
        dm = (1 << (hi - lo)) - 1
        one = prefix[3] == prefix[0] and cnt == n
        in_bins, seen = 0, set()
        new_prefix = list(prefix)
        for k in range(4):
            grp = cur[(cur & mask) == prefix[k]]
            hist = np.bincount((grp >> lo) & dm, minlength=dm + 1)
            cum = np.cumsum(hist)
            b = int(np.searchsorted(cum, rank[k], side="right"))
            below = int(cum[b - 1]) if b > 0 else 0
            if (prefix[k], b) not in seen:
                seen.add((prefix[k], b))
                in_bins += int(hist[b])
            new_prefix[k] = prefix[k] | (b << lo)
            rank[k] -= below
        prefix = new_prefix
        mask |= dm << lo
        hi = lo
        if hi == 0:
            break
        if one and in_bins <= DIRECT:
            return "gather"
        cur = cur[np.isin(cur & mask, prefix)]
        cnt = cur.size
        if cnt <= DIRECT:
            return "compact"
    return "passes"


def route(row, m=None, offset=0):
    """The path of one series through seqik_mid_quantile_f32.  row: (n,) float32; m: the count (None: n); offset: the
    row's start in floats past a 16-byte boundary.  -> dict(route ('empty' for m <= 0), end (warp_select4's, or None),
    aligned, reason (of a hand-off to the general kernel, or None), shift, below, cand)."""
    keys = order_key(row)
    n = keys.size
    m = n if m is None else int(m)
    info = dict(route=None, end=None, aligned=offset % 4 == 0, reason=None, shift=None, below=None, cand=None)
    if m <= 0:                                                 # every kernel writes NaN before it reads the series
        info["route"] = "empty"
        return info
    ranks = mid_quantile_ranks(np.array([m]))[0][:, 0]
    if n <= LQ_CAND:
        info["route"] = "warp" if n <= WQ_N else "long-small"
        info["end"] = select_end(keys, ranks)
        return info
    retry = "retry-cached" if n <= SEL_CACHE else "retry-global"
    stride = n // LQ_SAMPLE
    sample = keys[np.arange(LQ_SAMPLE, dtype=np.int64) * stride]
    sample = sample[sample < KEY_INF]
    if sample.size == 0:
        info.update(route=retry, reason="empty-sample")
        return info
    smin, smax = int(sample.min()), int(sample.max())
    shift = max(0, _bitlen(smax - smin) - 12)
    k64 = keys.astype(np.int64)
    below = int((k64 < smin).sum())
    inr = k64[(k64 >= smin) & (k64 <= smax)]
    bins = (inr - smin) >> shift
    hist = np.bincount(bins, minlength=LQ_BINS)
    cum = np.cumsum(hist)
    info.update(shift=shift, below=below)
    b = []
    for r in ranks:
        if r < below or r - below >= inr.size:
            info.update(route=retry, reason="rank-outside-range")
            return info
        b.append(int(np.searchsorted(cum, r - below, side="right")))
    distinct = sorted(set(b))
    c = int(sum(hist[d] for d in distinct))
    info["cand"] = c
    if shift > 0 and c > LQ_CAND:
        info.update(route=retry, reason="too-many-candidates")
        return info
    if shift == 0:
        info["route"] = "long-direct"
        return info
    cand = inr[np.isin(bins, distinct)]
    lrank, before = [], 0
    for t in range(4):
        if t > 0 and b[t] != b[t - 1]:
            before += int(hist[b[t - 1]])
        lrank.append(before + int(ranks[t]) - below - (int(cum[b[t] - 1]) if b[t] > 0 else 0))
    info.update(route="long-sweep", end=select_end(cand, lrank))
    return info


def routes(x, counts=None, offset=0):
    """``route`` of every row of x (rows, n), row 0 starting ``offset`` floats past a 16-byte boundary."""
    x = np.asarray(x, dtype=np.float32)
    n = x.shape[1]
    m = _counts(x, counts)
    return [route(x[r], m[r], offset + r * n) for r in range(x.shape[0])]


# ------------------------------------------------------------------------------------------------------------ alignment rows
def leg_series_exact(pose):
    """pose (n_chain, n_frame, 5, 3) float32 -> (n_chain, 7, n_frame) float32: ``leg_series_kernel``'s series (coxa x, y,
    z; the four segment lengths as sqrt((dx dx + dy dy) + dz dz), every operation rounded to float32)."""
    p = np.asarray(pose, dtype=np.float32)
    d = p[:, :, 1:] - p[:, :, :-1]                                             # (chain, frame, 4, 3)
    sq = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
    return np.concatenate([p[:, :, 0].transpose(0, 2, 1), np.sqrt(sq).transpose(0, 2, 1)], axis=1).astype(np.float32)


def leg_stats_exact(pose, consts, include_claw):
    """-> (series (n_chain, 7, n_frame), stats (n_chain, 7), affine (n_chain, 8)) as the leg statistics kernels compute
    them: ``len = (s3 + s4) + s5 [+ s6]``, ``a3 = k3 / len``, row (s0, s1, s2, a3, k0, k1, k2, 0)."""
    series = leg_series_exact(pose)
    n_chain, _, n_frame = series.shape
    stats = mid_quantile_exact(series.reshape(n_chain * 7, n_frame)).reshape(n_chain, 7)
    k = np.asarray(consts, dtype=np.float32)
    length = (stats[:, 3] + stats[:, 4]) + stats[:, 5]
    if include_claw:
        length = length + stats[:, 6]
    aff = np.zeros((n_chain, 8), dtype=np.float32)
    aff[:, :3] = stats[:, :3]
    with np.errstate(all="ignore"):
        aff[:, 3] = k[:, 3] / length
    aff[:, 4:7] = k[:, :3]
    return series, stats, aff


def head_rows_exact(series, consts):
    """series: the five float32 series of one trial (model_head.head_stats: the stationary base x, y, z and distances, the
    |tip - base| of every frame), consts (5,) float32 -> the affine row (8,) float32 of ``head_affine_kernel``:
    (q0, q1, q2, k3 / q3, k0, k1, k2, k4 / q4), NaN statistics for empty series."""
    q = np.array([mid_quantile_exact(np.asarray(s, dtype=np.float32)[None])[0] if len(s) else np.float32(np.nan)
                  for s in series], dtype=np.float32)
    k = np.asarray(consts, dtype=np.float32)
    with np.errstate(all="ignore"):
        return np.array([q[0], q[1], q[2], k[3] / q[3], k[0], k[1], k[2], k[4] / q[4]], dtype=np.float32)
