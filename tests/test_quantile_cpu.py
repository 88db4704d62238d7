"""The exact mid-quantile model (tests/model_quantile.py) against numpy, its constants against the kernel source, and the
route coverage of the GPU cases (tests/test_gpu_quantile.py), all without a GPU."""
import re
from pathlib import Path

import numpy as np
import pytest

import model_quantile as MQ

U = 2.0 ** -24
SRC = Path(__file__).resolve().parent.parent / "sequential-inverse-kinematics_b200" / "csrc" / "seqik_kernels.cu"


def sample_rows(rng, n):
    r = rng.random(n)
    return np.stack([rng.normal(size=n), np.round(rng.normal(size=n), 1), np.where(r < 0.5, 0.0, -0.0),
                     np.where(r < 0.5, 1.5, 1.5000001), 1e30 * rng.normal(size=n), 1e-41 * rng.normal(size=n),
                     np.where(r < 0.2, np.inf, np.where(r > 0.8, -np.inf, rng.normal(size=n)))]).astype(np.float32)


@pytest.mark.parametrize("n", [1, 2, 3, 10, 64, 65, 1000, 4097])
def test_order_statistics_equal_sort_and_partition(n):
    rng = np.random.default_rng(n)
    x = sample_rows(rng, n)
    vals, _, _ = MQ.order_statistics(x)
    ranks, _, _ = MQ.mid_quantile_ranks(np.full(x.shape[0], n))
    s = np.sort(x, axis=1)
    for t in range(4):
        ref = np.take_along_axis(s, ranks[t][:, None], axis=1)[:, 0]
        assert np.array_equal(vals[t], ref), t
        part = np.array([np.partition(x[r], ranks[t][r])[ranks[t][r]] for r in range(x.shape[0])])
        assert np.array_equal(vals[t], part), t
    # the m smallest: the same as the order statistics of the sorted prefix
    m = rng.integers(1, n + 1, size=x.shape[0])
    got = MQ.mid_quantile_exact(x, m)
    ref = np.array([MQ.mid_quantile_exact(s[r, :m[r]][None])[0] for r in range(x.shape[0])])
    assert np.array_equal(got, ref, equal_nan=True)


def test_key_order_of_zeros_and_nans():
    """-0 sorts below +0; a NaN with the sign bit clear above +inf, one with it set below -inf."""
    neg_nan = np.array([0xFFC00000], dtype=np.uint32).view(np.float32)[0]
    x = np.array([np.nan, 0.0, -0.0, np.inf, -np.inf, neg_nan, 1.0], dtype=np.float32)
    order = np.argsort(MQ.order_key(x), kind="stable")
    assert order.tolist() == [5, 4, 2, 1, 6, 3, 0]
    assert np.array_equal(MQ.key_value(MQ.order_key(x)).view(np.uint32), x.view(np.uint32))
    assert np.isnan(MQ.mid_quantile_exact(np.zeros((1, 4), np.float32), np.array([0]))[0])


@pytest.mark.parametrize("n", [2, 3, 7, 100, 1000, 4097, 30011])
def test_model_within_two_units_of_numpy_quantile(n):
    """The float32 interpolation stays within 2 u |q| of numpy's float64 mid-quantile on same-sign series, and within
    2 u of the largest order statistic when the four straddle zero (where q itself may cancel)."""
    rng = np.random.default_rng(100 + n)
    x = np.stack([0.7312 + 1e-3 * rng.normal(size=n), 1.0 + rng.random(n), -1.0 - rng.random(n), 3.0 * rng.random(n),
                  rng.normal(size=n), 1e30 * rng.normal(size=n), rng.choice([1.5, 1.5000001], size=n)]).astype(np.float32)
    got = MQ.mid_quantile_exact(x).astype(np.float64)
    x64 = x.astype(np.float64)
    ref = 0.5 * (np.quantile(x64, 0.45, axis=1) + np.quantile(x64, 0.55, axis=1))
    vals, _, _ = MQ.order_statistics(x)
    same_sign = (np.sign(vals).min(axis=0) == np.sign(vals).max(axis=0))
    bound = np.where(same_sign, 2 * U * np.abs(ref), 2 * U * np.abs(vals).max(axis=0))
    assert (np.abs(got - ref) <= bound).all(), (np.abs(got - ref) / np.maximum(np.abs(ref), 1e-300) / U)


def test_model_constants_are_the_kernels():
    src = SRC.read_text()
    for name, value in (("WQ_N", MQ.WQ_N), ("LQ_CAND", MQ.LQ_CAND), ("LQ_SAMPLE", MQ.LQ_SAMPLE), ("LQ_BINS", MQ.LQ_BINS),
                        ("SEL_CACHE", MQ.SEL_CACHE)):
        m = re.search(rf"\b{name}\s*=\s*(\d+)", src)
        assert m and int(m.group(1)) == value, name
    assert re.search(r"KEY_INF\s*=\s*0xff800000u", src)
    assert re.search(r"cnt\s*<=\s*64\)", src) and re.search(r"in_bins\s*<=\s*64u\)", src)
    assert int(MQ.order_key(np.array([np.inf], np.float32))[0]) == MQ.KEY_INF


def test_select_end_model():
    """warp_select4's endings on hand-made series."""
    k = lambda a: MQ.order_key(np.asarray(a, dtype=np.float32))
    r = lambda n: MQ.mid_quantile_ranks(np.array([n]))[0][:, 0]
    assert MQ.select_end(k(np.full(50, 2.0)), r(50)) == "constant"
    assert MQ.select_end(k(np.arange(200) * 1e-3 + 1.0), r(200)) == "gather"
    rng = np.random.default_rng(1)
    assert MQ.select_end(k(rng.normal(size=1000)), r(1000)) in ("gather", "compact")
    ties = np.sort(np.random.default_rng(2).normal(size=1000))
    ties[300:700] = 0.25
    assert MQ.select_end(k(ties), r(1000)) == "passes"


def test_leg_and_head_models_near_float64():
    rng = np.random.default_rng(9)
    pose = (rng.normal(size=(3, 1, 5, 3)) + 0.02 * rng.normal(size=(3, 301, 5, 3))).astype(np.float32)
    consts = (1.0 + rng.random((3, 4))).astype(np.float32)
    series, stats, aff = MQ.leg_stats_exact(pose, consts, True)
    p64 = pose.astype(np.float64)
    seg = np.linalg.norm(np.diff(p64, axis=2), axis=-1)
    mid = lambda a: 0.5 * (np.quantile(a, 0.45, axis=1) + np.quantile(a, 0.55, axis=1))
    assert np.allclose(series[:, 3:].transpose(0, 2, 1), seg, rtol=4 * U, atol=0)
    assert np.allclose(aff[:, :3], mid(p64[:, :, 0]), rtol=0, atol=4 * U * np.abs(p64).max())
    assert np.allclose(aff[:, 3], consts[:, 3] / mid(seg).sum(1), rtol=16 * U)
    row = MQ.head_rows_exact([series[0, 0], series[0, 1], np.zeros(0, np.float32), series[0, 3], series[0, 4]],
                             np.float32([1, 2, 3, 4, 5]))
    assert np.isnan(row[2]) and row[4:7].tolist() == [1, 2, 3] and row[3] == np.float32(4) / stats[0, 3]


# ------------------------------------------------------------------------------------------------------------ route coverage
def test_gpu_cases_reach_every_route_and_ending():
    """The cases of tests/test_gpu_quantile.py reach every route of the select, every way warp_select4 ends, every reason
    of a hand-off to the general kernel, and both the float4 and the scalar sweeps of the long kernel; the forced cases
    take the route they were built for."""
    import test_gpu_quantile as G
    got = G.reached(G.CASES)
    routes = {r for r, _, _, _ in got}
    assert routes >= set(MQ.ROUTES), set(MQ.ROUTES) - routes
    ends = {e for r, e, _, _ in got if e is not None}
    assert ends == set(MQ.ENDS), set(MQ.ENDS) - ends
    for route in ("warp", "long-small", "long-sweep"):
        seen = {e for r, e, _, _ in got if r == route}
        assert len(seen) >= (4 if route == "warp" else 2), (route, seen)
    assert {why for _, _, _, why in got if why} == set(MQ.RETRY_REASONS)
    for route in ("long-direct", "long-sweep", "retry-cached", "retry-global"):
        assert {a for r, _, a, _ in got if r == route} == {True, False}, route
    assert ("empty", None, True, None) in got or ("empty", None, False, None) in got
    for case in G.CASES:
        if "route" in case:
            info = MQ.routes(case["x"], case["counts"], case["offset"])[0]
            assert (info["route"], info["reason"]) == (case["route"], case["reason"]), case["name"]
