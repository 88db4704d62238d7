"""The alignment statistics -- seqik_mid_quantile_f32 and the leg / head affine rows built on it -- bit for bit against the
exact models of tests/model_quantile.py, on every path of the select.

The launcher and the kernels choose among several routes by length, data range, tie count and row alignment:
``mid_quantile_warp_kernel`` (n <= 1024), ``mid_quantile_long_kernel`` with its keys-to-shared-memory path (n <= 4096), its
direct read-off (sampled range of fewer than 4096 keys) and its two sweeps (float4 or scalar, by row alignment), and the
hand-off (MQ_RETRY) to ``mid_quantile_kernel``, cached (n <= 8192) or not.  ``warp_select4`` ends on a constant span, a
first-pass gather, a compaction or the last histogram pass.  ``quantile_cases`` builds series that reach every one of these
(``model_quantile.route`` says which; tests/test_quantile_cpu.py checks without a GPU that the set is complete), and every
result must equal the model value for value: NaN equals NaN and -0 equals +0.
"""
import numpy as np
import pytest

import model_head
import model_quantile as MQ

pytestmark = pytest.mark.gpu

LENGTHS = (1, 2, 3, 4, 5, 31, 32, 33, 63, 64, 65, 1023, 1024, 1025, 4095, 4096, 4097, 6143, 6144, 8192, 8193, 30011, 100003)
COUNT_LENGTHS = (5, 33, 65, 1000, 1025, 4097, 6144, 8193, 30011)


def families(rng, n):
    """(name, float32 row of n samples): the data families of every length.  14 rows: the warp kernel's last block of four
    series is partial."""
    r = rng.random(n)
    normal = rng.normal(size=n)
    ties = np.sort(normal)
    ties[int(0.35 * n):int(0.65 * n)] = 0.25                     # > 64 exact ties at the rank positions once n > 220
    nan = normal.copy()
    nan[r < 0.03] = np.nan
    nan[(r >= 0.03) & (r < 0.06)] = -np.nan                      # sign bit set: sorts below -inf
    rows = [
        ("narrow", 0.7312 + 1e-3 * normal),                       # a segment length: a sliver of one octave
        ("constant", np.full(n, -3.25)),
        ("two-valued", np.where(r < 0.5, 1.5, 1.5000001)),       # one ulp apart
        ("four-valued", 0.4 + 1e-6 * rng.integers(0, 4, size=n)),
        ("signed-zeros", np.where(r < 0.5, 0.0, -0.0)),
        ("zeros-and-small", np.where(r < 0.35, 0.0, np.where(r < 0.7, -0.0, 1e-3 * normal))),
        ("all-negative", -1.0 - np.abs(normal)),
        ("scale-1e30", 1e30 * normal),
        ("subnormal", 1e-41 * normal),
        ("with-inf", np.where(r < 0.15, np.inf, np.where(r > 0.85, -np.inf, normal))),
        ("with-nan", nan),
        ("ties-at-ranks", rng.permutation(ties)),
        ("wide", normal),
        ("drift", np.linspace(-1.0, 3.0, n) + 0.05 * normal),
    ]
    return [(name, np.asarray(row).astype(np.float32)) for name, row in rows]


def forced_cases(rng):
    """(name, row, count or None, expected route, expected reason): series that must leave the long kernel's fast paths."""
    out = []
    for n, want in ((6000, "retry-cached"), (20000, "retry-global")):
        x = rng.normal(size=n)
        x[np.arange(MQ.LQ_SAMPLE) * (n // MQ.LQ_SAMPLE)] = 1e6 + rng.normal(size=MQ.LQ_SAMPLE)   # only the sample is large
        out.append((f"high-samples-{n}", x.astype(np.float32), None, want, "rank-outside-range"))
    for n, k, want in ((8000, 4500, "retry-cached"), (30011, 5000, "retry-global")):
        x = 10.0 * rng.normal(size=n)
        x[rng.choice(n, size=k, replace=False)] = 0.0            # > 4096 copies of the median value in a wide range
        out.append((f"heavy-ties-{n}", x.astype(np.float32), None, want, "too-many-candidates"))
    for n, want in ((6144, "retry-cached"), (9000, "retry-global")):
        x = rng.normal(size=n)
        idx = np.arange(MQ.LQ_SAMPLE) * (n // MQ.LQ_SAMPLE)
        x[idx] = np.inf                                          # +inf padding at every sampled position
        out.append((f"inf-at-samples-{n}", x.astype(np.float32), n - MQ.LQ_SAMPLE, want, "empty-sample"))
    return out


def quantile_cases():
    """Every mid-quantile case: dicts of name, x (rows, n) float32, counts (rows,) int32 or None, offset (row 0 starts
    this many floats past a 16-byte boundary) and, for the forced ones, the route and reason they must take."""
    rng = np.random.default_rng(2024)
    cases = []
    for i, n in enumerate(LENGTHS):
        fam = families(rng, n)
        x = np.stack([row for _, row in fam])
        names = [name for name, _ in fam]
        for offset in (0, 1 + i % 3):
            cases.append(dict(name=f"families-{n}", rows=names, x=x, counts=None, offset=offset))
    for i, n in enumerate(COUNT_LENGTHS):
        fam = families(rng, n)
        x = np.stack([row for _, row in fam])
        m = rng.integers(1, n + 1, size=x.shape[0])
        m[:3] = (0, 1, n)
        m = m.astype(np.int32)
        padded = x.copy()                                         # +inf padding: the m smallest, then +inf, shuffled
        for r in range(padded.shape[0]):
            row = np.sort(padded[r])
            row[m[r]:] = np.inf
            padded[r] = rng.permutation(row)
        names = [f"{name}/m={m[r]}" for r, (name, _) in enumerate(fam)]
        cases.append(dict(name=f"counts-inf-{n}", rows=names, x=padded, counts=m, offset=i % 4))
        cases.append(dict(name=f"counts-finite-{n}", rows=names, x=x, counts=m, offset=(i + 2) % 4))
    for name, row, m, want, reason in forced_cases(rng):
        counts = None if m is None else np.array([m], dtype=np.int32)
        for offset in (0, 3):
            cases.append(dict(name=name, rows=[name], x=row[None], counts=counts, offset=offset, route=want, reason=reason))
    return cases


def reached(cases):
    """{(route, end, aligned, reason)} over every row of every case."""
    out = set()
    for c in cases:
        for info in MQ.routes(c["x"], c["counts"], c["offset"]):
            out.add((info["route"], info["end"], info["aligned"], info["reason"]))
    return out


# ------------------------------------------------------------------------------------------------------------ helpers
@pytest.fixture(scope="module")
def eng():
    import torch
    assert torch.cuda.is_available(), "these tests need the B200"
    from seqikpy_b200 import _native as N, engine
    N.load_library()
    return torch, engine, N


def offset_view(torch, t, k):
    """A contiguous copy of ``t`` that starts ``k`` elements past a 256-byte aligned allocation."""
    buf = torch.empty(t.numel() + 8, dtype=t.dtype, device=t.device)
    v = buf[k:k + t.numel()].view(t.shape)
    v.copy_(t)
    assert v.is_contiguous() and v.data_ptr() % 16 == 4 * k % 16
    return v


def dev(torch, a, offset=0):
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return offset_view(torch, t, offset) if offset else t


def same_values(got, ref):
    """Element-wise: equal (-0 == +0) or both NaN."""
    got, ref = np.asarray(got), np.asarray(ref)
    return (got == ref) | (np.isnan(got) & np.isnan(ref))


def assert_mid_quantiles(got, case):
    ref = MQ.mid_quantile_exact(case["x"], case["counts"])
    ok = same_values(got, ref)
    if ok.all():
        return
    vals, _, _ = MQ.order_statistics(case["x"], case["counts"])
    infos = MQ.routes(case["x"], case["counts"], case["offset"])
    bad = [dict(row=int(r), family=case["rows"][r], n=case["x"].shape[1], offset=case["offset"], route=infos[r]["route"],
                end=infos[r]["end"], aligned=infos[r]["aligned"], got=float(got[r]), want=float(ref[r]),
                order_statistics=vals[:, r].tolist()) for r in np.flatnonzero(~ok)]
    raise AssertionError(f"{case['name']}: {len(bad)} rows differ from the exact model: {bad[:6]}")


# ------------------------------------------------------------------------------------------------------------ mid-quantile
CASES = quantile_cases()


@pytest.mark.parametrize("name", sorted({c["name"] for c in CASES}, key=lambda s: (s.split("-")[0], len(s), s)))
def test_mid_quantile_equals_exact_model(eng, name):
    torch, E, _ = eng
    for case in (c for c in CASES if c["name"] == name):
        x = dev(torch, case["x"], case["offset"])
        counts = None if case["counts"] is None else dev(torch, case["counts"])
        got = E.mid_quantile(x, counts).cpu().numpy()
        assert_mid_quantiles(got, case)
        if "route" in case:
            assert [i["route"] for i in MQ.routes(case["x"], case["counts"], case["offset"])] == [case["route"]]
        # a second call on the same buffers gives the same bits (no state survives a launch)
        again = E.mid_quantile(x, counts).cpu().numpy()
        assert np.array_equal(got.view(np.uint32), again.view(np.uint32)), name


def test_cases_reach_every_route():
    got = reached(CASES)
    assert {r for r, _, _, _ in got} >= set(MQ.ROUTES)
    assert {e for _, e, _, _ in got} >= set(MQ.ENDS)
    assert {why for _, _, _, why in got} >= set(MQ.RETRY_REASONS)


# ------------------------------------------------------------------------------------------------------------ leg rows
def leg_poses(rng, n_chain, n_frame):
    """Key points around a per-chain rest pose, with coincident key points (chain 0: a zero-length femur on every frame;
    chain 1: a zero-length tibia on every third frame) and repeated frames (every fourth frame repeats the one before)."""
    p = rng.normal(size=(n_chain, 1, 5, 3)) + 0.02 * rng.normal(size=(n_chain, n_frame, 5, 3))
    p[0, :, 2] = p[0, :, 1]
    if n_chain > 1:
        p[1, ::3, 3] = p[1, ::3, 2]
    idx = np.arange(n_frame)
    idx[3::4] = idx[2::4][:idx[3::4].size]
    return np.ascontiguousarray(p[:, idx]).astype(np.float32)


def assert_rows(got, ref, what):
    ok = same_values(got, ref).all(axis=1)
    assert ok.all(), (what, np.flatnonzero(~ok)[:8].tolist(), got[~ok][:3].tolist(), ref[~ok][:3].tolist())


@pytest.mark.parametrize("n_frame", [1, 2, 7, 223, 224, 225, 448, 449, 1023, 1024])
def test_fused_leg_rows_equal_exact_model(eng, n_frame):
    """The fused per-chain kernel (staging tiles of LA_TILE = 224 frames, float4 or scalar by chain alignment) and the
    three separate kernels."""
    torch, E, _ = eng
    rng = np.random.default_rng(1000 + n_frame)
    n_chain = 5
    pose = leg_poses(rng, n_chain, n_frame)
    consts = (1.0 + rng.random((n_chain, 4))).astype(np.float32)
    d_consts = dev(torch, consts)
    for offset in (0, 1):
        d_pose = dev(torch, pose, offset)
        for claw in (False, True):
            _, _, ref = MQ.leg_stats_exact(pose, consts, claw)
            assert_rows(E.leg_affine(d_pose, d_consts, include_claw=claw).cpu().numpy(), ref, ("fused", offset, claw))
            assert_rows(E.leg_affine_unfused(d_pose, d_consts, include_claw=claw).cpu().numpy(), ref, ("unfused", offset, claw))


@pytest.mark.parametrize("n_frame", [1025, 4097, 30011])
def test_long_leg_rows_equal_exact_model(eng, n_frame):
    torch, E, _ = eng
    rng = np.random.default_rng(2000 + n_frame)
    n_chain = 3
    pose = leg_poses(rng, n_chain, n_frame)
    consts = (1.0 + rng.random((n_chain, 4))).astype(np.float32)
    _, _, ref = MQ.leg_stats_exact(pose, consts, True)
    d_pose, d_consts = dev(torch, pose, 2), dev(torch, consts)
    assert_rows(E.leg_affine(d_pose, d_consts, include_claw=True).cpu().numpy(), ref, "from_pose")
    assert_rows(E.leg_affine_unfused(d_pose, d_consts, include_claw=True).cpu().numpy(), ref, "unfused")


def test_leg_rows_at_grid_scale(eng):
    torch, E, _ = eng
    rng = np.random.default_rng(5)
    pose = leg_poses(rng, 2000, 1000)
    consts = (1.0 + rng.random((2000, 4))).astype(np.float32)
    _, _, ref = MQ.leg_stats_exact(pose, consts, False)
    assert_rows(E.leg_affine(dev(torch, pose), dev(torch, consts)).cpu().numpy(), ref, "2000 x 1000")


@pytest.mark.parametrize("n_frame", [300, 1024, 2000])
def test_strided_leg_entry_points_equal_exact_model(eng, n_frame):
    """Frame stride 18 floats and a chain stride padded by 5 (not a multiple of four): the fused kernel's scalar staging
    path, which engine.leg_affine never takes, and the series kernel on the same layout, series bit for bit.  The padding
    is NaN, so a read of it would show."""
    torch, _, N = eng
    lib = N.load_library()
    rng = np.random.default_rng(3000 + n_frame)
    n_chain, fs = 4, 18
    cs = n_frame * fs + 5
    pose = leg_poses(rng, n_chain, n_frame)
    consts = (1.0 + rng.random((n_chain, 4))).astype(np.float32)
    buf = torch.full((n_chain * cs,), float("nan"), dtype=torch.float32, device="cuda")
    buf.as_strided((n_chain, n_frame, 15), (cs, fs, 1)).copy_(dev(torch, pose.reshape(n_chain, n_frame, 15)))
    d_consts = dev(torch, consts)
    st = N.stream_ptr(torch, buf.device)
    series = torch.empty((n_chain * 7, n_frame), dtype=torch.float32, device="cuda")
    N.check(lib.seqik_leg_series_f32(N.ptr(buf), cs, fs, N.ptr(series), n_chain, n_frame, st), "seqik_leg_series_f32")
    ref_series, _, _ = MQ.leg_stats_exact(pose, consts, False)
    got = series.cpu().numpy().reshape(n_chain, 7, n_frame)
    assert np.array_equal(got.view(np.uint32), ref_series.view(np.uint32))
    scratch = torch.empty((n_chain * 7 * (n_frame + 1),), dtype=torch.float32, device="cuda")
    for claw in (False, True):
        _, _, ref = MQ.leg_stats_exact(pose, consts, claw)
        aff = torch.empty((n_chain, 8), dtype=torch.float32, device="cuda")
        N.check(lib.seqik_leg_affine_from_pose_f32(N.ptr(buf), cs, fs, N.ptr(d_consts), int(claw), N.ptr(scratch), N.ptr(aff),
                                                   n_chain, n_frame, st), "seqik_leg_affine_from_pose_f32")
        assert_rows(aff.cpu().numpy(), ref, ("strided", claw))


# ------------------------------------------------------------------------------------------------------------ head rows
@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("n_frame", [1, 3, 33, 1000, 1025, 4097])
def test_head_rows_equal_exact_model(eng, n_frame, dtype):
    from test_gpu_stream import head_stat_trials
    torch, E, _ = eng
    dt = np.dtype(dtype)
    rng = np.random.default_rng(4000 + n_frame + dt.itemsize)
    thr = 5e-5
    thr_dev = float(np.float32(thr)) if dt == np.float32 else thr           # the f32 entry point takes a float threshold
    n_trial = 7
    head, thorax = head_stat_trials(rng, n_trial, n_frame, 3, dt, 3)
    consts = np.float32(rng.uniform(0.5, 1.5, (n_trial, 5)))
    aff, counts = E.head_affine(dev(torch, head), dev(torch, thorax), dev(torch, consts), threshold=thr)
    aff, counts = aff.cpu().numpy(), counts.cpu().numpy()
    for tr in range(n_trial):
        m, _, series = model_head.head_stats(head[tr], thorax[tr], consts[tr], thr_dev)
        assert counts[tr].tolist() == [m] * 4 + [n_frame]
        ref = MQ.head_rows_exact(series, consts[tr])
        assert same_values(aff[tr], ref).all(), (tr, m, aff[tr].tolist(), ref.tolist())
