"""The streaming kernels -- FK, align / head apply, head angles, head statistics, pchip -- on every code path their launchers
choose between, against plain references.

Each launcher in csrc/seqik_kernels.cu picks a path from the shape and the pointer alignment: a persistent TMA tile pipeline
over the full tiles (every CTA walks several tiles once the grid is capped at SMs x CTAs that fit), the ragged tail through
the plain kernel, and the plain kernel alone for a total below one tile or for an input that is not 16-byte aligned (here: a
contiguous view at a 1-, 2- or 3-float offset).  The shapes below put chain boundaries inside tiles and inside the tail, and
one large case per kernel gives every CTA at least four tiles (4 x 148 x 4 tiles: whatever the CTAs per SM, both stages,
the mbarrier phase flip and the reuse of a stage's output buffer are exercised).

References:
* FK: oracle.seqik_oracle.fk_closed_form (float64) of the float32 inputs, on a sample of leg-frames (every tile's first and
  last one, every chain boundary, a seeded random set); the paths must agree bit for bit among themselves.
* align / head apply: the header's formulas in numpy float32, in the kernel's operation order ((p - a0) * s + a4; the build
  has no fma contraction), bit for bit.
* head angles: tests/model_head.py (float64 restatement of the reference), and float64 arctangents on a sweep.
* head statistics: numpy (np.quantile) on the frames that tests/model_head.py classifies as stationary; counts exactly.
* pchip: scipy.interpolate.pchip_interpolate, as tests/test_gpu_resample.py.
"""
import numpy as np
import pytest
from scipy.interpolate import pchip_interpolate

import model_head
from oracle import seqik_oracle as O

pytestmark = pytest.mark.gpu

U = 2.0 ** -24                      # unit roundoff of float32
TILE = 256                          # units per tile of the FK / align pipelines (leg-frames)
HEAD_TILE = 1024                    # frames per tile of the head-apply pipeline
N_LARGE_TILES = 4 * 148 * 4


@pytest.fixture(scope="module")
def eng():
    import torch
    assert torch.cuda.is_available(), "these tests need the B200"
    from seqikpy_b200 import _native as N, engine
    N.load_library()
    return torch, engine, N


def dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def offset_view(torch, t, k):
    """A contiguous copy of ``t`` that starts ``k`` elements past a 256-byte aligned allocation."""
    buf = torch.empty(t.numel() + 8, dtype=t.dtype, device=t.device)
    v = buf[k:k + t.numel()].view(t.shape)
    v.copy_(t)
    assert v.is_contiguous() and v.data_ptr() % 16 == 4 * k % 16
    return v


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def n_large(unit, n_frame):
    """Chains of ``n_frame`` for at least N_LARGE_TILES full tiles of ``unit`` plus a ragged tail."""
    n_chain = -(-N_LARGE_TILES * unit // n_frame)
    assert (n_chain * n_frame) // unit >= N_LARGE_TILES and (n_chain * n_frame) % unit
    return n_chain


# (n_chain, n_frame) in leg-frames: below one tile, exactly one tile, chain boundaries inside tiles and the tail, large
LEG_SHAPES = [(2, 50), (1, 256), (300, 1), (100, 7), (5, 255), (5, 257), (n_large(TILE, 1009), 1009)]


# ------------------------------------------------------------------------------------------------------------ FK
def fk_inputs(rng, n_chain, n_frame):
    ang = rng.uniform(-2 * np.pi, 2 * np.pi, (n_chain, n_frame, 7)).astype(np.float32)
    # the branch points of sincosv_: the quadrant-0 switch at 0.78, the quadrant edges k pi/4, the ends of its domain
    two_pi = np.float32(2 * np.pi)
    special = np.array([0.78, -0.78, np.nextafter(np.float32(0.78), np.float32(0)), np.nextafter(np.float32(0.78), np.float32(1)),
                        two_pi, -two_pi, np.nextafter(two_pi, np.float32(0)), 0.0, -0.0]
                       + [k * np.pi / 4 for k in range(-8, 9)], dtype=np.float32)
    flat = ang.reshape(-1)
    idx = rng.choice(flat.size, size=max(1, flat.size // 8), replace=False)
    flat[idx] = special[np.arange(idx.size) % special.size]
    org = rng.uniform(-2.0, 2.0, (n_chain, n_frame, 3)).astype(np.float32)
    params = np.zeros((n_chain, 32), dtype=np.float32)
    params[:, :4] = rng.uniform(0.1, 1.0, (n_chain, 4))                 # a different chain per row: a wrong index shows
    params[:, 4:] = rng.normal(size=(n_chain, 28))                       # (not read by FK)
    return ang, org, params


def fk_sample(rng, n_chain, n_frame):
    total = n_chain * n_frame
    full = total // TILE
    idx = [k * TILE for k in range(full)] + [k * TILE + TILE - 1 for k in range(full)]
    idx += [min(full * TILE, total - 1), total - 1]                          # the tail (if any)
    idx += [c * n_frame for c in range(n_chain)] + [c * n_frame - 1 for c in range(1, n_chain)]
    idx += list(rng.integers(0, total, size=min(total, 1000)))
    return np.unique(np.asarray(idx, dtype=np.int64))


def fk_bound(org, params):
    """Per chain, per coordinate: 32 u (|origin|_max + sum of the segment lengths).

    Each stage composes the running frame with at most two rotations whose sin / cos carry <= 2 u; a product of a unit
    matrix with a rotation adds <= 3 u per entry, so after the seven rotations the frame's columns are off by <= 7 (2 + 3) u
    = 35 u in the worst case, and ~ sqrt(7) 5 u typically; a joint position adds l_k times its column's error and one
    rounding of |p| <= |o| + sum l per multiply-add.  The worst case is far from reached (errors do not align); 32 u of
    the chain's extent is 16 times the largest error observed on a B200 at 1000 W (2 u of the extent)."""
    return 32 * U * (np.abs(org).reshape(org.shape[0], -1).max(axis=1) + params[:, :4].sum(axis=1))


def check_fk_vs_oracle(fk, ang, org_rows, params, sample, bound):
    n_frame = ang.shape[1]
    c_of, t_of = sample // n_frame, sample % n_frame
    worst = 0.0
    for c in np.unique(c_of):
        t = t_of[c_of == c]
        ref = O.fk_closed_form(ang[c, t].astype(np.float64), params[c, :4].astype(np.float64),
                               org_rows[c, t].astype(np.float64))
        err = np.abs(fk[c, t] - ref).max()
        assert err <= bound[c], (int(c), err, bound[c])
        worst = max(worst, err / bound[c])
    return worst


@pytest.mark.parametrize("n_chain,n_frame", LEG_SHAPES)
def test_fk_paths_bitwise_and_vs_float64(eng, n_chain, n_frame):
    torch, E, _ = eng
    rng = np.random.default_rng(1000 + n_frame)
    ang, org, params = fk_inputs(rng, n_chain, n_frame)
    d_ang, d_org, d_prm = dev(torch, ang), dev(torch, org), dev(torch, params)
    fk = E.forward_kinematics(d_ang, d_org, d_prm)                                   # TMA tiles (if any) + tail
    for k in (1, 2, 3):                                                              # plain kernel: angles unaligned
        assert torch.equal(E.forward_kinematics(offset_view(torch, d_ang, k), d_org, d_prm).view(torch.int32), fk.view(torch.int32)), k
    assert torch.equal(E.forward_kinematics(d_ang, offset_view(torch, d_org, 1), d_prm).view(torch.int32), fk.view(torch.int32))
    # constant origin per chain (stride 0): its alignment does not select the path
    org0 = org[:, 0].copy()
    fk0 = E.forward_kinematics(d_ang, dev(torch, org0), d_prm)
    assert torch.equal(E.forward_kinematics(offset_view(torch, d_ang, 3), dev(torch, org0), d_prm).view(torch.int32), fk0.view(torch.int32))
    fk, fk0 = fk.cpu().numpy(), fk0.cpu().numpy()
    sample = fk_sample(rng, n_chain, n_frame)
    bound = fk_bound(org, params)
    check_fk_vs_oracle(fk, ang, org, params, sample, bound)
    check_fk_vs_oracle(fk0, ang, np.repeat(org0[:, None], n_frame, axis=1), params, sample, bound)


# ------------------------------------------------------------------------------------------------------------ align apply
def align_ref(pose, aff):
    """out[:, :, 0] = template; out[:, :, i] = (pose - fixed) * scale + template, numpy float32 in the kernel's order."""
    a = aff[:, None, None, :]
    out = (pose - a[..., 0:3]) * a[..., 3:4] + a[..., 4:7]
    out[:, :, 0] = np.broadcast_to(aff[:, None, 4:7], out[:, :, 0].shape)
    return out


def align_affine(rng, n_chain):
    aff = np.zeros((n_chain, 8), dtype=np.float32)
    aff[:, 0:3] = rng.normal(size=(n_chain, 3))
    aff[:, 3] = rng.uniform(0.5, 2.0, n_chain)
    aff[:, 4:7] = rng.normal(size=(n_chain, 3))
    return aff


@pytest.mark.parametrize("n_chain,n_frame", LEG_SHAPES)
def test_align_apply_paths_bitwise(eng, n_chain, n_frame):
    torch, E, N = eng
    rng = np.random.default_rng(2000 + n_frame)
    pose = rng.normal(size=(n_chain, n_frame, 5, 3)).astype(np.float32)
    aff = align_affine(rng, n_chain)
    ref = align_ref(pose, aff)
    d_pose, d_aff = dev(torch, pose), dev(torch, aff)
    assert same_bits(E.align_apply(d_pose, d_aff).cpu().numpy(), ref)                           # TMA tiles + tail
    for k in (1, 2):
        assert same_bits(E.align_apply(offset_view(torch, d_pose, k), d_aff).cpu().numpy(), ref), k   # plain (unaligned)
    # the strided path: frame stride 18 floats, chain stride padded -- through the C ABI, as the engine only passes dense
    fs, cs = 18, n_frame * 18 + 5
    strided = np.zeros(n_chain * cs, dtype=np.float32)
    view = np.lib.stride_tricks.as_strided(strided, shape=(n_chain, n_frame, 15), strides=(4 * cs, 4 * fs, 4))
    view[...] = pose.reshape(n_chain, n_frame, 15)
    d_strided = dev(torch, strided)
    out = torch.empty((n_chain, n_frame, 5, 3), dtype=torch.float32, device="cuda")
    lib = N.load_library()
    N.check(lib.seqik_align_apply_f32(d_strided.data_ptr(), cs, fs, d_aff.data_ptr(), out.data_ptr(), n_chain, n_frame,
                                      torch.cuda.current_stream().cuda_stream), "seqik_align_apply_f32")
    assert same_bits(out.cpu().numpy(), ref)


# ------------------------------------------------------------------------------------------------------------ head apply
def head_apply_ref(head, aff):
    """Base rows scaled by aff[3], tip rows by aff[7] (numpy float32, the kernel's order)."""
    a = aff[:, None, :]
    out = np.empty_like(head)
    out[:, :, 0] = (head[:, :, 0] - a[..., 0:3]) * a[..., 3:4] + a[..., 4:7]
    out[:, :, 1] = (head[:, :, 1] - a[..., 0:3]) * a[..., 7:8] + a[..., 4:7]
    return out


HEAD_SHAPES = [(1, 1001), (1, 1024), (3000, 1), (500, 7), (9, 255), (9, 257), (5, 1025), (n_large(HEAD_TILE, 1023), 1023)]


@pytest.mark.parametrize("n_trial,n_frame", HEAD_SHAPES)
def test_head_apply_paths_bitwise(eng, n_trial, n_frame):
    torch, E, _ = eng
    rng = np.random.default_rng(3000 + n_frame)
    head = rng.normal(size=(n_trial, n_frame, 2, 3)).astype(np.float32)
    aff = align_affine(rng, n_trial)
    aff[:, 7] = rng.uniform(2.5, 4.0, n_trial)                          # scale_tip far from scale_base
    ref = head_apply_ref(head, aff)
    d_head, d_aff = dev(torch, head), dev(torch, aff)
    assert same_bits(E.head_apply(d_head, d_aff).cpu().numpy(), ref)
    for k in (1, 3):
        assert same_bits(E.head_apply(offset_view(torch, d_head, k), d_aff).cpu().numpy(), ref), k


# ------------------------------------------------------------------------------------------------------------ head angles
def atan_sweep_operands():
    """(y, z) float32 pairs whose signed angle is one atan2_pos call: a seeded sweep of the circle, the octant edges, the
    tan(pi/8) switch of the second reduction (and the float32 neighbours of all of these), the axes, det = +-0."""
    rng = np.random.default_rng(41)
    f = np.float32
    th = np.concatenate([rng.uniform(-np.pi, np.pi, 100_000), np.arange(-8, 9) * np.pi / 8])
    yz = [np.stack([np.cos(th), np.sin(th)], 1).astype(f)]
    t8 = f(0.4142135679721832)
    edges = []
    for a, b in ((1, 1), (1, t8), (t8, 1)):
        for da in (-1, 0, 1):
            for db in (-1, 0, 1):
                a2, b2 = f(a), f(b)
                for _ in range(abs(da)):
                    a2 = np.nextafter(a2, f(da * 2))
                for _ in range(abs(db)):
                    b2 = np.nextafter(b2, f(db * 2))
                for sy in (1, -1):
                    for sz in (1, -1):
                        edges.append((sy * a2, sz * b2))
    for y, z in ((1, 0), (1, -0.0), (-1, 0), (-1, -0.0), (0, 1), (-0.0, 1), (0, -1), (-0.0, -1), (1e-30, 1), (-1e-30, -1)):
        edges.append((y, z))
    yz.append(np.asarray(edges, dtype=f))
    return np.concatenate(yz)


def test_head_angles_arctangent_sweep(eng):
    """Right antenna base at 0, left base at r (0, y, z): the head roll is signed_angle(y, z), and with the left base at
    r (-z, y, 0) the head yaw is the same call -- one atan2_pos on exactly the float32 operands.  Error against the float64
    arctangent of those operands: at most half an ulp of the float32 result (its unavoidable rounding) + 2e-7 rad, i.e.
    < 3.2e-7 rad for results near pi and < 2.6e-7 rad below 2 rad.  (Measured on a B200 at 1000 W: 1.7e-7 beyond the half ulp,
    2.9e-7 rad in all.  The flat 3e-7 rad once documented does not hold near pi: pi - a rounds by up to 1.2e-7 there and
    the float32 pi is 8.7e-8 off; a float32 model of the function reaches 3.04e-7 on a denser sweep.)"""
    torch, E, _ = eng
    yz = atan_sweep_operands()
    for r in (np.float32(1e-3), np.float32(1.0), np.float32(1e3)):
        y, z = (yz[:, 0] * r).astype(np.float32), (yz[:, 1] * r).astype(np.float32)
        n = y.size
        head = np.zeros((2, n, 2, 2, 3), dtype=np.float32)             # (trial, frame, side R/L, base/tip, xyz)
        head[0, :, 1, 0, 1], head[0, :, 1, 0, 2] = y, z                 # trial 0: roll sweep
        head[1, :, 1, 0, 0], head[1, :, 1, 0, 1] = -z, y                # trial 1: yaw sweep
        head[:, :, :, 1] = head[:, :, :, 0] + np.float32([0.1, 0.2, -0.3])
        r_head, l_head = dev(torch, head[:, :, 0]), dev(torch, head[:, :, 1])
        neck = dev(torch, np.float32([[-1.0, 0.0, 0.0], [-1.0, 0.0, 0.0]]))
        out = E.head_angles(r_head, l_head, neck, dev(torch, np.zeros((2, 2), np.float32))).cpu().numpy()
        got = np.stack([out[0, 0], out[1, 2]])
        y64, z64 = y.astype(np.float64), z.astype(np.float64)
        ref = np.arctan2(np.abs(z64), y64) * np.where(z64 > 0, 1.0, -1.0)
        err = np.abs(got - ref)
        bound = 0.5 * np.spacing(np.abs(got)).astype(np.float64) + 2e-7
        assert (err <= bound).all(), (float(r), err.max(), yz[np.argmax((err - bound).max(axis=0))])
        # det = 0 with dot < 0: -pi, the reference's arccos(-1) * -1
        anti = (y < 0) & (z == 0)
        assert anti.sum() == 2 and (got[:, anti] == np.float32(-np.pi)).all()


def realistic_heads(n_trial, n_frame):
    from seqikpy_b200 import synthetic as S
    rs, ls, necks = [], [], []
    for tr in range(n_trial):
        r, l, _, neck = S.make_head_trial(tr, n_frame)
        rs.append(r); ls.append(l); necks.append(neck)
    return np.stack(rs).astype(np.float32), np.stack(ls).astype(np.float32), np.stack(necks).astype(np.float32)


def head_point_f32(p, aff, tip):
    """head_point of the kernel in numpy float32 (bit for bit)."""
    sc = aff[:, None, 7:8] if tip else aff[:, None, 3:4]
    return (p - aff[:, None, 0:3]) * sc + aff[:, None, 4:7]


def wrap(a):
    return (a + np.pi) % (2 * np.pi) - np.pi


@pytest.mark.parametrize("neck_per_frame", [False, True])
@pytest.mark.parametrize("with_affine", [False, True])
def test_head_angles_vs_float64_model(eng, neck_per_frame, with_affine):
    """Synthetic head motion (0.2 rad head roll / pitch / yaw, 0.3 rad antenna pitch), 3 trials of an odd frame count,
    against tests/model_head.py on the float32 points the kernel sees (the affine rows applied in float32 first).

    Bound per frame: 2e-6 rad + 16 u P / V, P = the largest coordinate, V = the shortest vector that enters an angle.  The
    five arctangents each carry < 4e-7 rad (test above) and the antenna angles inherit the roll's error through the
    de-rotation; the coordinates of a vector are float32 differences (and dot / det float32 sums) with errors of a few u
    of P, which turn an angle by that over V.  Differences are taken modulo 2 pi (an angle at +-pi may change sides)."""
    torch, E, _ = eng
    n_trial, n_frame = 3, 1001
    rng = np.random.default_rng(51)
    r, l, neck = realistic_heads(n_trial, n_frame)
    necks = neck[:, None] + rng.normal(0, 0.01, (n_trial, n_frame, 3)).astype(np.float32) if neck_per_frame else neck
    rest = np.float32([[0.3, -0.2], [0.1, 0.25], [-0.05, 0.0]])
    aff = None
    if with_affine:
        aff = [align_affine(rng, n_trial) for _ in range(2)]
        for a in aff:
            a[:, 0:3] = rng.normal(0, 0.1, (n_trial, 3))
            a[:, 3], a[:, 7] = rng.uniform(0.9, 1.1, n_trial), rng.uniform(0.9, 1.1, n_trial)
            a[:, 4:7] = rng.normal(0, 0.1, (n_trial, 3))
    out = E.head_angles(dev(torch, r), dev(torch, l), dev(torch, necks), dev(torch, rest),
                        *(dev(torch, a) for a in (aff or []))).cpu().numpy()
    if with_affine:
        r = np.stack([head_point_f32(r[:, :, 0], aff[0], False), head_point_f32(r[:, :, 1], aff[0], True)], 2)
        l = np.stack([head_point_f32(l[:, :, 0], aff[1], False), head_point_f32(l[:, :, 1], aff[1], True)], 2)
    for tr in range(n_trial):
        nk = (necks[tr] if neck_per_frame else necks[tr][None]).astype(np.float64)
        ref = model_head.head_angles(r[tr], l[tr], nk, float(rest[tr, 0]), float(rest[tr, 1]))
        nk = np.broadcast_to(nk, (n_frame, 3))
        pts = np.concatenate([r[tr].reshape(n_frame, 6), l[tr].reshape(n_frame, 6), nk], 1)
        vecs = [l[tr][:, 0] - r[tr][:, 0], r[tr][:, 1] - r[tr][:, 0], l[tr][:, 1] - l[tr][:, 0],
                0.5 * (r[tr][:, 0] + l[tr][:, 0]) - nk, nk - r[tr][:, 0], nk - l[tr][:, 0]]
        v_min = np.min([np.linalg.norm(v, axis=1) for v in vecs], axis=0)
        bound = 2e-6 + 16 * U * np.abs(pts).max(axis=1) / v_min
        err = np.abs(wrap(out[tr].astype(np.float64) - ref))
        assert (err <= bound).all(), (tr, err.max(axis=1), bound.max())


def test_head_angles_unaligned_inputs_give_the_same_bits(eng):
    """r_head / l_head at 4 mod 8 bytes take the scalar-load kernel: the same arithmetic, the same bits."""
    torch, E, _ = eng
    r, l, neck = realistic_heads(3, 777)
    d_r, d_l, d_n = dev(torch, r), dev(torch, l), dev(torch, neck)
    rest = dev(torch, np.float32([[0.3, -0.2]] * 3))
    ref = E.head_angles(d_r, d_l, d_n, rest)
    for k_r, k_l in ((1, 0), (0, 3), (1, 1), (3, 2)):
        rr = offset_view(torch, d_r, k_r) if k_r else d_r
        ll = offset_view(torch, d_l, k_l) if k_l else d_l
        assert torch.equal(E.head_angles(rr, ll, d_n, rest).view(torch.int32), ref.view(torch.int32)), (k_r, k_l)


# ------------------------------------------------------------------------------------------------------------ head statistics
def head_stat_trials(rng, n_trial, n_frame, n_kp, dtype, accelerating):
    """Antenna base at distance d(t) from the thorax mid point: 1 + 1e-4 noise (about 60 % stationary frames at the
    5e-5 threshold), or -- trial ``accelerating`` -- t (t + 1) / 2048 exactly (second difference 1 / 1024: none)."""
    thorax = (rng.normal(0, 0.2, (n_trial, 1, n_kp, 3)) + rng.normal(0, 0.01, (n_trial, n_frame, n_kp, 3))).astype(dtype)
    mid = 0.5 * (thorax[:, :, 0].astype(np.float64) + thorax[:, :, -1])
    u = rng.normal(size=(n_trial, 1, 3))
    u /= np.linalg.norm(u, axis=2, keepdims=True)
    d = 1.0 + 1e-4 * rng.normal(size=(n_trial, n_frame, 1))
    head = np.empty((n_trial, n_frame, 2, 3))
    head[:, :, 0] = mid + d * u
    head[:, :, 1] = head[:, :, 0] + 0.27 * u + rng.normal(0, 0.01, (n_trial, n_frame, 3))
    if accelerating is not None:
        t = np.arange(n_frame, dtype=np.float64)
        thorax[accelerating] = 0
        head[accelerating, :, 0] = 0
        head[accelerating, :, 0, 0] = t * (t + 1) / 2048
        head[accelerating, :, 1] = head[accelerating, :, 0] + 0.27
    return head.astype(dtype), thorax


@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("n_frame", [1, 2, 3, 31, 33, 1000, 1025, 4097])
def test_head_affine_counts_and_rows(eng, n_frame, dtype):
    """Stationary counts exactly equal to numpy's (warps that straddle two trials count through per-lane atomics), the
    affine rows within the float32 bound of the mid-quantile tests (3e-7 of the series' largest magnitude, plus one
    rounding of the scale's division); NaN where a trial has no stationary frame."""
    torch, E, _ = eng
    dt = np.dtype(dtype)
    rng = np.random.default_rng(n_frame * 10 + dt.itemsize)
    thr = 5e-5
    thr_dev = float(np.float32(thr)) if dt == np.float32 else thr           # the f32 entry point takes a float threshold
    for n_trial in (1, 3, 7):
        for n_kp in (1, 3):
            head, thorax = head_stat_trials(rng, n_trial, n_frame, n_kp, dt, n_trial // 2 if n_trial > 1 else None)
            consts = np.float32(rng.uniform(0.5, 1.5, (n_trial, 5)))
            aff, counts = E.head_affine(dev(torch, head), dev(torch, thorax), dev(torch, consts), threshold=thr)
            aff, counts = aff.cpu().numpy(), counts.cpu().numpy()
            for tr in range(n_trial):
                m, row, series = model_head.head_stats(head[tr], thorax[tr], consts[tr], thr_dev)
                assert counts[tr].tolist() == [m] * 4 + [n_frame], (n_trial, n_kp, tr, counts[tr], m)
                if n_trial > 1 and tr == n_trial // 2:
                    assert m == 0
                assert np.array_equal(aff[tr, 4:7], consts[tr, :3])
                for k, (col, s) in enumerate(((0, 0), (1, 1), (2, 2), (3, 3), (7, 4))):
                    if series[s].size == 0:
                        assert np.isnan(aff[tr, col]), (n_trial, n_kp, tr, col)
                        continue
                    scale = float(np.abs(series[s]).max())
                    if col < 3:
                        assert abs(aff[tr, col] - row[col]) <= 3e-7 * scale, (n_trial, n_kp, tr, col, aff[tr, col], row[col])
                    else:
                        q = consts[tr, 3 if col == 3 else 4] / row[col]
                        assert abs(aff[tr, col] / row[col] - 1) <= 3e-7 * scale / abs(q) + U, (n_trial, n_kp, tr, col)


def test_head_alignment_without_stationary_frames_raises(eng):
    """The dict API refuses an antenna with no stationary frame (the reference's assertion), rather than NaN rows."""
    from seqikpy_b200.alignment import AlignPose
    rng = np.random.default_rng(77)
    head, thorax = head_stat_trials(rng, 1, 200, 3, np.float64, 0)
    with pytest.raises(AssertionError):
        AlignPose({"R_head": head[0], "Thorax": thorax[0]}, legs_list=["RF", "LF"], log_level="ERROR").align_pose()


# ------------------------------------------------------------------------------------------------------------ pchip
TOL = {"float64": 1e-11, "float32": 2e-6}


def pchip_ref(y, ts, new_ts):
    """y (n_block, n, width) -> scipy's pchip_interpolate along the samples, as utils.interpolate_signal calls it."""
    n = y.shape[1]
    total = n * ts
    x = np.arange(0, total, ts)
    assert x.size == n
    return np.stack([pchip_interpolate(x, b, np.arange(0, total, new_ts), axis=0) for b in y.astype(np.float64)])


def run_pchip(eng, dtype, n_block, n, width, ts, new_ts, seed):
    torch, E, _ = eng
    rng = np.random.default_rng(seed)
    y = rng.normal(size=(n_block, n, width)).cumsum(axis=1)
    y[:, n // 3: n // 2] = y[:, n // 3: n // 3 + 1]                       # plateaus: zero secant slopes
    y = y.astype(dtype)
    got = E.pchip_resample(dev(torch, y), ts, new_ts).cpu().numpy()
    ref = pchip_ref(y, ts, new_ts)
    assert got.shape == ref.shape
    assert np.abs(got - ref).max() <= TOL[dtype] * max(1.0, np.abs(ref).max()), (n_block, n, width, ts, new_ts)


@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("width", [3, 14, 256])
def test_pchip_runtime_width(eng, dtype, width):
    """Widths other than 1 and 7 run the run-time-width instantiation (W = 0), up to 256 interleaved channels."""
    run_pchip(eng, dtype, 3, 50, width, 0.01, 0.001, width)


@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_pchip_edges_of_the_launch(eng, dtype):
    # 100x up-sampling: a CTA's output range exceeds the 32 KB staging buffer, the samples are stored directly
    run_pchip(eng, dtype, 2, 60, 7, 0.01, 0.0001, 1)
    # 300 blocks of 1000 samples x 7: more rows than grid.y, each thread walks several rows
    run_pchip(eng, dtype, 300, 1000, 7, 0.01, 0.005, 2)
    # m * width odd: consecutive rows alternate between the 128-bit and the scalar copy-out
    run_pchip(eng, dtype, 4, 41, 3, 0.01, 0.002, 3)
    run_pchip(eng, dtype, 5, 33, 1, 0.01, 0.003, 4)


def test_pchip_width_limit(eng):
    torch, E, _ = eng
    with pytest.raises(ValueError, match="256"):
        E.pchip_resample(torch.zeros((1, 10, 257), dtype=torch.float32, device="cuda"), 0.01, 0.001)
