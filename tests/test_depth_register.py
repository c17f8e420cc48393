"""Registration of a depth image into its colour camera, as the depth_image_proc/register nodelet does it
(RegisterNodelet::convert<T>), restated in Python: the reference of tests/test_gpu_depth_register.py.

`register_literal` is steps 1-5 of pft.h's pft_cloud_upload_depth_images_reg, a scalar loop over the depth pixels in
raster order with upstream's z-buffer test, every double operation in Python floats and every float one in numpy
float32.  `register_fast` computes the same image with numpy: the candidates of every pixel at once, then each colour
pixel's smallest candidate after its last reset.  It is used at camera sizes only, and checked here against the
literal loop.  Where upstream is undefined C++ (a double -> int cast of NaN or outside int, a 16UC1 fromMeters outside
0 .. 65535) or a 32FC1 candidate is NaN, both drop the candidate."""
import numpy as np
import pytest

F32 = np.float32
INT_LO, INT_HI = -2147483649.0, 2147483648.0


def _to_int(x):
    return int(x) if INT_LO < x < INT_HI else None  # int() truncates toward zero, as the C cast


def _project(pu, pv, depth, dcam, ccam, M):
    fx, fy, cx, cy, tx, ty = dcam
    X = ((pu - cx) * depth - tx) * (1.0 / fx)
    Y = ((pv - cy) * depth - ty) * (1.0 / fy)
    p = [((M[r][0] * X + M[r][1] * Y) + M[r][2] * depth) + M[r][3] for r in range(3)]
    inv_z = 1.0 / p[2] if p[2] != 0.0 else (np.inf if np.copysign(1.0, p[2]) > 0 else -np.inf)
    cfx, cfy, ccx, ccy, ctx, cty = ccam
    with np.errstate(invalid="ignore"):
        u = _to_int(((cfx * p[0] + ctx) * inv_z + ccx) + 0.5)
        v = _to_int(((cfy * p[1] + cty) * inv_z + ccy) + 0.5)
    return u, v, p[2]


def _from_metres(z, metres):
    with np.errstate(over="ignore", invalid="ignore"):
        m = F32(z)
        if metres:
            return None if np.isnan(m) else m
        t = m * F32(1000.0) + F32(0.5)
    return np.uint16(int(t)) if -1.0 < t < 65536.0 else None


def register_literal(depth, metres, dcam, ccam, width, height, M, fill):
    """The registered (height, width) image of `depth` (uint16 mm or float32 m): dcam, ccam = (fx, fy, cx, cy, Tx, Ty)
    of the depth and colour cameras, M the 3x4 depth -> colour matrix (nested lists or array of float64)."""
    M = [[float(x) for x in row] for row in np.asarray(M, dtype=np.float64)[:3]]
    dcam, ccam = [float(x) for x in dcam], [float(x) for x in ccam]
    reg = np.full((height, width), np.nan if metres else 0, dtype=F32 if metres else np.uint16)
    valid = (lambda x: np.isfinite(x)) if metres else (lambda x: x != 0)
    h, w = depth.shape
    for v in range(h):
        for u in range(w):
            d = depth[v, u]
            if not valid(d):
                continue
            dm = float(d) if metres else float(F32(d) * F32(0.001))
            if fill:
                u1, v1, z1 = _project(float(F32(u) - F32(0.5)), float(F32(v) - F32(0.5)), dm, dcam, ccam, M)
                u2, v2, z2 = _project(float(F32(u) + F32(0.5)), float(F32(v) + F32(0.5)), dm, dcam, ccam, M)
                if None in (u1, v1, u2, v2) or u1 < 0 or u2 >= width or v1 < 0 or v2 >= height:
                    continue
                new = _from_metres(0.5 * (z1 + z2), metres)
            else:
                u1, v1, z1 = _project(float(u), float(v), dm, dcam, ccam, M)
                if None in (u1, v1) or u1 < 0 or u1 >= width or v1 < 0 or v1 >= height:
                    continue
                u2, v2 = u1, v1
                new = _from_metres(z1, metres)
            if new is None:
                continue
            for nv in range(v1, v2 + 1):
                for nu in range(u1, u2 + 1):
                    if not valid(reg[nv, nu]) or reg[nv, nu] > new:
                        reg[nv, nu] = new
    return reg


def _project_np(pu, pv, depth, dcam, ccam, M):
    fx, fy, cx, cy, tx, ty = dcam
    X = ((pu - cx) * depth - tx) * (1.0 / fx)
    Y = ((pv - cy) * depth - ty) * (1.0 / fy)
    p = [((M[r, 0] * X + M[r, 1] * Y) + M[r, 2] * depth) + M[r, 3] for r in range(3)]
    cfx, cfy, ccx, ccy, ctx, cty = ccam
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        inv_z = 1.0 / p[2]
        uf = ((cfx * p[0] + ctx) * inv_z + ccx) + 0.5
        vf = ((cfy * p[1] + cty) * inv_z + ccy) + 0.5
    ok = (uf > INT_LO) & (uf < INT_HI) & (vf > INT_LO) & (vf < INT_HI)
    u = np.where(ok, np.trunc(np.where(ok, uf, 0.0)), 0).astype(np.int64)
    v = np.where(ok, np.trunc(np.where(ok, vf, 0.0)), 0).astype(np.int64)
    return u, v, p[2], ok


def register_fast(depth, metres, dcam, ccam, width, height, M, fill):
    """register_literal in numpy."""
    M = np.asarray(M, dtype=np.float64)[:3]
    dcam, ccam = [float(x) for x in dcam], [float(x) for x in ccam]
    h, w = depth.shape
    vv, uu = np.mgrid[0:h, 0:w]
    d = depth.ravel()
    idx = np.arange(h * w)
    uu, vv = uu.ravel(), vv.ravel()
    keep = np.isfinite(d) if metres else d != 0
    d, idx, uu, vv = d[keep], idx[keep], uu[keep], vv[keep]
    dm = d.astype(np.float64) if metres else (d.astype(F32) * F32(0.001)).astype(np.float64)
    if fill:
        lo_u, lo_v = (uu.astype(F32) - F32(0.5)).astype(np.float64), (vv.astype(F32) - F32(0.5)).astype(np.float64)
        hi_u, hi_v = (uu.astype(F32) + F32(0.5)).astype(np.float64), (vv.astype(F32) + F32(0.5)).astype(np.float64)
        u1, v1, z1, ok1 = _project_np(lo_u, lo_v, dm, dcam, ccam, M)
        u2, v2, z2, ok2 = _project_np(hi_u, hi_v, dm, dcam, ccam, M)
        ok = ok1 & ok2 & (u1 >= 0) & (u2 < width) & (v1 >= 0) & (v2 < height)
        with np.errstate(invalid="ignore"):
            z = 0.5 * (z1 + z2)
    else:
        u1, v1, z, ok = _project_np(uu.astype(np.float64), vv.astype(np.float64), dm, dcam, ccam, M)
        ok &= (u1 >= 0) & (u1 < width) & (v1 >= 0) & (v1 < height)
        u2, v2 = u1, v1
    with np.errstate(over="ignore", invalid="ignore"):
        m = z.astype(F32)
        if metres:
            ok &= ~np.isnan(m)
            val = m
        else:
            t = m * F32(1000.0) + F32(0.5)
            ok &= (t > -1.0) & (t < 65536.0)
            val = np.where(ok, t, 0).astype(np.int64).astype(np.uint16)
    u1, v1, u2, v2, val, idx = u1[ok], v1[ok], u2[ok], v2[ok], val[ok], idx[ok]
    # every (target, candidate) pair of the rectangles
    nu, nv = np.maximum(u2 - u1 + 1, 0), np.maximum(v2 - v1 + 1, 0)
    cnt = nu * nv
    rep = np.repeat(np.arange(len(cnt)), cnt)
    k = np.arange(cnt.sum()) - np.repeat(np.cumsum(cnt) - cnt, cnt)
    tu = u1[rep] + k % np.maximum(nu[rep], 1)
    tv = v1[rep] + k // np.maximum(nu[rep], 1)
    t = tv * width + tu
    cv, ci = val[rep], idx[rep]
    reset = (cv == -np.inf) if metres else (cv == 0)
    last = np.full(width * height, -1, dtype=np.int64)
    np.maximum.at(last, t[reset], ci[reset])
    reg = np.full(width * height, np.nan if metres else 0, dtype=F32 if metres else np.uint16)
    reg[last >= 0] = -np.inf if metres else 0
    after = ~reset & (ci > last[t])
    t, cv, ci = t[after], cv[after], ci[after]
    order = np.lexsort((ci, cv.astype(np.float64), t))  # per target: the least value, the earliest of equal ones
    t, cv = t[order], cv[order]
    first = np.ones(len(t), dtype=bool)
    first[1:] = t[1:] != t[:-1]
    reg[t[first]] = cv[first]
    return reg.reshape(height, width)


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32 if a.dtype == F32 else np.uint16)


def both(*args):
    """register_literal, checked bit for bit against register_fast."""
    a = register_literal(*args)
    b = register_fast(*args)
    assert np.array_equal(_bits(a), _bits(b))
    return a


EYE = np.eye(4)[:3]
NAN = F32(np.nan)


def _translation(tx=0.0, ty=0.0, tz=0.0):
    m = EYE.copy()
    m[:, 3] = (tx, ty, tz)
    return m


def test_identity_extrinsic_gives_the_depth_image():
    cam = (100.0, 100.0, 1.5, 1.0, 0.0, 0.0)
    d32 = np.array([[0.5, 1.0, 2.0, 4.0], [np.nan, 1.0, 0.25, -1.0], [2.0, np.inf, 8.0, 0.5]], dtype=F32)
    d16 = np.array([[1000, 2000, 0, 500], [250, 1000, 4000, 8000], [0, 0, 1000, 2000]], dtype=np.uint16)
    # u' = (int)((u - cx) + cx + 0.5) = u, also for z < 0 (x and 1 / z change sign together); invalid stays invalid
    assert np.array_equal(both(d32, True, cam, cam, 4, 3, EYE, False), np.where(np.isfinite(d32), d32, NAN), equal_nan=True)
    assert np.array_equal(both(d16, False, cam, cam, 4, 3, EYE, False), d16)


def test_pure_x_translation_shifts_by_fx_tx_over_z():
    cam = (100.0, 100.0, 2.0, 0.0, 0.0, 0.0)
    got = both(np.ones((1, 6), F32), True, cam, cam, 6, 1, _translation(tx=0.02), False)  # + fx * tx / z = 2 pixels
    assert np.isnan(got[0, :2]).all() and (got[0, 2:] == 1.0).all()
    # pixel u lands on u + 2 / z: u=0 -> 2, u=1 -> 2 (z 2: collides, the nearer stays), u=2 -> 4, u=3 -> 7 (outside),
    # u=4 -> 5, u=5 -> 7 (outside)
    got = both(F32([[1.0, 2.0, 1.0, 0.5, 2.0, 1.0]]), True, cam, cam, 6, 1, _translation(tx=0.02), False)
    assert np.array_equal(got[0], F32([np.nan, np.nan, 1.0, np.nan, 1.0, 2.0]), equal_nan=True)


@pytest.mark.parametrize("fill", [False, True])
def test_projection_in_minus_one_to_zero_lands_in_column_zero(fill):
    dcam = (100.0, 100.0, 0.0, 0.0, 0.0, 0.0)
    ccam = (100.0, 100.0, 0.0, 0.2, 0.0, 0.0)  # rows: v' = (int)(0.2 + 0.5) = 0; corners (int)(0.2) = 0, (int)(1.2) = 1
    depth = F32([[1.0, np.nan, np.nan]])
    # u' = (int)(0 - 1.2 + 0.5) = (int)(-0.7) = 0: column 0, where floor would drop it
    got = both(depth, True, dcam, ccam, 3, 2, _translation(tx=-0.012), fill)
    if not fill:
        assert got[0, 0] == 1.0 and np.isnan(got.ravel()[1:]).all()
    else:
        # corners: u1 = (int)(-0.5 - 1.2 + 0.5) = (int)(-1.2) = -1 < 0: skipped
        assert np.isnan(got).all()
        got = both(depth, True, dcam, ccam, 3, 2, _translation(tx=-0.006), fill)  # u1 = (int)(-0.6) = 0, u2 = (int)(0.4) = 0
        assert (got[:, 0] == 1.0).all() and np.isnan(got[:, 1:]).all()
    # a projection at or below -1 is dropped
    assert np.isnan(both(depth, True, dcam, ccam, 3, 2, _translation(tx=-0.016), False)).all()


def test_fill_upsampling_rectangles():
    dcam = (10.0, 10.0, 0.0, 0.0, 0.0, 0.0)
    ccam = (20.0, 20.0, 0.0, 0.0, 0.0, 0.0)
    depth = F32([[1.0, 2.0], [4.0, 0.5]])
    # pixel u covers columns [(int)(2u - 0.5), (int)(2u + 1.5)] = [0, 1] (u = 0), [1, 3] (u = 1); rows likewise
    want = F32([[1.0, 1.0, 2.0, 2.0],
                [1.0, 0.5, 0.5, 0.5],
                [4.0, 0.5, 0.5, 0.5],
                [4.0, 0.5, 0.5, 0.5]])
    assert np.array_equal(both(depth, True, dcam, ccam, 4, 4, EYE, True), want)
    # 3x3: the rectangles of u = 1 or v = 1 end at 3, outside: those pixels are skipped whole
    assert np.array_equal(both(depth, True, dcam, ccam, 3, 3, EYE, True), F32([[1, 1, np.nan], [1, 1, np.nan], [np.nan] * 3]), equal_nan=True)
    # without fill the same cameras leave holes: pixel u lands on (int)(2u + 0.5) = 2u
    assert np.array_equal(both(depth, True, dcam, ccam, 4, 4, EYE, False),
                          F32([[1, np.nan, 2, np.nan], [np.nan] * 4, [4, np.nan, 0.5, np.nan], [np.nan] * 4]), equal_nan=True)


def test_zbuffer_collision_keeps_the_nearest():
    dcam = (20.0, 20.0, 0.0, 0.0, 0.0, 0.0)
    ccam = (10.0, 10.0, 0.0, 0.0, 0.0, 0.0)
    # u' = (int)(u / 2 + 0.5): u = 1 and u = 2 both land on column 1
    for a, b in ((3.0, 2.0), (2.0, 3.0)):
        got = both(F32([[1.0, a, b, 1.0]]), True, dcam, ccam, 3, 1, EYE, False)
        assert np.array_equal(got, F32([[1.0, 2.0, 1.0]]))
    got = both(np.array([[1000, 3000, 2000, 1000]], np.uint16), False, dcam, ccam, 3, 1, EYE, False)
    assert np.array_equal(got, np.array([[1000, 2000, 1000]], np.uint16))


# colour fx so small that every depth pixel lands on colour pixel (2, 2)
SPOT = (1e-6, 1e-6, 2.0, 2.0, 0.0, 0.0)
DSPOT = (500.0, 500.0, 1.0, 0.0, 0.0, 0.0)


def test_16uc1_reset_then_a_larger_value():
    m = _translation(tz=-0.4999)
    # 1000 mm -> z 0.5001 -> 500; 500 mm -> z 1e-4 -> (uint16)(0.6) = 0, a reset; 1300 mm -> 800
    got = both(np.array([[1000, 500, 1300]], np.uint16), False, DSPOT, SPOT, 4, 4, m, False)
    assert got[2, 2] == 800 and np.count_nonzero(got) == 1
    assert both(np.array([[1000, 0, 1300]], np.uint16), False, DSPOT, SPOT, 4, 4, m, False)[2, 2] == 500
    assert both(np.array([[1300, 1000, 500]], np.uint16), False, DSPOT, SPOT, 4, 4, m, False)[2, 2] == 0
    # z * 1000 + 0.5 at or below -1, or at 65536 and above, is undefined upstream: dropped
    assert both(np.array([[1000, 498]], np.uint16), False, DSPOT, SPOT, 4, 4, m, False)[2, 2] == 500
    assert both(np.array([[1000]], np.uint16), False, DSPOT, SPOT, 4, 4, _translation(tz=65.0), False)[2, 2] == 0
    assert both(np.array([[1000]], np.uint16), False, DSPOT, SPOT, 4, 4, _translation(tz=64.0), False)[2, 2] == 65000


@pytest.mark.parametrize("seq,want", [
    ("P", np.inf), ("P1", 1.0), ("1P", 1.0), ("1N", -np.inf), ("NP", np.inf), ("PN", -np.inf), ("N1P", 1.0), ("1NP", np.inf), ("N", -np.inf),
])
def test_32fc1_infinite_candidates(seq, want):
    m = EYE.copy()
    m[2, 2] = 10.0  # z' = 10 z: 3e38 -> +inf, -3e38 -> -inf, 0.1 -> 1
    depth = F32([[{"P": 3e38, "N": -3e38, "1": 0.1}[c] for c in seq]])
    got = both(depth, True, DSPOT, SPOT, 4, 4, m, False)
    one = F32(10.0 * float(F32(0.1)))
    assert got[2, 2] == (one if want == 1.0 else want)
    assert np.isnan(np.delete(got.ravel(), 10)).all()


@pytest.mark.parametrize("first", [1.0, -1.0])
def test_signed_zero_ties_keep_the_earlier(first):
    m = EYE.copy()
    m[2, 2] = 1e-50  # z' = +-1e-50, which is +-0.0 as a float
    dcam = (1e60, 1e60, 0.0, 0.0, 0.0, 0.0)
    ccam = (1.0, 1.0, 2.0, 2.0, 0.0, 0.0)
    got = both(F32([[first, -first, 3.0]]), True, dcam, ccam, 4, 4, m, False)
    assert got[2, 2] == 0.0 and np.signbit(got[2, 2]) == (first < 0)
    # a smaller value still wins over both
    got = both(F32([[first, -first, -2.0]]), True, dcam, ccam, 4, 4, m, False)
    assert got[2, 2] == F32(-2e-50)


def _random_case(rng, metres, fill, dw, dh, cw, ch):
    depth = rng.uniform(0.3, 3.0, (dh, dw)).astype(F32)
    odd = rng.random((dh, dw)) < 0.1
    if metres:
        depth[odd] = rng.choice(F32([np.nan, np.inf, -np.inf, 0.0, -0.0, -0.5, 3e38, -3e38, 1e-3]), int(odd.sum()))
    else:
        depth = (depth * 1000).astype(np.uint16)
        depth[odd] = 0
    dcam = (dw * 0.9, dw * 0.9, dw / 2 - 0.3, dh / 2 + 0.2, 0.0, 0.0)
    ccam = (cw * 0.95, cw * 0.95, cw / 2 + 0.1, ch / 2 - 0.4, rng.uniform(-0.05, 0.05), rng.uniform(-0.05, 0.05))
    a = rng.uniform(-0.2, 0.2, 3)
    from scipy.spatial.transform import Rotation
    M = np.zeros((3, 4))
    M[:, :3] = Rotation.from_rotvec(a).as_matrix()
    M[:, 3] = rng.uniform(-0.1, 0.1, 3)
    M[2, 3] = rng.choice([0.0, -0.6])  # -0.6: some candidates reach z <= 0.0005 (16UC1 resets) or behind the camera
    return depth, metres, dcam, ccam, cw, ch, M, fill


@pytest.mark.parametrize("metres", [False, True])
@pytest.mark.parametrize("fill", [False, True])
def test_fast_restatement_equals_the_literal_loop(metres, fill):
    rng = np.random.default_rng(11 + 2 * metres + fill)
    for dw, dh, cw, ch in ((17, 13, 23, 11), (40, 30, 20, 15), (9, 31, 33, 7)):
        case = _random_case(rng, metres, fill, dw, dh, cw, ch)
        got = both(*case)
        assert (~np.isnan(got) if metres else got != 0).any()
