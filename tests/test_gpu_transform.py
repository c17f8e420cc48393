"""pcl::transformPointCloud on the device (pft_transform_cloud), the model builder's removeZeroPoints
(pft_remove_zero_points) and the tracked object's cloud (pft_tracker_get_result_cloud), each against a numpy
restatement: float32, one rounded operation at a time, compared bit for bit."""
import ctypes as C

import numpy as np
import pytest

from pcl_tracking_b200 import _capi as capi
from pcl_tracking_b200 import pcl
from tests import util

pytestmark = pytest.mark.gpu


def np_transform(pts, m):
    """pcl::transformPointCloud (PCL 1.8.0, not dense) in float32: x' = ((m00 x + m01 y) + m02 z) + m03 for a point
    whose three coordinates are finite; any other point is copied unchanged (bits included)."""
    m = np.asarray(m, dtype=np.float32)[:3, :4]
    out = np.array(pts, dtype=pcl.POINT, copy=True)
    x, y, z = (np.asarray(pts[k], dtype=np.float32) for k in ("x", "y", "z"))
    fin = np.isfinite(x) & np.isfinite(y) & np.isfinite(z)
    with np.errstate(all="ignore"):
        for r, k in enumerate(("x", "y", "z")):
            v = ((m[r, 0] * x + m[r, 1] * y) + m[r, 2] * z) + m[r, 3]
            out[k][fin] = v[fin]
    return out


def np_keep_nonzero(pts):
    """removeZeroPoints: keep finite points unless |x|, |y| and |z| are all below 0.01 (compared in double)."""
    x, y, z = (np.asarray(pts[k], dtype=np.float64) for k in ("x", "y", "z"))
    fin = np.isfinite(x) & np.isfinite(y) & np.isfinite(z)
    with np.errstate(invalid="ignore"):
        zero = (np.abs(x) < 0.01) & (np.abs(y) < 0.01) & (np.abs(z) < 0.01)
    return fin & ~zero


def rigid(seed, t_scale=1.0):
    rng = np.random.default_rng(seed)
    q, _ = np.linalg.qr(rng.normal(size=(3, 3)))
    q *= np.sign(np.linalg.det(q))
    m = np.eye(4)
    m[:3, :3], m[:3, 3] = q, rng.uniform(-1, 1, 3) * t_scale
    return m.astype(np.float32)


def random_cloud(n, seed, scale=2.0):
    rng = np.random.default_rng(seed)
    pts = np.zeros(n, dtype=pcl.POINT)
    for k in ("x", "y", "z"):
        pts[k] = rng.uniform(-scale, scale, n)
    pts["rgba"] = rng.integers(0, 2 ** 32, n, dtype=np.uint64).astype(np.uint32)
    return pts


def same_bits(a, b):
    return np.ascontiguousarray(a).tobytes() == np.ascontiguousarray(b).tobytes()


@pytest.mark.parametrize("n", [1, 255, 256, 4097, 200_000])
def test_random_clouds_bit_for_bit(n):
    pts = random_cloud(n, n)
    m = rigid(n)
    got = pcl.transformPointCloud(pcl.PointCloud(pts), m).to_numpy()
    assert same_bits(got, np_transform(pts, m))
    # a general (non-rigid) 3x4 matrix, given as 3x4
    g = np.random.default_rng(n + 1).normal(size=(3, 4)).astype(np.float32)
    assert same_bits(pcl.transformPointCloud(pcl.PointCloud(pts), g).to_numpy(), np_transform(pts, g))


def test_non_finite_coordinates_negative_zero_and_far_points():
    pts = random_cloud(64, 5)
    specials = [np.nan, np.inf, -np.inf]
    i = 0
    for v in specials:              # each special value in each coordinate on its own
        for k in ("x", "y", "z"):
            pts[k][i] = v
            i += 1
    pts["x"][i] = pts["y"][i] = pts["z"][i] = np.nan; i += 1
    nan_payload = np.array([0x7fc01234], dtype=np.uint32).view(np.float32)[0]
    pts["y"][i] = nan_payload; i += 1
    pts["x"][i], pts["y"][i], pts["z"][i] = -0.0, -0.0, -0.0; i += 1
    pts["x"][i], pts["y"][i], pts["z"][i] = 0.0, -0.0, 0.0; i += 1
    for j in range(8):              # coordinates around 1e4 m
        pts["x"][i], pts["y"][i], pts["z"][i] = 1e4 + j * 0.37, -1e4 - j * 1.1, 9999.99 + j
        i += 1
    m = rigid(11, t_scale=500.0)
    got = pcl.transformPointCloud(pcl.PointCloud(pts), m).to_numpy()
    want = np_transform(pts, m)
    assert same_bits(got, want)
    assert np.array_equal(got["rgba"], pts["rgba"])                     # colour of every point, finite or not
    bad = ~(np.isfinite(pts["x"]) & np.isfinite(pts["y"]) & np.isfinite(pts["z"]))
    assert bad.sum() == 11 and same_bits(got[bad], pts[bad])            # non-finite points copied unchanged
    # the identity keeps every point, -0.0 included
    assert same_bits(pcl.transformPointCloud(pcl.PointCloud(pts), np.eye(4)).to_numpy(), np_transform(pts, np.eye(4)))


def test_in_place_equals_out_of_place():
    pts = random_cloud(10_000, 2)
    pts["z"][::97] = np.nan
    m = rigid(3)
    a = pcl.PointCloud(pts)
    out = pcl.transformPointCloud(a, m).to_numpy()
    b = pcl.PointCloud(pts)
    assert pcl.transformPointCloud(b, m, out=b) is b
    assert same_bits(b.to_numpy(), out) and same_bits(out, np_transform(pts, m))
    # twice in place = the numpy composition of two transforms
    m2 = rigid(4)
    pcl.transformPointCloud(b, m2, out=b)
    assert same_bits(b.to_numpy(), np_transform(np_transform(pts, m), m2))


def test_empty_input_gives_empty_output():
    empty = pcl.PointCloud(np.zeros(0, dtype=pcl.POINT))
    out = pcl.PointCloud(random_cloud(10, 1))          # a stale output of another size is overwritten
    pcl.transformPointCloud(empty, rigid(1), out=out)
    assert out.size() == 0
    assert pcl.transformPointCloud(pcl.PointCloud(), rigid(1)).size() == 0


def test_input_straight_from_the_downsample():
    """The count of a pft_passthrough_voxel_grid output lives on the device only; the transform reads it there (one
    kernel launch, no host read in between)."""
    pts = random_cloud(50_000, 9, scale=0.5)
    pts["x"][::13] = np.nan
    vg = pcl.VoxelGrid()
    vg.setLeafSize(0.01)
    vg.setPassThrough("z", -0.3, 0.4)
    vg.setInputCloud(pcl.PointCloud(pts))
    ds = vg.filter()
    m = rigid(21)
    moved = pcl.PointCloud()                            # (creating a cloud launches a header write of its own)
    before = pcl.kernel_launch_count()
    pcl.transformPointCloud(ds, m, out=moved)
    assert pcl.kernel_launch_count() - before == 1
    got = moved.to_numpy()
    down = ds.to_numpy()
    assert len(down) > 1000 and same_bits(got, np_transform(down, m))


def test_errors():
    lib = capi.load()
    ctx = pcl.Context.default()
    a, b = pcl.PointCloud(random_cloud(10, 1)), pcl.PointCloud()
    m = np.ascontiguousarray(rigid(1)[:3], dtype=np.float32)
    assert lib.pft_transform_cloud(None, a._h, b._h, capi.ptr(m)) == capi.ERR_INVALID
    assert lib.pft_transform_cloud(ctx._h, None, b._h, capi.ptr(m)) == capi.ERR_INVALID
    assert lib.pft_transform_cloud(ctx._h, a._h, None, capi.ptr(m)) == capi.ERR_INVALID
    assert lib.pft_transform_cloud(ctx._h, a._h, b._h, None) == capi.ERR_INVALID
    for v in (np.nan, np.inf, -np.inf):
        for k in (0, 5, 11):
            bad = m.copy()
            bad.reshape(-1)[k] = v
            assert lib.pft_transform_cloud(ctx._h, a._h, b._h, capi.ptr(bad)) == capi.ERR_INVALID
            assert b"not finite" in lib.pft_last_error()
    other = pcl.Context(0)
    c = pcl.PointCloud(random_cloud(10, 2), ctx=other)
    assert lib.pft_transform_cloud(ctx._h, c._h, b._h, capi.ptr(m)) == capi.ERR_INVALID
    assert lib.pft_transform_cloud(ctx._h, a._h, c._h, capi.ptr(m)) == capi.ERR_INVALID
    with pytest.raises(ValueError):
        pcl.transformPointCloud(a, np.eye(3))
    # removeZeroPoints: null arguments, in place, another context
    assert lib.pft_remove_zero_points(None, a._h, b._h) == capi.ERR_INVALID
    assert lib.pft_remove_zero_points(ctx._h, None, b._h) == capi.ERR_INVALID
    assert lib.pft_remove_zero_points(ctx._h, a._h, None) == capi.ERR_INVALID
    assert lib.pft_remove_zero_points(ctx._h, a._h, a._h) == capi.ERR_INVALID
    assert lib.pft_remove_zero_points(ctx._h, c._h, b._h) == capi.ERR_INVALID
    # the result cloud: null arguments, no result yet, a cloud of another context
    t = pcl.KLDAdaptiveParticleFilterOMPTracker(16)
    assert lib.pft_tracker_get_result_cloud(None, 0.0, b._h) == capi.ERR_INVALID
    assert lib.pft_tracker_get_result_cloud(t._h, 0.0, None) == capi.ERR_INVALID
    assert lib.pft_tracker_get_result_cloud(t._h, 0.0, b._h) == capi.ERR_STATE
    assert lib.pft_tracker_get_result_cloud(t._h, 0.0, c._h) == capi.ERR_INVALID
    # a valid call after the failures still works
    assert same_bits(pcl.transformPointCloud(a, m).to_numpy(), np_transform(a.to_numpy(), m))


def test_remove_zero_points_at_the_edges():
    vals = [0.0, -0.0, 0.0099, -0.0099, 0.00999999, 0.01, -0.01, np.float32(0.01), 0.0100001, 0.5]
    grid = np.array(np.meshgrid(vals, vals, vals, indexing="ij")).reshape(3, -1).T
    pts = np.zeros(len(grid) + 9, dtype=pcl.POINT)
    pts["x"][:len(grid)], pts["y"][:len(grid)], pts["z"][:len(grid)] = grid.T
    pts["rgba"] = np.arange(len(pts), dtype=np.uint32) * 2654435761
    for j, (k, v) in enumerate([(k, v) for k in ("x", "y", "z") for v in (np.nan, np.inf, -np.inf)]):
        row = len(grid) + j                      # one non-finite coordinate, the others far from zero / at zero
        pts["x"][row], pts["y"][row], pts["z"][row] = (0.5, 0.0, 0.3) if j % 2 else (0.0, 0.0, 0.0)
        pts[k][row] = v
    got = pcl.removeZeroPoints(pcl.PointCloud(pts)).to_numpy()
    keep = np_keep_nonzero(pts)
    assert same_bits(got, pts[keep])
    assert 0 < keep.sum() < len(grid)
    # |v| < 0.01 decides in double: float32(0.01) lies just below 0.01 and is dropped, the next float32 up is kept
    one = np.zeros(3, dtype=pcl.POINT)
    one["x"] = [np.float32(0.0099), np.float32(0.01), np.nextafter(np.float32(0.01), np.float32(1))]
    assert same_bits(pcl.removeZeroPoints(pcl.PointCloud(one)).to_numpy(), one[2:])


def test_result_cloud_is_the_reference_at_the_result_pose():
    scene, model, centre = util.small_case(31, n_scene=3000, n_model=500)
    t = pcl.KLDAdaptiveParticleFilterOMPTracker(16)
    pcl.configure_like_reference(t, particle_num=100, max_particle_num=150, use_hsv=False)
    m = np.eye(4, dtype=np.float32)
    m[:3, 3] = centre
    t.setTrans(m)
    t.seed(5)
    t.setReferenceCloud(model)
    t.setInputCloud(pcl.PointCloud(scene))
    t.compute(); t.compute()
    r = t.getResult()
    ref = pcl.PointCloud(model)
    for z in (-0.005, 0.0, 0.02):
        got = t.getResultCloud(z).to_numpy()
        M = t.toEigenMatrix(r)
        M[2, 3] = np.float32(M[2, 3]) + np.float32(z)
        assert len(got) == len(model)
        assert same_bits(got, pcl.transformPointCloud(ref, M).to_numpy())
        assert same_bits(got, np_transform(model, M))          # order and colours of the reference as given
        box = t.getResultBox(z)
        mean = np.array([got[k].astype(np.float64).mean() for k in ("x", "y", "z")])
        assert np.abs(mean - box["centroid"]).max() < 1e-6
    # getResultBox keeps its output when getResultCloud runs in between
    b0 = t.getResultBox()
    t.getResultCloud()
    assert t.getResultBox().tobytes() == b0.tobytes()
    # into a given cloud, which is overwritten
    out = pcl.PointCloud(random_cloud(7, 3))
    assert t.getResultCloud(0.0, out=out) is out
    assert same_bits(out.to_numpy(), np_transform(model, t.toEigenMatrix(r)))
