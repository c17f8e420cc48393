"""Frame ingest from registered depth + colour images (pft_cloud_upload_depth_image(_async), depth_image_kernel).

The contract is depth_image_proc::convert<uint16_t> plus the colour copy of the point_cloud_xyzrgb nodelet, the code
that computes the points topic the reference subscribes to (ref: src/auto_tracking.cpp:775); `restate` below is that
contract in numpy, every fp32 operation rounded on its own.  The device cloud must equal it bit for bit (NaNs
included), and tracking on it must equal tracking on the PointCloud2 payload built from the same images."""
import subprocess

import numpy as np
import pytest

from pcl_tracking_b200 import pcl, synth
from pcl_tracking_b200._capi import POINT
from tests.test_shim_depth import build_depth_ingest

pytestmark = pytest.mark.gpu


def restate(depth, bgr, fx, fy, cx, cy):
    """The organised cloud (H * W POINT records, row-major) of a uint16 mm depth image and a bgr8 image."""
    h, w = depth.shape
    cxf, cyf = np.float32(cx), np.float32(cy)
    kx = np.float32(np.float64(np.float32(0.001)) / fx)
    ky = np.float32(np.float64(np.float32(0.001)) / fy)
    d = depth.astype(np.float32)
    u = np.arange(w, dtype=np.float32)[None, :]
    v = np.arange(h, dtype=np.float32)[:, None]
    x = ((u - cxf) * d) * kx
    y = ((v - cyf) * d) * ky
    z = d * np.float32(0.001)
    bad = depth == 0
    for a in (x, y, z):
        a[bad] = np.float32(np.nan)
    c = bgr.astype(np.uint32)
    out = np.zeros(h * w, dtype=POINT)
    out["x"], out["y"], out["z"] = x.ravel(), y.ravel(), z.ravel()
    out["rgba"] = (c[..., 0] | (c[..., 1] << 8) | (c[..., 2] << 16) | np.uint32(255 << 24)).ravel()
    return out


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32).reshape(len(a), 4)


def _random_images(w, h, seed):
    rng = np.random.default_rng(seed)
    depth = rng.integers(0, 65536, (h, w), dtype=np.uint32).astype(np.uint16)
    depth[rng.random((h, w)) < 0.1] = 0
    depth.flat[0], depth.flat[-1] = 65535, 0
    bgr = rng.integers(0, 256, (h, w, 3), dtype=np.uint32).astype(np.uint8)
    return depth, bgr


def _padded_rows(img, pad_bytes):
    """The bytes of `img` in rows `pad_bytes` longer than its pixels (a padded image of step row + pad_bytes)."""
    h, row = img.shape[0], img[0].nbytes
    buf = np.full((h, row + pad_bytes), 0xA5, dtype=np.uint8)
    buf[:, :row] = np.ascontiguousarray(img).reshape(h, -1).view(np.uint8)
    return buf


def _padded(img, pad_bytes):
    """`img` as a numpy view into padded rows: its row stride is the step."""
    v = _padded_rows(img, pad_bytes)[:, :img[0].nbytes].view(img.dtype).reshape(img.shape)
    assert v.strides[0] == img[0].nbytes + pad_bytes
    return v


def _pinned(img, pad_bytes):
    """(PinnedBuffer, step): `img` in page-locked memory with padded rows."""
    rows = _padded_rows(img, pad_bytes)
    return pcl.PinnedBuffer.of(rows), rows.shape[1]


INTRINSICS = [(365.0, 365.0, 256.0, 212.0), (540.0, 540.0, 480.0, 270.0), (366.193, 365.817, 255.409, 208.786)]


@pytest.mark.parametrize("w,h,pad_d,pad_c", [(512, 424, 0, 0), (960, 540, 0, 0), (512, 424, 64, 13), (961, 540, 2, 5), (7, 3, 6, 1), (1, 1, 0, 0)])
def test_matches_restatement(w, h, pad_d, pad_c):
    depth, bgr = _random_images(w, h, w * 7 + h)
    for k, (fx, fy, cx, cy) in enumerate(INTRINSICS):
        want = _bits(restate(depth, bgr, fx, fy, cx, cy))
        # numpy images: packed, or views into padded rows (the row stride is the step)
        dv, cv = (depth, bgr) if k == 0 else (_padded(depth, pad_d), _padded(bgr, pad_c))
        got = pcl.PointCloud().fromDepthImage(dv, cv, fx, fy, cx, cy)
        assert got.size() == w * h
        assert np.array_equal(_bits(got.to_numpy()), want), (w, h, k)
        # pinned pointers with explicit steps, synchronous and on the copy stream
        (bd, sd), (bc, sc) = _pinned(depth, pad_d), _pinned(bgr, pad_c)
        for asynchronous in (False, True):
            c = pcl.PointCloud().fromDepthImage(bd.ptr, bc.ptr, fx, fy, cx, cy, asynchronous=asynchronous, width=w, height=h,
                                                depth_step=sd, bgr_step=sc)
            assert np.array_equal(_bits(c.to_numpy()), want), (w, h, k, asynchronous)


def _pcl32_payload(pts):
    return np.ascontiguousarray(synth.to_pcl32(pts)).view(np.uint8)


def _tracker(model, centre):
    t = pcl.KLDAdaptiveParticleFilterOMPTracker(16)
    pcl.configure_like_reference(t, particle_num=300, max_particle_num=400, use_hsv=True)
    m = np.eye(4, dtype=np.float32)
    m[:3, 3] = centre
    t.setTrans(m)
    t.seed(77)
    t.setReferenceCloud(model)
    return t


def _voxel_grid():
    vg = pcl.ApproximateVoxelGrid()
    vg.setLeafSize(0.01, 0.01, 0.01)
    vg.setPassThrough("z", 0.0, 10.0)
    return vg


@pytest.mark.parametrize("sensor", ["sd", "qhd"])
def test_tracking_equals_pointcloud2_ingest(sensor):
    s = synth.KINECT2_SD if sensor == "sd" else synth.KINECT2_QHD
    w, h = s["width"], s["height"]
    objs = synth.default_objects(1)
    rendered = [synth.render(f, objs, sensor=s)[0] for f in range(6)]
    images = [synth.depth_images(p, s) for p in rendered]
    depth0, bgr0, K = images[0]
    fx, fy, cx, cy = K[0, 0], K[1, 1], K[0, 2], K[1, 2]
    _, oid0 = synth.render(0, objs, sensor=s)
    model, centre = pcl.prepare_model(pcl.PointCloud(synth.model_points(restate(depth0, bgr0, fx, fy, cx, cy), oid0, 0)), 0.01)
    ta, tb = _tracker(model, centre), _tracker(model, centre)
    vg = _voxel_grid()
    ca, cb, da, db = pcl.PointCloud(), pcl.PointCloud(), pcl.PointCloud(), pcl.PointCloud()
    for k, (depth, bgr, _) in enumerate(images):
        ca.fromDepthImage(depth, bgr, fx, fy, cx, cy)
        cb.fromPointCloud2(_pcl32_payload(restate(depth, bgr, fx, fy, cx, cy)), w, h, 32)
        assert np.array_equal(_bits(ca.to_numpy()), _bits(cb.to_numpy())), k
        vg.setInputCloud(ca)
        vg.filter(da)
        vg.setInputCloud(cb)
        vg.filter(db)
        assert da.size() > 1000
        assert np.array_equal(_bits(da.to_numpy()), _bits(db.to_numpy())), k
        for t, d in ((ta, da), (tb, db)):
            t.setInputCloud(d)
            t.compute()
        pa, pb = ta.getParticles(), tb.getParticles()
        assert np.array_equal(pa.view(np.uint32), pb.view(np.uint32)), k
        assert np.array_equal(ta.rawWeights().view(np.uint32), tb.rawWeights().view(np.uint32)), k
        ra, rb = np.array(ta.getResult()), np.array(tb.getResult())
        assert ra.tobytes() == rb.tobytes(), k
    # the images came through: the tracker sits on the object
    r = ta.getResult()
    assert np.isfinite([r["x"], r["y"], r["z"]]).all()


def _frame_loop(bufs, shape, K, model, centre, pipelined):
    w, h = shape
    fx, fy, cx, cy = K[0, 0], K[1, 1], K[0, 2], K[1, 2]
    t = _tracker(model, centre)
    vg = _voxel_grid()
    clouds, ds = [pcl.PointCloud(), pcl.PointCloud()], pcl.PointCloud()
    poses = []

    def up(k, asynchronous):
        clouds[k % 2].fromDepthImage(bufs[k][0].ptr, bufs[k][1].ptr, fx, fy, cx, cy, asynchronous=asynchronous, width=w, height=h)

    if pipelined:
        up(0, True)
    for k in range(len(bufs)):
        if pipelined:
            if k + 1 < len(bufs):  # frame k + 1 travels while frame k is tracked
                up(k + 1, True)
        else:
            up(k, False)
        vg.setInputCloud(clouds[k % 2])
        vg.filter(ds)
        t.setInputCloud(ds)
        t.compute()
        poses.append(np.array(t.getResult()).tobytes() + t.getParticles().tobytes() + ds.to_numpy().tobytes())
    return poses


def test_async_double_buffered_equals_synchronous():
    s = synth.KINECT2_QHD
    objs = synth.default_objects(1)
    images = [synth.depth_images(synth.render(f, objs, sensor=s)[0], s) for f in range(6)]
    bufs = [(pcl.PinnedBuffer.of(d), pcl.PinnedBuffer.of(c)) for d, c, _ in images]
    depth0, bgr0, K = images[0]
    _, oid0 = synth.render(0, objs, sensor=s)
    raw = restate(depth0, bgr0, K[0, 0], K[1, 1], K[0, 2], K[1, 2])
    model, centre = pcl.prepare_model(pcl.PointCloud(synth.model_points(raw, oid0, 0)), 0.01)
    shape = (s["width"], s["height"])
    serial = _frame_loop(bufs, shape, K, model, centre, pipelined=False)
    piped = _frame_loop(bufs, shape, K, model, centre, pipelined=True)
    assert serial == piped


def test_malformed_arguments_are_rejected():
    lib = pcl.capi.load()
    cloud = pcl.PointCloud()
    w, h = 8, 4
    depth, bgr = _random_images(w, h, 5)
    d, c = depth.ctypes.data, bgr.ctypes.data
    good = (d, 2 * w, c, 3 * w, w, h, 365.0, 365.0, 4.0, 2.0)
    inf, nan = float("inf"), float("nan")
    bad = [
        (None, 2 * w, c, 3 * w, w, h, 365.0, 365.0, 4.0, 2.0),     # null depth
        (d, 2 * w, None, 3 * w, w, h, 365.0, 365.0, 4.0, 2.0),     # null colour
        (d, 2 * w - 2, c, 3 * w, w, h, 365.0, 365.0, 4.0, 2.0),    # depth step too small
        (d, 2 * w + 1, c, 3 * w, w, h, 365.0, 365.0, 4.0, 2.0),    # odd depth step
        (d, 2 * w, c, 3 * w - 1, w, h, 365.0, 365.0, 4.0, 2.0),    # colour step too small
        (d, 2 * w, c, 3 * w, w, h, 0.0, 365.0, 4.0, 2.0),          # fx zero
        (d, 2 * w, c, 3 * w, w, h, 365.0, 0.0, 4.0, 2.0),          # fy zero
        (d, 2 * w, c, 3 * w, w, h, inf, 365.0, 4.0, 2.0),          # fx not finite
        (d, 2 * w, c, 3 * w, w, h, 365.0, nan, 4.0, 2.0),          # fy not finite
        (d, 2 * w, c, 3 * w, w, h, 365.0, 365.0, nan, 2.0),        # cx not finite
        (d, 2 * w, c, 3 * w, w, h, 365.0, 365.0, 4.0, -inf),       # cy not finite
        (d, 2 * 65536, c, 3 * 65536, 65536, 32768, 365.0, 365.0, 4.0, 2.0),  # 2^31 pixels
    ]
    for fn in (lib.pft_cloud_upload_depth_image, lib.pft_cloud_upload_depth_image_async):
        assert fn(None, *good) == pcl.capi.ERR_INVALID
        for k, args in enumerate(bad):
            assert fn(cloud._h, *args) == pcl.capi.ERR_INVALID, (fn, k)
        assert fn(cloud._h, *good) == pcl.capi.OK
        assert cloud.size() == w * h
        for ew, eh in ((0, h), (w, 0), (0, 0)):
            assert fn(cloud._h, None, 0, None, 0, ew, eh, 365.0, 365.0, 4.0, 2.0) == pcl.capi.OK
            assert cloud.size() == 0
    e = pcl.PointCloud().fromDepthImage(np.zeros((0, 5), np.uint16), np.zeros((0, 5, 3), np.uint8), 365.0, 365.0, 2.0, 0.0)
    assert e.size() == 0
    with pytest.raises(pcl.PftError):
        pcl.PointCloud().fromDepthImage(depth, bgr, 0.0, 365.0, 4.0, 2.0)
    with pytest.raises(TypeError):
        pcl.PointCloud().fromDepthImage(depth.astype(np.float32), bgr, 365.0, 365.0, 4.0, 2.0)


def test_shim_program_prints_the_same_cloud(tmp_path):
    exe = build_depth_ingest(tmp_path)
    w, h, pad_d, pad_c = 961, 540, 4, 7
    depth, bgr = _random_images(w, h, 11)
    fx, fy, cx, cy = INTRINSICS[2]
    (bd, sd), (bc, sc) = _pinned(depth, pad_d), _pinned(bgr, pad_c)
    (tmp_path / "d.raw").write_bytes(bd.numpy().tobytes())
    (tmp_path / "c.raw").write_bytes(bc.numpy().tobytes())
    out = tmp_path / "out.raw"
    r = _stdout([exe, str(tmp_path / "d.raw"), str(tmp_path / "c.raw"), str(w), str(h), str(sd), str(sc), repr(fx), repr(fy), repr(cx), repr(cy), str(out)])
    assert r.splitlines() == ["%d %d %d" % (w * h, w, h)] * 2
    rec = np.frombuffer(out.read_bytes(), dtype=synth.to_pcl32(np.zeros(0, POINT)).dtype)
    assert len(rec) == 2 * w * h
    want = restate(depth, bgr, fx, fy, cx, cy)
    for half in (rec[:w * h], rec[w * h:]):
        got = np.zeros(w * h, dtype=POINT)
        for k in ("x", "y", "z", "rgba"):
            got[k] = half[k]
        assert np.array_equal(_bits(got), _bits(want))


def _stdout(cmd):
    return subprocess.run(cmd, capture_output=True, text=True, check=True).stdout

