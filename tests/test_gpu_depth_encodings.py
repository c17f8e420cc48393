"""Frame ingest from depth images in every encoding the depth_image_proc nodelets take (pft_cloud_upload_depth_images_enc
(_async)): 16UC1 or 32FC1 depth with bgr8, rgb8, bgra8, rgba8 or mono8 colour (point_cloud_xyzrgb), or depth alone
(point_cloud_xyz).

`restate` below is depth_image_proc::convert<T> plus the colour copy in numpy, every fp32 operation rounded on its own
in the nodelet's order; the device cloud must equal it bit for bit, NaN points and their colour included.  Every
colour image has four different bytes in every pixel, so any swapped channel offset changes the cloud."""
import ctypes as C
import subprocess

import numpy as np
import pytest

from pcl_tracking_b200 import _capi, pcl, synth
from pcl_tracking_b200._capi import POINT
from tests.test_gpu_depth import INTRINSICS, _bits, _padded, _pinned, _voxel_grid
from tests.test_gpu_depth_cameras import _rigid, pcl_transform
from tests.test_shim_depth_encodings import build_depth_encodings, run_depth_encodings

DEPTHS = ["16UC1", "32FC1"]
COLOURS = ["bgr8", "rgb8", "bgra8", "rgba8", "mono8", "none"]
# byte offsets of r, g, b in a colour pixel, and its bytes
LAYOUT = {"bgr8": ((2, 1, 0), 3), "rgb8": ((0, 1, 2), 3), "bgra8": ((2, 1, 0), 4), "rgba8": ((0, 1, 2), 4), "mono8": ((0, 0, 0), 1), "none": (None, 0)}


def restate(depth, colour, depth_encoding, colour_encoding, fx, fy, cx, cy):
    """The organised cloud (H * W POINT records, row-major) of one camera: depth_image_proc::convert<T> in fp32."""
    h, w = depth.shape
    cxf, cyf = np.float32(cx), np.float32(cy)
    u = np.arange(w, dtype=np.float32)[None, :]
    v = np.arange(h, dtype=np.float32)[:, None]
    if depth_encoding == "32FC1":
        assert depth.dtype == np.float32
        kx, ky = np.float32(1.0 / fx), np.float32(1.0 / fy)
        d = depth
        valid = np.isfinite(d)
    else:
        assert depth.dtype == np.uint16
        kx = np.float32(np.float64(np.float32(0.001)) / fx)
        ky = np.float32(np.float64(np.float32(0.001)) / fy)
        d = depth.astype(np.float32)
        valid = depth != 0
    with np.errstate(invalid="ignore", over="ignore"):
        x = ((u - cxf) * d) * kx
        y = ((v - cyf) * d) * ky
        z = d.copy() if depth_encoding == "32FC1" else d * np.float32(0.001)
    for a in (x, y, z):
        a[~valid] = np.float32(np.nan)
    out = np.zeros(h * w, dtype=POINT)
    out["x"], out["y"], out["z"] = x.ravel(), y.ravel(), z.ravel()
    offs, bpp = LAYOUT[colour_encoding]
    if bpp:
        c = colour.reshape(h, w, bpp).astype(np.uint32)
        r, g, b = (c[..., o] for o in offs)
        out["rgba"] = (b | (g << 8) | (r << 16) | np.uint32(255 << 24)).ravel()
    return out


SPECIALS = np.array([0.0, -0.0, -1.25, -7e3, 1e-40, -1e-45, np.float32(1.17549435e-38), np.nan, np.inf, -np.inf, 3e38, -3e38, 65.535],
                    dtype=np.float32)


def _images(w, h, depth_encoding, colour_encoding, seed):
    """Random depth in `depth_encoding` (16UC1: with 0 and 65535; 32FC1: with every value of SPECIALS) and a colour
    image whose channels differ from each other in every pixel."""
    rng = np.random.default_rng(seed)
    if depth_encoding == "32FC1":
        depth = rng.uniform(-0.5, 9.0, (h, w)).astype(np.float32)
        flat = depth.reshape(-1)
        k = min(len(flat), len(SPECIALS))
        flat[:k] = SPECIALS[:k]
        pick = rng.random(flat.shape) < 0.1
        flat[pick] = rng.choice(SPECIALS, int(pick.sum()))
    else:
        depth = rng.integers(0, 65536, (h, w), dtype=np.uint32).astype(np.uint16)
        depth[rng.random((h, w)) < 0.1] = 0
        depth.flat[0], depth.flat[-1] = 65535, 0
    _, bpp = LAYOUT[colour_encoding]
    colour = None
    if bpp:
        base = rng.integers(0, 256, (h, w, 1), dtype=np.uint32).astype(np.uint8)
        colour = base ^ np.array([0x00, 0x5A, 0xA5, 0xFF], dtype=np.uint8)[:bpp]
        if bpp == 1:
            colour = colour[..., 0]
    return depth, colour


def test_colour_channels_differ_in_every_pixel():
    # any two of the four bytes of a pixel differ, so a swapped r / g / b offset cannot go unnoticed
    _, c = _images(33, 5, "16UC1", "rgba8", 1)
    for i in range(4):
        for j in range(i + 1, 4):
            assert (c[..., i] != c[..., j]).all()
    d, c = _images(33, 5, "16UC1", "bgr8", 2)
    bgr, rgb = (restate(d, c, "16UC1", e, 365.0, 365.0, 16.0, 2.0)["rgba"] for e in ("bgr8", "rgb8"))
    assert (bgr != rgb).all()


def test_unknown_encodings_and_mismatched_arrays_are_rejected_on_the_host():
    keep = []
    d16, d32 = np.zeros((2, 3), np.uint16), np.zeros((2, 3), np.float32)
    c3, c4, c1 = np.zeros((2, 3, 3), np.uint8), np.zeros((2, 3, 4), np.uint8), np.zeros((2, 3), np.uint8)
    args = (None, None, None, None, 365.0, 365.0, 1.0, 1.0, None, keep)
    for depth, colour, denc, cenc, err in [
        (d16, c3, "16UC2", "bgr8", ValueError), (d16, c3, "16UC1", "BGR8", ValueError), (d16, c3, "16UC1", None, ValueError),
        (d16, c3, "32FC1", "bgr8", TypeError), (d32, c3, "16UC1", "bgr8", TypeError), (d32, c3, "mono16", "bgr8", TypeError),
        (d16, c4, "16UC1", "rgb8", TypeError), (d16, c3, "16UC1", "rgba8", TypeError), (d16, c3, "16UC1", "mono8", TypeError),
        (d16, c1, "16UC1", "bgra8", TypeError), (d16, c3.astype(np.uint16), "16UC1", "bgr8", TypeError), (d16, c1[:1], "16UC1", "mono8", ValueError),
    ]:
        with pytest.raises(err):
            pcl._depth_camera(depth, colour, *args[:4], denc, cenc, *args[4:])
    for depth, colour, denc, cenc, want in [(d16, c3, "16UC1", "bgr8", (0, 0)), (d16, c3, "mono16", "rgb8", (0, 1)), (d32, c4, "32FC1", "bgra8", (1, 2)),
                                            (d32, c4, "32FC1", "rgba8", (1, 3)), (d16, c1, "16UC1", "mono8", (0, 4)), (d32, None, "32FC1", "none", (1, 5))]:
        e = pcl._depth_camera(depth, colour, *args[:4], denc, cenc, *args[4:])
        assert (e.depth_encoding, e.colour_encoding) == want
        assert e.cam.depth_step == 3 * depth.itemsize and e.cam.bgr_step == (0 if colour is None else 3 * colour[0, 0].nbytes)
        assert (e.cam.bgr is None) == (colour is None)


def _camera(w, h, denc, cenc, seed, k, pose=None, pad=(0, 0)):
    depth, colour = _images(w, h, denc, cenc, seed)
    fx, fy, cx, cy = INTRINSICS[k % len(INTRINSICS)]
    if pad != (0, 0):
        depth = _padded(depth, pad[0])
        colour = None if colour is None else _padded(colour, pad[1])
    return dict(depth=depth, bgr=colour, fx=fx, fy=fy, cx=cx, cy=cy, pose=pose, depth_encoding=denc, colour_encoding=cenc)


def restate_fused(cams):
    parts = []
    for c in cams:
        colour = None if c["bgr"] is None else np.ascontiguousarray(c["bgr"])
        p = restate(np.ascontiguousarray(c["depth"]), colour, c["depth_encoding"], c["colour_encoding"], c["fx"], c["fy"], c["cx"], c["cy"])
        if c.get("pose") is not None:
            p = pcl_transform(p, np.asarray(c["pose"], dtype=np.float32)[:3, :4])
        parts.append(p)
    return np.concatenate(parts)


def _pointer_camera(c, pinned):
    """`c` as pinned pointers with explicit (padded) steps."""
    d = c["depth"]
    h, w = d.shape
    bd, sd = _pinned(np.ascontiguousarray(d), d.strides[0] - d[0].nbytes)
    pinned.append(bd)
    out = dict(c, depth=bd.ptr, width=w, height=h, depth_step=sd, bgr=None)
    if c["bgr"] is not None:
        bc, sc = _pinned(np.ascontiguousarray(c["bgr"]), c["bgr"].strides[0] - c["bgr"][0].nbytes)
        pinned.append(bc)
        out.update(bgr=bc.ptr, bgr_step=sc)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("denc", DEPTHS)
@pytest.mark.parametrize("cenc", COLOURS)
def test_every_encoding_pair_matches_restatement(denc, cenc):
    for k, (w, h, pad) in enumerate([(961, 540, (12, 7)), (101, 37, (4, 1)), (7, 3, (0, 0)), (1, 1, (0, 0))]):
        c = _camera(w, h, denc, cenc, 7 * w + h + len(cenc), k, pad=pad)
        want = _bits(restate_fused([c]))
        a = pcl.PointCloud().fromDepthImage(c["depth"], c["bgr"], c["fx"], c["fy"], c["cx"], c["cy"], depth_encoding=denc, colour_encoding=cenc)
        assert a.size() == w * h
        assert np.array_equal(_bits(a.to_numpy()), want), (denc, cenc, w, h)
        pinned = []
        p = _pointer_camera(c, pinned)
        for asynchronous in (False, True):
            b = pcl.PointCloud().fromDepthImage(p["depth"], p["bgr"], c["fx"], c["fy"], c["cx"], c["cy"], asynchronous=asynchronous, width=w,
                                                height=h, depth_step=p["depth_step"], bgr_step=p.get("bgr_step"), depth_encoding=denc,
                                                colour_encoding=cenc)
            assert np.array_equal(_bits(b.to_numpy()), want), (denc, cenc, w, h, asynchronous)
            f = pcl.PointCloud().fromDepthImages([p], asynchronous=asynchronous)
            assert np.array_equal(_bits(f.to_numpy()), want), (denc, cenc, w, h, asynchronous)


@pytest.mark.gpu
def test_32fc1_special_depths():
    # 0, -0, negative, subnormal, the smallest normal, NaN, +-inf, values whose x overflows to inf, in every colour
    w, h = 13, 1
    depth = SPECIALS.reshape(h, w)
    for k, cenc in enumerate(COLOURS):
        c = _camera(w, h, "32FC1", cenc, 40 + k, 1)
        c["depth"] = depth
        got = pcl.PointCloud().fromDepthImages([c]).to_numpy()
        want = restate_fused([c])
        assert np.array_equal(_bits(got), _bits(want)), cenc
        bad = ~np.isfinite(SPECIALS)
        assert np.isnan(got["z"][bad]).all() and np.array_equal(got["z"][~bad].view(np.uint32), SPECIALS[~bad].view(np.uint32))
        assert np.signbit(got["z"][1]) and got["z"][4] != 0  # -0 and the subnormal come through as they are
        # with a matrix: finite points moved, the overflowed ones (x = +-inf) and the invalid ones copied untouched
        c["pose"] = _rigid(np.random.default_rng(k))
        got = pcl.PointCloud().fromDepthImages([c]).to_numpy()
        assert np.array_equal(_bits(got), _bits(restate_fused([c]))), cenc


def _mixed_cameras():
    rng = np.random.default_rng(99)
    return [_camera(960, 540, "32FC1", "rgb8", 1, 0, pose=_rigid(rng), pad=(8, 5)),
            _camera(512, 424, "16UC1", "bgra8", 2, 1, pose=None),
            _camera(101, 37, "32FC1", "none", 3, 2, pose=_rigid(rng), pad=(4, 0)),
            _camera(512, 424, "16UC1", "bgr8", 4, 0, pose=_rigid(rng)),
            _camera(33, 9, "16UC1", "mono8", 5, 1, pose=None, pad=(2, 3)),
            _camera(64, 48, "32FC1", "rgba8", 6, 2, pose=_rigid(rng))]


@pytest.mark.gpu
def test_mixed_cameras_in_one_call():
    cams = _mixed_cameras()[:3]
    want = _bits(restate_fused(cams))
    # the per-camera clouds, concatenated and transformed on the host
    parts = []
    for c in cams:
        p = pcl.PointCloud().fromDepthImage(c["depth"], c["bgr"], c["fx"], c["fy"], c["cx"], c["cy"], depth_encoding=c["depth_encoding"],
                                            colour_encoding=c["colour_encoding"]).to_numpy()
        parts.append(p if c["pose"] is None else pcl_transform(p, c["pose"][:3]))
    assert np.array_equal(_bits(np.concatenate(parts)), want)
    pinned = []
    ptr_cams = [_pointer_camera(c, pinned) for c in cams]
    for asynchronous in (False, True):
        for cc in (cams, ptr_cams):
            got = pcl.PointCloud().fromDepthImages(cc, asynchronous=asynchronous)
            assert got.size() == len(want)
            assert np.array_equal(_bits(got.to_numpy()), want), asynchronous
    six = _mixed_cameras()
    assert np.array_equal(_bits(pcl.PointCloud().fromDepthImages(six).to_numpy()), _bits(restate_fused(six)))


@pytest.mark.gpu
def test_one_conversion_launch_per_frame():
    six = _mixed_cameras()
    grown = {}
    cloud = pcl.PointCloud()
    for asynchronous in (False, True):
        for n in (1, 3, 6):
            cloud.fromDepthImages(six[:n], asynchronous=asynchronous)  # staging and cloud storage in place
            cloud.ctx.synchronize()
            before = pcl.kernel_launch_count()
            cloud.fromDepthImages(six[:n], asynchronous=asynchronous)
            grown[(asynchronous, n)] = pcl.kernel_launch_count() - before
            assert cloud.size() == sum(c["depth"].size for c in six[:n])
    assert set(grown.values()) == {2}, grown  # the conversion and the header write


def _old_camera(c):
    d, b = c["depth"], c["bgr"]
    h, w = d.shape
    m12 = None
    if c["pose"] is not None:
        m = np.ascontiguousarray(np.asarray(c["pose"], np.float32)[:3])
        c["_m"] = m
        m12 = m.ctypes.data_as(C.POINTER(C.c_float))
    return _capi.DepthCamera(d.ctypes.data, d.strides[0], b.ctypes.data, b.strides[0], w, h, c["fx"], c["fy"], c["cx"], c["cy"], m12)


@pytest.mark.gpu
def test_calls_without_encodings_equal_16uc1_bgr8():
    lib = _capi.load()
    rng = np.random.default_rng(5)
    cams = [_camera(961, 540, "16UC1", "bgr8", 8, 0, pose=None, pad=(6, 7)), _camera(512, 424, "16UC1", "bgr8", 9, 1, pose=_rigid(rng)),
            _camera(7, 3, "16UC1", "bgr8", 10, 2, pose=_rigid(rng), pad=(2, 1))]
    old = (_capi.DepthCamera * 3)(*[_old_camera(c) for c in cams])
    enc = (_capi.DepthCameraEnc * 3)(*[_capi.DepthCameraEnc(old[k], _capi.DEPTH_16UC1, _capi.COLOUR_BGR8) for k in range(3)])
    c0 = cams[0]
    d, b = c0["depth"], c0["bgr"]
    args = (d.ctypes.data, d.strides[0], b.ctypes.data, b.strides[0], d.shape[1], d.shape[0], c0["fx"], c0["fy"], c0["cx"], c0["cy"])
    for asynchronous in (False, True):
        sfx = "_async" if asynchronous else ""
        x, y = pcl.PointCloud(), pcl.PointCloud()
        _capi.check(getattr(lib, "pft_cloud_upload_depth_image" + sfx)(x._h, *args))
        _capi.check(getattr(lib, "pft_cloud_upload_depth_images_enc" + sfx)(y._h, enc, 1))
        assert np.array_equal(_bits(x.to_numpy()), _bits(y.to_numpy()))
        assert np.array_equal(_bits(x.to_numpy()), _bits(restate_fused(cams[:1])))
        _capi.check(getattr(lib, "pft_cloud_upload_depth_images" + sfx)(x._h, old, 3))
        _capi.check(getattr(lib, "pft_cloud_upload_depth_images_enc" + sfx)(y._h, enc, 3))
        assert np.array_equal(_bits(x.to_numpy()), _bits(y.to_numpy()))
        assert np.array_equal(_bits(x.to_numpy()), _bits(restate_fused(cams)))


@pytest.mark.gpu
def test_malformed_encodings_are_rejected():
    lib = _capi.load()
    cloud = pcl.PointCloud()
    w, h = 8, 4
    d16, _ = _images(w, h, "16UC1", "none", 1)
    d32, _ = _images(w, h, "32FC1", "none", 2)
    col = np.zeros((h, 4 * w), np.uint8)

    def cam(denc=_capi.DEPTH_16UC1, cenc=_capi.COLOUR_BGR8, **kw):
        depth = d32 if denc == _capi.DEPTH_32FC1 else d16
        bpp = {_capi.COLOUR_BGR8: 3, _capi.COLOUR_RGB8: 3, _capi.COLOUR_BGRA8: 4, _capi.COLOUR_RGBA8: 4, _capi.COLOUR_MONO8: 1}.get(cenc, 0)
        a = dict(depth=depth.ctypes.data, depth_step=depth.strides[0], bgr=col.ctypes.data, bgr_step=bpp * w, width=w, height=h, fx=365.0, fy=365.0,
                 cx=4.0, cy=2.0, m12=None)
        a.update(kw)
        return _capi.DepthCameraEnc(_capi.DepthCamera(**a), denc, cenc)

    def arr(cams):
        return (_capi.DepthCameraEnc * len(cams))(*cams)

    F, N = _capi.DEPTH_32FC1, _capi.COLOUR_NONE
    bad = [
        ([cam(denc=2)], "camera 0"),                                                   # unknown depth encoding
        ([cam(), cam(denc=-1)], "camera 1"),
        ([cam(), cam(), cam(cenc=6)], "camera 2"),                                     # unknown colour encoding
        ([cam(cenc=-1)], "camera 0"),
        ([cam(), cam(F, depth_step=4 * w + 2)], "camera 1"),                           # 32FC1 step not a multiple of 4
        ([cam(), cam(), cam(), cam(F, depth_step=4 * w - 4)], "camera 3"),             # 32FC1 step below 4 * width
        ([cam(F, _capi.COLOUR_RGB8, bgr_step=3 * w - 1)], "camera 0"),                 # colour steps below bytes-per-pixel * width
        ([cam(), cam(F, _capi.COLOUR_BGRA8, bgr_step=4 * w - 1)], "camera 1"),
        ([cam(), cam(cenc=_capi.COLOUR_RGBA8, bgr_step=3 * w)], "camera 1"),
        ([cam(), cam(), cam(cenc=_capi.COLOUR_MONO8, bgr_step=w - 1)], "camera 2"),
        ([cam(F, _capi.COLOUR_MONO8, bgr=None)], "camera 0"),                          # null colour with pixels
        ([cam(), cam(F, _capi.COLOUR_RGB8, bgr=None)], "camera 1"),
        ([cam(), cam(F, N, depth=None)], "camera 1"),                                  # null depth, depth alone
    ]
    for fn in (lib.pft_cloud_upload_depth_images_enc, lib.pft_cloud_upload_depth_images_enc_async):
        assert fn(None, arr([cam()]), 1) == _capi.ERR_INVALID
        assert fn(cloud._h, None, 1) == _capi.ERR_INVALID
        assert fn(cloud._h, arr([cam()] * 9), 9) == _capi.ERR_INVALID
        for k, (cams, who) in enumerate(bad):
            assert fn(cloud._h, arr(cams), len(cams)) == _capi.ERR_INVALID, (fn, k)
            assert who in lib.pft_last_error().decode(), (k, lib.pft_last_error())
        # depth alone: the colour pointer and step are ignored; a camera without pixels needs no images
        ok = [cam(cenc=N, bgr=None, bgr_step=0), cam(F, N, bgr=12345, bgr_step=1), cam(F, _capi.COLOUR_MONO8),
              cam(F, _capi.COLOUR_RGBA8, width=0, depth=None, bgr=None)]
        assert fn(cloud._h, arr(ok), 4) == _capi.OK, lib.pft_last_error()
        assert cloud.size() == 3 * w * h
    want = restate_fused([dict(depth=d16, bgr=None, depth_encoding="16UC1", colour_encoding="none", fx=365.0, fy=365.0, cx=4.0, cy=2.0),
                          dict(depth=d32, bgr=None, depth_encoding="32FC1", colour_encoding="none", fx=365.0, fy=365.0, cx=4.0, cy=2.0),
                          dict(depth=d32, bgr=col[:, :w], depth_encoding="32FC1", colour_encoding="mono8", fx=365.0, fy=365.0, cx=4.0, cy=2.0)])
    assert np.array_equal(_bits(cloud.to_numpy()), _bits(want))


@pytest.mark.gpu
@pytest.mark.parametrize("denc", DEPTHS)
def test_distance_only_tracking_on_depth_alone(denc):
    s = synth.KINECT2_QHD
    objs = synth.default_objects(1)
    frames = []
    for f in range(5):
        depth, _, K = synth.depth_images(synth.render(f, objs, sensor=s)[0], s)
        if denc == "32FC1":
            metres = depth.astype(np.float32) * np.float32(0.001)
            depth = np.where(depth == 0, np.float32(np.nan), metres).astype(np.float32)
        frames.append(depth)
    fx, fy, cx, cy = K[0, 0], K[1, 1], K[0, 2], K[1, 2]
    _, oid0 = synth.render(0, objs, sensor=s)
    raw = restate(frames[0], None, denc, "none", fx, fy, cx, cy)
    model, centre = pcl.prepare_model(pcl.PointCloud(synth.model_points(raw, oid0, 0)), 0.01)

    def tracker():  # DistanceCoherence alone: the points carry no colour
        t = pcl.KLDAdaptiveParticleFilterOMPTracker(16)
        pcl.configure_like_reference(t, particle_num=300, max_particle_num=400, use_hsv=False)
        m = np.eye(4, dtype=np.float32)
        m[:3, 3] = centre
        t.setTrans(m)
        t.seed(77)
        t.setReferenceCloud(model)
        return t

    ta, tb = tracker(), tracker()
    vg = _voxel_grid()
    ca, cb, da, db = pcl.PointCloud(), pcl.PointCloud(), pcl.PointCloud(), pcl.PointCloud()
    for k, depth in enumerate(frames):
        ca.fromDepthImage(depth, None, fx, fy, cx, cy, depth_encoding=denc, colour_encoding="none")
        pts = restate(depth, None, denc, "none", fx, fy, cx, cy)
        assert (pts["rgba"] == 0).all()
        cb.upload(pts)
        assert np.array_equal(_bits(ca.to_numpy()), _bits(pts)), k
        for c, d in ((ca, da), (cb, db)):
            vg.setInputCloud(c)
            vg.filter(d)
        assert da.size() > 1000
        for t, d in ((ta, da), (tb, db)):
            t.setInputCloud(d)
            t.compute()
        assert np.array_equal(ta.getParticles().view(np.uint32), tb.getParticles().view(np.uint32)), k
        assert np.array(ta.getResult()).tobytes() == np.array(tb.getResult()).tobytes(), k
    r = ta.getResult()
    assert np.isfinite([r["x"], r["y"], r["z"]]).all()


@pytest.mark.gpu
def test_shim_program_prints_the_same_cloud(tmp_path):
    exe = build_depth_encodings(tmp_path)
    for denc, cenc in (("16UC2", "bgr8"), ("32FC1", "BGR8"), ("", "rgb8"), ("mono16", "yuv422")):
        r = run_depth_encodings(exe, tmp_path, denc, cenc)
        assert r.returncode == 4 and "pft error -1: unknown" in r.stderr, (denc, cenc, r.stderr)

    def files(k, c):
        d = np.ascontiguousarray(c["depth"])
        bd, sd = _pinned(d, 4 * (k + 1))
        (tmp_path / ("d%d.raw" % k)).write_bytes(bd.numpy().tobytes())
        cpath, sc = "-", "0"
        if c["bgr"] is not None:
            b = np.ascontiguousarray(c["bgr"])
            bc, sc = _pinned(b, k + 3)
            cpath = str(tmp_path / ("c%d.raw" % k))
            (tmp_path / ("c%d.raw" % k)).write_bytes(bc.numpy().tobytes())
        mpath = "-"
        if c["pose"] is not None:
            mpath = str(tmp_path / ("m%d.raw" % k))
            (tmp_path / ("m%d.raw" % k)).write_bytes(np.ascontiguousarray(c["pose"][:3], dtype=np.float32).tobytes())
        h, w = d.shape
        spelled = "mono16" if c["depth_encoding"] == "16UC1" and k % 2 else c["depth_encoding"]
        return [str(tmp_path / ("d%d.raw" % k)), spelled, cpath, c["colour_encoding"], str(w), str(h), str(sd), str(sc), repr(c["fx"]),
                repr(c["fy"]), repr(c["cx"]), repr(c["cy"]), mpath]

    def records(out, n, clouds):
        rec = np.frombuffer(out.read_bytes(), dtype=synth.to_pcl32(np.zeros(0, POINT)).dtype)
        assert len(rec) == clouds * n
        for i in range(clouds):
            got = np.zeros(n, dtype=POINT)
            for k in ("x", "y", "z", "rgba"):
                got[k] = rec[i * n:(i + 1) * n][k]
            yield got

    six = _mixed_cameras()
    out = tmp_path / "out.raw"
    # one camera per encoding pair: fromDepthImages, fromDepthImagesAsync and the two encoding overloads of fromDepthImage
    for denc in DEPTHS:
        for i, cenc in enumerate(COLOURS):
            c = _camera(61, 9, denc, cenc, 70 + i, i)
            r = subprocess.run([exe, str(out)] + files(i, c), capture_output=True, text=True, check=True).stdout
            assert r.splitlines() == ["549 549 1"] * 2 + ["549 61 9"] * 2, (denc, cenc)
            want = pcl.PointCloud().fromDepthImage(c["depth"], c["bgr"], c["fx"], c["fy"], c["cx"], c["cy"], depth_encoding=denc,
                                                   colour_encoding=cenc).to_numpy()
            assert np.array_equal(_bits(want), _bits(restate_fused([c])))
            for got in records(out, 549, 4):
                assert np.array_equal(_bits(got), _bits(want)), (denc, cenc)
    # six cameras of mixed encodings with poses
    args = sum((files(k, c) for k, c in enumerate(six)), [])
    n = sum(c["depth"].size for c in six)
    r = subprocess.run([exe, str(out)] + args, capture_output=True, text=True, check=True).stdout
    assert r.splitlines() == ["%d %d 1" % (n, n)] * 2
    want = pcl.PointCloud().fromDepthImages(six).to_numpy()
    for got in records(out, n, 2):
        assert np.array_equal(_bits(got), _bits(want))
