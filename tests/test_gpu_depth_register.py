"""Depth images registered into their colour camera on the device (pft_cloud_upload_depth_images_reg(_async)): the
depth_image_proc/register -> point_cloud_xyzrgb nodelet chain.

The reference is tests/test_depth_register.py's restatement of RegisterNodelet::convert<T> followed by
tests/test_gpu_depth_encodings.py's restatement of the conversion; the device cloud must equal it bit for bit, NaN
points and their colour included."""
import ctypes as C
import subprocess

import numpy as np
import pytest

from pcl_tracking_b200 import _capi, pcl, synth
from pcl_tracking_b200._capi import POINT
from tests.test_depth_register import DSPOT, EYE, SPOT, _random_case, _translation, register_fast
from tests.test_gpu_depth import _bits, _padded, _pinned, _voxel_grid
from tests.test_gpu_depth_cameras import _rigid, pcl_transform
from tests.test_gpu_depth_encodings import _images, restate, restate_fused
from tests.test_shim_depth_register import build_depth_register

pytestmark = pytest.mark.gpu
F32 = np.float32


def reg_camera(depth, denc, dcam, colour, cenc, ccam, width, height, M, fill, pose=None):
    """A camera mapping of fromDepthImages with a `registration`: dcam, ccam = (fx, fy, cx, cy, Tx, Ty)."""
    reg = dict(depth_fx=dcam[0], depth_fy=dcam[1], depth_cx=dcam[2], depth_cy=dcam[3], depth_Tx=dcam[4], depth_Ty=dcam[5], colour_Tx=ccam[4],
               colour_Ty=ccam[5], depth_to_colour=np.asarray(M, np.float64), fill_upsampling=fill)
    return dict(depth=depth, bgr=colour, fx=ccam[0], fy=ccam[1], cx=ccam[2], cy=ccam[3], width=width, height=height, pose=pose, depth_encoding=denc,
                colour_encoding=cenc, registration=reg)


def registered_image(c):
    r = c["registration"]
    dcam = (r["depth_fx"], r["depth_fy"], r["depth_cx"], r["depth_cy"], r["depth_Tx"], r["depth_Ty"])
    ccam = (c["fx"], c["fy"], c["cx"], c["cy"], r["colour_Tx"], r["colour_Ty"])
    return register_fast(np.ascontiguousarray(c["depth"]), c["depth_encoding"] == "32FC1", dcam, ccam, c["width"], c["height"], r["depth_to_colour"],
                         r["fill_upsampling"])


def restate_cams(cams):
    """The fused cloud of registered and already-registered cameras: registration, then the conversion."""
    plain = []
    for c in cams:
        if c.get("registration") is not None:
            c = dict(c, depth=registered_image(c))
        plain.append(c)
    return restate_fused(plain)


def pointer_camera(c, pinned, pad=(4, 3)):
    """`c` as pinned pointers with padded steps."""
    out = dict(c)
    d = np.ascontiguousarray(c["depth"])
    bd, sd = _pinned(d, pad[0] * d.itemsize)
    pinned.append(bd)
    out.update(depth=bd.ptr, depth_step=sd)
    if c.get("registration") is not None:
        out["registration"] = dict(c["registration"], depth_width=d.shape[1], depth_height=d.shape[0])
    else:
        out.update(width=d.shape[1], height=d.shape[0])
    if c["bgr"] is not None:
        b = np.ascontiguousarray(c["bgr"])
        bc, sc = _pinned(b, pad[1])
        pinned.append(bc)
        out.update(bgr=bc.ptr, bgr_step=sc)
    return out


def check_all_ways(cams, want=None):
    """fromDepthImages from arrays and from pinned pointers, sync and async, each equal to the restatement."""
    want = _bits(restate_cams(cams)) if want is None else want
    pinned = []
    ptr = [pointer_camera(c, pinned) for c in cams]
    for asynchronous in (False, True):
        for cc in (cams, ptr):
            got = pcl.PointCloud().fromDepthImages(cc, asynchronous=asynchronous)
            assert got.size() == len(want)
            assert np.array_equal(_bits(got.to_numpy()), want), asynchronous
    return want


def kinect2_rig(frame, denc, fill, objects=None):
    """sd depth from the default camera, qhd colour from a camera 52 mm to its right, as a Kinect2's two sensors."""
    sd, qhd = synth.KINECT2_SD, synth.KINECT2_QHD
    objects = objects or synth.default_objects(1)
    depth, _, Kd = synth.depth_images(synth.render(frame, objects, sensor=sd)[0], sd)
    offset = np.array([0.052, 0.0015, -0.002])
    _, bgr, Kc = synth.depth_images(synth.render(frame, objects, sensor=qhd, camera=(np.eye(3), offset))[0], qhd)
    if denc == "32FC1":
        depth = np.where(depth == 0, F32(np.nan), depth.astype(F32) * F32(0.001)).astype(F32)
    M = _translation(*(-offset))
    dcam = (Kd[0, 0], Kd[1, 1], Kd[0, 2], Kd[1, 2], 0.0, 0.0)
    ccam = (Kc[0, 0], Kc[1, 1], Kc[0, 2], Kc[1, 2], 0.0, 0.0)
    return reg_camera(depth, denc, dcam, bgr, "bgr8", ccam, qhd["width"], qhd["height"], M, fill)


@pytest.mark.parametrize("denc", ["16UC1", "32FC1"])
@pytest.mark.parametrize("fill", [False, True])
def test_kinect2_sd_depth_into_qhd_colour(denc, fill):
    c = kinect2_rig(0, denc, fill)
    reg = registered_image(c)
    valid = ~np.isnan(reg) if denc == "32FC1" else reg != 0
    assert valid.mean() > (0.4 if fill else 0.15)  # sd depth covers a part of the qhd grid; fill_upsampling closes the holes
    check_all_ways([c])


@pytest.mark.parametrize("fill", [False, True])
def test_depth_finer_than_colour_collides(fill):
    sd, qhd = synth.KINECT2_SD, synth.KINECT2_QHD
    objs = synth.default_objects(2)
    depth, _, Kd = synth.depth_images(synth.render(3, objs, sensor=qhd)[0], qhd)
    offset = np.array([-0.03, 0.01, 0.005])
    _, bgr, Kc = synth.depth_images(synth.render(3, objs, sensor=sd, camera=(np.eye(3), offset))[0], sd)
    c = reg_camera(depth, "16UC1", (Kd[0, 0], Kd[1, 1], Kd[0, 2], Kd[1, 2], 0.0, 0.0), bgr, "bgr8", (Kc[0, 0], Kc[1, 1], Kc[0, 2], Kc[1, 2], 0.0, 0.0),
                   sd["width"], sd["height"], _translation(*(-offset)), fill)
    check_all_ways([c])


@pytest.mark.parametrize("denc", ["16UC1", "32FC1"])
@pytest.mark.parametrize("fill", [False, True])
def test_odd_sizes_padded_steps_and_special_depths(denc, fill):
    rng = np.random.default_rng(5 + fill)
    for dw, dh, cw, ch in ((61, 37, 45, 29), (33, 9, 97, 41), (7, 3, 5, 11), (1, 1, 3, 2)):
        depth, metres, dcam, ccam, w, h, M, _ = _random_case(rng, denc == "32FC1", fill, dw, dh, cw, ch)
        cenc = ["rgb8", "bgra8", "mono8", "none"][dw % 4]
        _, colour = _images(w, h, "16UC1", cenc, dw + ch)
        c = reg_camera(_padded(depth, 6 * depth.itemsize), denc, dcam, None if colour is None else _padded(colour, 5), cenc, ccam, w, h, M, fill)
        check_all_ways([c])


# the known answers of tests/test_depth_register.py, through the device
def _spot(depth, metres, m, dcam=DSPOT, ccam=SPOT, w=4, h=4, fill=False):
    return reg_camera(depth, "32FC1" if metres else "16UC1", dcam, None, "none", ccam, w, h, m, fill)


def _known_cases():
    m_inf = EYE.copy()
    m_inf[2, 2] = 10.0
    m_zero = EYE.copy()
    m_zero[2, 2] = 1e-50
    cam = (100.0, 100.0, 2.0, 0.0, 0.0, 0.0)
    yield _spot(np.array([[1000, 500, 1300]], np.uint16), False, _translation(tz=-0.4999))    # 16UC1 reset, then larger
    yield _spot(np.array([[1300, 1000, 500]], np.uint16), False, _translation(tz=-0.4999))    # reset last
    for seq in ("P", "P1", "1P", "1N", "NP", "PN", "N1P", "1NP"):                             # 32FC1 +-inf
        yield _spot(F32([[{"P": 3e38, "N": -3e38, "1": 0.1}[k] for k in seq]]), True, m_inf)
    for first in (1.0, -1.0):                                                                 # +0 / -0 ties
        yield _spot(F32([[first, -first, 3.0]]), True, m_zero, dcam=(1e60, 1e60, 0.0, 0.0, 0.0, 0.0), ccam=(1.0, 1.0, 2.0, 2.0, 0.0, 0.0))
    yield _spot(F32([[1.0, 2.0, 1.0, 0.5, 2.0, 1.0]]), True, _translation(tx=0.02), cam, cam, 6, 1)  # x-translation
    for fill in (False, True):                                                                # u' in (-1, 0)
        yield _spot(F32([[1.0, np.nan, np.nan]]), True, _translation(tx=-0.006 if fill else -0.012), (100.0, 100.0, 0.0, 0.0, 0.0, 0.0),
                    (100.0, 100.0, 0.0, 0.2, 0.0, 0.0), 3, 2, fill)
    yield _spot(F32([[1.0, 2.0], [4.0, 0.5]]), True, EYE, (10.0, 10.0, 0.0, 0.0, 0.0, 0.0), (20.0, 20.0, 0.0, 0.0, 0.0, 0.0), 4, 4, True)  # rectangles


def test_known_answers_on_the_device():
    cases = list(_known_cases())
    for c in cases:
        check_all_ways([c])
    # the +0 / -0 tie keeps the sign of the earlier candidate in z
    z = [pcl.PointCloud().fromDepthImages([c]).to_numpy()["z"][10] for c in cases[10:12]]
    assert z[0] == 0 and z[1] == 0 and not np.signbit(z[0]) and np.signbit(z[1])


def _three(rng):
    a = kinect2_rig(1, "16UC1", True)
    a["pose"] = _rigid(rng)
    d, col = _images(64, 48, "32FC1", "rgba8", 3)
    b = dict(depth=d, bgr=col, fx=60.0, fy=61.0, cx=31.5, cy=23.0, pose=_rigid(rng), depth_encoding="32FC1", colour_encoding="rgba8")
    depth, metres, dcam, ccam, w, h, M, fill = _random_case(rng, True, False, 80, 60, 50, 40)
    _, colour = _images(w, h, "16UC1", "mono8", 4)
    c = reg_camera(depth, "32FC1", dcam, colour, "mono8", ccam, w, h, M, fill)
    return [a, b, c]


def test_three_cameras_with_and_without_registration():
    cams = _three(np.random.default_rng(8))
    check_all_ways(cams)
    check_all_ways(cams[::-1])


def test_identity_registration_equals_the_enc_cloud():
    lib = _capi.load()
    d, col = _images(97, 31, "16UC1", "bgr8", 12)
    plain = dict(depth=d, bgr=col, fx=80.0, fy=80.0, cx=48.0, cy=15.0, depth_encoding="16UC1", colour_encoding="bgr8")
    want = _bits(pcl.PointCloud().fromDepthImages([plain]).to_numpy())
    c = reg_camera(d, "16UC1", (80.0, 80.0, 48.0, 15.0, 0.0, 0.0), col, "bgr8", (80.0, 80.0, 48.0, 15.0, 0.0, 0.0), 97, 31, np.eye(4), False)
    assert np.array_equal(registered_image(c), d)
    check_all_ways([c], want)
    # every depth_to_colour NULL: the _enc call, bit for bit and launch for launch
    rng = np.random.default_rng(9)
    cams = [dict(plain, pose=_rigid(rng)), _three(rng)[1]]  # two cameras, neither registered on the device
    keep = []
    enc = [pcl._depth_camera(c["depth"], c["bgr"], None, None, None, None, c["depth_encoding"], c["colour_encoding"], c["fx"], c["fy"], c["cx"], c["cy"],
                             pcl._pose_m12(c, k, keep), keep) for k, c in enumerate(cams)]
    e = (_capi.DepthCameraEnc * 2)(*enc)
    r = (_capi.DepthCameraReg * 2)(*[_capi.DepthCameraReg(x, None) for x in enc])
    for sfx in ("", "_async"):
        x, y = pcl.PointCloud(), pcl.PointCloud()
        _capi.check(getattr(lib, "pft_cloud_upload_depth_images_enc" + sfx)(x._h, e, 2))
        x.ctx.synchronize()
        before = pcl.kernel_launch_count()
        _capi.check(getattr(lib, "pft_cloud_upload_depth_images_reg" + sfx)(y._h, r, 2))
        assert pcl.kernel_launch_count() - before == 2
        assert np.array_equal(_bits(x.to_numpy()), _bits(y.to_numpy()))
        assert np.array_equal(_bits(x.to_numpy()), _bits(restate_cams(cams)))


def test_launches_per_frame_do_not_depend_on_the_cameras():
    rng = np.random.default_rng(10)
    base = _three(rng)
    grown = {}
    cloud = pcl.PointCloud()
    for n in (1, 2, 8):
        cams = [base[2] if k % 2 == 0 else base[k % 2] for k in range(n)]
        for asynchronous in (False, True):
            cloud.fromDepthImages(cams, asynchronous=asynchronous)
            cloud.ctx.synchronize()
            before = pcl.kernel_launch_count()
            cloud.fromDepthImages(cams, asynchronous=asynchronous)
            grown[(n, asynchronous)] = pcl.kernel_launch_count() - before
            assert np.array_equal(_bits(cloud.to_numpy()), _bits(restate_cams(cams)))
    assert set(grown.values()) == {5}, grown  # reset scatter, z-buffer scatter, finalise, conversion, header


def test_registered_camera_without_depth_pixels_gives_nan_points_with_colour():
    _, col = _images(9, 4, "16UC1", "rgb8", 2)
    for depth in (np.zeros((0, 5), np.uint16), np.zeros((3, 0), F32)):
        c = reg_camera(depth, "32FC1" if depth.dtype == F32 else "16UC1", (5.0, 5.0, 2.0, 1.0, 0.0, 0.0), col, "rgb8", (9.0, 9.0, 4.0, 2.0, 0.0, 0.0), 9,
                       4, np.eye(4), True)
        got = pcl.PointCloud().fromDepthImages([c]).to_numpy()
        assert len(got) == 36 and np.isnan(got["z"]).all()
        assert np.array_equal(_bits(got), _bits(restate_cams([c])))


def test_malformed_registrations_are_rejected():
    lib = _capi.load()
    cloud = pcl.PointCloud()
    d16, _ = _images(8, 4, "16UC1", "none", 1)
    d10 = np.ones((6, 10), np.uint16)  # registered already: the colour camera's size
    col = np.zeros((6, 3 * 10), np.uint8)
    eye = np.ascontiguousarray(np.eye(4)[:3])

    def cam(m=eye, denc=_capi.DEPTH_16UC1, **kw):
        e = _capi.DepthCameraEnc(_capi.DepthCamera(d16.ctypes.data, d16.strides[0], col.ctypes.data, 30, 10, 6, 9.0, 9.0, 5.0, 3.0, None), denc,
                                 _capi.COLOUR_BGR8)
        a = dict(depth_width=8, depth_height=4, depth_fx=7.0, depth_fy=7.0, depth_cx=4.0, depth_cy=2.0, depth_tx=0.0, depth_ty=0.0, colour_tx=0.0,
                 colour_ty=0.0, fill_upsampling=0)
        for k in ("depth", "depth_step", "width", "fx", "cx"):
            if k in kw:
                setattr(e.cam, k, kw.pop(k))
        a.update(kw)
        return _capi.DepthCameraReg(e, None if m is None else m.ctypes.data_as(C.POINTER(C.c_double)), **a)

    bad_m = [eye.copy() for _ in range(3)]
    bad_m[0][1, 2], bad_m[1][2, 3], bad_m[2][0, 0] = np.nan, np.inf, -np.inf
    nan, inf = float("nan"), float("inf")
    bad = [
        ([cam(bad_m[0])], "camera 0"), ([cam(), cam(bad_m[1])], "camera 1"), ([cam(), cam(), cam(bad_m[2])], "camera 2"),  # matrix entries
        ([cam(depth_fx=0.0)], "camera 0"), ([cam(), cam(depth_fy=nan)], "camera 1"), ([cam(depth_fx=inf)], "camera 0"),      # depth fx / fy
        ([cam(depth_cx=nan)], "camera 0"), ([cam(), cam(depth_cy=inf)], "camera 1"), ([cam(depth_tx=nan)], "camera 0"),      # cx, cy, Tx, Ty
        ([cam(depth_ty=-inf)], "camera 0"), ([cam(), cam(colour_tx=nan)], "camera 1"), ([cam(colour_ty=inf)], "camera 0"),
        ([cam(cx=nan)], "camera 0"),
        ([cam(fill_upsampling=2)], "camera 0"), ([cam(), cam(fill_upsampling=-1)], "camera 1"),                               # fill_upsampling
        ([cam(depth_step=15)], "camera 0"), ([cam(), cam(depth_step=14)], "camera 1"),                                        # depth steps
        ([cam(denc=_capi.DEPTH_32FC1, depth_step=30)], "camera 0"), ([cam(denc=_capi.DEPTH_32FC1, depth_step=16)], "camera 0"),
        ([cam(depth=None)], "camera 0"), ([cam(), cam(depth=None, depth_height=1)], "camera 1"),                              # null depth
        ([cam(depth_width=65536, depth_height=32768, depth_step=131072)], "camera 0"),                                        # 2^31 pixels
        ([cam(fx=0.0)], "camera 0"), ([cam(), cam(denc=5)], "camera 1"),                                                      # colour side
    ]
    arr = lambda cams: (_capi.DepthCameraReg * len(cams))(*cams)
    for fn in (lib.pft_cloud_upload_depth_images_reg, lib.pft_cloud_upload_depth_images_reg_async):
        assert fn(None, arr([cam()]), 1) == _capi.ERR_INVALID
        assert fn(cloud._h, None, 1) == _capi.ERR_INVALID
        assert fn(cloud._h, arr([cam()] * 9), 9) == _capi.ERR_INVALID
        assert fn(cloud._h, arr([cam()]), 0) == _capi.ERR_INVALID
        for k, (cams, who) in enumerate(bad):
            assert fn(cloud._h, arr(cams), len(cams)) == _capi.ERR_INVALID, (fn, k)
            assert who in lib.pft_last_error().decode(), (k, lib.pft_last_error())
        # no depth pixels: no depth image needed; no colour pixels: nothing added; an unregistered camera ignores the fields
        ok = [cam(depth=None, depth_width=0), cam(width=0), cam(None, depth=d10.ctypes.data, depth_step=20, fill_upsampling=7, depth_fx=nan),
              cam(fill_upsampling=1)]
        assert fn(cloud._h, arr(ok), 4) == _capi.OK, lib.pft_last_error()
        assert cloud.size() == 3 * 60
    with pytest.raises(ValueError):  # the depth array's shape against the registration's depth size
        c = reg_camera(d16, "16UC1", (7.0, 7.0, 4.0, 2.0, 0.0, 0.0), col[:, :30].reshape(6, 10, 3), "bgr8", (9.0, 9.0, 5.0, 3.0, 0.0, 0.0), 10, 6, eye, 0)
        c["registration"]["depth_width"] = 9
        pcl.PointCloud().fromDepthImages([c])


def test_tracking_on_registered_frames():
    objs = synth.default_objects(1)
    frames = [kinect2_rig(f, "16UC1", True, objs) for f in range(6)]
    raw = restate_cams(frames[:1])
    _, oid = synth.render(0, objs, sensor=synth.KINECT2_SD)
    # the model from the depth camera's own cloud (the object's points), centred as the reference does
    sd = synth.KINECT2_SD
    pts0 = synth.render(0, objs, sensor=sd)[0]
    model, centre = pcl.prepare_model(pcl.PointCloud(synth.model_points(pts0, oid, 0)), 0.01)

    def tracker():
        t = pcl.KLDAdaptiveParticleFilterOMPTracker(16)
        pcl.configure_like_reference(t, particle_num=300, max_particle_num=400)
        m = np.eye(4, dtype=np.float32)
        m[:3, 3] = centre
        t.setTrans(m)
        t.seed(78)
        t.setReferenceCloud(model)
        return t

    ta, tb = tracker(), tracker()
    vg = _voxel_grid()
    ca, cb, da, db = pcl.PointCloud(), pcl.PointCloud(), pcl.PointCloud(), pcl.PointCloud()
    assert np.isfinite(raw["z"]).sum() > 100_000
    for k, c in enumerate(frames):
        ca.fromDepthImages([c], asynchronous=k % 2 == 1)
        pts = restate_cams([c])
        cb.upload(pts)
        assert np.array_equal(_bits(ca.to_numpy()), _bits(pts)), k
        for src, dst in ((ca, da), (cb, db)):
            vg.setInputCloud(src)
            vg.filter(dst)
        for t, d in ((ta, da), (tb, db)):
            t.setInputCloud(d)
            t.compute()
        assert np.array_equal(ta.getParticles().view(np.uint32), tb.getParticles().view(np.uint32)), k
        assert np.array(ta.getResult()).tobytes() == np.array(tb.getResult()).tobytes(), k


def test_shim_program_prints_the_same_cloud(tmp_path):
    exe = build_depth_register(tmp_path)
    rng = np.random.default_rng(21)
    cams = [kinect2_rig(2, "32FC1", False), _three(rng)[1]]
    cams[0]["pose"] = _rigid(rng)
    args = []
    for k, c in enumerate(cams):
        d = np.ascontiguousarray(c["depth"])
        (tmp_path / ("d%d.raw" % k)).write_bytes(d.tobytes())
        (tmp_path / ("c%d.raw" % k)).write_bytes(np.ascontiguousarray(c["bgr"]).tobytes())
        (tmp_path / ("p%d.raw" % k)).write_bytes(np.ascontiguousarray(c["pose"][:3], np.float32).tobytes())
        r = c.get("registration")
        h, w = np.asarray(c["bgr"]).shape[:2]
        cpp = np.asarray(c["bgr"]).shape[2] if np.asarray(c["bgr"]).ndim == 3 else 1
        args += [str(tmp_path / ("d%d.raw" % k)), c["depth_encoding"], str(d.shape[1]), str(d.shape[0]), str(d.strides[0]),
                 str(tmp_path / ("c%d.raw" % k)), c["colour_encoding"], str(w), str(h), str(w * cpp), repr(float(c["fx"])), repr(float(c["fy"])), repr(float(c["cx"])),
                 repr(float(c["cy"])), str(tmp_path / ("p%d.raw" % k))]
        if r is None:
            args.append("-")
        else:
            mpath = tmp_path / ("m%d.raw" % k)
            mpath.write_bytes(np.ascontiguousarray(np.asarray(r["depth_to_colour"], np.float64)[:3, :4]).tobytes())
            args += [str(mpath)] + [repr(float(r[x])) for x in ("depth_fx", "depth_fy", "depth_cx", "depth_cy", "depth_Tx", "depth_Ty", "colour_Tx",
                                                                  "colour_Ty")] + [str(int(r["fill_upsampling"]))]
    out = tmp_path / "out.raw"
    res = subprocess.run([exe, str(out)] + args, capture_output=True, text=True, check=True).stdout
    want = restate_cams(cams)
    n = len(want)
    assert res.splitlines() == ["%d %d 1" % (n, n)] * 2
    rec = np.frombuffer(out.read_bytes(), dtype=synth.to_pcl32(np.zeros(0, POINT)).dtype)
    assert len(rec) == 2 * n
    for i in range(2):
        got = np.zeros(n, dtype=POINT)
        for k in ("x", "y", "z", "rgba"):
            got[k] = rec[i * n:(i + 1) * n][k]
        assert np.array_equal(_bits(got), _bits(want)), i
