"""Several calibrated depth cameras fused into one scene cloud (pft_cloud_upload_depth_images(_async), the
multi-camera form of depth_image_kernel).

The contract is the PCL composition over the nodelet's clouds: for each camera k, pcl::transformPointCloud(cloud_k,
T_k) (PCL 1.8.0: finite points only, x' = ((m00 x + m01 y) + m02 z) + m03, every fp32 operation rounded on its own),
then scene += cloud_k.  `restate_fused` below is that contract in numpy on top of test_gpu_depth.restate; the device
cloud must equal it bit for bit, and tracking on it must equal tracking on the same composition done on the host."""
import ctypes as C
import subprocess

import numpy as np
import pytest

import oracle
from pcl_tracking_b200 import _capi, pcl, synth
from pcl_tracking_b200._capi import POINT
from tests.test_gpu_depth import INTRINSICS, _bits, _padded, _pinned, _random_images, _tracker, _voxel_grid, restate
from tests.test_shim_depth_cameras import build_depth_cameras

pytestmark = pytest.mark.gpu


def pcl_transform(pts, m):
    """pcl::transformPointCloud of a cloud that is not dense: finite points moved by the 3x4 fp32 matrix, one rounded
    fp32 operation at a time; the others copied as they are."""
    m = np.asarray(m, dtype=np.float32)
    out = pts.copy()
    x, y, z = pts["x"], pts["y"], pts["z"]
    finite = np.isfinite(x) & np.isfinite(y) & np.isfinite(z)
    with np.errstate(invalid="ignore", over="ignore"):
        for r, k in enumerate(("x", "y", "z")):
            v = ((m[r, 0] * x + m[r, 1] * y) + m[r, 2] * z) + m[r, 3]
            out[k][finite] = v[finite]
    return out


def restate_fused(cams):
    """The fused cloud of the camera dicts (depth, bgr, fx, fy, cx, cy, pose or None), concatenated in camera order."""
    parts = []
    for c in cams:
        p = restate(np.ascontiguousarray(c["depth"]), np.ascontiguousarray(c["bgr"]), c["fx"], c["fy"], c["cx"], c["cy"])
        if c.get("pose") is not None:
            p = pcl_transform(p, np.asarray(c["pose"], dtype=np.float32)[:3, :4])
        parts.append(p)
    return np.concatenate(parts) if parts else np.zeros(0, POINT)


def _rigid(rng):
    """A random rigid transform (4x4 float32) with negative entries."""
    q, r = np.linalg.qr(rng.standard_normal((3, 3)))
    q = q * np.sign(np.diag(r))
    if np.linalg.det(q) < 0:
        q[:, 0] = -q[:, 0]
    m = np.eye(4, dtype=np.float32)
    m[:3, :3] = q
    m[:3, 3] = rng.uniform(-2.0, 2.0, 3)
    assert (m[:3, :] < 0).any()
    return m


def _camera(w, h, seed, k, pose, pad=(0, 0)):
    if w * h == 0:
        depth, bgr = np.zeros((h, w), np.uint16), np.zeros((h, w, 3), np.uint8)
    else:
        depth, bgr = _random_images(w, h, seed)
    fx, fy, cx, cy = INTRINSICS[k % len(INTRINSICS)]
    if pad != (0, 0):
        depth, bgr = _padded(depth, pad[0]), _padded(bgr, pad[1])
    return dict(depth=depth, bgr=bgr, fx=fx, fy=fy, cx=cx, cy=cy, pose=pose)


SD, QHD = (512, 424), (960, 540)


def _cases():
    rng = np.random.default_rng(2024)
    R = lambda: _rigid(rng)  # noqa: E731
    return {
        "1": [(SD, (0, 0), R())],
        "2": [(SD, (0, 0), None), (QHD, (6, 3), R())],
        "3": [(QHD, (0, 0), R()), ((961, 540), (2, 5), R()), ((7, 3), (6, 1), None)],
        "8": [(SD, (0, 0), R()), (QHD, (0, 0), None), ((961, 540), (4, 7), R()), ((7, 3), (6, 1), R()), ((0, 0), (0, 0), R()),
              (SD, (64, 13), None), ((1, 1), (0, 0), R()), (QHD, (2, 2), R())],
    }


@pytest.mark.parametrize("case", ["1", "2", "3", "8"])
def test_matches_restatement(case):
    cams = [_camera(w, h, 31 * k + w + h, k, pose, pad) for k, ((w, h), pad, pose) in enumerate(_cases()[case])]
    want = _bits(restate_fused(cams))
    got = pcl.PointCloud().fromDepthImages(cams)
    assert got.size() == len(want)
    assert np.array_equal(_bits(got.to_numpy()), want), case
    # K instead of fx, fy, cx, cy; 3x4 poses; pinned pointers with explicit steps, synchronous and on the copy stream
    pinned, ptr_cams = [], []
    for c in cams:
        K = np.array([[c["fx"], 0, c["cx"]], [0, c["fy"], c["cy"]], [0, 0, 1]])
        h, w = c["depth"].shape
        pose = None if c["pose"] is None else c["pose"][:3]
        if w * h == 0:
            ptr_cams.append(dict(depth=0, bgr=0, width=w, height=h, K=K, pose=pose))
            continue
        (bd, sd) = _pinned(c["depth"], c["depth"].strides[0] - c["depth"][0].nbytes)
        (bc, sc) = _pinned(c["bgr"], c["bgr"].strides[0] - c["bgr"][0].nbytes)
        pinned += [bd, bc]
        ptr_cams.append(dict(depth=bd.ptr, bgr=bc.ptr, width=w, height=h, depth_step=sd, bgr_step=sc, K=K, pose=pose))
    for asynchronous in (False, True):
        c = pcl.PointCloud().fromDepthImages(ptr_cams, asynchronous=asynchronous)
        assert np.array_equal(_bits(c.to_numpy()), want), (case, asynchronous)


@pytest.mark.parametrize("w,h,pad_d,pad_c", [(512, 424, 0, 0), (960, 540, 0, 0), (961, 540, 4, 7)])
def test_one_camera_without_matrix_equals_single_image_ingest(w, h, pad_d, pad_c):
    depth, bgr = _random_images(w, h, 3 * w + h)
    dv, cv = _padded(depth, pad_d), _padded(bgr, pad_c)
    for fx, fy, cx, cy in INTRINSICS:
        for asynchronous in (False, True):
            a = pcl.PointCloud().fromDepthImage(dv, cv, fx, fy, cx, cy, asynchronous=asynchronous)
            b = pcl.PointCloud().fromDepthImages([dict(depth=dv, bgr=cv, fx=fx, fy=fy, cx=cx, cy=cy)], asynchronous=asynchronous)
            assert b.size() == w * h
            assert np.array_equal(_bits(a.to_numpy()), _bits(b.to_numpy()))


def _two_views(n_frames, objs):
    """Frames of the default camera (qhd) and of synth.side_camera() (sd), as images; the common frame is camera 0's."""
    side = synth.side_camera()
    pose = synth.pose_matrix(side).astype(np.float32)
    frames = []
    for f in range(n_frames):
        d0, c0, K0 = synth.depth_images(synth.render(f, objs, sensor=synth.KINECT2_QHD)[0], synth.KINECT2_QHD)
        d1, c1, K1 = synth.depth_images(synth.render(f, objs, sensor=synth.KINECT2_SD, camera=side)[0], synth.KINECT2_SD)
        frames.append([dict(depth=d0, bgr=c0, K=K0, pose=None), dict(depth=d1, bgr=c1, K=K1, pose=pose)])
    return frames


def _k(c):
    K = c["K"]
    return dict(c, fx=K[0, 0], fy=K[1, 1], cx=K[0, 2], cy=K[1, 2])


def host_composition(cams):
    """The path a caller takes without the fused ingest: every camera through fromDepthImage, downloaded, moved by
    pcl_transform on the host, concatenated (16-byte records, uploaded as PACKED16)."""
    parts = []
    for c in map(_k, cams):
        p = pcl.PointCloud().fromDepthImage(c["depth"], c["bgr"], c["fx"], c["fy"], c["cx"], c["cy"]).to_numpy()
        parts.append(p if c["pose"] is None else pcl_transform(p, c["pose"][:3]))
    return np.concatenate(parts)


def _model(frames, objs):
    c0 = _k(frames[0][0])
    _, oid0 = synth.render(0, objs, sensor=synth.KINECT2_QHD)
    raw = restate(c0["depth"], c0["bgr"], c0["fx"], c0["fy"], c0["cx"], c0["cy"])
    return pcl.prepare_model(pcl.PointCloud(synth.model_points(raw, oid0, 0)), 0.01)


def test_tracking_equals_host_composition():
    objs = synth.default_objects(1)
    frames = _two_views(6, objs)
    model, centre = _model(frames, objs)
    ta, tb = _tracker(model, centre), _tracker(model, centre)
    vg = _voxel_grid()
    ca, cb, da, db = pcl.PointCloud(), pcl.PointCloud(), pcl.PointCloud(), pcl.PointCloud()
    for k, cams in enumerate(frames):
        host = host_composition(cams)
        ca.fromDepthImages(cams)
        cb.upload(host)
        assert np.array_equal(_bits(ca.to_numpy()), _bits(host)), k
        assert np.array_equal(_bits(host), _bits(restate_fused([_k(c) for c in cams]))), k
        vg.setInputCloud(ca)
        vg.filter(da)
        vg.setInputCloud(cb)
        vg.filter(db)
        assert da.size() > 1000
        assert np.array_equal(_bits(da.to_numpy()), _bits(db.to_numpy())), k
        for t, d in ((ta, da), (tb, db)):
            t.setInputCloud(d)
            t.compute()
        assert np.array_equal(ta.getParticles().view(np.uint32), tb.getParticles().view(np.uint32)), k
        assert np.array(ta.getResult()).tobytes() == np.array(tb.getResult()).tobytes(), k
    r = ta.getResult()
    assert np.isfinite([r["x"], r["y"], r["z"]]).all()


def test_voxel_grid_at_the_fused_size():
    # four qhd cameras (2.07 M points): K1's tables are sized from the cloud capacity
    rng = np.random.default_rng(5)
    objs = synth.default_objects(3)
    n = synth.table_frame()[2]
    views = [None, synth.side_camera(), synth.look_at([-1.3, -0.2, 0.9], [0.0, 0.25, 1.15], n), synth.look_at([0.3, -0.9, 0.2], [0.0, 0.3, 1.2], n)]
    cams = []
    for k, view in enumerate(views):
        d, c, K = synth.depth_images(synth.render(k, objs, sensor=synth.KINECT2_QHD, camera=view)[0], synth.KINECT2_QHD)
        pose = None if view is None else synth.pose_matrix(view).astype(np.float32)
        if k == 3:
            pose = _rigid(rng) @ pose  # a common frame that is not camera 0's
        cams.append(dict(depth=d, bgr=c, K=K, pose=pose))
    fused = pcl.PointCloud().fromDepthImages(cams)
    assert fused.size() == 4 * 960 * 540
    pts = fused.to_numpy()
    assert np.array_equal(_bits(pts), _bits(restate_fused([_k(c) for c in cams])))
    vg = _voxel_grid()
    vg.setInputCloud(fused)
    ds = vg.filter()
    want = oracle.voxel_grid_exact(pts, 0.01, 2, 0.0, 10.0)
    assert len(want) > 10000
    assert np.array_equal(ds.to_numpy().view(np.uint32), want.view(np.uint32))


def test_one_conversion_launch_per_frame():
    depth, bgr = _random_images(512, 424, 9)
    cam = dict(depth=depth, bgr=bgr, fx=365.0, fy=365.0, cx=256.0, cy=212.0)
    pose = _rigid(np.random.default_rng(1))
    grown = {}
    cloud = pcl.PointCloud()
    for asynchronous in (False, True):
        for n in (1, 2, 8):
            cams = [dict(cam, pose=pose if k % 2 else None) for k in range(n)]
            cloud.fromDepthImages(cams, asynchronous=asynchronous)  # staging and cloud storage in place
            cloud.ctx.synchronize()
            before = pcl.kernel_launch_count()
            cloud.fromDepthImages(cams, asynchronous=asynchronous)
            grown[(asynchronous, n)] = pcl.kernel_launch_count() - before
            assert cloud.size() == n * 512 * 424
    assert len(set(grown.values())) == 1, grown
    assert grown[(False, 1)] == 2  # the conversion and the header write


def _frame_loop(bufs, cams0, model, centre, pipelined):
    t = _tracker(model, centre)
    vg = _voxel_grid()
    clouds, ds = [pcl.PointCloud(), pcl.PointCloud()], pcl.PointCloud()
    poses = []

    def up(k, asynchronous):
        cams = [dict(c, depth=b[0].ptr, bgr=b[1].ptr, width=c["depth"].shape[1], height=c["depth"].shape[0]) for c, b in zip(cams0, bufs[k])]
        clouds[k % 2].fromDepthImages(cams, asynchronous=asynchronous)

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
    objs = synth.default_objects(1)
    frames = _two_views(6, objs)
    model, centre = _model(frames, objs)
    bufs = [[(pcl.PinnedBuffer.of(c["depth"]), pcl.PinnedBuffer.of(c["bgr"])) for c in cams] for cams in frames]
    serial = _frame_loop(bufs, frames[0], model, centre, pipelined=False)
    piped = _frame_loop(bufs, frames[0], model, centre, pipelined=True)
    assert serial == piped


def test_malformed_arguments_are_rejected():
    lib = _capi.load()
    cloud = pcl.PointCloud()
    w, h = 8, 4
    depth, bgr = _random_images(w, h, 5)
    m = np.ascontiguousarray(_rigid(np.random.default_rng(3))[:3])
    fp = C.POINTER(C.c_float)

    def cam(**kw):
        a = dict(depth=depth.ctypes.data, depth_step=2 * w, bgr=bgr.ctypes.data, bgr_step=3 * w, width=w, height=h, fx=365.0, fy=365.0,
                 cx=4.0, cy=2.0, m12=m.ctypes.data_as(fp))
        a.update(kw)
        return _capi.DepthCamera(**a)

    def arr(cams):
        return (_capi.DepthCamera * max(len(cams), 1))(*cams)

    inf, nan = float("inf"), float("nan")
    bad_m = [m.copy(), m.copy()]
    bad_m[0][1, 2] = nan
    bad_m[1][2, 3] = -inf
    big = dict(depth_step=2 * 65536, bgr_step=3 * 65536, width=65536, height=16384)  # 2^30 pixels each
    bad = [
        ([cam()], 0, None),                                                        # n < 1
        ([cam()] * 9, 9, None),                                                    # n > PFT_MAX_DEPTH_CAMERAS
        ([cam(), cam(m12=bad_m[0].ctypes.data_as(fp))], 2, "camera 1"),            # NaN matrix entry
        ([cam(m12=bad_m[1].ctypes.data_as(fp))], 1, "camera 0"),                   # infinite matrix entry
        ([cam(**big), cam(**big)], 2, "in total"),                                 # 2^31 pixels in total
        ([cam(), cam(), cam(depth=None)], 3, "camera 2"),                          # null depth
        ([cam(), cam(), cam(), cam(bgr=None)], 4, "camera 3"),                     # null colour
        ([cam(), cam(depth_step=2 * w + 1)], 2, "camera 1"),                       # odd depth step
        ([cam(), cam(bgr_step=3 * w - 1)], 2, "camera 1"),                         # colour step too small
        ([cam(), cam(), cam(), cam(), cam(), cam(fx=0.0)], 6, "camera 5"),         # fx zero
        ([cam(), cam(cy=inf)], 2, "camera 1"),                                     # cy not finite
        ([cam(), cam(width=65536, height=32768, depth_step=2 * 65536, bgr_step=3 * 65536)], 2, "camera 1"),  # 2^31 in one camera
    ]
    for fn in (lib.pft_cloud_upload_depth_images, lib.pft_cloud_upload_depth_images_async):
        assert fn(None, arr([cam()]), 1) == _capi.ERR_INVALID
        assert fn(cloud._h, None, 1) == _capi.ERR_INVALID
        for k, (cams, n, who) in enumerate(bad):
            assert fn(cloud._h, arr(cams), n) == _capi.ERR_INVALID, (fn, k)
            if who:
                assert who in lib.pft_last_error().decode(), (k, lib.pft_last_error())
        assert fn(cloud._h, arr([cam(), cam(m12=None), cam(width=0, height=0, depth=None, bgr=None)]), 3) == _capi.OK
        assert cloud.size() == 2 * w * h
        assert fn(cloud._h, arr([cam(width=0, depth=None, bgr=None)]), 1) == _capi.OK
        assert cloud.size() == 0
    with pytest.raises(pcl.PftError):
        pcl.PointCloud().fromDepthImages([])
    with pytest.raises(ValueError):
        pcl.PointCloud().fromDepthImages([dict(depth=depth, bgr=bgr, fx=365.0, fy=365.0, cx=4.0, cy=2.0, pose=np.eye(3))])


def test_shim_program_prints_the_same_cloud(tmp_path):
    exe = build_depth_cameras(tmp_path)
    rng = np.random.default_rng(17)
    spec = [((961, 540), (4, 7), _rigid(rng)), ((512, 424), (0, 0), None), ((7, 3), (6, 1), _rigid(rng))]
    args, cams = [], []
    for k, ((w, h), (pad_d, pad_c), pose) in enumerate(spec):
        depth, bgr = _random_images(w, h, 11 + k)
        fx, fy, cx, cy = INTRINSICS[k]
        (bd, sd), (bc, sc) = _pinned(depth, pad_d), _pinned(bgr, pad_c)
        (tmp_path / ("d%d.raw" % k)).write_bytes(bd.numpy().tobytes())
        (tmp_path / ("c%d.raw" % k)).write_bytes(bc.numpy().tobytes())
        mpath = "-"
        if pose is not None:
            mpath = str(tmp_path / ("m%d.raw" % k))
            (tmp_path / ("m%d.raw" % k)).write_bytes(np.ascontiguousarray(pose[:3], dtype=np.float32).tobytes())
        args += [str(tmp_path / ("d%d.raw" % k)), str(tmp_path / ("c%d.raw" % k)), str(w), str(h), str(sd), str(sc), repr(fx), repr(fy),
                 repr(cx), repr(cy), mpath]
        cams.append(dict(depth=depth, bgr=bgr, fx=fx, fy=fy, cx=cx, cy=cy, pose=pose))
    n = sum(w * h for (w, h), _, _ in spec)
    out = tmp_path / "out.raw"
    r = subprocess.run([exe, str(out)] + args, capture_output=True, text=True, check=True).stdout
    assert r.splitlines() == ["%d %d 1" % (n, n)] * 2
    rec = np.frombuffer(out.read_bytes(), dtype=synth.to_pcl32(np.zeros(0, POINT)).dtype)
    assert len(rec) == 2 * n
    want = pcl.PointCloud().fromDepthImages(cams).to_numpy()
    assert np.array_equal(_bits(want), _bits(restate_fused(cams)))
    for half in (rec[:n], rec[n:]):
        got = np.zeros(n, dtype=POINT)
        for k in ("x", "y", "z", "rgba"):
            got[k] = half[k]
        assert np.array_equal(_bits(got), _bits(want))
