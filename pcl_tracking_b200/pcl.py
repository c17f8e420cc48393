"""Host-side mirror of the PCL surface that ref: src/auto_tracking.cpp drives, over the C ABI.

Class and method names are PCL's (pcl::PassThrough, pcl::ApproximateVoxelGrid, pcl::VoxelGrid,
pcl::tracking::{KLDAdaptiveParticleFilterOMPTracker, ParticleFilterOMPTracker,
ApproxNearestPairPointCloudCoherence, NearestPairPointCloudCoherence, DistanceCoherence,
HSVColorCoherence}, pcl::search::Octree) so that code written against the reference reads the same:

    tracker = KLDAdaptiveParticleFilterOMPTracker(16)          # ref :209-210
    tracker.setMaximumParticleNum(500); tracker.setDelta(0.99) # ref :211-212
    ...
    coherence = ApproxNearestPairPointCloudCoherence()         # ref :235
    coherence.addPointCoherence(DistanceCoherence())           # ref :240-242
    tracker.setCloudCoherence(coherence)                       # ref :254
    tracker.setReferenceCloud(model); tracker.setInputCloud(scene); tracker.compute()

Everything computes on the GPU through libpft.so; this module holds no arithmetic.
"""
import ctypes as C

import numpy as np

from . import _capi as capi
from ._capi import PARTICLE, POINT, POINT_PCL32, PftError, check, ptr  # noqa: F401


# ------------------------------------------------------------------ context / clouds
class Context:
    """One CUDA device + stream (pft_context)."""

    _default = {}

    def __init__(self, device=0):
        self._h = C.c_void_p()
        check(capi.load().pft_context_create(int(device), C.byref(self._h)))
        self.device = int(device)

    @classmethod
    def default(cls, device=0):
        if device not in cls._default:
            cls._default[device] = cls(device)
        return cls._default[device]

    def synchronize(self):
        check(capi.load().pft_context_synchronize(self._h))

    @property
    def stream(self):
        return capi.load().pft_context_stream(self._h)

    def commInit(self, nranks, rank, unique_id):
        buf = (C.c_char * 128).from_buffer_copy(bytes(unique_id))
        check(capi.load().pft_context_comm_init(self._h, int(nranks), int(rank), buf))

    def commDestroy(self):
        check(capi.load().pft_context_comm_destroy(self._h))

    def close(self):
        if self._h:
            capi.load().pft_context_destroy(self._h)
            self._h = C.c_void_p()


class PinnedBuffer:
    """Page-locked host memory (pft_host_alloc) for frame buffers: what upload_raw / upload_raw_async copy from."""

    def __init__(self, nbytes):
        self.nbytes = int(nbytes)
        self._p = C.c_void_p()
        check(capi.load().pft_host_alloc(C.byref(self._p), self.nbytes))

    @classmethod
    def of(cls, array):
        a = np.ascontiguousarray(array)
        b = cls(a.nbytes)
        if a.nbytes:
            C.memmove(b._p, a.ctypes.data, a.nbytes)
        return b

    @property
    def ptr(self):
        return self._p.value

    def numpy(self, dtype=np.uint8):
        n = self.nbytes // np.dtype(dtype).itemsize
        return np.ctypeslib.as_array(C.cast(self._p, C.POINTER(C.c_uint8)), shape=(self.nbytes,)).view(dtype)[:n]

    def free(self):
        if self._p:
            capi.load().pft_host_free(self._p)
            self._p = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def _image_arg(img, dtype, channels, step, width, height, keep):
    """(pointer, width, height, step in bytes) of one image: an array (rows may be padded: the row stride is the step),
    appended to `keep`, or a raw host pointer (int) with width, height and the step (default: packed rows)."""
    pixel = np.dtype(dtype).itemsize * channels
    if isinstance(img, int):
        if width is None or height is None:
            raise ValueError("a pointer image needs width and height")
        return C.c_void_p(img), int(width), int(height), int(width) * pixel if step is None else int(step)
    a = np.asarray(img)
    shape = "(H, W)" if channels == 1 else "(H, W, %d)" % channels
    if a.dtype != dtype or a.ndim != (2 if channels == 1 else 3) or (channels > 1 and a.shape[2] != channels):
        raise TypeError("image must be a %s array of shape %s, got %s %r" % (np.dtype(dtype), shape, a.dtype, a.shape))
    # padded rows (a view into a wider buffer) go as they are, with the row stride as the step
    packed = a.strides[1] == pixel and (channels == 1 or a.strides[2] == a.itemsize)
    if not packed or a.shape[0] < 2 or a.strides[0] < a.shape[1] * pixel:
        a = np.ascontiguousarray(a)
    keep.append(a)
    return C.c_void_p(a.ctypes.data if a.size else None), a.shape[1], a.shape[0], a.strides[0]


# sensor_msgs/Image encodings the depth-image ingest takes: name -> (pft_depth_encoding, numpy dtype) of the depth image
# and name -> (pft_colour_encoding, channels of uint8) of the colour image; colour "none" is depth alone
DEPTH_ENCODINGS = {"16UC1": (capi.DEPTH_16UC1, np.uint16), "mono16": (capi.DEPTH_16UC1, np.uint16), "32FC1": (capi.DEPTH_32FC1, np.float32)}
COLOUR_ENCODINGS = {"bgr8": (capi.COLOUR_BGR8, 3), "rgb8": (capi.COLOUR_RGB8, 3), "bgra8": (capi.COLOUR_BGRA8, 4), "rgba8": (capi.COLOUR_RGBA8, 4),
                    "mono8": (capi.COLOUR_MONO8, 1), "none": (capi.COLOUR_NONE, 0)}


def _depth_camera(depth, bgr, width, height, depth_step, bgr_step, depth_encoding, colour_encoding, fx, fy, cx, cy, m12, keep):
    """pft_depth_camera_enc of a depth + colour image pair in the named encodings (colour "none": `bgr` is ignored)."""
    if depth_encoding not in DEPTH_ENCODINGS:
        raise ValueError("unknown depth encoding %r (one of %s)" % (depth_encoding, ", ".join(DEPTH_ENCODINGS)))
    if colour_encoding not in COLOUR_ENCODINGS:
        raise ValueError("unknown colour encoding %r (one of %s)" % (colour_encoding, ", ".join(COLOUR_ENCODINGS)))
    denc, dtype = DEPTH_ENCODINGS[depth_encoding]
    cenc, channels = COLOUR_ENCODINGS[colour_encoding]
    dp, w, h, dstep = _image_arg(depth, dtype, 1, depth_step, width, height, keep)
    bp, bstep = C.c_void_p(None), 0
    if channels:
        bp, w2, h2, bstep = _image_arg(bgr, np.uint8, channels, bgr_step, width, height, keep)
        if (w, h) != (w2, h2):
            raise ValueError("depth is %dx%d, colour %dx%d" % (w, h, w2, h2))
    cam = capi.DepthCamera(dp.value, dstep, bp.value, bstep, w, h, float(fx), float(fy), float(cx), float(cy), m12)
    return capi.DepthCameraEnc(cam, denc, cenc)


def _intrinsics(cam):
    """fx, fy, cx, cy of a camera mapping: from `K` (3x3 camera_info matrix) or its own keys."""
    if "K" in cam:
        K = np.asarray(cam["K"], dtype=np.float64)
        return K[0, 0], K[1, 1], K[0, 2], K[1, 2]
    return cam["fx"], cam["fy"], cam["cx"], cam["cy"]


def _pose_m12(cam, k, keep):
    """The float32 3x4 pointer of a camera mapping's optional `pose`, or None."""
    if cam.get("pose") is None:
        return None
    pose = np.asarray(cam["pose"], dtype=np.float32)
    if pose.shape not in ((4, 4), (3, 4)):
        raise ValueError("camera %d: pose must be 4x4 or 3x4, got %r" % (k, pose.shape))
    m = np.ascontiguousarray(pose[:3, :4])
    keep.append(m)
    return m.ctypes.data_as(C.POINTER(C.c_float))


def _registration(cam, reg, m12, keep, k):
    """pft_depth_camera_reg of camera mapping `cam` (its depth image in the depth camera's geometry) and its
    `registration` mapping `reg` (see PointCloud.fromDepthImages)."""
    depth_encoding, colour_encoding = cam.get("depth_encoding", "16UC1"), cam.get("colour_encoding", "bgr8")
    if depth_encoding not in DEPTH_ENCODINGS:
        raise ValueError("unknown depth encoding %r (one of %s)" % (depth_encoding, ", ".join(DEPTH_ENCODINGS)))
    if colour_encoding not in COLOUR_ENCODINGS:
        raise ValueError("unknown colour encoding %r (one of %s)" % (colour_encoding, ", ".join(COLOUR_ENCODINGS)))
    denc, dtype = DEPTH_ENCODINGS[depth_encoding]
    cenc, channels = COLOUR_ENCODINGS[colour_encoding]
    dw, dh = reg.get("depth_width"), reg.get("depth_height")
    dp, w_d, h_d, dstep = _image_arg(cam["depth"], dtype, 1, cam.get("depth_step"), dw, dh, keep)
    if (dw is not None and int(dw) != w_d) or (dh is not None and int(dh) != h_d):
        raise ValueError("camera %d: the depth image is %dx%d, the registration says %sx%s" % (k, w_d, h_d, dw, dh))
    bp, bstep = C.c_void_p(None), 0
    if channels:
        bp, w, h, bstep = _image_arg(cam.get("bgr"), np.uint8, channels, cam.get("bgr_step"), cam.get("width"), cam.get("height"), keep)
    elif cam.get("width") is None or cam.get("height") is None:
        raise ValueError("camera %d: without a colour image the colour camera's width and height are needed" % k)
    else:
        w, h = int(cam["width"]), int(cam["height"])
    fx, fy, cx, cy = _intrinsics(cam)
    if "depth_K" in reg:
        K = np.asarray(reg["depth_K"], dtype=np.float64)
        dfx, dfy, dcx, dcy = K[0, 0], K[1, 1], K[0, 2], K[1, 2]
    else:
        dfx, dfy, dcx, dcy = reg["depth_fx"], reg["depth_fy"], reg["depth_cx"], reg["depth_cy"]
    t = np.asarray(reg["depth_to_colour"], dtype=np.float64)
    if t.shape not in ((4, 4), (3, 4)):
        raise ValueError("camera %d: depth_to_colour must be 4x4 or 3x4, got %r" % (k, t.shape))
    t = np.ascontiguousarray(t[:3, :4])
    keep.append(t)
    fill = reg.get("fill_upsampling", False)
    if fill not in (0, 1):
        raise ValueError("camera %d: fill_upsampling must be a bool, got %r" % (k, fill))
    cam_enc = capi.DepthCameraEnc(capi.DepthCamera(dp.value, dstep, bp.value, bstep, w, h, float(fx), float(fy), float(cx), float(cy), m12), denc, cenc)
    return capi.DepthCameraReg(cam_enc, t.ctypes.data_as(C.POINTER(C.c_double)), w_d, h_d, float(dfx), float(dfy), float(dcx), float(dcy),
                               float(reg.get("depth_Tx", 0.0)), float(reg.get("depth_Ty", 0.0)), float(reg.get("colour_Tx", 0.0)),
                               float(reg.get("colour_Ty", 0.0)), int(fill))


class PointCloud:
    """pcl::PointCloud<pcl::PointXYZRGBA> resident in HBM as float4 {x, y, z, rgba}."""

    def __init__(self, points=None, ctx=None):
        self.ctx = ctx or Context.default()
        self._h = C.c_void_p()
        check(capi.load().pft_cloud_create(self.ctx._h, C.byref(self._h)))
        if points is not None:
            self.upload(points)

    def upload(self, points):
        """points: numpy array of POINT (16 B packed) or POINT_PCL32 (the 32 B PCL struct)."""
        a = np.ascontiguousarray(points)
        if a.dtype == POINT:
            layout = capi.LAYOUT_PACKED16
        elif a.dtype == POINT_PCL32:
            layout = capi.LAYOUT_PCL32
        else:
            raise TypeError("points must have dtype POINT or POINT_PCL32, got %r" % (a.dtype,))
        check(capi.load().pft_cloud_upload(self._h, ptr(a), a.shape[0], layout))
        return self

    def upload_raw(self, host_ptr, n, layout=capi.LAYOUT_PACKED16):
        """Upload from a raw host pointer (e.g. pinned memory from host_alloc)."""
        check(capi.load().pft_cloud_upload(self._h, C.c_void_p(host_ptr), n, layout))
        return self

    def upload_raw_async(self, host_ptr, n, layout=capi.LAYOUT_PACKED16):
        """Like upload_raw, on the context's copy stream: overlaps the work enqueued after this call (the previous
        frame's compute); consumers of this cloud wait for the copy on the device.  `host_ptr` must be pinned."""
        check(capi.load().pft_cloud_upload_async(self._h, C.c_void_p(host_ptr), n, layout))
        return self

    def waitUpload(self):
        check(capi.load().pft_cloud_wait_upload(self._h))
        return self

    def fromPointCloud2(self, data, width, height, point_step, row_step=None, off_x=0, off_y=4, off_z=8, off_rgb=16, is_bigendian=False,
                        asynchronous=False):
        """sensor_msgs/PointCloud2 payload -> device cloud (pcl::fromPCLPointCloud2, ref: src/auto_tracking.cpp:619-622).
        `data`: bytes / uint8 array of height x row_step bytes, or a raw host pointer (int)."""
        row_step = int(width) * int(point_step) if row_step is None else int(row_step)
        if isinstance(data, int):
            p = C.c_void_p(data)
        else:
            a = np.ascontiguousarray(np.frombuffer(data, dtype=np.uint8) if isinstance(data, (bytes, bytearray, memoryview)) else data)
            if a.nbytes < row_step * int(height):
                raise ValueError("PointCloud2 data holds %d bytes, need %d" % (a.nbytes, row_step * int(height)))
            self._keep = a
            p = ptr(a)
        fn = capi.load().pft_cloud_upload_pointcloud2_async if asynchronous else capi.load().pft_cloud_upload_pointcloud2
        check(fn(self._h, p, int(width), int(height), int(point_step), row_step, int(off_x), int(off_y),
                 int(off_z), int(off_rgb), 1 if is_bigendian else 0))
        return self

    def fromDepthImage(self, depth, bgr, fx, fy, cx, cy, asynchronous=False, width=None, height=None, depth_step=None, bgr_step=None,
                       depth_encoding="16UC1", colour_encoding="bgr8"):
        """Registered depth + colour images -> organised device cloud (pft_cloud_upload_depth_images_enc, one camera):
        what the depth_image_proc/point_cloud_xyzrgb nodelet computes for the points topic of ref:
        src/auto_tracking.cpp:775, or point_cloud_xyz with colour_encoding "none" (rgba = 0, `bgr` is ignored).
        `depth`: (H, W) uint16 millimetres ("16UC1" or "mono16") or float32 metres ("32FC1"); `bgr`: the colour image,
        (H, W, 3) uint8 for "bgr8" or "rgb8", (H, W, 4) for "bgra8" or "rgba8", (H, W) for "mono8".  The encodings are
        spelled as sensor_msgs/Image::encoding.  Each image is an array (rows may be padded: the row stride is the step)
        or a raw host pointer (int; pinned for `asynchronous`) with width, height and the steps in bytes (default:
        packed rows).  fx, fy, cx, cy: camera_info.K[0], K[4], K[2], K[5]."""
        keep = []
        arr = (capi.DepthCameraEnc * 1)(_depth_camera(depth, bgr, width, height, depth_step, bgr_step, depth_encoding, colour_encoding,
                                                      fx, fy, cx, cy, None, keep))
        self._keep = keep
        fn = capi.load().pft_cloud_upload_depth_images_enc_async if asynchronous else capi.load().pft_cloud_upload_depth_images_enc
        check(fn(self._h, arr, 1))
        return self

    def fromDepthImages(self, cameras, asynchronous=False):
        """Several calibrated cameras fused into one unorganised device cloud (pft_cloud_upload_depth_images_enc): for
        each camera k the cloud fromDepthImage makes, moved by pcl::transformPointCloud(cloud_k, T_k) into the common
        frame, then scene += cloud_k, all converted in one kernel launch.  `cameras`: up to 8 mappings, each with
        `depth` and `bgr` as for fromDepthImage (and `width`, `height`, `depth_step`, `bgr_step` for pointer images),
        optionally `depth_encoding` and `colour_encoding` (defaults "16UC1" and "bgr8"; with "none", `bgr` may be
        absent), either `K` (3x3 camera_info matrix) or `fx`, `fy`, `cx`, `cy`, and an optional `pose`: the 4x4 or 3x4
        matrix from the camera's optical frame to the common frame, cast to float32 (absent or None: the camera's own
        frame).  Cameras may mix encodings.

        A camera whose depth image is not registered to its colour camera carries a `registration` mapping: its `depth`
        image is then in the depth camera's geometry and is registered into the colour camera on the device, as the
        depth_image_proc/register nodelet does, before the conversion (pft_cloud_upload_depth_images_reg).  The mapping
        holds the depth camera's `depth_K` (3x3) or `depth_fx`, `depth_fy`, `depth_cx`, `depth_cy`, optionally
        `depth_Tx`, `depth_Ty`, `colour_Tx`, `colour_Ty` (P[3], P[7] of each camera_info; default 0),
        `depth_to_colour`, the 4x4 or 3x4 matrix from the depth optical frame to the colour optical frame in float64,
        `fill_upsampling` (default False), and `depth_width`, `depth_height` (needed for a pointer depth image; checked
        against a depth array).  `K` / `fx` .. `cy`, the colour image, `width`, `height` (needed without a colour image)
        and `pose` are the colour camera's, and the camera's points are organised in its geometry.  Cameras with and
        without a registration may be mixed."""
        keep = []
        cams = list(cameras)
        if any(cam.get("registration") is not None for cam in cams):
            return self._from_registered(cams, keep, asynchronous)
        arr = (capi.DepthCameraEnc * len(cams))()
        for k, cam in enumerate(cams):
            fx, fy, cx, cy = _intrinsics(cam)
            m12 = _pose_m12(cam, k, keep)
            arr[k] = _depth_camera(cam["depth"], cam.get("bgr"), cam.get("width"), cam.get("height"), cam.get("depth_step"), cam.get("bgr_step"),
                                   cam.get("depth_encoding", "16UC1"), cam.get("colour_encoding", "bgr8"), fx, fy, cx, cy, m12, keep)
        self._keep = keep
        fn = capi.load().pft_cloud_upload_depth_images_enc_async if asynchronous else capi.load().pft_cloud_upload_depth_images_enc
        check(fn(self._h, arr, len(cams)))
        return self

    def _from_registered(self, cams, keep, asynchronous):
        arr = (capi.DepthCameraReg * len(cams))()
        for k, cam in enumerate(cams):
            m12 = _pose_m12(cam, k, keep)
            if cam.get("registration") is not None:
                arr[k] = _registration(cam, cam["registration"], m12, keep, k)
                continue
            fx, fy, cx, cy = _intrinsics(cam)
            arr[k].cam = _depth_camera(cam["depth"], cam.get("bgr"), cam.get("width"), cam.get("height"), cam.get("depth_step"), cam.get("bgr_step"),
                                       cam.get("depth_encoding", "16UC1"), cam.get("colour_encoding", "bgr8"), fx, fy, cx, cy, m12, keep)
        self._keep = keep
        fn = capi.load().pft_cloud_upload_depth_images_reg_async if asynchronous else capi.load().pft_cloud_upload_depth_images_reg
        check(fn(self._h, arr, len(cams)))
        return self

    def broadcast(self, capacity, root=0):
        """NVLink broadcast of this cloud from `root` over the context communicator."""
        check(capi.load().pft_cloud_broadcast(self._h, int(capacity), int(root)))
        return self

    # scene distribution by peer stores: one rank owns the sensor, its kernel stores the cloud into every rank's copy
    def peerExport(self, capacity):
        """Fixes this cloud's storage at `capacity` points (the same on every rank) and returns its CUDA IPC handles (bytes)."""
        buf = C.create_string_buffer(capi.CLOUD_PEER_HANDLE_BYTES)
        check(capi.load().pft_cloud_peer_export(self._h, int(capacity), buf))
        return bytes(buf.raw)

    def peerAttach(self, handles, rank):
        """`handles`: the peerExport() results of all ranks in rank order (e.g. dist.all_gather_object)."""
        blob = b"".join(bytes(h) for h in handles)
        buf = C.create_string_buffer(blob, len(blob))
        check(capi.load().pft_cloud_peer_attach(self._h, buf, len(handles), int(rank)))
        return self

    def peerBroadcast(self, root=0):
        """Stream ordered; every rank calls it once per scene: the root pushes its contents over NVLink, the others wait for them."""
        check(capi.load().pft_cloud_peer_broadcast(self._h, int(root)))
        return self

    def peerDetach(self):
        check(capi.load().pft_cloud_peer_detach(self._h))

    def size(self):
        n = C.c_size_t()
        check(capi.load().pft_cloud_size(self._h, C.byref(n)))
        return n.value

    __len__ = size

    def to_numpy(self, pcl32=False):
        n = self.size()
        out = np.zeros(n, dtype=POINT_PCL32 if pcl32 else POINT)
        got = C.c_size_t()
        check(capi.load().pft_cloud_download(self._h, ptr(out), n, capi.LAYOUT_PCL32 if pcl32 else capi.LAYOUT_PACKED16, C.byref(got)))
        return out

    def __del__(self):
        try:
            if self._h:
                capi.load().pft_cloud_destroy(self._h)
                self._h = C.c_void_p()
        except Exception:
            pass


_FIELDS = {"x": 0, "y": 1, "z": 2}


class PassThrough:
    """pcl::PassThrough<PointXYZRGBA> (ref: src/auto_tracking.cpp:539-545)."""

    def __init__(self, ctx=None):
        self.ctx = ctx or Context.default()
        self._field, self._lo, self._hi, self._in = 2, -3.4028234663852886e38, 3.4028234663852886e38, None

    def setFilterFieldName(self, name):
        if name not in _FIELDS:
            raise ValueError("filter field must be 'x', 'y' or 'z'")
        self._field = _FIELDS[name]

    def setFilterLimits(self, lo, hi):
        self._lo, self._hi = float(lo), float(hi)

    def setKeepOrganized(self, keep):
        if keep:
            raise NotImplementedError("setKeepOrganized(true) is not on the reference's path (ref :542 passes false)")

    def setInputCloud(self, cloud):
        self._in = cloud

    def filter(self, out=None):
        out = PointCloud(ctx=self.ctx) if out is None else out
        check(capi.load().pft_passthrough(self.ctx._h, self._in._h, out._h, self._field, self._lo, self._hi))
        return out


class EuclideanClusterExtraction:
    """pcl::EuclideanClusterExtraction<PointXYZRGBA> as the model builder configures it (ref: src/create_model.cpp:169-179).
    extract() returns the clusters as index arrays (sorted indices, largest cluster first), cluster_cloud(k) the k-th
    cluster as a device cloud (what create_model returns to auto_tracking, ref: src/create_model.cpp:209-230)."""

    def __init__(self, ctx=None):
        self.ctx = ctx or Context.default()
        self._tol, self._min, self._max, self._in = 0.0, 1, 2 ** 31 - 1, None
        self.labels, self.sizes = None, None

    def setClusterTolerance(self, tol):
        self._tol = float(tol)

    def setMinClusterSize(self, n):
        self._min = int(n)

    def setMaxClusterSize(self, n):
        self._max = int(n)

    def setSearchMethod(self, tree):
        pass  # the KdTree of ref :169-173 is replaced by the uniform grid built inside extract()

    def setInputCloud(self, cloud):
        self._in = cloud

    def extract(self):
        n = self._in.size()
        labels = np.full(n, -1, dtype=np.int32)
        sizes = np.zeros(4096, dtype=np.int32)
        k = C.c_size_t()
        check(capi.load().pft_euclidean_clusters(self.ctx._h, self._in._h, self._tol, self._min, self._max, ptr(labels) if n else None, n,
                                                 ptr(sizes), len(sizes), C.byref(k)))
        self.labels, self.sizes = labels, sizes[:k.value].copy()
        return [np.flatnonzero(labels == c).astype(np.int32) for c in range(k.value)]

    def cluster_cloud(self, k, out=None):
        out = PointCloud(ctx=self.ctx) if out is None else out
        check(capi.load().pft_cloud_select_cluster(self.ctx._h, self._in._h, int(k), out._h))
        return out


class SACSegmentation:
    """pcl::SACSegmentation<PointXYZRGBA> configured as the model builder's plane variant does (SACMODEL_PLANE, SAC_RANSAC;
    ref: src/create_model_planar_segmentation.cpp:157-163) fused with the two pcl::ExtractIndices passes that follow it
    (ref :166-174): segment() returns (coefficients[4], inlier count) and leaves the plane / everything-else clouds in
    .plane and .rest.  setSamples() injects the RANSAC draws (rows of three point indices), otherwise they are generated
    on the device from setSeed()."""

    def __init__(self, ctx=None):
        self.ctx = ctx or Context.default()
        self._thr, self._max_it, self._prob, self._opt, self._in = 0.0, 50, 0.99, True, None
        self._samples, self._seed = None, 0x5EED
        self.plane, self.rest, self.iterations = None, None, 0

    def setModelType(self, model="SACMODEL_PLANE"):
        if model not in ("SACMODEL_PLANE", 0):
            raise NotImplementedError("only SACMODEL_PLANE is on the reference's path")

    def setMethodType(self, method="SAC_RANSAC"):
        if method not in ("SAC_RANSAC", 0):
            raise NotImplementedError("only SAC_RANSAC is on the reference's path")

    def setMaxIterations(self, n):
        self._max_it = int(n)

    def setDistanceThreshold(self, t):
        self._thr = float(t)

    def setProbability(self, p):
        self._prob = float(p)

    def setOptimizeCoefficients(self, on):
        self._opt = bool(on)

    def setSamples(self, samples3):
        self._samples = None if samples3 is None else np.ascontiguousarray(samples3, dtype=np.int32).reshape(-1, 3)

    def setSeed(self, seed):
        self._seed = int(seed)

    def setInputCloud(self, cloud):
        self._in = cloud

    def segment(self):
        coeff = np.zeros(4, dtype=np.float32)
        it, n_in = C.c_int32(), C.c_size_t()
        self.plane, self.rest = PointCloud(ctx=self.ctx), PointCloud(ctx=self.ctx)
        s = self._samples
        check(capi.load().pft_segment_plane(self.ctx._h, self._in._h, self._thr, self._max_it, self._prob, ptr(s) if s is not None else None,
                                            len(s) if s is not None else 0, self._seed, 1 if self._opt else 0, ptr(coeff), C.byref(it),
                                            self.plane._h, self.rest._h, C.byref(n_in)))
        self.iterations = it.value
        return coeff, n_in.value


class VoxelGrid:
    """pcl::VoxelGrid / pcl::ApproximateVoxelGrid (ref: src/auto_tracking.cpp:553-557, :568-571): one
    centroid per occupied voxel of the lattice floor(coord / leaf).  setPassThrough() folds the
    preceding PassThrough (ref :637) into the same pass."""

    def __init__(self, ctx=None):
        self.ctx = ctx or Context.default()
        self._leaf, self._in = 0.01, None
        self._field, self._lo, self._hi = -1, 0.0, 0.0
        self._pcl_approx = False

    def setPclApproximateMode(self, on=True):
        """Parity mode: reproduce pcl::ApproximateVoxelGrid exactly (512-entry cache, partial centroids on eviction,
        input-order dependent; sequential on one GPU thread) instead of one exact centroid per voxel."""
        self._pcl_approx = bool(on)

    def setLeafSize(self, lx, ly=None, lz=None):
        ly = lx if ly is None else ly
        lz = lx if lz is None else lz
        if not (np.float32(lx) == np.float32(ly) == np.float32(lz)):
            raise NotImplementedError("anisotropic leaf sizes are not on the reference's path (ref :555, :569 pass one size)")
        self._leaf = float(lx)

    def setPassThrough(self, field, lo, hi):
        self._field = -1 if field is None else _FIELDS[field]
        self._lo, self._hi = float(lo), float(hi)

    def setInputCloud(self, cloud):
        self._in = cloud

    def filter(self, out=None):
        out = PointCloud(ctx=self.ctx) if out is None else out
        fn = capi.load().pft_approx_voxel_grid_pcl if self._pcl_approx else capi.load().pft_passthrough_voxel_grid
        check(fn(self.ctx._h, self._in._h, out._h, self._leaf, self._field, self._lo, self._hi))
        return out


ApproximateVoxelGrid = VoxelGrid


def prepare_model(raw_cloud, leaf=0.01, ctx=None):
    """removeZeroPoints + compute3DCentroid + translate by -centroid + VoxelGrid(leaf)
    (ref: src/auto_tracking.cpp:656-674).  Returns (model_cloud, centroid[3])."""
    ctx = ctx or raw_cloud.ctx
    out = PointCloud(ctx=ctx)
    c = np.zeros(3, dtype=np.float32)
    check(capi.load().pft_prepare_model(ctx._h, raw_cloud._h, out._h, float(leaf), ptr(c)))
    return out, c


def transformPointCloud(cloud, m, out=None):
    """pcl::transformPointCloud(cloud, out, m) (PCL 1.8.0): every point moved by the affine `m` (4x4 or 3x4, cast to
    float32 entry by entry, as pcl_ros does with a tf matrix), in order, colours kept; a point with a non-finite
    coordinate is copied as it is.  `out` may be `cloud` itself (in place).  Returns the output cloud."""
    a = np.asarray(m)
    if a.shape not in ((4, 4), (3, 4)):
        raise ValueError("m must be 4x4 or 3x4, got %r" % (a.shape,))
    m12 = np.ascontiguousarray(a[:3, :4], dtype=np.float32)
    out = PointCloud(ctx=cloud.ctx) if out is None else out
    check(capi.load().pft_transform_cloud(cloud.ctx._h, cloud._h, out._h, ptr(m12)))
    return out


def removeZeroPoints(cloud, out=None):
    """removeZeroPoints of the model builder (ref: src/create_model.cpp:59-77): drops the points with a non-finite
    coordinate and those with |x|, |y| and |z| all below 0.01, order preserving.  Returns the output cloud."""
    out = PointCloud(ctx=cloud.ctx) if out is None else out
    check(capi.load().pft_remove_zero_points(cloud.ctx._h, cloud._h, out._h))
    return out


# ------------------------------------------------------------------ coherence configuration objects
class DistanceCoherence:
    """pcl::tracking::DistanceCoherence (ref :240-242)."""

    def __init__(self):
        self.weight = 1.0

    def setWeight(self, w):
        self.weight = float(w)


class HSVColorCoherence:
    """pcl::tracking::HSVColorCoherence (ref :244-247)."""

    def __init__(self):
        self.weight, self.h_weight, self.s_weight, self.v_weight = 1.0, 1.0, 1.0, 0.0

    def setWeight(self, w):
        self.weight = float(w)

    def setHWeight(self, w):
        self.h_weight = float(w)

    def setSWeight(self, w):
        self.s_weight = float(w)

    def setVWeight(self, w):
        self.v_weight = float(w)


class Octree:
    """pcl::search::Octree(resolution) (ref :250): here the cell size of the uniform-grid index."""

    def __init__(self, resolution):
        self.resolution = float(resolution)


class NearestPairPointCloudCoherence:
    """pcl::tracking::NearestPairPointCloudCoherence (ref :237-238)."""

    def __init__(self):
        self.point_coherences = []
        self.search = None
        self.maximum_distance = 1.79769313486231570815e308

    def addPointCoherence(self, c):
        self.point_coherences.append(c)

    def setSearchMethod(self, search):
        self.search = search

    def setMaximumDistance(self, d):
        self.maximum_distance = float(d)


class ApproxNearestPairPointCloudCoherence(NearestPairPointCloudCoherence):
    """pcl::tracking::ApproxNearestPairPointCloudCoherence (ref :235-236).  By default the GPU index answers the
    exact nearest neighbour for both coherence classes (DESIGN.md, "Approx vs exact");
    setPclApproximateSearch(True) selects the parity mode that reproduces upstream's greedy octree descent
    (approxNearestSearch), misses included -- far slower, for result comparisons against a PCL run only."""

    def __init__(self):
        super().__init__()
        self.pcl_approximate_search = False

    def setPclApproximateSearch(self, on=True):
        self.pcl_approximate_search = bool(on)


# ------------------------------------------------------------------ trackers
def _particle(rec):
    out = np.zeros(1, dtype=PARTICLE)
    out[0] = rec
    return out


class ParticleFilterOMPTracker:
    """pcl::tracking::ParticleFilterOMPTracker<PointXYZRGBA, ParticleXYZRPY> (ref :201-206)."""

    _KLD = 0

    def __init__(self, nr_threads=0, ctx=None, devices=None):
        """devices: single-process multi-device mode -- this one tracker object drives these GPUs (devices[0] = the device
        of `ctx`), see setDevices."""
        self.ctx = ctx or Context.default()
        self._h = C.c_void_p()
        check(capi.load().pft_tracker_create(self.ctx._h, self._KLD, C.byref(self._h)))
        self._input = None
        if devices is not None and len(devices) > 1:
            self.setDevices(devices)
        self._si(capi.THREADS, nr_threads)

    # -- plumbing
    def _si(self, k, v):
        check(capi.load().pft_tracker_set_i(self._h, k, int(v)))

    def _sd(self, k, v):
        check(capi.load().pft_tracker_set_d(self._h, k, float(v)))

    def _sv(self, k, v):
        a = np.ascontiguousarray(v, dtype=np.float64)
        if a.shape != (6,):
            raise ValueError("expected 6 values")
        check(capi.load().pft_tracker_set_vec6(self._h, k, ptr(a)))

    # -- the PCL setters the reference calls
    def setNumberOfThreads(self, n):
        self._si(capi.THREADS, n)

    def setParticleNum(self, n):
        self._si(capi.PARTICLE_NUM, n)

    def setIterationNum(self, n):
        self._si(capi.ITERATION_NUM, n)

    def setTrans(self, affine):
        m = np.ascontiguousarray(np.asarray(affine, dtype=np.float32).reshape(-1)[:12])
        check(capi.load().pft_tracker_set_trans(self._h, ptr(m)))

    def setStepNoiseCovariance(self, v):
        self._sv(capi.STEP_NOISE_COV, v)

    def setInitialNoiseCovariance(self, v):
        self._sv(capi.INIT_NOISE_COV, v)

    def setInitialNoiseMean(self, v):
        self._sv(capi.INIT_NOISE_MEAN, v)

    def setResampleLikelihoodThr(self, v):
        self._sd(capi.RESAMPLE_LIKELIHOOD_THR, v)

    def setUseNormal(self, use):
        self._si(capi.USE_NORMAL, 1 if use else 0)

    def setMinIndices(self, n):
        self._si(capi.MIN_INDICES, n)

    # change detector of pcl::tracking::ParticleFilterTracker (off by default and in the reference, SURVEY 8 f-4)
    def setUseChangeDetector(self, use):
        self._si(capi.USE_CHANGE_DETECTOR, 1 if use else 0)

    def setIntervalOfChangeDetection(self, n):
        self._si(capi.CHANGE_DETECTOR_INTERVAL, int(n))

    def setMinPointsOfChangeDetection(self, n):
        self._si(capi.CHANGE_DETECTOR_MIN_POINTS, int(n))

    def setResolutionOfChangeDetection(self, r):
        self._sd(capi.CHANGE_DETECTOR_RESOLUTION, float(r))

    def changeDetectorInfo(self):
        out = np.zeros(4, dtype=np.int32)
        check(capi.load().pft_tracker_get_change_detector_info(self._h, ptr(out)))
        return {"counter": int(out[0]), "tests": int(out[1]), "last_found": int(out[2]), "changed": bool(out[3])}

    def setAlpha(self, a):
        self._sd(capi.ALPHA, a)

    def setMotionRatio(self, r):
        self._sd(capi.MOTION_RATIO, r)

    def setCloudCoherence(self, coherence):
        use_d = use_h = 0
        for pc in coherence.point_coherences:
            if isinstance(pc, DistanceCoherence):
                use_d = 1
                self._sd(capi.DIST_WEIGHT, pc.weight)
            elif isinstance(pc, HSVColorCoherence):
                use_h = 1
                self._sd(capi.HSV_WEIGHT, pc.weight)
                self._sd(capi.H_WEIGHT, pc.h_weight)
                self._sd(capi.S_WEIGHT, pc.s_weight)
                self._sd(capi.V_WEIGHT, pc.v_weight)
            else:
                raise NotImplementedError("point coherence %r is not on the reference's path" % (pc,))
        self._si(capi.USE_DISTANCE, use_d)
        self._si(capi.USE_HSV, use_h)
        self._si(capi.NN_MODE, capi.NN_PCL_APPROX if getattr(coherence, "pcl_approximate_search", False) else capi.NN_EXACT)
        self._sd(capi.MAX_DIST, coherence.maximum_distance)
        if coherence.search is not None:
            self._sd(capi.SEARCH_RESOLUTION, coherence.search.resolution)
        self._coherence = coherence

    def setReferenceCloud(self, cloud):
        if isinstance(cloud, PointCloud):
            check(capi.load().pft_tracker_set_reference_cloud(self._h, cloud._h))
        else:
            a = np.ascontiguousarray(cloud)
            layout = capi.LAYOUT_PACKED16 if a.dtype == POINT else capi.LAYOUT_PCL32
            check(capi.load().pft_tracker_set_reference_points(self._h, ptr(a), a.shape[0], layout))

    def setInputCloud(self, cloud):
        """The cloud may belong to another context than the tracker's, also on another GPU: the tracker's context then
        reads a replica of it, refreshed once per change (one object per GPU; not for sharded trackers)."""
        self._input = cloud  # keep the handle alive: the tracker borrows it
        check(capi.load().pft_tracker_set_input_cloud(self._h, cloud._h if cloud is not None else None))

    def compute(self):
        check(capi.load().pft_tracker_compute(self._h))

    def getResult(self):
        out = np.zeros(1, dtype=PARTICLE)
        check(capi.load().pft_tracker_get_result(self._h, ptr(out)))
        return out[0]

    def getResultBox(self, z_offset=-0.005):
        """Centroid + PCA oriented bounding box of the model at the result pose (viz_cb, ref: src/auto_tracking.cpp:432-466)."""
        out = np.zeros(1, dtype=capi.RESULT_BOX)
        check(capi.load().pft_tracker_get_result_box(self._h, float(z_offset), ptr(out)))
        return out[0]

    def getResultCloud(self, z_offset=-0.005, out=None):
        """The reference cloud moved to the result pose, translation z + z_offset (viz_cb, ref: src/auto_tracking.cpp:
        309-316): the tracked object's points, as a device cloud of the tracker's context."""
        out = PointCloud(ctx=self.ctx) if out is None else out
        check(capi.load().pft_tracker_get_result_cloud(self._h, float(z_offset), out._h))
        return out

    def getParticles(self):
        n = C.c_size_t()
        rc = capi.load().pft_tracker_get_particles(self._h, None, 0, C.byref(n))
        if rc not in (capi.OK, capi.ERR_CAPACITY):
            check(rc)
        out = np.zeros(n.value, dtype=PARTICLE)
        if n.value:
            check(capi.load().pft_tracker_get_particles(self._h, ptr(out), n.value, C.byref(n)))
        return out[: n.value]

    def toEigenMatrix(self, particle):
        """ParticleXYZRPY::toEigenMatrix (ref :310): 4x4 affine."""
        p = _particle(particle)
        m = np.zeros(12, dtype=np.float32)
        check(capi.load().pft_particle_to_matrix(self.ctx._h, ptr(p), ptr(m)))
        out = np.eye(4, dtype=np.float32)
        out[:3, :] = m.reshape(3, 4)
        return out

    def resetTracking(self):
        check(capi.load().pft_tracker_reset(self._h))

    def getFitRatio(self):
        v = C.c_double()
        check(capi.load().pft_tracker_get_fit_ratio(self._h, C.byref(v)))
        return v.value

    # -- reproducibility / parity hooks (no PCL equivalent: upstream seeds its RNGs with time(0))
    def setParticles(self, parts):
        a = np.ascontiguousarray(parts, dtype=PARTICLE)
        check(capi.load().pft_tracker_set_particles(self._h, ptr(a), a.shape[0]))

    def setResult(self, rep=None, motion=None):
        r = _particle(rep) if rep is not None else None
        m = _particle(motion) if motion is not None else None
        check(capi.load().pft_tracker_set_result(self._h, ptr(r) if r is not None else None, ptr(m) if m is not None else None))

    def getMotion(self):
        out = np.zeros(1, dtype=PARTICLE)
        check(capi.load().pft_tracker_get_motion(self._h, ptr(out)))
        return out[0]

    def injectDraws(self, usel, normals6, umotion):
        if usel is None:
            check(capi.load().pft_tracker_inject_draws(self._h, None, None, None, 0, 0))
            return
        usel = np.ascontiguousarray(usel, dtype=np.float32)
        slots, stride = usel.shape
        normals6 = np.ascontiguousarray(normals6, dtype=np.float32).reshape(slots, stride, 6)
        umotion = np.ascontiguousarray(umotion, dtype=np.float32).reshape(slots, stride)
        check(capi.load().pft_tracker_inject_draws(self._h, ptr(usel), ptr(normals6), ptr(umotion), slots, stride))

    def seed(self, s):
        check(capi.load().pft_tracker_seed(self._h, int(s)))

    def setSampler(self, s):
        self._si(capi.SAMPLER, s)

    def setQuaternionSampling(self, on):
        self._si(capi.QUAT_SAMPLE, 1 if on else 0)

    def setCandidateLists(self, mode):
        """0 never, 1 automatic, 2 always (internal to the search; results do not depend on it)."""
        self._si(capi.CANDIDATE_LISTS, mode)

    def setDebugNN(self, k):
        self._si(capi.DEBUG_NN, k)

    def setChanged(self, c):
        check(capi.load().pft_tracker_set_changed(self._h, 1 if c else 0))

    def initParticles(self):
        check(capi.load().pft_tracker_init_particles(self._h))

    def resample(self, slot=0):
        check(capi.load().pft_tracker_resample(self._h, int(slot)))

    def weight(self):
        check(capi.load().pft_tracker_weight(self._h))

    def weightPhase(self, phase):
        check(capi.load().pft_tracker_weight_phase(self._h, int(phase)))

    def update(self):
        check(capi.load().pft_tracker_update(self._h))

    def aabb(self):
        a = np.zeros(6, dtype=np.float32)
        check(capi.load().pft_tracker_get_aabb(self._h, ptr(a)))
        return a

    def cropBox(self):
        a = np.zeros(6, dtype=np.float32)
        check(capi.load().pft_tracker_get_crop_box(self._h, ptr(a)))
        return a

    def setCropBox(self, a):
        a = np.ascontiguousarray(a, dtype=np.float32)
        check(capi.load().pft_tracker_set_crop_box(self._h, ptr(a)))

    def rawSlice(self, rank):
        n = C.c_size_t()
        capi.load().pft_tracker_get_raw_slice(self._h, int(rank), None, 0, C.byref(n))
        out = np.zeros(n.value, dtype=np.float32)
        check(capi.load().pft_tracker_get_raw_slice(self._h, int(rank), ptr(out), n.value, C.byref(n)))
        return out

    def setRawSlice(self, rank, values):
        a = np.ascontiguousarray(values, dtype=np.float32)
        check(capi.load().pft_tracker_set_raw_slice(self._h, int(rank), ptr(a), a.shape[0]))

    def setShard(self, nranks, rank):
        check(capi.load().pft_tracker_set_shard(self._h, int(nranks), int(rank)))

    def croppedCount(self):
        n = C.c_size_t()
        check(capi.load().pft_tracker_get_cropped_count(self._h, C.byref(n)))
        return n.value

    def indexInfo(self):
        a = np.zeros(8, dtype=np.int32)
        check(capi.load().pft_tracker_get_index_info(self._h, ptr(a)))
        return dict(zip(("dim_x", "dim_y", "dim_z", "level", "n_cropped", "n_cells", "use_lists", "list_cells"), a.tolist()))

    def rawWeights(self):
        n = C.c_size_t()
        rc = capi.load().pft_tracker_get_raw_weights(self._h, None, 0, C.byref(n))
        if rc not in (capi.OK, capi.ERR_CAPACITY):
            check(rc)
        out = np.zeros(n.value, dtype=np.float32)
        if n.value:
            check(capi.load().pft_tracker_get_raw_weights(self._h, ptr(out), n.value, C.byref(n)))
        return out

    def ancestors(self):
        n = C.c_size_t()
        rc = capi.load().pft_tracker_get_ancestors(self._h, None, 0, C.byref(n))
        if rc not in (capi.OK, capi.ERR_CAPACITY):
            check(rc)
        out = np.zeros(n.value, dtype=np.int32)
        if n.value:
            check(capi.load().pft_tracker_get_ancestors(self._h, ptr(out), n.value, C.byref(n)))
        return out

    def nn(self, particle, m):
        idx = np.zeros(m, dtype=np.int32)
        d2 = np.zeros(m, dtype=np.float32)
        check(capi.load().pft_tracker_get_nn(self._h, int(particle), ptr(idx), ptr(d2), m))
        return idx, d2

    def enableTiming(self, on=True):
        check(capi.load().pft_tracker_enable_timing(self._h, 1 if on else 0))

    def timing(self):
        w, c = C.c_float(), C.c_float()
        check(capi.load().pft_tracker_get_timing(self._h, C.byref(w), C.byref(c)))
        return w.value, c.value

    def kernelTimes(self):
        """[(kernel name, ms)] of the last compute() in launch order (timing mode)."""
        cap = 256
        names = (C.c_char_p * cap)()
        ms = (C.c_float * cap)()
        n = C.c_int()
        check(capi.load().pft_tracker_get_kernel_times(self._h, names, ms, cap, C.byref(n)))
        return [(names[i].decode(), float(ms[i])) for i in range(n.value)]

    def evalCount(self):
        n = C.c_uint64()
        check(capi.load().pft_tracker_get_eval_count(self._h, C.byref(n)))
        return n.value

    def graphReplays(self):
        n = C.c_uint64()
        check(capi.load().pft_tracker_graph_replays(self._h, C.byref(n)))
        return n.value

    def commInit(self, nranks, rank, unique_id):
        buf = (C.c_char * 128).from_buffer_copy(bytes(unique_id))
        check(capi.load().pft_tracker_comm_init(self._h, int(nranks), int(rank), buf))

    def commDestroy(self):
        check(capi.load().pft_tracker_comm_destroy(self._h))

    def setDevices(self, devices):
        """Single-process multi-device mode: this one tracker object drives the GPUs `devices` (devices[0] = the device of
        its context).  Must be the first call on a new tracker; everything else stays as with one GPU."""
        arr = (C.c_int * len(devices))(*[int(d) for d in devices])
        check(capi.load().pft_tracker_set_devices(self._h, len(devices), arr))

    def follower(self, rank):
        """Multi-device mode: a borrowed view of the library-owned tracker of `rank` (1 .. n-1), for the getters."""
        v = object.__new__(type(self))
        v.ctx, v._input, v._h = self.ctx, None, C.c_void_p()
        check(capi.load().pft_tracker_get_follower(self._h, int(rank), C.byref(v._h)))
        v._borrowed = True
        return v

    # NVLink peer exchange: the collectives of weight() as peer stores from the producing kernels
    def peerExport(self):
        """Allocates this rank's exchange window and returns its CUDA IPC handle (bytes).  Needs the rank
        layout (setShard / commInit) and the particle numbers to be set."""
        buf = C.create_string_buffer(capi.PEER_HANDLE_BYTES)
        check(capi.load().pft_tracker_peer_export(self._h, buf))
        return bytes(buf.raw)

    def peerAttach(self, handles):
        """`handles`: the peerExport() results of all ranks in rank order (e.g. dist.all_gather_object)."""
        blob = b"".join(bytes(h) for h in handles)
        buf = C.create_string_buffer(blob, len(blob))
        check(capi.load().pft_tracker_peer_attach(self._h, buf))

    def peerDetach(self):
        check(capi.load().pft_tracker_peer_detach(self._h))

    def __del__(self):
        try:
            if self._h and not getattr(self, "_borrowed", False):
                capi.load().pft_tracker_destroy(self._h)
                self._h = C.c_void_p()
        except Exception:
            pass


class KLDAdaptiveParticleFilterOMPTracker(ParticleFilterOMPTracker):
    """pcl::tracking::KLDAdaptiveParticleFilterOMPTracker<PointXYZRGBA, ParticleXYZRPY> (ref :209-222)."""

    _KLD = 1

    def setMaximumParticleNum(self, n):
        self._si(capi.MAX_PARTICLE_NUM, n)

    def setDelta(self, d):
        self._sd(capi.DELTA, d)

    def setEpsilon(self, e):
        self._sd(capi.EPSILON, e)

    def setBinSize(self, b):
        """b: 6 values x,y,z,roll,pitch,yaw or a PARTICLE record (ref :214-221)."""
        if isinstance(b, np.void) or (isinstance(b, np.ndarray) and b.dtype == PARTICLE):
            b = [float(b[k]) for k in ("x", "y", "z", "roll", "pitch", "yaw")]
        self._sv(capi.BIN_SIZE, b)


def comm_unique_id():
    """128-byte NCCL unique id (rank 0 creates it, the host framework ships it to the other ranks)."""
    buf = (C.c_char * 128)()
    check(capi.load().pft_comm_get_unique_id(buf))
    return bytes(buf.raw)


def loadPCDFile(path, ctx=None):
    """pcl::io::loadPCDFile<PointXYZRGBA> -> device cloud (host-side parsing in pcd.py)."""
    from . import pcd
    pts, _, _ = pcd.loadPCDFile(path)
    return PointCloud(pts, ctx=ctx)


def savePCDFile(path, cloud, binary=False):
    """pcl::PCDWriter::write(path, cloud, binary) (ref: src/create_model.cpp:223): `cloud` is a PointCloud or a point array."""
    from . import pcd
    pcd.savePCDFile(path, cloud.to_numpy() if isinstance(cloud, PointCloud) else cloud, binary=binary)


def compute_batch(trackers):
    """compute() of several trackers that share one scene (ref :688-697).  The trackers may sit on other contexts than
    the scene, and on several (one object per GPU): each context's trackers run concurrently on its own stream."""
    arr = (C.c_void_p * len(trackers))(*[t._h for t in trackers])
    check(capi.load().pft_compute_batch(arr, len(trackers)))


def kernel_launch_count():
    return capi.load().pft_kernel_launch_count()


def configure_like_reference(tracker, coherence_cls=ApproxNearestPairPointCloudCoherence, particle_num=400, max_particle_num=500,
                             use_hsv=True, iteration_num=2):
    """Apply the knob values of ref: src/auto_tracking.cpp:187-254 (SURVEY 5.6) to a tracker."""
    step = [0.015 * 0.015] * 6
    for k in (3, 4, 5):
        step[k] *= 40.0
    if isinstance(tracker, KLDAdaptiveParticleFilterOMPTracker):
        tracker.setMaximumParticleNum(max_particle_num)
        tracker.setDelta(0.99)
        tracker.setEpsilon(0.2)
        tracker.setBinSize([0.1] * 6)
    tracker.setTrans(np.eye(4, dtype=np.float32))
    tracker.setStepNoiseCovariance(step)
    tracker.setInitialNoiseCovariance([0.00001] * 6)
    tracker.setInitialNoiseMean([0.0] * 6)
    tracker.setIterationNum(iteration_num)
    tracker.setParticleNum(particle_num)
    tracker.setResampleLikelihoodThr(0.0)
    tracker.setUseNormal(False)
    coherence = coherence_cls()
    coherence.addPointCoherence(DistanceCoherence())
    if use_hsv:
        hsv = HSVColorCoherence()
        hsv.setWeight(0.1)
        coherence.addPointCoherence(hsv)
    coherence.setSearchMethod(Octree(0.01))
    coherence.setMaximumDistance(0.1)
    tracker.setCloudCoherence(coherence)
    return tracker
