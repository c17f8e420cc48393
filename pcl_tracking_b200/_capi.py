"""ctypes binding of include/pft/pft.h (the C ABI of libpft.so).

This is the only way Python reaches the tracker: there is no CPU fallback and no second code path.
If the library has not been built, or no CUDA device is present, calls fail loudly.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PFT_LIB") or os.path.join(_HERE, "lib", "libpft.so")  # PFT_LIB: kernel-tuning builds only
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "pft", "pft.h")

POINT = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("rgba", "<u4")])
POINT_PCL32 = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("w", "<f4"), ("rgba", "<u4"), ("pad", "<u4", (3,))])
PARTICLE = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("one", "<f4"),
                     ("roll", "<f4"), ("pitch", "<f4"), ("yaw", "<f4"), ("weight", "<f4")])

RESULT_BOX = np.dtype([("centroid", "<f4", (3,)), ("axes", "<f4", (3, 3)), ("extent", "<f4", (3,)), ("center", "<f4", (3,)),
                       ("quat", "<f4", (4,)), ("eigenvalues", "<f4", (3,)), ("n", "<i4")])

LAYOUT_PACKED16, LAYOUT_PCL32 = 0, 1
OK, ERR_INVALID, ERR_CUDA, ERR_STATE, ERR_CAPACITY, ERR_COMM = 0, -1, -2, -3, -4, -5

# pft_key
THREADS, PARTICLE_NUM, MAX_PARTICLE_NUM, ITERATION_NUM, NN_MODE, USE_HSV, USE_DISTANCE, SAMPLER, QUAT_SAMPLE, USE_NORMAL, MIN_INDICES, DEBUG_NN, CANDIDATE_LISTS = range(13)
(DELTA, EPSILON, ALPHA, MOTION_RATIO, MAX_DIST, DIST_WEIGHT, HSV_WEIGHT, H_WEIGHT, S_WEIGHT, V_WEIGHT, SEARCH_RESOLUTION,
 RESAMPLE_LIKELIHOOD_THR) = range(20, 32)
STEP_NOISE_COV, INIT_NOISE_COV, INIT_NOISE_MEAN, BIN_SIZE = range(40, 44)
USE_CHANGE_DETECTOR, CHANGE_DETECTOR_INTERVAL, CHANGE_DETECTOR_MIN_POINTS = 13, 14, 15
CHANGE_DETECTOR_RESOLUTION = 32
NN_EXACT, NN_PCL_APPROX = 0, 1
PEER_HANDLE_BYTES = 64
CLOUD_PEER_HANDLE_BYTES = 192
SAMPLER_ALIAS_PCL, SAMPLER_CDF, SAMPLER_CDF_VDC = 0, 1, 2


class PftError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("pft error %d: %s" % (code, msg))
        self.code = code


MAX_DEPTH_CAMERAS = 8


class DepthCamera(C.Structure):
    """pft_depth_camera: one calibrated camera of pft_cloud_upload_depth_images (m12 NULL: no transform)."""
    _fields_ = [("depth", C.c_void_p), ("depth_step", C.c_uint32), ("bgr", C.c_void_p), ("bgr_step", C.c_uint32),
                ("width", C.c_uint32), ("height", C.c_uint32), ("fx", C.c_double), ("fy", C.c_double), ("cx", C.c_double),
                ("cy", C.c_double), ("m12", C.POINTER(C.c_float))]


# pft_depth_encoding, pft_colour_encoding
DEPTH_16UC1, DEPTH_32FC1 = 0, 1
COLOUR_BGR8, COLOUR_RGB8, COLOUR_BGRA8, COLOUR_RGBA8, COLOUR_MONO8, COLOUR_NONE = range(6)


class DepthCameraEnc(C.Structure):
    """pft_depth_camera_enc: a pft_depth_camera with its depth and colour encodings (pft_cloud_upload_depth_images_enc)."""
    _fields_ = [("cam", DepthCamera), ("depth_encoding", C.c_int32), ("colour_encoding", C.c_int32)]


class DepthCameraReg(C.Structure):
    """pft_depth_camera_reg: a pft_depth_camera_enc whose depth image is in a separate depth camera's geometry, registered
    into the colour camera on the device (depth_to_colour NULL: already registered)."""
    _fields_ = [("cam", DepthCameraEnc), ("depth_to_colour", C.POINTER(C.c_double)), ("depth_width", C.c_uint32), ("depth_height", C.c_uint32),
                ("depth_fx", C.c_double), ("depth_fy", C.c_double), ("depth_cx", C.c_double), ("depth_cy", C.c_double), ("depth_tx", C.c_double),
                ("depth_ty", C.c_double), ("colour_tx", C.c_double), ("colour_ty", C.c_double), ("fill_upsampling", C.c_int32)]


_vp, _i, _f, _d, _sz, _u64 = C.c_void_p, C.c_int, C.c_float, C.c_double, C.c_size_t, C.c_uint64
_pp = C.POINTER(C.c_void_p)
_psz = C.POINTER(C.c_size_t)

# name -> (restype, argtypes); every PFT_API function of pft.h is listed (tests/test_abi.py checks it)
SIGNATURES = {
    "pft_last_error": (C.c_char_p, []),
    "pft_version": (C.c_char_p, []),
    "pft_device_count": (_i, []),
    "pft_context_create": (_i, [_i, _pp]),
    "pft_context_destroy": (None, [_vp]),
    "pft_context_synchronize": (_i, [_vp]),
    "pft_context_stream": (_vp, [_vp]),
    "pft_host_alloc": (_i, [_pp, _sz]),
    "pft_host_free": (_i, [_vp]),
    "pft_kernel_launch_count": (_u64, []),
    "pft_cloud_create": (_i, [_vp, _pp]),
    "pft_cloud_destroy": (None, [_vp]),
    "pft_cloud_upload": (_i, [_vp, _vp, _sz, _i]),
    "pft_cloud_upload_pointcloud2": (_i, [_vp, _vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _i]),
    "pft_cloud_upload_async": (_i, [_vp, _vp, _sz, _i]),
    "pft_cloud_upload_pointcloud2_async": (_i, [_vp, _vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _i]),
    "pft_cloud_upload_depth_image": (_i, [_vp, _vp, C.c_uint32, _vp, C.c_uint32, C.c_uint32, C.c_uint32, _d, _d, _d, _d]),
    "pft_cloud_upload_depth_image_async": (_i, [_vp, _vp, C.c_uint32, _vp, C.c_uint32, C.c_uint32, C.c_uint32, _d, _d, _d, _d]),
    "pft_cloud_upload_depth_images": (_i, [_vp, C.POINTER(DepthCamera), _i]),
    "pft_cloud_upload_depth_images_async": (_i, [_vp, C.POINTER(DepthCamera), _i]),
    "pft_cloud_upload_depth_images_enc": (_i, [_vp, C.POINTER(DepthCameraEnc), _i]),
    "pft_cloud_upload_depth_images_enc_async": (_i, [_vp, C.POINTER(DepthCameraEnc), _i]),
    "pft_cloud_upload_depth_images_reg": (_i, [_vp, C.POINTER(DepthCameraReg), _i]),
    "pft_cloud_upload_depth_images_reg_async": (_i, [_vp, C.POINTER(DepthCameraReg), _i]),
    "pft_cloud_wait_upload": (_i, [_vp]),
    "pft_cloud_size": (_i, [_vp, _psz]),
    "pft_cloud_download": (_i, [_vp, _vp, _sz, _i, _psz]),
    "pft_passthrough": (_i, [_vp, _vp, _vp, _i, _f, _f]),
    "pft_passthrough_voxel_grid": (_i, [_vp, _vp, _vp, _f, _i, _f, _f]),
    "pft_approx_voxel_grid_pcl": (_i, [_vp, _vp, _vp, _f, _i, _f, _f]),
    "pft_prepare_model": (_i, [_vp, _vp, _vp, _f, _vp]),
    "pft_transform_cloud": (_i, [_vp, _vp, _vp, _vp]),
    "pft_remove_zero_points": (_i, [_vp, _vp, _vp]),
    "pft_euclidean_clusters": (_i, [_vp, _vp, _d, _i, _i, _vp, _sz, _vp, _sz, _psz]),
    "pft_cloud_select_cluster": (_i, [_vp, _vp, _i, _vp]),
    "pft_segment_plane": (_i, [_vp, _vp, _d, _i, _d, _vp, _i, _u64, _i, _vp, C.POINTER(C.c_int32), _vp, _vp, _psz]),
    "pft_tracker_create": (_i, [_vp, _i, _pp]),
    "pft_tracker_destroy": (None, [_vp]),
    "pft_tracker_set_i": (_i, [_vp, _i, _i]),
    "pft_tracker_set_d": (_i, [_vp, _i, _d]),
    "pft_tracker_set_vec6": (_i, [_vp, _i, _vp]),
    "pft_tracker_set_trans": (_i, [_vp, _vp]),
    "pft_tracker_set_reference_cloud": (_i, [_vp, _vp]),
    "pft_tracker_set_reference_points": (_i, [_vp, _vp, _sz, _i]),
    "pft_tracker_set_input_cloud": (_i, [_vp, _vp]),
    "pft_tracker_compute": (_i, [_vp]),
    "pft_compute_batch": (_i, [_pp, _i]),
    "pft_tracker_get_result": (_i, [_vp, _vp]),
    "pft_tracker_get_particles": (_i, [_vp, _vp, _sz, _psz]),
    "pft_particle_to_matrix": (_i, [_vp, _vp, _vp]),
    "pft_tracker_get_result_box": (_i, [_vp, _f, _vp]),
    "pft_tracker_get_result_cloud": (_i, [_vp, _f, _vp]),
    "pft_tracker_reset": (_i, [_vp]),
    "pft_tracker_get_eval_count": (_i, [_vp, C.POINTER(C.c_uint64)]),
    "pft_tracker_get_fit_ratio": (_i, [_vp, C.POINTER(C.c_double)]),
    "pft_tracker_set_particles": (_i, [_vp, _vp, _sz]),
    "pft_tracker_set_result": (_i, [_vp, _vp, _vp]),
    "pft_tracker_get_motion": (_i, [_vp, _vp]),
    "pft_tracker_inject_draws": (_i, [_vp, _vp, _vp, _vp, _i, _i]),
    "pft_tracker_seed": (_i, [_vp, _u64]),
    "pft_tracker_init_particles": (_i, [_vp]),
    "pft_tracker_resample": (_i, [_vp, _i]),
    "pft_tracker_weight": (_i, [_vp]),
    "pft_tracker_update": (_i, [_vp]),
    "pft_tracker_set_changed": (_i, [_vp, _i]),
    "pft_tracker_get_change_detector_info": (_i, [_vp, _vp]),
    "pft_tracker_get_aabb": (_i, [_vp, _vp]),
    "pft_tracker_get_cropped_count": (_i, [_vp, _psz]),
    "pft_tracker_get_raw_weights": (_i, [_vp, _vp, _sz, _psz]),
    "pft_tracker_get_ancestors": (_i, [_vp, _vp, _sz, _psz]),
    "pft_tracker_get_nn": (_i, [_vp, _i, _vp, _vp, _sz]),
    "pft_tracker_get_timing": (_i, [_vp, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "pft_tracker_enable_timing": (_i, [_vp, _i]),
    "pft_tracker_get_kernel_times": (_i, [_vp, _vp, _vp, _i, C.POINTER(C.c_int)]),
    "pft_tracker_get_index_info": (_i, [_vp, _vp]),
    "pft_tracker_graph_replays": (_i, [_vp, C.POINTER(C.c_uint64)]),
    "pft_tracker_weight_phase": (_i, [_vp, _i]),
    "pft_tracker_get_crop_box": (_i, [_vp, _vp]),
    "pft_tracker_set_crop_box": (_i, [_vp, _vp]),
    "pft_tracker_get_raw_slice": (_i, [_vp, _i, _vp, _sz, _psz]),
    "pft_tracker_set_raw_slice": (_i, [_vp, _i, _vp, _sz]),
    "pft_tracker_set_shard": (_i, [_vp, _i, _i]),
    "pft_comm_get_unique_id": (_i, [_vp]),
    "pft_context_comm_init": (_i, [_vp, _i, _i, _vp]),
    "pft_context_comm_destroy": (_i, [_vp]),
    "pft_cloud_broadcast": (_i, [_vp, _sz, _i]),
    "pft_tracker_comm_init": (_i, [_vp, _i, _i, _vp]),
    "pft_tracker_comm_destroy": (_i, [_vp]),
    "pft_cloud_peer_export": (_i, [_vp, _sz, _vp]),
    "pft_cloud_peer_attach": (_i, [_vp, _vp, _i, _i]),
    "pft_cloud_peer_broadcast": (_i, [_vp, _i]),
    "pft_cloud_peer_detach": (_i, [_vp]),
    "pft_tracker_set_devices": (_i, [_vp, _i, _vp]),
    "pft_tracker_get_follower": (_i, [_vp, _i, _vp]),
    "pft_tracker_peer_export": (_i, [_vp, _vp]),
    "pft_tracker_peer_attach": (_i, [_vp, _vp]),
    "pft_tracker_peer_detach": (_i, [_vp]),
}

_lib = None


def load():
    """dlopen libpft.so and bind every entry point.  Raises if the library has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "%s is missing: build it with `python -m pcl_tracking_b200.build` (nvcc, sm_100a). "
                "There is no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise PftError(rc, load().pft_last_error().decode("utf-8", "replace"))


def ptr(a):
    return a.ctypes.data_as(C.c_void_p)
