/*
 * pft.h -- C ABI of the B200-native particle-filter point-cloud tracker.
 *
 * Drop-in boundary for the one hot path cmaestre/pcl_tracking drives through PCL 1.8.0:
 *   scene filters  -> ref: src/auto_tracking.cpp:536-575 (PassThrough, VoxelGrid, ApproximateVoxelGrid)
 *   tracker set-up -> ref: src/auto_tracking.cpp:198-258 (KLDAdaptiveParticleFilterOMPTracker knobs)
 *   frame loop     -> ref: src/auto_tracking.cpp:683-697 (gridSampleApprox, setInputCloud, compute)
 *   read-out       -> ref: src/auto_tracking.cpp:270, :309-310 (getParticles, getResult, toEigenMatrix)
 * The reference has no FFI layer (it links PCL templates directly, ref: CMakeLists.txt:68-69); every
 * entry point below names the PCL method it replaces.  include/pft/pcl_shim.hpp maps the PCL class
 * names onto this ABI.  Plain C: opaque handles, POD structs, pointers and sizes; no exceptions
 * cross the boundary; every function returns a pft_status (0 = ok, < 0 = error, text in
 * pft_last_error()).  PCL's own convention is kept where it matters: compute() on an empty
 * input/reference cloud is a silent no-op (PFT_OK), as Tracker::initCompute does.
 *
 * There is NO CPU fallback: every call that computes runs hand-written sm_100a CUDA kernels and
 * fails with PFT_ERR_CUDA when no device is present.
 *
 * Threading: a tracker is not thread safe; distinct trackers may be driven from distinct threads.
 * Calls are asynchronous on the owning context's stream unless they return data to the host.
 */
#ifndef PFT_PFT_H_
#define PFT_PFT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PFT_API __attribute__((visibility("default")))

typedef enum {
  PFT_OK = 0,
  PFT_ERR_INVALID = -1,   /* bad argument / unknown key */
  PFT_ERR_CUDA = -2,      /* CUDA runtime error or no device */
  PFT_ERR_STATE = -3,     /* call order (e.g. compute before setReferenceCloud on a non-empty input) */
  PFT_ERR_CAPACITY = -4,  /* caller buffer too small */
  PFT_ERR_COMM = -5       /* NCCL error / NCCL not loadable / NVLink peer exchange failed (IPC mapping, a peer that never arrived) */
} pft_status;

/* 16-byte packed point {x,y,z,rgba}; rgba bytes are b,g,r,a as in pcl::PointXYZRGBA */
typedef struct { float x, y, z; uint32_t rgba; } pft_point;
/* the 32-byte in-memory layout of pcl::PointXYZRGBA (ref: src/auto_tracking.cpp:139-140) */
typedef struct { float x, y, z, w; uint32_t rgba; uint32_t pad[3]; } pft_point_pcl32;
/* the 32-byte layout of pcl::tracking::ParticleXYZRPY (ref: src/auto_tracking.cpp:142) */
typedef struct { float x, y, z, one, roll, pitch, yaw, weight; } pft_particle;

typedef enum { PFT_LAYOUT_PACKED16 = 0, PFT_LAYOUT_PCL32 = 1 } pft_layout;

typedef struct pft_context pft_context; /* one CUDA device + stream + scratch */
typedef struct pft_cloud pft_cloud;     /* device-resident point cloud (pcl::PointCloud<PointXYZRGBA>) */
typedef struct pft_tracker pft_tracker; /* pcl::tracking::(KLDAdaptive)ParticleFilterOMPTracker */

/* ---------------------------------------------------------------- context */
PFT_API const char* pft_last_error(void);
PFT_API const char* pft_version(void);
PFT_API int pft_device_count(void);
PFT_API int pft_context_create(int device, pft_context** out);
PFT_API void pft_context_destroy(pft_context* ctx);
PFT_API int pft_context_synchronize(pft_context* ctx);
/* raw cudaStream_t of the context, so that a host framework can order its own work after ours */
PFT_API void* pft_context_stream(pft_context* ctx);
/* pinned host memory for frame buffers (H2D of a pageable buffer is staged by the driver) */
PFT_API int pft_host_alloc(void** ptr, size_t bytes);
PFT_API int pft_host_free(void* ptr);
/* number of kernels this library has launched since load (bench.py's gpu_launches) */
PFT_API uint64_t pft_kernel_launch_count(void);

/* ---------------------------------------------------------------- clouds */
PFT_API int pft_cloud_create(pft_context* ctx, pft_cloud** out);
PFT_API void pft_cloud_destroy(pft_cloud* cloud);
/* replaces pcl::fromPCLPointCloud2 / cloud assignment (ref: src/auto_tracking.cpp:619-622) */
PFT_API int pft_cloud_upload(pft_cloud* cloud, const void* host_points, size_t n, int layout);
/* frame ingest: a sensor_msgs/PointCloud2 payload as it arrives from the camera driver -> device cloud.  Replaces
 * pcl_conversions::toPCL + pcl::fromPCLPointCloud2 (ref: src/auto_tracking.cpp:619-622): `data` holds `height` rows of
 * `row_step` bytes with `width` records of `point_step` bytes each; off_* are the byte offsets of the float32 fields
 * x, y, z and of the packed rgb/rgba word inside a record (off_rgb < 0: no colour, rgba = 0).  Point order is
 * row-major, NaN points are kept (the PassThrough that follows drops them, ref :637). */
PFT_API int pft_cloud_upload_pointcloud2(pft_cloud* cloud, const void* data, uint32_t width, uint32_t height, uint32_t point_step,
                                         uint32_t row_step, int32_t off_x, int32_t off_y, int32_t off_z, int32_t off_rgb, int is_bigendian);
/* frame ingest one step earlier: the registered depth and colour images the points topic is computed from (kinect2_bridge
 * <res>/image_depth_rect, <res>/image_color_rect, <res>/camera_info), 5 bytes per pixel instead of a 32-byte record.
 * Replaces the depth_image_proc/point_cloud_xyzrgb nodelet behind the topic of ref: src/auto_tracking.cpp:775, with its
 * rounding: `depth` holds `height` rows of `depth_step` bytes (even) of uint16 millimetres, `bgr` `height` rows of
 * `bgr_step` bytes of bgr8 pixels; fx, fy, cx, cy are camera_info.K[0], K[4], K[2], K[5].  Pixel (u, v) with depth d
 * becomes x = ((u - (float)cx) * d) * (float)(0.001f / fx), y likewise with v, fy, cy, z = d * 0.001f, all in fp32;
 * d == 0 gives x = y = z = NaN.  rgba = b | g << 8 | r << 16 | 255 << 24 for every pixel.  The cloud is organised,
 * width * height points in row-major order, as pft_cloud_upload_pointcloud2 leaves it.  Only (height - 1) * step +
 * width * bytes-per-pixel bytes of each image are read.  PFT_ERR_INVALID: a null image with pixels, a step below
 * width * bytes-per-pixel or an odd depth step, fx or fy zero or not finite, cx or cy not finite, 2^31 pixels or more. */
PFT_API int pft_cloud_upload_depth_image(pft_cloud* cloud, const void* depth, uint32_t depth_step, const void* bgr, uint32_t bgr_step,
                                         uint32_t width, uint32_t height, double fx, double fy, double cx, double cy);
/* One calibrated camera of a fused frame: the images and intrinsics of pft_cloud_upload_depth_image, and `m12`, the
 * fp32 3x4 row-major matrix from the camera's optical frame to the common frame (Eigen::Affine3f rows 0-2, the
 * convention of pft_tracker_set_trans; e.g. tf2 lookupTransform(target, camera_optical_frame)), or NULL to keep the
 * camera's own frame. */
typedef struct {
  const void* depth;
  uint32_t depth_step;
  const void* bgr;
  uint32_t bgr_step;
  uint32_t width, height;
  double fx, fy, cx, cy;
  const float* m12;
} pft_depth_camera;
#define PFT_MAX_DEPTH_CAMERAS 8
/* Several calibrated cameras fused into one scene cloud: for each camera k, pcl::transformPointCloud(cloud_k, T_k) of
 * the nodelet's cloud, then scene += cloud_k.  Pixel (u, v) of camera k becomes the point pft_cloud_upload_depth_image
 * makes of it; with a matrix, each finite point is then transformed as PCL 1.8.0 does, x' = ((m00 x + m01 y) + m02 z)
 * + m03, every fp32 operation rounded on its own.  Depth-0 (NaN) points are kept as they are, colour included.  The
 * cloud is unorganised: camera 0's width * height points in row-major order, then camera 1's, and so on.  Cameras
 * may differ in size; one with no pixels adds nothing.  All images are converted by one kernel launch.  One camera
 * without a matrix gives exactly the cloud of pft_cloud_upload_depth_image.  PFT_ERR_INVALID: n < 1 or n >
 * PFT_MAX_DEPTH_CAMERAS, null `cams`, any camera that pft_cloud_upload_depth_image would reject (the message names
 * its index), a non-finite matrix entry, 2^31 pixels or more in total. */
PFT_API int pft_cloud_upload_depth_images(pft_cloud* cloud, const pft_depth_camera* cams, int n);
/* The calls above take 16UC1 depth and bgr8 colour.  Every encoding the depth_image_proc nodelets accept
 * (point_cloud_xyzrgb, and point_cloud_xyz for depth alone) goes through pft_cloud_upload_depth_images_enc: each camera
 * names its pair, `cam.bgr` / `cam.bgr_step` then hold the colour image in `colour_encoding`, and any mix of pairs is
 * converted by the same one launch.  Pixel (u, v) becomes depth_image_proc::convert<T>'s point, every fp32 operation
 * rounded on its own:
 *   depth encoding    bytes  valid when      x (y likewise with v, cy, fy)                               z
 *   PFT_DEPTH_16UC1   2      d != 0          ((u - (float)cx) * (float)d) * (float)((double)0.001f / fx)  (float)d * 0.001f
 *   PFT_DEPTH_32FC1   4      isfinite(d)     ((u - (float)cx) * d) * (float)(1.0 / fx)                   d
 * (16UC1 is millimetres, 32FC1 metres; 32FC1 keeps 0 and negative depths, as upstream.)  An invalid pixel gives a
 * quiet-NaN x, y, z; its colour is still written.  rgba = b | g << 8 | r << 16 | 255 << 24, with r, g, b read at these
 * byte offsets of the colour pixel:
 *   colour encoding     bytes  r, g, b
 *   PFT_COLOUR_BGR8     3      2, 1, 0
 *   PFT_COLOUR_RGB8     3      0, 1, 2
 *   PFT_COLOUR_BGRA8    4      2, 1, 0   (alpha ignored)
 *   PFT_COLOUR_RGBA8    4      0, 1, 2   (alpha ignored)
 *   PFT_COLOUR_MONO8    1      0, 0, 0
 *   PFT_COLOUR_NONE     0      rgba = 0 (point_cloud_xyz; `bgr` and `bgr_step` are ignored and nothing is copied)
 * sensor_msgs/Image "mono16" is 16UC1.  Camera k with {16UC1, bgr8} gives exactly the points of
 * pft_cloud_upload_depth_images; one camera without a matrix those of pft_cloud_upload_depth_image.  PFT_ERR_INVALID,
 * naming the camera: any rejection of pft_cloud_upload_depth_images, an unknown encoding, a 32FC1 depth step that is
 * not a multiple of 4 or below 4 * width, a colour step below bytes-per-pixel * width, a null colour image with pixels
 * (unless PFT_COLOUR_NONE).  Images are little-endian and of equal size. */
typedef enum { PFT_DEPTH_16UC1 = 0, PFT_DEPTH_32FC1 = 1 } pft_depth_encoding;
typedef enum { PFT_COLOUR_BGR8 = 0, PFT_COLOUR_RGB8 = 1, PFT_COLOUR_BGRA8 = 2, PFT_COLOUR_RGBA8 = 3, PFT_COLOUR_MONO8 = 4, PFT_COLOUR_NONE = 5 } pft_colour_encoding;
typedef struct {
  pft_depth_camera cam;
  int32_t depth_encoding;   /* pft_depth_encoding */
  int32_t colour_encoding;  /* pft_colour_encoding */
} pft_depth_camera_enc;
PFT_API int pft_cloud_upload_depth_images_enc(pft_cloud* cloud, const pft_depth_camera_enc* cams, int n);
/* Frame ingest overlapped with the previous frame's compute (SURVEY 8 f-1).  Same arguments as the five uploads above,
 * but the copy (and the unpack kernel) run on a copy stream of the context instead of its compute stream: the call
 * returns at once, the copy starts when everything enqueued on the context BEFORE this call has finished (so earlier
 * readers of `cloud` are safe), and it overlaps whatever is enqueued AFTER it.  The first library call that consumes
 * `cloud` orders the compute stream behind the copy by itself (no host wait); pft_cloud_wait_upload does the same
 * explicitly, e.g. before handing the context stream to foreign code.  The host buffer must be pinned
 * (pft_host_alloc) and stay untouched until a consumer of the cloud has completed.  Typical frame loop with two
 * clouds A/B: upload_async(B, frame k+1); filter(A) + compute (frame k); read the result; swap A and B. */
PFT_API int pft_cloud_upload_async(pft_cloud* cloud, const void* host_points, size_t n, int layout);
PFT_API int pft_cloud_upload_pointcloud2_async(pft_cloud* cloud, const void* data, uint32_t width, uint32_t height, uint32_t point_step,
                                               uint32_t row_step, int32_t off_x, int32_t off_y, int32_t off_z, int32_t off_rgb, int is_bigendian);
PFT_API int pft_cloud_upload_depth_image_async(pft_cloud* cloud, const void* depth, uint32_t depth_step, const void* bgr, uint32_t bgr_step,
                                               uint32_t width, uint32_t height, double fx, double fy, double cx, double cy);
PFT_API int pft_cloud_upload_depth_images_async(pft_cloud* cloud, const pft_depth_camera* cams, int n);
PFT_API int pft_cloud_upload_depth_images_enc_async(pft_cloud* cloud, const pft_depth_camera_enc* cams, int n);
/* Depth images that are NOT registered to the colour camera: the depth_image_proc/register nodelet
 * (RegisterNodelet::convert<T>) on the device, followed by the conversion of pft_cloud_upload_depth_images_enc, i.e.
 * the register -> point_cloud_xyzrgb nodelet chain.  A camera with `depth_to_colour` set has its depth image
 * (`cam.depth`, `cam.depth_step`, `cam.depth_encoding`) in the depth camera's geometry, depth_width x depth_height;
 * `cam.width`, `cam.height`, `cam.fx` .. `cam.cy`, the colour image and `cam.m12` are the colour camera's, as for
 * pft_cloud_upload_depth_images_enc, and so is the cloud: width * height points, organised in the colour camera's
 * geometry.  Intrinsics are image_geometry::PinholeCameraModel's, P[0], P[5], P[2], P[6], and Tx = P[3], Ty = P[7] (a
 * monocular camera: K's, Tx = Ty = 0); full resolution (no binning, no ROI).  depth_to_colour: double 3x4 row-major,
 * Eigen::Affine3d rows 0-2 of tf2 lookupTransform(colour_frame, depth_frame).  Every operation is in double unless
 * stated, each rounded on its own:
 *   1. the registered image starts all invalid: 0 (16UC1), quiet NaN (32FC1);
 *   2. depth pixels (u, v) in raster order; an invalid raw depth (16UC1 0, 32FC1 non-finite) is skipped, otherwise
 *      depth = (double)toMeters(d), toMeters = the float d * 0.001f (16UC1) or d (32FC1);
 *   3. without fill_upsampling: X = ((u - cx_d) * depth - Tx_d) * (1.0 / fx_d), Y likewise with v, cy_d, Ty_d, fy_d,
 *      Z = depth; p = M (X, Y, Z, 1), each row ((m0 X + m1 Y) + m2 Z) + m3; u' = (int)(((fx_c p.x + Tx_c) * (1.0 / p.z)
 *      + cx_c) + 0.5), v' likewise (truncation toward zero: (-1, 0) lands on column 0); skipped unless 0 <= u' < width
 *      and 0 <= v' < height; candidate fromMeters((float)p.z): (uint16_t)((float)p.z * 1000.0f + 0.5f) in float for
 *      16UC1, (float)p.z for 32FC1;
 *   4. with fill_upsampling: the same for the corners (u - 0.5f, v - 0.5f) and (u + 0.5f, v + 0.5f) (float sums), giving
 *      (u1, v1) and (u2, v2) and z1, z2; skipped if u1 < 0 || u2 >= width || v1 < 0 || v2 >= height; otherwise every
 *      pixel of [u1, u2] x [v1, v2] (possibly empty) gets the candidate fromMeters((float)(0.5 * (z1 + z2)));
 *   5. z-buffer at the target: if (!valid(reg) || reg > new) reg = new.
 * So a pixel holds the smallest valid candidate after its last reset (a 16UC1 0 or 32FC1 -inf candidate, which
 * replaces anything), the earliest of equal ones (+0 before -0 if it came first); else +inf, if a +inf candidate came
 * after that reset; else the reset value; else the initial one.  Where upstream is undefined C++ the candidate is
 * dropped: a double -> int cast of NaN or of a value whose truncation does not fit an int, a 16UC1 fromMeters whose
 * z * 1000.0f + 0.5f is NaN or truncates outside 0 .. 65535.  A 32FC1 candidate that is NaN (only a corner at +inf and
 * one at -inf make one) is dropped as well.  The registered image is then converted exactly as
 * pft_cloud_upload_depth_images_enc converts a registered one.  A registered camera without depth pixels gives width *
 * height NaN points with their colour.  depth_to_colour NULL: the camera is exactly the pft_depth_camera_enc `cam`, and
 * the other fields are ignored; registered and already-registered cameras mix in one call.  Kernel launches per frame:
 * 2 (conversion and header) when no camera is registered, 5 when any is (reset scatter, z-buffer scatter, finalise),
 * whatever the number of cameras.  PFT_ERR_INVALID, naming the camera: any rejection of
 * pft_cloud_upload_depth_images_enc for the colour side, a non-finite matrix entry, depth fx or fy zero or not finite,
 * a non-finite cx, cy, Tx or Ty on either camera, fill_upsampling not 0 or 1, a depth step that is not a multiple of the
 * depth pixel or below depth_width pixels, a null depth image with pixels, 2^31 depth pixels or more. */
typedef struct {
  pft_depth_camera_enc cam;
  const double* depth_to_colour;  /* 3x4 row-major; NULL: the depth is already registered */
  uint32_t depth_width, depth_height;
  double depth_fx, depth_fy, depth_cx, depth_cy, depth_tx, depth_ty;
  double colour_tx, colour_ty;
  int32_t fill_upsampling;        /* 0 or 1 */
} pft_depth_camera_reg;
PFT_API int pft_cloud_upload_depth_images_reg(pft_cloud* cloud, const pft_depth_camera_reg* cams, int n);
PFT_API int pft_cloud_upload_depth_images_reg_async(pft_cloud* cloud, const pft_depth_camera_reg* cams, int n);
PFT_API int pft_cloud_wait_upload(pft_cloud* cloud);
PFT_API int pft_cloud_size(pft_cloud* cloud, size_t* n);
PFT_API int pft_cloud_download(pft_cloud* cloud, void* host_points, size_t capacity, int layout, size_t* n);

/* ---------------------------------------------------------------- filters (kernel K1) */
/* pcl::PassThrough::filter, !keepOrganized: keep finite points with lo <= field <= hi, order
 * preserving (ref: src/auto_tracking.cpp:536-547).  field: 0=x 1=y 2=z. */
PFT_API int pft_passthrough(pft_context* ctx, const pft_cloud* in, pft_cloud* out, int field, float lo, float hi);
/* PassThrough + voxel-grid centroid in one pass: replaces filterPassThrough + gridSampleApprox /
 * gridSample (ref: src/auto_tracking.cpp:637, :683, :641).  Exactly one centroid per occupied voxel
 * of the lattice floor(coord * (1/leaf)); voxels are emitted in order of first appearance.
 * field < 0 disables the PassThrough predicate (finite check only). */
PFT_API int pft_passthrough_voxel_grid(pft_context* ctx, const pft_cloud* in, pft_cloud* out, float leaf,
                                       int field, float lo, float hi);
/* Parity mode: pcl::ApproximateVoxelGrid::applyFilter reproduced exactly -- the 512-entry direct-mapped cache walked in
 * input order, partial centroids emitted on every eviction, sequential fp32 sums (ref: src/auto_tracking.cpp:563-575,
 * PCL-1.8.0 filters/impl/approximate_voxel_grid.hpp).  The algorithm is a sequential scan and runs on one GPU thread
 * (~10 ms for a Kinect2 frame): use it to reproduce the reference's downsampled cloud bit for bit, and
 * pft_passthrough_voxel_grid in production. */
PFT_API int pft_approx_voxel_grid_pcl(pft_context* ctx, const pft_cloud* in, pft_cloud* out, float leaf, int field, float lo, float hi);
/* removeZeroPoints + compute3DCentroid + transformPointCloud(-centroid) + VoxelGrid(leaf): the model
 * preparation of ref: src/auto_tracking.cpp:656-674.  centroid3 receives the translation that the
 * caller passes to pft_tracker_set_trans. */
PFT_API int pft_prepare_model(pft_context* ctx, const pft_cloud* raw, pft_cloud* out, float leaf, float* centroid3);
/* pcl::transformPointCloud (PCL 1.8.0, common/impl/transforms.hpp) as the model builder moves a frame into the robot base
 * frame and its clusters back to the camera (ref: src/create_model.cpp:107-123, :184-204 through pcl_ros).  `m12` is
 * the fp32 3x4 row-major [R|t], the convention of pft_tracker_set_trans and pft_depth_camera.m12 (pcl_ros rounds each
 * entry of the double tf matrix to float: do the same).  `out` receives every point of `in` in the same order, rgba
 * copied.  A point whose x, y and z are finite becomes x' = ((m00 x + m01 y) + m02 z) + m03 (y', z' likewise), every
 * fp32 operation rounded on its own; a point with a non-finite coordinate is copied unchanged.  That is PCL's non-dense
 * branch; for a cloud of finite points it equals the dense one, so the result differs from PCL only for a cloud flagged
 * is_dense that nevertheless holds non-finite points (PCL then transforms them too).  in == out is allowed (in place);
 * both clouds belong to `ctx`.  The point count is read from `in`'s device header: the call never waits for the host
 * and may follow a filter whose count has not been read back.  One kernel launch.  PFT_ERR_INVALID: a null argument,
 * a non-finite matrix entry, a cloud of another context. */
PFT_API int pft_transform_cloud(pft_context* ctx, const pft_cloud* in, pft_cloud* out, const float* m12);
/* removeZeroPoints of the model builder (ref: src/create_model.cpp:59-77) and of pft_prepare_model (ref:
 * src/auto_tracking.cpp:577-595): drops a point if any coordinate is not finite, or if |x|, |y| and |z| are all < 0.01
 * (compared in double); order preserving.  in != out.  The same kernel as the first step of pft_prepare_model. */
PFT_API int pft_remove_zero_points(pft_context* ctx, const pft_cloud* in, pft_cloud* out);

/* ---------------------------------------------------------------- model acquisition */
/* pcl::EuclideanClusterExtraction::extract as the model builder runs it (ref: src/create_model.cpp:169-179:
 * tolerance 0.02, min 500, max 25000): connected components of "closer than `tolerance`" (squared fp32 distance <
 * (float)(tolerance^2), as FLANN's radius search), kept when min_size <= size <= max_size, ranked by size descending
 * (ties: lower first point index).  labels[i] (host, may be NULL) = cluster rank of point i or -1; sizes[k] (host, may
 * be NULL) = points of cluster k.  Non-finite points belong to no cluster.  The labels stay on the device for
 * pft_cloud_select_cluster, which extracts cluster k as a cloud in input order (= the sorted indices upstream): the
 * clouds create_model writes to models/<time>/<k>.pcd and returns to auto_tracking (ref: src/create_model.cpp:209-230). */
PFT_API int pft_euclidean_clusters(pft_context* ctx, const pft_cloud* in, double tolerance, int min_size, int max_size, int32_t* labels,
                                   size_t labels_capacity, int32_t* sizes, size_t sizes_capacity, size_t* n_clusters);
PFT_API int pft_cloud_select_cluster(pft_context* ctx, const pft_cloud* in, int k, pft_cloud* out);
/* pcl::SACSegmentation(SACMODEL_PLANE, SAC_RANSAC)::segment + pcl::ExtractIndices of the model builder's plane variant
 * (ref: src/create_model_planar_segmentation.cpp:157-174: setMaxIterations(1000), setDistanceThreshold(0.015); upstream
 * defaults probability 0.99, optimize_coefficients true).  samples3 (host, n_samples x 3 point indices) injects the
 * RANSAC draws in draw order (upstream uses rand(): not reproducible); NULL: generated on the device from `seed`.
 * Every hypothesis is scored, then the sequential accept / adapt-k / stop rule is replayed over the scores: the same
 * plane as upstream's loop for the same draws (a collinear sample is skipped without counting as an iteration).
 * coefficients4 = (a, b, c, d) of the (refined) plane; plane_out / rest_out (may be NULL) = ExtractIndices with
 * setNegative(false) / (true), both in input order; non-finite points are never inliers. */
PFT_API int pft_segment_plane(pft_context* ctx, const pft_cloud* in, double distance_threshold, int max_iterations, double probability,
                              const int32_t* samples3, int n_samples, uint64_t seed, int optimize_coefficients, float* coefficients4,
                              int32_t* iterations, pft_cloud* plane_out, pft_cloud* rest_out, size_t* n_inliers);

/* ---------------------------------------------------------------- tracker configuration */
typedef enum {
  /* int keys */
  PFT_THREADS = 0,            /* ctor(nr_threads) / setNumberOfThreads: accepted, ignored (ref :204,:210) */
  PFT_PARTICLE_NUM = 1,       /* setParticleNum           (ref :231) */
  PFT_MAX_PARTICLE_NUM = 2,   /* setMaximumParticleNum    (ref :211) */
  PFT_ITERATION_NUM = 3,      /* setIterationNum          (ref :229) */
  PFT_NN_MODE = 4,            /* pft_nn_mode: Nearest- vs ApproxNearestPairPointCloudCoherence (ref :235-238) */
  PFT_USE_HSV = 5,            /* addPointCoherence(HSVColorCoherence) (ref :244-247) */
  PFT_USE_DISTANCE = 6,       /* addPointCoherence(DistanceCoherence) (ref :240-242) */
  PFT_SAMPLER = 7,            /* pft_sampler */
  PFT_QUAT_SAMPLE = 8,        /* 1: PCL>=1.8.0 quaternion rotation noise; 0: additive RPY noise */
  PFT_USE_NORMAL = 9,         /* setUseNormal: only 0 is supported (ref :233) */
  PFT_MIN_INDICES = 10,       /* setMinIndices: accepted, inert without normals (ref :676) */
  PFT_DEBUG_NN = 11,          /* record per-point NN indices for the first K particles of weight() */
  PFT_CANDIDATE_LISTS = 12,   /* exact-NN lookup tables per weight(): 0 never, 1 when they pay off (default), 2 always.
                                 Internal to the search: results are identical in all three modes. */
  PFT_USE_CHANGE_DETECTOR = 13,        /* setUseChangeDetector (upstream default false; the reference never sets it).  On: every
                                          `interval` weight() calls the cropped cloud goes through an
                                          OctreePointCloudChangeDetector; no new voxel => the weights are not recomputed,
                                          resample() and update() are skipped until something changes.  compute() then
                                          runs stream-launched with one read-back per test (no graph replay). */
  PFT_CHANGE_DETECTOR_INTERVAL = 14,   /* setIntervalOfChangeDetection (default 10) */
  PFT_CHANGE_DETECTOR_MIN_POINTS = 15, /* setMinPointsOfChangeDetection (default 10): new voxels with fewer points are ignored */
  /* double keys */
  PFT_DELTA = 20,             /* setDelta                 (ref :212) */
  PFT_EPSILON = 21,           /* setEpsilon               (ref :213) */
  PFT_ALPHA = 22,             /* setAlpha (upstream default 15) */
  PFT_MOTION_RATIO = 23,      /* setMotionRatio (upstream default 0.25) */
  PFT_MAX_DIST = 24,          /* coherence->setMaximumDistance (ref :253) */
  PFT_DIST_WEIGHT = 25,       /* DistanceCoherence::setWeight */
  PFT_HSV_WEIGHT = 26,        /* HSVColorCoherence::setWeight (ref :246) */
  PFT_H_WEIGHT = 27, PFT_S_WEIGHT = 28, PFT_V_WEIGHT = 29,
  PFT_SEARCH_RESOLUTION = 30, /* pcl::search::Octree(resolution) -> index cell size (ref :250) */
  PFT_RESAMPLE_LIKELIHOOD_THR = 31, /* setResampleLikelihoodThr: accepted, inert upstream (ref :232) */
  PFT_CHANGE_DETECTOR_RESOLUTION = 32, /* setResolutionOfChangeDetection (default 0.01) */
  /* 6-vector keys */
  PFT_STEP_NOISE_COV = 40,    /* setStepNoiseCovariance    (ref :226) */
  PFT_INIT_NOISE_COV = 41,    /* setInitialNoiseCovariance (ref :227) */
  PFT_INIT_NOISE_MEAN = 42,   /* setInitialNoiseMean       (ref :228) */
  PFT_BIN_SIZE = 43           /* setBinSize                (ref :214-221) */
} pft_key;

typedef enum {
  PFT_NN_EXACT = 0,      /* true nearest neighbour, ties to the lower index (the product path) */
  PFT_NN_PCL_APPROX = 1  /* parity mode: pcl::octree approxNearestSearch of ApproxNearestPairPointCloudCoherence
                            (ref: src/auto_tracking.cpp:235-238) -- greedy descent, may miss the nearest point; the
                            octree is rebuilt sequentially by every weight(), far slower than PFT_NN_EXACT */
} pft_nn_mode;
/* PFT_SAMPLER_ALIAS_PCL: upstream's Walker alias table (genAliasTable / sampleWithReplacement), built sequentially on
 * one GPU thread -- parity mode: same ancestors as PCL for the same uniforms.  PFT_SAMPLER_CDF (default): inverse-CDF on
 * a fixed-point cumulative table built in parallel (same distribution).  PFT_SAMPLER_CDF_VDC: one uniform + van der
 * Corput offsets (low-variance selection). */
typedef enum { PFT_SAMPLER_ALIAS_PCL = 0, PFT_SAMPLER_CDF = 1, PFT_SAMPLER_CDF_VDC = 2 } pft_sampler;

/* kld != 0: KLDAdaptiveParticleFilterOMPTracker (ref :209-222); kld == 0: ParticleFilterOMPTracker (ref :201-206) */
PFT_API int pft_tracker_create(pft_context* ctx, int kld, pft_tracker** out);
PFT_API void pft_tracker_destroy(pft_tracker* t);
PFT_API int pft_tracker_set_i(pft_tracker* t, int key, int value);
PFT_API int pft_tracker_set_d(pft_tracker* t, int key, double value);
PFT_API int pft_tracker_set_vec6(pft_tracker* t, int key, const double* v6);
/* setTrans(Eigen::Affine3f): row-major 3x4 [R|t] (ref :225, :674) */
PFT_API int pft_tracker_set_trans(pft_tracker* t, const float* m12);
/* setReferenceCloud (ref :673): copied into the tracker */
/* the cloud may belong to another context, as for pft_tracker_set_input_cloud (read once, through a replica) */
PFT_API int pft_tracker_set_reference_cloud(pft_tracker* t, const pft_cloud* cloud);
PFT_API int pft_tracker_set_reference_points(pft_tracker* t, const void* host_points, size_t n, int layout);
/* setInputCloud (ref :691): the cloud handle is borrowed until the next set_input/compute pair.  The cloud may belong
 * to another context, on the same device or another one (one object per GPU): the tracker's context then reads a
 * replica of it, shared by all its trackers and refreshed by one fan-out launch on the cloud's stream when a library
 * call has written the cloud since.  This call enables peer access from the cloud's device to the tracker's (and its
 * followers') devices: PFT_ERR_COMM where that is impossible.  A tracker attached to a communicator, a shard
 * (pft_tracker_set_shard) or peer windows refuses a cloud of another context with PFT_ERR_INVALID. */
PFT_API int pft_tracker_set_input_cloud(pft_tracker* t, const pft_cloud* cloud);

/* ---------------------------------------------------------------- tracker execution */
/* Tracker::compute (ref :693): iteration_num x { resample (if changed) ; weight ; update }.
 * Enqueued on the context stream; results are read with the getters below (which synchronise). */
PFT_API int pft_tracker_compute(pft_tracker* t);
/* compute() of n independent trackers that share one scene (ref :688-697 loops them serially).  The trackers may sit
 * on several contexts: stale scene replicas are refreshed first (one launch per source cloud), then every context's
 * trackers run concurrently on streams forked from and joined to that context's stream.  The host waits for no device. */
PFT_API int pft_compute_batch(pft_tracker** trackers, int n);
/* getResult (ref :309) */
PFT_API int pft_tracker_get_result(pft_tracker* t, pft_particle* out);
/* getParticles (ref :270) */
PFT_API int pft_tracker_get_particles(pft_tracker* t, pft_particle* out, size_t capacity, size_t* n);
/* ParticleXYZRPY::toEigenMatrix (ref :310): row-major 3x4, computed by the same device routine as weight() */
PFT_API int pft_particle_to_matrix(pft_context* ctx, const pft_particle* p, float* m12);
/* Result post-processing, what viz_cb derives from getResult() per object (ref: src/auto_tracking.cpp:309-316,
 * :432-466, :481-515): the reference cloud moved to the result pose (translation.z + z_offset; the reference passes
 * -0.005), its compute3DCentroid (the position published on /visual/cam_frame_obj_pos_vector), the eigenvectors of
 * its normalised covariance (ascending eigenvalues, third axis = first x second; the sign of an eigenvector is
 * unspecified in Eigen, here the largest component of the first two axes is positive) and the oriented bounding box
 * in that frame: edge lengths, centre (tfinal) and orientation quaternion (qfinal: w, x, y, z). */
typedef struct {
  float centroid[3];
  float axes[9];      /* row-major 3x3, columns = box axes */
  float extent[3];
  float center[3];
  float quat[4];
  float eigenvalues[3];
  int32_t n;          /* model points */
} pft_result_box;
PFT_API int pft_tracker_get_result_box(pft_tracker* t, float z_offset, pft_result_box* out);
/* The cloud pft_tracker_get_result_box measures (ref: src/auto_tracking.cpp:309-316): the reference cloud, in the order
 * and with the colours it was given, moved by toEigenMatrix(getResult()) with translation.z += z_offset -- the tracked
 * object's points, e.g. for a grasp planner.  Bit for bit pft_transform_cloud(reference, M) with M =
 * pft_particle_to_matrix(result) and M[11] += z_offset in fp32.  `out` belongs to the tracker's context; asynchronous,
 * one kernel launch, outside compute().  PFT_ERR_STATE before a reference cloud and a compute(). */
PFT_API int pft_tracker_get_result_cloud(pft_tracker* t, float z_offset, pft_cloud* out);
/* resetTracking */
PFT_API int pft_tracker_reset(pft_tracker* t);
/* likelihood evaluations so far (sum over weight() calls of live particles x model points; counted on the device,
 * the particle count of a KLD tracker never travels to the host) */
PFT_API int pft_tracker_get_eval_count(pft_tracker* t, uint64_t* out);
/* getFitRatio */
PFT_API int pft_tracker_get_fit_ratio(pft_tracker* t, double* out);

/* ---------------------------------------------------------------- reproducibility / parity hooks */
/* Replace the particle set (checkpoint restore, parity tests). */
PFT_API int pft_tracker_set_particles(pft_tracker* t, const pft_particle* p, size_t n);
PFT_API int pft_tracker_set_result(pft_tracker* t, const pft_particle* representative, const pft_particle* motion);
PFT_API int pft_tracker_get_motion(pft_tracker* t, pft_particle* out);
/* Fixed RNG draws (the reference seeds three RNGs with time(0)/rand(), SURVEY A.9): per resample slot
 * (= iteration index within one compute) `stride` selection uniforms, stride x 6 standard normals,
 * stride motion uniforms.  Pass NULLs to return to the on-device Philox generator. */
PFT_API int pft_tracker_inject_draws(pft_tracker* t, const float* u_select, const float* normals6,
                                     const float* u_motion, int slots, int stride);
PFT_API int pft_tracker_seed(pft_tracker* t, uint64_t seed);
/* Stage-level entry points (each is one stage of computeTracking): */
PFT_API int pft_tracker_init_particles(pft_tracker* t);      /* initParticles(true) */
PFT_API int pft_tracker_resample(pft_tracker* t, int slot);  /* resample()          */
PFT_API int pft_tracker_weight(pft_tracker* t);              /* weight() incl. normalizeWeight() */
PFT_API int pft_tracker_update(pft_tracker* t);              /* update()            */
PFT_API int pft_tracker_set_changed(pft_tracker* t, int changed);
/* change detector state: out4 = { change_counter_, tests run so far, point indices the last test reported (-1: no test
 * yet), changed_ } */
PFT_API int pft_tracker_get_change_detector_info(pft_tracker* t, int32_t* out4);
/* Inspection of the last weight(): crop AABB (minx,miny,minz,maxx,maxy,maxz), number of cropped scene
 * points, raw (un-normalised) weights, ancestors chosen by the last resample. */
PFT_API int pft_tracker_get_aabb(pft_tracker* t, float* aabb6);
PFT_API int pft_tracker_get_cropped_count(pft_tracker* t, size_t* n);
PFT_API int pft_tracker_get_raw_weights(pft_tracker* t, float* out, size_t capacity, size_t* n);
PFT_API int pft_tracker_get_ancestors(pft_tracker* t, int32_t* out, size_t capacity, size_t* n);
/* NN results recorded by weight() when PFT_DEBUG_NN = K > 0: for particle < K and every model point (in
 * the order of the reference cloud as given), the index of the nearest scene point IN THE INPUT CLOUD
 * (-1: none inside the crop) and its squared distance. */
PFT_API int pft_tracker_get_nn(pft_tracker* t, int particle, int32_t* idx, float* d2, size_t capacity);
/* Device time in ms of the stages of the last compute(): weight kernel only, whole compute. */
PFT_API int pft_tracker_get_timing(pft_tracker* t, float* weight_kernel_ms, float* compute_ms);
PFT_API int pft_tracker_enable_timing(pft_tracker* t, int on);
/* timing mode: device time in ms of every kernel of the last compute(), in launch order (static name strings) */
PFT_API int pft_tracker_get_kernel_times(pft_tracker* t, const char** names, float* ms, int capacity, int* n);

/* dims[3], level (cell edge = resolution x 2^level), n_cropped, n_cells, use_lists, list_cells of the scene index built by the last weight() */
PFT_API int pft_tracker_get_index_info(pft_tracker* t, int* info8);
/* number of compute() calls served by replaying the captured CUDA graph */
PFT_API int pft_tracker_graph_replays(pft_tracker* t, uint64_t* n);

/* weight() in its three parts with both exchange points exposed (sharded runs without a communicator,
 * used by the single-GPU emulation tests): phase 0 = transforms + this rank's crop box, 1 = index build +
 * coherence of this rank's particles, 2 = normalizeWeight.  The crop box is read/written between 0 and
 * 1, the raw-weight slices ([nranks][slice], particle i -> rank i % nranks, position i / nranks)
 * between 1 and 2.  A tracker attached to peer windows (pft_tracker_peer_attach, or pft_tracker_set_devices
 * after its first compute()) exchanges inside its kernels: it refuses every phase with PFT_ERR_STATE. */
PFT_API int pft_tracker_weight_phase(pft_tracker* t, int phase);
PFT_API int pft_tracker_get_crop_box(pft_tracker* t, float* aabb6);
PFT_API int pft_tracker_set_crop_box(pft_tracker* t, const float* aabb6);
PFT_API int pft_tracker_get_raw_slice(pft_tracker* t, int rank, float* out, size_t capacity, size_t* n);
PFT_API int pft_tracker_set_raw_slice(pft_tracker* t, int rank, const float* in, size_t n);
/* sharding without a communicator: this rank evaluates particles i % nranks == rank */
PFT_API int pft_tracker_set_shard(pft_tracker* t, int nranks, int rank);

/* ---------------------------------------------------------------- multi-GPU (particle sharding) */
/* One process per GPU.  Rank 0 calls pft_comm_get_unique_id and ships the 128 bytes to the other
 * ranks with the host framework's own plumbing (torch.distributed in bench.py); every rank then calls
 * pft_tracker_comm_init (before the first compute).  weight() evaluates only this rank's particles
 * (i % nranks == rank); the crop AABB is all-reduced and the raw weights all-gathered over NCCL/NVLink;
 * resample/normalise/update run replicated from identical draws (same seed or same injected arrays). */
PFT_API int pft_comm_get_unique_id(void* id128);
/* one NCCL communicator per context, shared by its clouds and trackers */
PFT_API int pft_context_comm_init(pft_context* ctx, int nranks, int rank, const void* id128);
PFT_API int pft_context_comm_destroy(pft_context* ctx);
/* NVLink broadcast of a (downsampled) scene cloud from `root`: header + `capacity` points; the point
 * count stays on the device.  Every rank passes the same capacity and root. */
PFT_API int pft_cloud_broadcast(pft_cloud* cloud, size_t capacity, int root);
/* attach the tracker to the context communicator (creates it on first use); detach */
PFT_API int pft_tracker_comm_init(pft_tracker* t, int nranks, int rank, const void* id128);
PFT_API int pft_tracker_comm_destroy(pft_tracker* t);


/* ---------------------------------------------------------------- multi-GPU: NVLink peer exchange */
/* The exchange steps of weight() fused into the producing kernels: every rank owns a window in its HBM
 * that all peers map with CUDA IPC; aabb -> peer stores of the crop box + flag barrier, and normalizeWeight
 * sums this rank's raw weights, stores them straight into every rank's window (it IS the all-gather) and
 * waits on the flag.  No NCCL call is made per frame.  Call order on every rank (one
 * process per GPU, same node): pft_tracker_set_shard (or _comm_init) -> particle numbers ->
 * pft_tracker_peer_export -> the host framework all-gathers the PFT_PEER_HANDLE_BYTES handles in rank
 * order -> pft_tracker_peer_attach -> compute().  Results are bit-identical to the NCCL path and to the
 * unsharded run. */
#define PFT_PEER_HANDLE_BYTES 64
PFT_API int pft_tracker_peer_export(pft_tracker* t, void* handle64);
PFT_API int pft_tracker_peer_attach(pft_tracker* t, const void* handles /* nranks x PFT_PEER_HANDLE_BYTES */);
PFT_API int pft_tracker_peer_detach(pft_tracker* t);

/* Scene distribution by peer stores: ONE rank owns the sensor.  It uploads and downsamples the frame; its
 * push kernel stores the downsampled cloud (points + header) straight into the same cloud of every other
 * rank over NVLink and raises a flag there; the other ranks' streams wait on their flag.  One host->device
 * copy per frame for the whole job, no collective call.  Call order on every rank: pft_cloud_peer_export
 * (the same `capacity` everywhere; fixes the cloud's storage) -> the host framework all-gathers the
 * PFT_CLOUD_PEER_HANDLE_BYTES handles in rank order -> pft_cloud_peer_attach -> per frame the root fills
 * the cloud and EVERY rank calls pft_cloud_peer_broadcast (stream ordered).  The root must not refill the
 * cloud before its peers have finished with the previous scene: a peer-mode tracker loop implies that
 * (the last raw-weight exchange of a frame follows every rank's last read of the scene). */
#define PFT_CLOUD_PEER_HANDLE_BYTES 192
PFT_API int pft_cloud_peer_export(pft_cloud* cloud, size_t capacity, void* handles192);
PFT_API int pft_cloud_peer_attach(pft_cloud* cloud, const void* handles /* nranks x PFT_CLOUD_PEER_HANDLE_BYTES */, int nranks, int rank);
PFT_API int pft_cloud_peer_broadcast(pft_cloud* cloud, int root);
PFT_API int pft_cloud_peer_detach(pft_cloud* cloud);

/* Single-process multi-device mode: ONE tracker object drives n GPUs of the node (the reference is one process:
 * ref src/auto_tracking.cpp).  The tracker becomes rank 0 on devices[0] (= the device of its context); the
 * library creates a follower tracker per further device, shards the particles over them (particle i on rank
 * i % n), maps the exchange windows of weight() directly (cudaDeviceEnablePeerAccess; no IPC, no second
 * process) and copies the model and every frame's scene to the other devices itself.  Must be the first call
 * on a new tracker; the setters called afterwards are forwarded.  compute() enqueues one frame on every
 * device; results are bit-identical to the single-GPU run.  The stage-by-stage API is not forwarded. */
PFT_API int pft_tracker_set_devices(pft_tracker* t, int n, const int* devices);
/* the library-owned tracker of rank 1 .. n-1 (borrowed handle, for the getters: every rank holds the same replicated state) */
PFT_API int pft_tracker_get_follower(pft_tracker* t, int rank, pft_tracker** out);

#ifdef __cplusplus
}
#endif
#endif /* PFT_PFT_H_ */
