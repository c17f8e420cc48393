// pft_api.cu -- C ABI: context, device clouds and the filter entry points (include/pft/pft.h).
//
// Host-side plumbing only; the kernels live in pft_filters.cu / pft_tracker_kernels.cuh.  Everything
// here replaces glue the reference does on the CPU around PCL containers:
//   pft_cloud_upload        pcl::fromPCLPointCloud2 into PointCloud<PointXYZRGBA>  (ref: src/auto_tracking.cpp:619-622)
//   pft_cloud_upload_depth_image  depth_image_proc/point_cloud_xyzrgb, which computes the points topic of ref :775
//   pft_cloud_upload_depth_images  the same per calibrated camera + transformPointCloud(cloud_k, T_k), scene += cloud_k
//   pft_cloud_upload_depth_images_enc  the same in every encoding of point_cloud_xyzrgb / point_cloud_xyz
//   pft_cloud_upload_depth_images_reg  the same behind depth_image_proc/register, for unregistered depth images
//   pft_passthrough         filterPassThrough                                       (ref: src/auto_tracking.cpp:536-547)
//   pft_passthrough_voxel_grid  filterPassThrough + gridSampleApprox / gridSample   (ref: src/auto_tracking.cpp:637, :683, :641)
//   pft_prepare_model       removeZeroPoints + centroid + translate + gridSample    (ref: src/auto_tracking.cpp:656-674)
//   pft_transform_cloud     pcl(_ros)::transformPointCloud into / out of the base frame (ref: src/create_model.cpp:107-123, :184-204)
//   pft_remove_zero_points  removeZeroPoints                                        (ref: src/create_model.cpp:59-77)
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include "pft_internal.h"

namespace pft {

static thread_local char g_err[512] = "";
std::atomic<unsigned long long> g_launch_count{0};
static std::atomic<unsigned long long> g_cloud_serial{0};

void set_last_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int DevBuf::reserve(size_t need) {
  if (need <= bytes) return PFT_OK;
  // grow geometrically so that a slowly growing frame does not reallocate every call
  size_t want = need + need / 4 + 256;
  void* np = nullptr;
  PFT_CUDA_TRY(cudaMalloc(&np, want));
  if (p) {
    // callers never rely on the old contents across a reserve() except clouds, which copy explicitly
    cudaFree(p);
  }
  p = np;
  bytes = want;
  return PFT_OK;
}
void DevBuf::release() {
  if (p) cudaFree(p);
  p = nullptr;
  bytes = 0;
}

}  // namespace pft

int pft_cloud::ensure(size_t cap) {
  int rc = hdr.reserve(sizeof(pft::CloudHeader));
  if (rc) return rc;
  if (peer_exported && cap * sizeof(float4) > pts.bytes) {
    pft::set_last_error("the cloud is mapped by its peers with room for %zu points; %zu do not fit (export it with a larger capacity)", peer_capacity, cap);
    return PFT_ERR_CAPACITY;
  }
  if (cap > capacity || !pts.p) {
    rc = pts.reserve((cap ? cap : 1) * sizeof(float4));
    if (rc) return rc;
  }
  capacity = cap;
  return PFT_OK;
}

// Orders the context stream after an asynchronous upload into this cloud (no host wait).
int pft_cloud::join_upload() const {
  if (!upload_pending) return PFT_OK;
  PFT_CUDA_TRY(cudaStreamWaitEvent(ctx->stream, ready, 0));
  upload_pending = false;
  return PFT_OK;
}

using namespace pft;

namespace {

// Common front of the asynchronous uploads: the copy stream, ordered after everything the context stream holds so far
// (earlier readers of the cloud that is about to be overwritten).
int begin_async_upload(pft_cloud* c, size_t n, cudaStream_t* cs) {
  pft_context* ctx = c->ctx;
  PFT_CUDA_TRY(cudaSetDevice(ctx->device));
  if (!ctx->copy_stream) {
    PFT_CUDA_TRY(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    PFT_CUDA_TRY(cudaEventCreateWithFlags(&ctx->copy_fence, cudaEventDisableTiming));
  }
  if (!c->ready) PFT_CUDA_TRY(cudaEventCreateWithFlags(&c->ready, cudaEventDisableTiming));
  int rc = c->ensure(n);
  if (rc) return rc;
  PFT_CUDA_TRY(cudaEventRecord(ctx->copy_fence, ctx->stream));
  PFT_CUDA_TRY(cudaStreamWaitEvent(ctx->copy_stream, ctx->copy_fence, 0));
  *cs = ctx->copy_stream;
  return PFT_OK;
}

int end_async_upload(pft_cloud* c, size_t n, cudaStream_t cs) {
  int rc = launch_set_header(cs, c->d_hdr(), (int)n);
  if (rc) return rc;
  PFT_CUDA_TRY(cudaEventRecord(c->ready, cs));
  c->upload_pending = true;
  c->written((long long)n);
  return PFT_OK;
}

int check_pointcloud2_layout(size_t n, uint32_t width, uint32_t point_step, uint32_t row_step, int32_t off_x, int32_t off_y, int32_t off_z, int32_t off_rgb,
                             int is_bigendian) {
  if (n > 0x7fffffffull) { set_last_error("cloud too large"); return PFT_ERR_INVALID; }
  if (is_bigendian) { set_last_error("big-endian PointCloud2 data is not supported"); return PFT_ERR_INVALID; }
  if (n) {
    if (point_step < 12 || (point_step & 3) || (row_step & 3) || (size_t)row_step < (size_t)width * point_step) {
      set_last_error("bad PointCloud2 strides: point_step %u, row_step %u, width %u (4-byte multiples, row_step >= width * point_step)", point_step, row_step, width);
      return PFT_ERR_INVALID;
    }
    const int32_t offs[4] = {off_x, off_y, off_z, off_rgb};
    for (int k = 0; k < 4; ++k) {
      const bool optional = k == 3 && offs[k] < 0;  // no colour field: rgba = 0
      if (!optional && (offs[k] < 0 || (offs[k] & 3) || (uint32_t)offs[k] + 4 > point_step)) {
        set_last_error("bad PointCloud2 field offset %d (float32 x, y, z and the packed rgb(a) word, 4-byte aligned inside point_step %u)", offs[k], point_step);
        return PFT_ERR_INVALID;
      }
    }
  }
  return PFT_OK;
}

// A depth + colour frame of one or more cameras, checked and laid out for one staging buffer: per camera its depth
// rows, then its colour rows (none for depth alone), each from a 16-byte aligned offset.  Only the bytes an image
// occupies are copied, (height - 1) * step + width * bytes per pixel, so a caller's view into a larger buffer is never
// read past its last pixel.  `cams` holds the cameras with pixels, in order, as depth_image_kernel reads them; their points follow
// each other in the cloud.
// A registered camera (pft_cloud_upload_depth_images_reg) copies its raw depth image to its own slot instead, and the
// register kernels write the registered image to its depth slot; the z-buffers of all registered cameras follow the
// images, in one span that one memset clears.
struct DepthImageFrame {
  DepthCameras cams;
  const void* depth[PFT_MAX_DEPTH_CAMERAS];  // NULL: a registered camera, nothing is copied
  const void* bgr[PFT_MAX_DEPTH_CAMERAS];
  size_t depth_bytes[PFT_MAX_DEPTH_CAMERAS], bgr_bytes[PFT_MAX_DEPTH_CAMERAS];
  int n;               // cameras with pixels
  size_t points;       // points of the cloud
  size_t staging;      // bytes of the staging buffer
  RegCameras reg;      // cameras 0 .. n-1, `registered` set for those with a depth_to_colour matrix
  const void* raw[PFT_MAX_DEPTH_CAMERAS];
  size_t raw_bytes[PFT_MAX_DEPTH_CAMERAS];
  int n_reg;           // registered cameras
  size_t zbuf_off, zbuf_bytes;
};

inline size_t align16(size_t b) { return (b + 15) & ~(size_t)15; }

// Bytes per pixel of a colour encoding (pft_colour_encoding; 0: no colour image), -1 for an unknown one.
int colour_bytes(int32_t enc) {
  switch (enc) {
    case PFT_COLOUR_BGR8: case PFT_COLOUR_RGB8: return 3;
    case PFT_COLOUR_BGRA8: case PFT_COLOUR_RGBA8: return 4;
    case PFT_COLOUR_MONO8: return 1;
    case PFT_COLOUR_NONE: return 0;
    default: return -1;
  }
}

// Checks camera `cam` and appends it to `f`.  `cam` < 0: the single-image call, whose messages name no camera.
int check_depth_image(const char* fn, int cam, const pft_depth_camera_enc& e, DepthImageFrame* f) {
  const pft_depth_camera& c = e.cam;
  char who[24] = "";
  if (cam >= 0) snprintf(who, sizeof(who), ": camera %d", cam);
  if (e.depth_encoding != PFT_DEPTH_16UC1 && e.depth_encoding != PFT_DEPTH_32FC1) {
    set_last_error("%s%s: unknown depth encoding %d (PFT_DEPTH_16UC1 or PFT_DEPTH_32FC1)", fn, who, (int)e.depth_encoding);
    return PFT_ERR_INVALID;
  }
  const int cbytes = colour_bytes(e.colour_encoding);
  if (cbytes < 0) { set_last_error("%s%s: unknown colour encoding %d (PFT_COLOUR_BGR8 .. PFT_COLOUR_NONE)", fn, who, (int)e.colour_encoding); return PFT_ERR_INVALID; }
  const bool metres = e.depth_encoding == PFT_DEPTH_32FC1;
  const unsigned int dbytes = metres ? 4 : 2;
  const size_t n = (size_t)c.width * c.height;
  if (n > 0x7fffffffull) { set_last_error("%s%s: image too large", fn, who); return PFT_ERR_INVALID; }
  if (!(c.fx != 0.0 && c.fy != 0.0 && isfinite(c.fx) && isfinite(c.fy) && isfinite(c.cx) && isfinite(c.cy))) {
    set_last_error("%s%s: bad intrinsics fx %g fy %g cx %g cy %g (fx, fy finite and non-zero; cx, cy finite)", fn, who, c.fx, c.fy, c.cx, c.cy);
    return PFT_ERR_INVALID;
  }
  if (c.m12) {
    for (int i = 0; i < 12; ++i) {
      if (!isfinite(c.m12[i])) { set_last_error("%s%s: matrix entry %d is %g (must be finite)", fn, who, i, (double)c.m12[i]); return PFT_ERR_INVALID; }
    }
  }
  if (!n) return PFT_OK;
  if (!c.depth || (cbytes && !c.bgr)) { set_last_error("%s%s: null image", fn, who); return PFT_ERR_INVALID; }
  if (c.depth_step % dbytes || (size_t)c.depth_step < (size_t)c.width * dbytes || (size_t)c.bgr_step < (size_t)c.width * cbytes) {
    set_last_error("%s%s: bad steps: depth %u (a multiple of %u, >= %u * width), colour %u (>= %d * width), width %u", fn, who, c.depth_step, dbytes,
                   dbytes, c.bgr_step, cbytes, c.width);
    return PFT_ERR_INVALID;
  }
  if (f->points + n > 0x7fffffffull) { set_last_error("%s: 2^31 pixels or more in total (at camera %d)", fn, cam); return PFT_ERR_INVALID; }
  const int i = f->n++;
  DepthCamera& k = f->cams.cam[i];
  f->depth[i] = c.depth;
  f->bgr[i] = cbytes ? c.bgr : nullptr;
  f->depth_bytes[i] = (size_t)(c.height - 1) * c.depth_step + (size_t)c.width * dbytes;
  f->bgr_bytes[i] = cbytes ? (size_t)(c.height - 1) * c.bgr_step + (size_t)c.width * cbytes : 0;
  k.depth_off = f->staging;
  k.bgr_off = align16(k.depth_off + f->depth_bytes[i]);
  f->staging = align16(k.bgr_off + f->bgr_bytes[i]);
  k.out_off = f->points;
  f->points += n;
  k.width = c.width;
  k.height = c.height;
  k.depth_step = c.depth_step;
  k.bgr_step = cbytes ? c.bgr_step : 0;
  k.depth_enc = e.depth_encoding;
  k.colour_enc = e.colour_encoding;
  // the constants of depth_image_proc::convert<T>: float centre, float(unit / f) with the double unit
  // DepthTraits<T>::toMeters(T(1)), double(0.001f) for uint16_t millimetres and 1 for float metres
  const double unit = metres ? 1.0 : (double)0.001f;
  k.cx = (float)c.cx;
  k.cy = (float)c.cy;
  k.kx = (float)(unit / c.fx);
  k.ky = (float)(unit / c.fy);
  k.has_m = c.m12 != nullptr;
  if (c.m12) memcpy(k.m, c.m12, sizeof(k.m));
  return PFT_OK;
}

// Checks camera `cam` of a pft_cloud_upload_depth_images_reg call and appends it to `f`: check_depth_image for the
// colour side and the output, as if the registered image were its depth image, then the registration fields.
int check_registration(const char* fn, int cam, const pft_depth_camera_reg& r, DepthImageFrame* f) {
  if (!r.depth_to_colour) return check_depth_image(fn, cam, r.cam, f);
  pft_depth_camera_enc e = r.cam;
  const unsigned int dbytes = e.depth_encoding == PFT_DEPTH_32FC1 ? 4 : 2;
  e.cam.depth = f;  // the registered image: written on the device, never null, packed rows
  e.cam.depth_step = e.cam.width * dbytes;
  const int before = f->n;
  int rc = check_depth_image(fn, cam, e, f);
  if (rc) return rc;
  for (int i = 0; i < 12; ++i) {
    if (!isfinite(r.depth_to_colour[i])) { set_last_error("%s: camera %d: depth_to_colour entry %d is %g (must be finite)", fn, cam, i, r.depth_to_colour[i]); return PFT_ERR_INVALID; }
  }
  if (!(r.depth_fx != 0.0 && r.depth_fy != 0.0 && isfinite(r.depth_fx) && isfinite(r.depth_fy) && isfinite(r.depth_cx) && isfinite(r.depth_cy) &&
        isfinite(r.depth_tx) && isfinite(r.depth_ty) && isfinite(r.colour_tx) && isfinite(r.colour_ty))) {
    set_last_error("%s: camera %d: bad registration intrinsics: depth fx %g fy %g cx %g cy %g Tx %g Ty %g, colour Tx %g Ty %g (depth fx, fy finite and "
                   "non-zero; the rest finite)", fn, cam, r.depth_fx, r.depth_fy, r.depth_cx, r.depth_cy, r.depth_tx, r.depth_ty, r.colour_tx, r.colour_ty);
    return PFT_ERR_INVALID;
  }
  if (r.fill_upsampling != 0 && r.fill_upsampling != 1) { set_last_error("%s: camera %d: fill_upsampling %d (0 or 1)", fn, cam, (int)r.fill_upsampling); return PFT_ERR_INVALID; }
  const size_t dn = (size_t)r.depth_width * r.depth_height;
  if (dn > 0x7fffffffull) { set_last_error("%s: camera %d: depth image too large", fn, cam); return PFT_ERR_INVALID; }
  if (dn && !r.cam.cam.depth) { set_last_error("%s: camera %d: null depth image", fn, cam); return PFT_ERR_INVALID; }
  if (dn && (r.cam.cam.depth_step % dbytes || (size_t)r.cam.cam.depth_step < (size_t)r.depth_width * dbytes)) {
    set_last_error("%s: camera %d: bad depth step %u (a multiple of %u, >= %u * depth_width %u)", fn, cam, r.cam.cam.depth_step, dbytes, dbytes, r.depth_width);
    return PFT_ERR_INVALID;
  }
  if (f->n == before) return PFT_OK;  // no colour pixels: the camera adds nothing
  const int i = f->n - 1;
  f->depth[i] = nullptr;
  f->raw[i] = r.cam.cam.depth;
  f->raw_bytes[i] = dn ? (size_t)(r.depth_height - 1) * r.cam.cam.depth_step + (size_t)r.depth_width * dbytes : 0;
  RegCamera& k = f->reg.cam[i];
  k.raw_off = f->staging;
  f->staging = align16(k.raw_off + f->raw_bytes[i]);
  k.reg_off = f->cams.cam[i].depth_off;
  k.depth_width = dn ? r.depth_width : 0;
  k.depth_height = dn ? r.depth_height : 0;
  k.depth_step = r.cam.cam.depth_step;
  k.width = e.cam.width;
  k.height = e.cam.height;
  k.registered = 1;
  k.depth_enc = e.depth_encoding;
  k.fill = r.fill_upsampling;
  k.inv_fx = 1.0 / r.depth_fx;
  k.inv_fy = 1.0 / r.depth_fy;
  k.cx = r.depth_cx; k.cy = r.depth_cy; k.tx = r.depth_tx; k.ty = r.depth_ty;
  k.rgb_fx = e.cam.fx; k.rgb_fy = e.cam.fy; k.rgb_cx = e.cam.cx; k.rgb_cy = e.cam.cy; k.rgb_tx = r.colour_tx; k.rgb_ty = r.colour_ty;
  memcpy(k.m, r.depth_to_colour, sizeof(k.m));
  ++f->n_reg;
  return PFT_OK;
}

// The z-buffers of the registered cameras, after every image of the frame: per camera a uint64 key and a uint32 reset
// per colour pixel.
void place_zbuffers(DepthImageFrame* f) {
  f->zbuf_off = align16(f->staging);
  size_t off = f->zbuf_off;
  for (int i = 0; i < f->n; ++i) {
    RegCamera& k = f->reg.cam[i];
    if (!k.registered) continue;
    const size_t px = (size_t)k.width * k.height;
    k.key_off = off;
    k.reset_off = off + px * sizeof(unsigned long long);
    off = align16(k.reset_off + px * sizeof(unsigned int));
  }
  f->zbuf_bytes = off - f->zbuf_off;
  f->staging = off;
}

int check_depth_cameras(const char* fn, const pft_depth_camera_enc* cams, int n, DepthImageFrame* f) {
  if (!cams) { set_last_error("%s: null cameras", fn); return PFT_ERR_INVALID; }
  if (n < 1 || n > PFT_MAX_DEPTH_CAMERAS) { set_last_error("%s: %d cameras (1 to %d)", fn, n, PFT_MAX_DEPTH_CAMERAS); return PFT_ERR_INVALID; }
  for (int k = 0; k < n; ++k) {
    int rc = check_depth_image(fn, k, cams[k], f);
    if (rc) return rc;
  }
  return PFT_OK;
}

// The frame's copies (two per camera) and its one conversion launch, on stream `s` through `staging`.
int enqueue_depth_image(cudaStream_t s, pft::DevBuf& staging, pft_cloud* c, const DepthImageFrame& f) {
  if (!f.n) return PFT_OK;
  int rc = staging.reserve(f.staging);
  if (rc) return rc;
  unsigned char* base = staging.as<unsigned char>();
  for (int k = 0; k < f.n; ++k) {
    if (f.depth[k]) PFT_CUDA_TRY(cudaMemcpyAsync(base + f.cams.cam[k].depth_off, f.depth[k], f.depth_bytes[k], cudaMemcpyHostToDevice, s));
    if (f.raw_bytes[k]) PFT_CUDA_TRY(cudaMemcpyAsync(base + f.reg.cam[k].raw_off, f.raw[k], f.raw_bytes[k], cudaMemcpyHostToDevice, s));
    if (f.bgr_bytes[k]) PFT_CUDA_TRY(cudaMemcpyAsync(base + f.cams.cam[k].bgr_off, f.bgr[k], f.bgr_bytes[k], cudaMemcpyHostToDevice, s));
  }
  if (f.n_reg) {
    PFT_CUDA_TRY(cudaMemsetAsync(base + f.zbuf_off, 0, f.zbuf_bytes, s));
    if ((rc = launch_register_depth(s, base, f.reg, f.n))) return rc;
  }
  return launch_depth_image(s, base, c->d_pts(), f.cams, f.n);
}

// A checked frame into `c`: on the context stream through its staging buffer, or (asynchronous) on the copy stream
// through the cloud's own.
int upload_depth_frame(pft_cloud* c, const DepthImageFrame& f, bool asynchronous) {
  int rc;
  if (asynchronous) {
    cudaStream_t cs = nullptr;
    if ((rc = begin_async_upload(c, f.points, &cs))) return rc;
    if ((rc = enqueue_depth_image(cs, c->raw_staging, c, f))) return rc;
    return end_async_upload(c, f.points, cs);
  }
  pft_context* ctx = c->ctx;
  PFT_CUDA_TRY(cudaSetDevice(ctx->device));
  if ((rc = c->join_upload())) return rc;
  if ((rc = c->ensure(f.points))) return rc;
  cudaStream_t s = ctx->stream;
  if ((rc = enqueue_depth_image(s, ctx->staging, c, f))) return rc;
  if ((rc = launch_set_header(s, c->d_hdr(), (int)f.points))) return rc;
  c->written((long long)f.points);
  return PFT_OK;
}

int upload_depth_image(const char* fn, pft_cloud* c, const void* depth, uint32_t depth_step, const void* bgr, uint32_t bgr_step, uint32_t width,
                       uint32_t height, double fx, double fy, double cx, double cy, bool asynchronous) {
  if (!c) { set_last_error("%s: null cloud", fn); return PFT_ERR_INVALID; }
  const pft_depth_camera_enc cam = {{depth, depth_step, bgr, bgr_step, width, height, fx, fy, cx, cy, nullptr}, PFT_DEPTH_16UC1, PFT_COLOUR_BGR8};
  DepthImageFrame f{};
  int rc = check_depth_image(fn, -1, cam, &f);
  if (rc) return rc;
  return upload_depth_frame(c, f, asynchronous);
}

int upload_depth_images(const char* fn, pft_cloud* c, const pft_depth_camera_enc* cams, int n, bool asynchronous) {
  if (!c) { set_last_error("%s: null cloud", fn); return PFT_ERR_INVALID; }
  DepthImageFrame f{};
  int rc = check_depth_cameras(fn, cams, n, &f);
  if (rc) return rc;
  return upload_depth_frame(c, f, asynchronous);
}

int upload_depth_images_reg(const char* fn, pft_cloud* c, const pft_depth_camera_reg* cams, int n, bool asynchronous) {
  if (!c) { set_last_error("%s: null cloud", fn); return PFT_ERR_INVALID; }
  if (!cams) { set_last_error("%s: null cameras", fn); return PFT_ERR_INVALID; }
  if (n < 1 || n > PFT_MAX_DEPTH_CAMERAS) { set_last_error("%s: %d cameras (1 to %d)", fn, n, PFT_MAX_DEPTH_CAMERAS); return PFT_ERR_INVALID; }
  DepthImageFrame f{};
  for (int k = 0; k < n; ++k) {
    int rc = check_registration(fn, k, cams[k], &f);
    if (rc) return rc;
  }
  place_zbuffers(&f);
  return upload_depth_frame(c, f, asynchronous);
}

// The cameras of pft_cloud_upload_depth_images(_async): 16UC1 depth, bgr8 colour.
int upload_depth_images_bgr8(const char* fn, pft_cloud* c, const pft_depth_camera* cams, int n, bool asynchronous) {
  pft_depth_camera_enc enc[PFT_MAX_DEPTH_CAMERAS];
  const bool valid = cams && n >= 1 && n <= PFT_MAX_DEPTH_CAMERAS;  // otherwise check_depth_cameras rejects the call
  for (int k = 0; valid && k < n; ++k) enc[k] = {cams[k], PFT_DEPTH_16UC1, PFT_COLOUR_BGR8};
  return upload_depth_images(fn, c, cams ? enc : nullptr, n, asynchronous);
}

}  // namespace

extern "C" {

const char* pft_last_error(void) { return g_err; }
const char* pft_version(void) { return "pft 0.1 (sm_100a)"; }

int pft_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

int pft_context_create(int device, pft_context** out) {
  if (!out) { set_last_error("pft_context_create: null out"); return PFT_ERR_INVALID; }
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    cudaGetLastError();
    set_last_error("no CUDA device available (%s); this library has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "count = 0");
    return PFT_ERR_CUDA;
  }
  if (device < 0 || device >= n) { set_last_error("device %d out of range [0,%d)", device, n); return PFT_ERR_INVALID; }
  PFT_CUDA_TRY(cudaSetDevice(device));
  pft_context* c = new pft_context();
  c->device = device;
  cudaDeviceProp prop;
  PFT_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  c->sm_count = prop.multiProcessorCount;
  PFT_CUDA_TRY(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  c->pinned_bytes = 4096;
  PFT_CUDA_TRY(cudaHostAlloc(&c->pinned, c->pinned_bytes, cudaHostAllocDefault));
  *out = c;
  return PFT_OK;
}

void pft_context_destroy(pft_context* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  release_replicas_in(c);
  pft_context_comm_destroy(c);
  pft::DevBuf* bufs[] = {&c->k1_keys, &c->k1_first, &c->k1_vid, &c->k1_slot_of, &c->k1_acc_xyz, &c->k1_acc_rgbc, &c->k1_blk, &c->staging, &c->tmp_cloud_pts, &c->tmp_hdr, &c->tmp_f,
                         &c->cl_grid, &c->cl_cells, &c->cl_work, &c->cl_sel};
  for (auto* b : bufs) b->release();
  if (c->pinned) cudaFreeHost(c->pinned);
  if (c->batch_fork) cudaEventDestroy(c->batch_fork);
  if (c->copy_stream) { cudaStreamSynchronize(c->copy_stream); cudaStreamDestroy(c->copy_stream); }
  if (c->copy_fence) cudaEventDestroy(c->copy_fence);
  for (int k = 0; k < pft_context::kK1Graphs; ++k) if (c->k1_exec[k]) cudaGraphExecDestroy(c->k1_exec[k]);
  cudaStreamDestroy(c->stream);
  delete c;
}

int pft_context_synchronize(pft_context* c) {
  if (!c) { set_last_error("null context"); return PFT_ERR_INVALID; }
  PFT_CUDA_TRY(cudaStreamSynchronize(c->stream));
  return PFT_OK;
}

void* pft_context_stream(pft_context* c) { return c ? (void*)c->stream : nullptr; }

int pft_host_alloc(void** ptr, size_t bytes) {
  if (!ptr) { set_last_error("null ptr"); return PFT_ERR_INVALID; }
  PFT_CUDA_TRY(cudaHostAlloc(ptr, bytes ? bytes : 1, cudaHostAllocDefault));
  return PFT_OK;
}
int pft_host_free(void* ptr) {
  if (ptr) PFT_CUDA_TRY(cudaFreeHost(ptr));
  return PFT_OK;
}

uint64_t pft_kernel_launch_count(void) { return (uint64_t)g_launch_count.load(); }

// ------------------------------------------------------------------ clouds
int pft_cloud_create(pft_context* ctx, pft_cloud** out) {
  if (!ctx || !out) { set_last_error("pft_cloud_create: null argument"); return PFT_ERR_INVALID; }
  PFT_CUDA_TRY(cudaSetDevice(ctx->device));
  pft_cloud* c = new pft_cloud();
  c->ctx = ctx;
  c->serial = ++g_cloud_serial;
  int rc = c->ensure(0);
  if (rc) { delete c; return rc; }
  rc = launch_set_header(ctx->stream, c->d_hdr(), 0);
  if (rc) { delete c; return rc; }
  c->host_n = 0;
  *out = c;
  return PFT_OK;
}

void pft_cloud_destroy(pft_cloud* c) {
  if (!c) return;
  cudaSetDevice(c->ctx->device);
  cudaStreamSynchronize(c->ctx->stream);
  if (c->ready) { cudaEventSynchronize(c->ready); cudaEventDestroy(c->ready); }
  release_replicas_of(c);
  pft_cloud_peer_detach(c);
  c->pts.release();
  c->hdr.release();
  c->raw_staging.release();
  delete c;
}

int pft_cloud_upload(pft_cloud* c, const void* host_points, size_t n, int layout) {
  if (!c || (n && !host_points)) { set_last_error("pft_cloud_upload: null argument"); return PFT_ERR_INVALID; }
  if (layout != PFT_LAYOUT_PACKED16 && layout != PFT_LAYOUT_PCL32) { set_last_error("unknown layout %d", layout); return PFT_ERR_INVALID; }
  if (n > 0x7fffffffull) { set_last_error("cloud too large"); return PFT_ERR_INVALID; }
  pft_context* ctx = c->ctx;
  PFT_CUDA_TRY(cudaSetDevice(ctx->device));
  int rc = c->join_upload();
  if (rc) return rc;
  if ((rc = c->ensure(n))) return rc;
  cudaStream_t s = ctx->stream;
  if (n) {
    if (layout == PFT_LAYOUT_PACKED16) {
      PFT_CUDA_TRY(cudaMemcpyAsync(c->d_pts(), host_points, n * sizeof(float4), cudaMemcpyHostToDevice, s));
    } else {
      // 32-byte pcl::PointXYZRGBA records: copy raw, repack to float4 {x,y,z,rgba} on the device
      if ((rc = ctx->staging.reserve(n * 32))) return rc;
      PFT_CUDA_TRY(cudaMemcpyAsync(ctx->staging.p, host_points, n * 32, cudaMemcpyHostToDevice, s));
      if ((rc = launch_unpack_pcl32(s, ctx->staging.p, c->d_pts(), n))) return rc;
    }
  }
  if ((rc = launch_set_header(s, c->d_hdr(), (int)n))) return rc;
  c->written((long long)n);
  return PFT_OK;
}

int pft_cloud_upload_pointcloud2(pft_cloud* c, const void* data, uint32_t width, uint32_t height, uint32_t point_step, uint32_t row_step,
                                 int32_t off_x, int32_t off_y, int32_t off_z, int32_t off_rgb, int is_bigendian) {
  if (!c) { set_last_error("pft_cloud_upload_pointcloud2: null cloud"); return PFT_ERR_INVALID; }
  const size_t n = (size_t)width * height;
  if (n && !data) { set_last_error("pft_cloud_upload_pointcloud2: null data"); return PFT_ERR_INVALID; }
  int rc = check_pointcloud2_layout(n, width, point_step, row_step, off_x, off_y, off_z, off_rgb, is_bigendian);
  if (rc) return rc;
  pft_context* ctx = c->ctx;
  PFT_CUDA_TRY(cudaSetDevice(ctx->device));
  if ((rc = c->join_upload())) return rc;
  if ((rc = c->ensure(n))) return rc;
  cudaStream_t s = ctx->stream;
  if (n) {
    const size_t bytes = (size_t)row_step * height;
    if ((rc = ctx->staging.reserve(bytes))) return rc;
    PFT_CUDA_TRY(cudaMemcpyAsync(ctx->staging.p, data, bytes, cudaMemcpyHostToDevice, s));
    if ((rc = launch_unpack_pointcloud2(s, ctx->staging.p, c->d_pts(), width, height, point_step, row_step, off_x, off_y, off_z, off_rgb))) return rc;
  }
  if ((rc = launch_set_header(s, c->d_hdr(), (int)n))) return rc;
  c->written((long long)n);
  return PFT_OK;
}

int pft_cloud_upload_async(pft_cloud* c, const void* host_points, size_t n, int layout) {
  if (!c || (n && !host_points)) { set_last_error("pft_cloud_upload_async: null argument"); return PFT_ERR_INVALID; }
  if (layout != PFT_LAYOUT_PACKED16 && layout != PFT_LAYOUT_PCL32) { set_last_error("unknown layout %d", layout); return PFT_ERR_INVALID; }
  if (n > 0x7fffffffull) { set_last_error("cloud too large"); return PFT_ERR_INVALID; }
  cudaStream_t cs = nullptr;
  int rc = begin_async_upload(c, n, &cs);
  if (rc) return rc;
  if (n) {
    if (layout == PFT_LAYOUT_PACKED16) {
      PFT_CUDA_TRY(cudaMemcpyAsync(c->d_pts(), host_points, n * sizeof(float4), cudaMemcpyHostToDevice, cs));
    } else {
      if ((rc = c->raw_staging.reserve(n * 32))) return rc;
      PFT_CUDA_TRY(cudaMemcpyAsync(c->raw_staging.p, host_points, n * 32, cudaMemcpyHostToDevice, cs));
      if ((rc = launch_unpack_pcl32(cs, c->raw_staging.p, c->d_pts(), n))) return rc;
    }
  }
  return end_async_upload(c, n, cs);
}

int pft_cloud_upload_pointcloud2_async(pft_cloud* c, const void* data, uint32_t width, uint32_t height, uint32_t point_step, uint32_t row_step,
                                       int32_t off_x, int32_t off_y, int32_t off_z, int32_t off_rgb, int is_bigendian) {
  if (!c) { set_last_error("pft_cloud_upload_pointcloud2_async: null cloud"); return PFT_ERR_INVALID; }
  const size_t n = (size_t)width * height;
  if (n && !data) { set_last_error("pft_cloud_upload_pointcloud2_async: null data"); return PFT_ERR_INVALID; }
  int rc = check_pointcloud2_layout(n, width, point_step, row_step, off_x, off_y, off_z, off_rgb, is_bigendian);
  if (rc) return rc;
  cudaStream_t cs = nullptr;
  if ((rc = begin_async_upload(c, n, &cs))) return rc;
  if (n) {
    const size_t bytes = (size_t)row_step * height;
    if ((rc = c->raw_staging.reserve(bytes))) return rc;
    PFT_CUDA_TRY(cudaMemcpyAsync(c->raw_staging.p, data, bytes, cudaMemcpyHostToDevice, cs));
    if ((rc = launch_unpack_pointcloud2(cs, c->raw_staging.p, c->d_pts(), width, height, point_step, row_step, off_x, off_y, off_z, off_rgb))) return rc;
  }
  return end_async_upload(c, n, cs);
}

int pft_cloud_upload_depth_image(pft_cloud* c, const void* depth, uint32_t depth_step, const void* bgr, uint32_t bgr_step, uint32_t width,
                                 uint32_t height, double fx, double fy, double cx, double cy) {
  return upload_depth_image("pft_cloud_upload_depth_image", c, depth, depth_step, bgr, bgr_step, width, height, fx, fy, cx, cy, false);
}

int pft_cloud_upload_depth_image_async(pft_cloud* c, const void* depth, uint32_t depth_step, const void* bgr, uint32_t bgr_step, uint32_t width,
                                       uint32_t height, double fx, double fy, double cx, double cy) {
  return upload_depth_image("pft_cloud_upload_depth_image_async", c, depth, depth_step, bgr, bgr_step, width, height, fx, fy, cx, cy, true);
}

int pft_cloud_upload_depth_images(pft_cloud* c, const pft_depth_camera* cams, int n) {
  return upload_depth_images_bgr8("pft_cloud_upload_depth_images", c, cams, n, false);
}

int pft_cloud_upload_depth_images_async(pft_cloud* c, const pft_depth_camera* cams, int n) {
  return upload_depth_images_bgr8("pft_cloud_upload_depth_images_async", c, cams, n, true);
}

int pft_cloud_upload_depth_images_enc(pft_cloud* c, const pft_depth_camera_enc* cams, int n) {
  return upload_depth_images("pft_cloud_upload_depth_images_enc", c, cams, n, false);
}

int pft_cloud_upload_depth_images_enc_async(pft_cloud* c, const pft_depth_camera_enc* cams, int n) {
  return upload_depth_images("pft_cloud_upload_depth_images_enc_async", c, cams, n, true);
}

int pft_cloud_upload_depth_images_reg(pft_cloud* c, const pft_depth_camera_reg* cams, int n) {
  return upload_depth_images_reg("pft_cloud_upload_depth_images_reg", c, cams, n, false);
}

int pft_cloud_upload_depth_images_reg_async(pft_cloud* c, const pft_depth_camera_reg* cams, int n) {
  return upload_depth_images_reg("pft_cloud_upload_depth_images_reg_async", c, cams, n, true);
}

int pft_cloud_wait_upload(pft_cloud* c) {
  if (!c) { set_last_error("pft_cloud_wait_upload: null cloud"); return PFT_ERR_INVALID; }
  PFT_CUDA_TRY(cudaSetDevice(c->ctx->device));
  return c->join_upload();
}

int pft_cloud_size(pft_cloud* c, size_t* n) {
  if (!c || !n) { set_last_error("pft_cloud_size: null argument"); return PFT_ERR_INVALID; }
  { int jrc = c->join_upload(); if (jrc) return jrc; }  // every consumer that sizes its work from the cloud passes here
  if (c->host_n < 0) {
    pft_context* ctx = c->ctx;
    PFT_CUDA_TRY(cudaSetDevice(ctx->device));
    PFT_CUDA_TRY(cudaMemcpyAsync(ctx->pinned, c->d_hdr(), sizeof(CloudHeader), cudaMemcpyDeviceToHost, ctx->stream));
    PFT_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    c->host_n = reinterpret_cast<CloudHeader*>(ctx->pinned)->n;
  }
  *n = (size_t)c->host_n;
  return PFT_OK;
}

int pft_cloud_download(pft_cloud* c, void* host_points, size_t capacity, int layout, size_t* n_out) {
  if (!c) { set_last_error("pft_cloud_download: null cloud"); return PFT_ERR_INVALID; }
  if (layout != PFT_LAYOUT_PACKED16 && layout != PFT_LAYOUT_PCL32) { set_last_error("unknown layout %d", layout); return PFT_ERR_INVALID; }
  size_t n = 0;
  int rc = pft_cloud_size(c, &n);
  if (rc) return rc;
  if (n_out) *n_out = n;
  if (n > capacity) { set_last_error("pft_cloud_download: %zu points, capacity %zu", n, capacity); return PFT_ERR_CAPACITY; }
  if (n == 0) return PFT_OK;
  if (!host_points) { set_last_error("pft_cloud_download: null buffer"); return PFT_ERR_INVALID; }
  pft_context* ctx = c->ctx;
  cudaStream_t s = ctx->stream;
  if ((rc = c->join_upload())) return rc;
  if (layout == PFT_LAYOUT_PACKED16) {
    PFT_CUDA_TRY(cudaMemcpyAsync(host_points, c->d_pts(), n * sizeof(float4), cudaMemcpyDeviceToHost, s));
  } else {
    if ((rc = ctx->staging.reserve(n * 32))) return rc;
    if ((rc = launch_pack_pcl32(s, c->d_pts(), ctx->staging.p, n))) return rc;
    PFT_CUDA_TRY(cudaMemcpyAsync(host_points, ctx->staging.p, n * 32, cudaMemcpyDeviceToHost, s));
  }
  PFT_CUDA_TRY(cudaStreamSynchronize(s));
  return PFT_OK;
}

// ------------------------------------------------------------------ filters
static int check_filter_args(pft_context* ctx, const pft_cloud* in, pft_cloud* out, const char* who, bool in_place_ok = false) {
  if (!ctx || !in || !out) { set_last_error("%s: null argument", who); return PFT_ERR_INVALID; }
  if (in == out && !in_place_ok) { set_last_error("%s: in-place filtering is not supported", who); return PFT_ERR_INVALID; }
  if (in->ctx != ctx || out->ctx != ctx) { set_last_error("%s: clouds belong to another context", who); return PFT_ERR_INVALID; }
  PFT_CUDA_TRY(cudaSetDevice(ctx->device));
  int rc = in->join_upload();  // an asynchronous upload into the input / output must land before the filter touches it
  if (rc) return rc;
  return out->join_upload();
}

int pft_passthrough(pft_context* ctx, const pft_cloud* in, pft_cloud* out, int field, float lo, float hi) {
  int rc = check_filter_args(ctx, in, out, "pft_passthrough");
  if (rc) return rc;
  if (field < 0 || field > 2) { set_last_error("pft_passthrough: field must be 0 (x), 1 (y) or 2 (z)"); return PFT_ERR_INVALID; }
  return run_passthrough(ctx, in, out, field, lo, hi, 0);
}

int pft_passthrough_voxel_grid(pft_context* ctx, const pft_cloud* in, pft_cloud* out, float leaf, int field, float lo, float hi) {
  int rc = check_filter_args(ctx, in, out, "pft_passthrough_voxel_grid");
  if (rc) return rc;
  if (field > 2) { set_last_error("pft_passthrough_voxel_grid: field must be <0 (off), 0, 1 or 2"); return PFT_ERR_INVALID; }
  return run_voxel_grid(ctx, in, out, leaf, field, lo, hi);
}

int pft_approx_voxel_grid_pcl(pft_context* ctx, const pft_cloud* in, pft_cloud* out, float leaf, int field, float lo, float hi) {
  int rc = check_filter_args(ctx, in, out, "pft_approx_voxel_grid_pcl");
  if (rc) return rc;
  if (field > 2) { set_last_error("pft_approx_voxel_grid_pcl: field must be <0 (off), 0, 1 or 2"); return PFT_ERR_INVALID; }
  return run_approx_voxel_grid_pcl(ctx, in, out, leaf, field, lo, hi);
}

int pft_transform_cloud(pft_context* ctx, const pft_cloud* in, pft_cloud* out, const float* m12) {
  if (!m12) { set_last_error("pft_transform_cloud: null matrix"); return PFT_ERR_INVALID; }
  for (int k = 0; k < 12; ++k)
    if (!isfinite(m12[k])) { set_last_error("pft_transform_cloud: matrix entry %d (row %d, column %d) is not finite", k, k / 4, k % 4); return PFT_ERR_INVALID; }
  int rc = check_filter_args(ctx, in, out, "pft_transform_cloud", true);
  if (rc) return rc;
  return run_transform_cloud(ctx, in, out, m12);
}

int pft_remove_zero_points(pft_context* ctx, const pft_cloud* in, pft_cloud* out) {
  int rc = check_filter_args(ctx, in, out, "pft_remove_zero_points");
  if (rc) return rc;
  return run_passthrough(ctx, in, out, -1, 0.f, 0.f, 1);
}

int pft_prepare_model(pft_context* ctx, const pft_cloud* raw, pft_cloud* out, float leaf, float* centroid3) {
  int rc = check_filter_args(ctx, raw, out, "pft_prepare_model");
  if (rc) return rc;
  // removeZeroPoints -> centroid -> translate by -centroid -> VoxelGrid(leaf)
  pft_cloud tmp;
  tmp.ctx = ctx;
  // scratch cloud backed by context buffers (kept across calls)
  tmp.pts = ctx->tmp_cloud_pts;
  tmp.hdr = ctx->tmp_hdr;
  tmp.capacity = tmp.pts.bytes / sizeof(float4);
  auto stash = [&]() { ctx->tmp_cloud_pts = tmp.pts; ctx->tmp_hdr = tmp.hdr; tmp.pts = DevBuf(); tmp.hdr = DevBuf(); };
  if ((rc = tmp.ensure(raw->capacity))) { stash(); return rc; }
  if ((rc = ctx->tmp_f.reserve(16 * sizeof(float)))) { stash(); return rc; }
  if ((rc = run_passthrough(ctx, raw, &tmp, -1, 0.f, 0.f, 1))) { stash(); return rc; }
  if ((rc = run_centre_on_centroid(ctx, &tmp, ctx->tmp_f.as<float>()))) { stash(); return rc; }
  rc = run_voxel_grid(ctx, &tmp, out, leaf, -1, 0.f, 0.f);
  stash();
  if (rc) return rc;
  if (centroid3) {
    PFT_CUDA_TRY(cudaMemcpyAsync(ctx->pinned, ctx->tmp_f.p, 3 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    PFT_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    memcpy(centroid3, ctx->pinned, 3 * sizeof(float));
  }
  return PFT_OK;
}

}  // extern "C"
