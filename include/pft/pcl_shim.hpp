// pcl_shim.hpp -- header-only C++ classes with PCL's names over the C ABI of libpft.so.
//
// What a maintainer of cmaestre/pcl_tracking includes INSTEAD of the PCL tracking/filter headers
// (ref: src/auto_tracking.cpp:38-109) so that initialize_trackers() (ref :181-259) and cloud_cb()
// (ref :597-727) compile unchanged against the B200 tracker.  Only the surface that file drives is
// provided (SURVEY.md section 8b); every method cites the reference line that calls it.
//
// The shim defines its own minimal pcl::PointXYZRGBA / pcl::PointCloud / ParticleXYZRPY when the PCL
// headers are absent (as in this repository's build image).  With PCL present, define
// PFT_SHIM_USE_PCL_TYPES before including it: the classes then live in namespace pft_pcl and take the
// real PCL point/cloud types (both are the same 32-byte records).
//
// Errors: PCL's compute()/filter() return void and log with PCL_ERROR; here a failing C-ABI call
// throws pft::Error (std::runtime_error) carrying pft_last_error().
#ifndef PFT_PCL_SHIM_HPP_
#define PFT_PCL_SHIM_HPP_

#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <fstream>
#include <memory>
#include <sstream>
#include <stdexcept>
#include <string>
#include <vector>

#include "pft.h"

// Smart pointers: PCL 1.8 hands clouds, coherences and trackers around as boost::shared_ptr, and so does the reference
// (ref: src/auto_tracking.cpp:199-254).  Define PFT_SHIM_USE_BOOST before including this header to make every Ptr of
// the shim a boost::shared_ptr (needs <boost/shared_ptr.hpp>); the default is std::shared_ptr.
#ifdef PFT_SHIM_USE_BOOST
#include <boost/make_shared.hpp>
#include <boost/pointer_cast.hpp>
#include <boost/shared_ptr.hpp>
#define PFT_SHIM_PTR_NS boost
#else
#define PFT_SHIM_PTR_NS std
#endif
// Eigen: define PFT_SHIM_USE_EIGEN (with <Eigen/Geometry> included first) to get Eigen::Affine3f from toEigenMatrix();
// setTrans() takes any affine type with operator()(row, col) either way (Eigen::Affine3f, pft::Affine3f).

namespace pft {
namespace sp {
using PFT_SHIM_PTR_NS::shared_ptr;
using PFT_SHIM_PTR_NS::make_shared;
using PFT_SHIM_PTR_NS::static_pointer_cast;
using PFT_SHIM_PTR_NS::dynamic_pointer_cast;
}  // namespace sp

struct Error : std::runtime_error {
  int code;
  Error(int c, const char* m) : std::runtime_error(std::string("pft error ") + std::to_string(c) + ": " + m), code(c) {}
};
inline void check(int rc) { if (rc != PFT_OK) throw Error(rc, pft_last_error()); }

// Stand-in for Eigen::Affine3f where Eigen is not available: column-major 4x4, like Eigen's storage.
struct Affine3f {
  float m[16];
  Affine3f() { setIdentity(); }
  void setIdentity() { std::memset(m, 0, sizeof(m)); m[0] = m[5] = m[10] = m[15] = 1.f; }
  static Affine3f Identity() { return Affine3f(); }
  float& operator()(int r, int c) { return m[c * 4 + r]; }
  float operator()(int r, int c) const { return m[c * 4 + r]; }
  void translation(float x, float y, float z) { m[12] = x; m[13] = y; m[14] = z; }
  const float* data() const { return m; }
  float* data() { return m; }
  const Affine3f& matrix() const { return *this; }  // (Eigen: t.matrix().data() is the column-major 4x4)
};
#ifdef PFT_SHIM_USE_EIGEN
typedef Eigen::Affine3f AffineResult;
#else
typedef Affine3f AffineResult;
#endif

// One context (device + stream) per process by default, like the implicit global state of a CPU library.
class Context {
 public:
  explicit Context(int device = 0) { check(pft_context_create(device, &h_)); }
  ~Context() { pft_context_destroy(h_); }
  Context(const Context&) = delete;
  Context& operator=(const Context&) = delete;
  pft_context* get() const { return h_; }
  void synchronize() { check(pft_context_synchronize(h_)); }
  static std::shared_ptr<Context>& Default() {
    static std::shared_ptr<Context> c;
    if (!c) c = std::make_shared<Context>(0);
    return c;
  }
 private:
  pft_context* h_ = nullptr;
};

// a device list "0,1,..." from the environment (empty when unset)
inline std::vector<int> devicesFromEnv(const char* name) {
  std::vector<int> v;
  if (const char* e = std::getenv(name)) {
    for (const char* p = e; *p;) {
      char* end = nullptr;
      const long d = std::strtol(p, &end, 10);
      if (end == p) break;
      v.push_back((int)d);
      p = (*end == ',') ? end + 1 : end;
    }
  }
  return v;
}

// GPUs driven by every tracker constructed afterwards (single-process multi-device mode, pft_tracker_set_devices)
inline std::vector<int>& trackerDevices() {
  static std::vector<int> devs = devicesFromEnv("PFT_DEVICES");
  return devs;
}
inline void setTrackerDevices(const std::vector<int>& devices) { trackerDevices() = devices; }

// One object per GPU: the k-th tracker constructed afterwards lives on devices[k % n], in one context per device (created
// on first use, apart from the default context).  Clouds and filters stay on the default context, the sensor's; every
// tracker takes the scene from there (pft_tracker_set_input_cloud with a cloud of another context), so the reference's
// loop setInputCloud(scene); compute() spreads over the GPUs unchanged.  The list comes from pft::setObjectDevices({0,
// 1, ...}) or the environment (PFT_OBJECT_DEVICES=0,1,...).  It excludes the multi-device mode of one tracker.
inline std::vector<int>& objectDevices() {
  static std::vector<int> devs = devicesFromEnv("PFT_OBJECT_DEVICES");
  return devs;
}
inline void setObjectDevices(const std::vector<int>& devices) { objectDevices() = devices; }
// the context of the next tracker: the default one without object devices
inline std::shared_ptr<Context> nextTrackerContext() {
  const std::vector<int>& devs = objectDevices();
  if (devs.empty()) return Context::Default();
  if (trackerDevices().size() > 1) throw Error(PFT_ERR_INVALID, "object devices (PFT_OBJECT_DEVICES) and tracker devices (PFT_DEVICES) exclude each other");
  static std::vector<std::shared_ptr<Context>> per_device;
  static size_t constructed = 0;
  const int dev = devs[constructed++ % devs.size()];
  if (dev < 0) throw Error(PFT_ERR_INVALID, "negative object device");
  if (per_device.size() <= (size_t)dev) per_device.resize(dev + 1);
  if (!per_device[dev]) per_device[dev] = std::make_shared<Context>(dev);
  return per_device[dev];
}

// sensor_msgs/Image::encoding of a depth image -> pft_depth_encoding: "16UC1" and "mono16" (the same bytes, uint16
// millimetres), "32FC1" (float metres).  Anything else throws pft::Error (PFT_ERR_INVALID).
inline int32_t depthEncoding(const std::string& e) {
  if (e == "16UC1" || e == "mono16") return PFT_DEPTH_16UC1;
  if (e == "32FC1") return PFT_DEPTH_32FC1;
  throw Error(PFT_ERR_INVALID, ("unknown depth encoding \"" + e + "\" (16UC1, mono16 or 32FC1)").c_str());
}
// ... of a colour image -> pft_colour_encoding: "bgr8", "rgb8", "bgra8", "rgba8", "mono8", or "none" for depth alone
// (depth_image_proc/point_cloud_xyz: rgba = 0, the colour pointer is ignored).  Anything else throws pft::Error.
inline int32_t colourEncoding(const std::string& e) {
  static const char* const names[] = {"bgr8", "rgb8", "bgra8", "rgba8", "mono8", "none"};  // in pft_colour_encoding order
  for (int32_t k = 0; k <= PFT_COLOUR_NONE; ++k) if (e == names[k]) return k;
  throw Error(PFT_ERR_INVALID, ("unknown colour encoding \"" + e + "\" (bgr8, rgb8, bgra8, rgba8, mono8 or none)").c_str());
}

// One calibrated camera of a fused frame (PointCloud::fromDepthImages): the registered images and intrinsics of
// fromDepthImage, and optionally the pose of its optical frame in the common frame, T_k of
// pcl::transformPointCloud(cloud_k, T_k) (e.g. tf2 lookupTransform(target, camera_optical_frame) as Eigen::Affine3f).
struct DepthCamera {
  const void* depth = nullptr;
  uint32_t depth_step = 0;  // bytes (msg.step)
  const uint8_t* bgr = nullptr;  // the colour image, in colour_encoding
  uint32_t bgr_step = 0;
  uint32_t width = 0, height = 0;
  double fx = 0, fy = 0, cx = 0, cy = 0;  // camera_info K[0], K[4], K[2], K[5]
  std::string depth_encoding = "16UC1";   // msg.encoding, as depthEncoding / colourEncoding take it
  std::string colour_encoding = "bgr8";
  bool has_pose = false;
  float pose[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0};  // 3x4 row-major
  // any affine type with operator()(row, col), as setTrans: Eigen::Affine3f, pft::Affine3f
  template <typename AffineT> void setPose(const AffineT& t) {
    for (int r = 0; r < 3; ++r) for (int c = 0; c < 4; ++c) pose[r * 4 + c] = t(r, c);
    has_pose = true;
  }
  void clearPose() { has_pose = false; }
  // Registration (depth_image_proc/register, on the device): set when `depth` is the image of a separate depth camera,
  // not yet registered to the colour camera.  `depth` / `depth_step` / `depth_encoding` are then the depth camera's
  // image, depth_width x depth_height; width, height, fx .. cy and the colour image stay the colour camera's, and the
  // cloud is organised in its geometry.  Intrinsics are camera_info P[0], P[5], P[2], P[6], Tx = P[3], Ty = P[7].
  bool has_registration = false;
  double depth_to_colour[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0};  // 3x4 row-major, depth optical -> colour optical
  uint32_t depth_width = 0, depth_height = 0;
  double depth_fx = 0, depth_fy = 0, depth_cx = 0, depth_cy = 0, depth_tx = 0, depth_ty = 0;
  double colour_tx = 0, colour_ty = 0;
  bool fill_upsampling = false;
  // any affine type with operator()(row, col), as setPose, with double entries: Eigen::Affine3d of tf2
  // lookupTransform(colour_frame, depth_frame)
  template <typename AffineT> void setDepthToColour(const AffineT& t) {
    for (int r = 0; r < 3; ++r) for (int c = 0; c < 4; ++c) depth_to_colour[r * 4 + c] = (double)t(r, c);
    has_registration = true;
  }
  void clearDepthToColour() { has_registration = false; }
};

}  // namespace pft

#ifndef PFT_SHIM_USE_PCL_TYPES
namespace pcl {

// the 32-byte pcl::PointXYZRGBA record (ref: src/auto_tracking.cpp:139-140)
struct alignas(16) PointXYZRGBA {
  float x = 0.f, y = 0.f, z = 0.f, data3 = 1.f;
  union { struct { uint8_t b, g, r, a; }; uint32_t rgba; };
  uint32_t pad_[3] = {0, 0, 0};
  PointXYZRGBA() : rgba(0) {}
};
static_assert(sizeof(PointXYZRGBA) == 32, "PointXYZRGBA must be the 32-byte PCL record");

// pcl::PointCloud<PointT>: host vector + a lazily synchronised device mirror
template <typename PointT>
class PointCloud {
 public:
  typedef pft::sp::shared_ptr<PointCloud<PointT>> Ptr;
  typedef pft::sp::shared_ptr<const PointCloud<PointT>> ConstPtr;
  std::vector<PointT> points;
  uint32_t width = 0, height = 1;
  bool is_dense = true;
  size_t size() const { return device_only_ ? device_size() : points.size(); }
  bool empty() const { return size() == 0; }
  void push_back(const PointT& p) { points.push_back(p); host_dirty_ = true; device_only_ = false; }
  void clear() { points.clear(); host_dirty_ = true; device_only_ = false; }
  void touch() { host_dirty_ = true; device_only_ = false; }  // call after editing `points` in place

  // ---- device side (used by the shim's filters/trackers)
  pft_cloud* device(const std::shared_ptr<pft::Context>& ctx = pft::Context::Default()) const {
    if (!dev_) { ctx_ = ctx; pft::check(pft_cloud_create(ctx_->get(), &dev_)); host_dirty_ = true; }
    if (host_dirty_ && !device_only_) {
      pft::check(pft_cloud_upload(dev_, points.data(), points.size(), PFT_LAYOUT_PCL32));
      host_dirty_ = false;
    }
    return dev_;
  }
  // Frame ingest straight from a sensor_msgs/PointCloud2 message, replacing pcl_conversions::toPCL +
  // pcl::fromPCLPointCloud2 (ref: src/auto_tracking.cpp:619-622): the payload is unpacked on the device; the host
  // vector stays empty until download().  off_* = byte offsets of the x, y, z and rgb/rgba fields (msg.fields).
  void fromPointCloud2(const void* data, uint32_t w, uint32_t h, uint32_t point_step, uint32_t row_step, int off_x, int off_y, int off_z,
                       int off_rgb, bool is_bigendian = false, const std::shared_ptr<pft::Context>& ctx = pft::Context::Default()) {
    if (!dev_) { ctx_ = ctx; pft::check(pft_cloud_create(ctx_->get(), &dev_)); }
    pft::check(pft_cloud_upload_pointcloud2(dev_, data, w, h, point_step, row_step, off_x, off_y, off_z, off_rgb, is_bigendian ? 1 : 0));
    points.clear();
    width = w; height = h;
    mark_device_written();
  }
  // The same on the context's copy stream (pft_cloud_upload_pointcloud2_async): returns at once, the copy overlaps the
  // tracking enqueued after the call, the first consumer of this cloud waits for it on the device.  `data` must be
  // pinned (pft_host_alloc) and stay untouched until that consumer has finished.  Use two clouds alternately.
  void fromPointCloud2Async(const void* data, uint32_t w, uint32_t h, uint32_t point_step, uint32_t row_step, int off_x, int off_y, int off_z,
                            int off_rgb, bool is_bigendian = false, const std::shared_ptr<pft::Context>& ctx = pft::Context::Default()) {
    if (!dev_) { ctx_ = ctx; pft::check(pft_cloud_create(ctx_->get(), &dev_)); }
    pft::check(pft_cloud_upload_pointcloud2_async(dev_, data, w, h, point_step, row_step, off_x, off_y, off_z, off_rgb, is_bigendian ? 1 : 0));
    points.clear();
    width = w; height = h;
    mark_device_written();
  }
  // Frame ingest from the registered images the points topic is computed from (kinect2_bridge <res>/image_depth_rect
  // 16UC1 mm, <res>/image_color_rect bgr8, <res>/camera_info), replacing the depth_image_proc/point_cloud_xyzrgb
  // nodelet behind ref: src/auto_tracking.cpp:775 (pft_cloud_upload_depth_image): the conversion runs on the device;
  // the host vector stays empty until download().  Steps in bytes (msg.step); fx, fy, cx, cy = K[0], K[4], K[2], K[5].
  void fromDepthImage(const uint16_t* depth, uint32_t depth_step, const uint8_t* bgr, uint32_t bgr_step, uint32_t w, uint32_t h, double fx,
                      double fy, double cx, double cy, const std::shared_ptr<pft::Context>& ctx = pft::Context::Default()) {
    if (!dev_) { ctx_ = ctx; pft::check(pft_cloud_create(ctx_->get(), &dev_)); }
    pft::check(pft_cloud_upload_depth_image(dev_, depth, depth_step, bgr, bgr_step, w, h, fx, fy, cx, cy));
    points.clear();
    width = w; height = h;
    mark_device_written();
  }
  // The same on the context's copy stream (pft_cloud_upload_depth_image_async): returns at once, the copy overlaps the
  // tracking enqueued after the call, the first consumer of this cloud waits for it on the device.  Both images must be
  // pinned (pft_host_alloc) and stay untouched until that consumer has finished.  Use two clouds alternately.
  void fromDepthImageAsync(const uint16_t* depth, uint32_t depth_step, const uint8_t* bgr, uint32_t bgr_step, uint32_t w, uint32_t h, double fx,
                           double fy, double cx, double cy, const std::shared_ptr<pft::Context>& ctx = pft::Context::Default()) {
    if (!dev_) { ctx_ = ctx; pft::check(pft_cloud_create(ctx_->get(), &dev_)); }
    pft::check(pft_cloud_upload_depth_image_async(dev_, depth, depth_step, bgr, bgr_step, w, h, fx, fy, cx, cy));
    points.clear();
    width = w; height = h;
    mark_device_written();
  }
  // Both of the above for images in any encoding the depth_image_proc nodelets take (pft_cloud_upload_depth_images_enc,
  // one camera), named as sensor_msgs/Image::encoding spells it, so that a callback passes its messages through:
  //   cloud->fromDepthImage(d->data.data(), d->step, d->encoding, c->data.data(), c->step, c->encoding, d->width,
  //                         d->height, K[0], K[4], K[2], K[5]);
  // Depth "16UC1" / "mono16" / "32FC1"; colour "bgr8", "rgb8", "bgra8", "rgba8", "mono8", or "none" for depth alone
  // (point_cloud_xyz: rgba = 0, `colour` is ignored).  An unknown encoding throws pft::Error (PFT_ERR_INVALID).
  void fromDepthImage(const void* depth, uint32_t depth_step, const std::string& depth_encoding, const uint8_t* colour, uint32_t colour_step,
                      const std::string& colour_encoding, uint32_t w, uint32_t h, double fx, double fy, double cx, double cy,
                      const std::shared_ptr<pft::Context>& ctx = pft::Context::Default()) {
    upload_depth_image(depth, depth_step, depth_encoding, colour, colour_step, colour_encoding, w, h, fx, fy, cx, cy, ctx, false);
  }
  void fromDepthImageAsync(const void* depth, uint32_t depth_step, const std::string& depth_encoding, const uint8_t* colour, uint32_t colour_step,
                           const std::string& colour_encoding, uint32_t w, uint32_t h, double fx, double fy, double cx, double cy,
                           const std::shared_ptr<pft::Context>& ctx = pft::Context::Default()) {
    upload_depth_image(depth, depth_step, depth_encoding, colour, colour_step, colour_encoding, w, h, fx, fy, cx, cy, ctx, true);
  }
  // Several calibrated cameras fused into one scene (pft_cloud_upload_depth_images): for each camera,
  // pcl::transformPointCloud(cloud_k, T_k) of the cloud fromDepthImage makes, then scene += cloud_k, in one kernel
  // launch.  The cloud is unorganised: width = all the cameras' pixels, height = 1.  Cameras with setDepthToColour are
  // registered into their colour camera on the device first (pft_cloud_upload_depth_images_reg).
  void fromDepthImages(const std::vector<pft::DepthCamera>& cams, const std::shared_ptr<pft::Context>& ctx = pft::Context::Default()) {
    upload_depth_cameras(cams, ctx, false);
  }
  // The same on the context's copy stream (pft_cloud_upload_depth_images_async), with the pinned-buffer rules of
  // fromDepthImageAsync for every image.
  void fromDepthImagesAsync(const std::vector<pft::DepthCamera>& cams, const std::shared_ptr<pft::Context>& ctx = pft::Context::Default()) {
    upload_depth_cameras(cams, ctx, true);
  }
  // a filter wrote the device mirror: the host vector is stale until download()
  void mark_device_written() { device_only_ = true; host_dirty_ = false; }
  void download() {
    if (!device_only_) return;
    size_t n = device_size();
    points.resize(n);
    if (n) pft::check(pft_cloud_download(dev_, points.data(), n, PFT_LAYOUT_PCL32, &n));
    width = (uint32_t)n; height = 1;
    device_only_ = false; host_dirty_ = false;
  }
  ~PointCloud() { if (dev_) pft_cloud_destroy(dev_); }
  PointCloud() = default;
  PointCloud(const PointCloud& o) : points(o.host_points()), width(o.width), height(o.height), is_dense(o.is_dense) {}
  PointCloud& operator=(const PointCloud& o) { points = o.host_points(); width = o.width; height = o.height; host_dirty_ = true; device_only_ = false; return *this; }

 private:
  void upload_depth_image(const void* depth, uint32_t depth_step, const std::string& depth_encoding, const uint8_t* colour, uint32_t colour_step,
                          const std::string& colour_encoding, uint32_t w, uint32_t h, double fx, double fy, double cx, double cy,
                          const std::shared_ptr<pft::Context>& ctx, bool asynchronous) {
    const pft_depth_camera_enc c = {{depth, depth_step, colour, colour_step, w, h, fx, fy, cx, cy, nullptr}, pft::depthEncoding(depth_encoding),
                                    pft::colourEncoding(colour_encoding)};
    if (!dev_) { ctx_ = ctx; pft::check(pft_cloud_create(ctx_->get(), &dev_)); }
    pft::check(asynchronous ? pft_cloud_upload_depth_images_enc_async(dev_, &c, 1) : pft_cloud_upload_depth_images_enc(dev_, &c, 1));
    points.clear();
    width = w; height = h;
    mark_device_written();
  }
  void upload_depth_cameras(const std::vector<pft::DepthCamera>& cams, const std::shared_ptr<pft::Context>& ctx, bool asynchronous) {
    std::vector<pft_depth_camera_enc> c(cams.size());
    size_t n = 0;
    bool registration = false;
    for (size_t k = 0; k < cams.size(); ++k) {
      const pft::DepthCamera& s = cams[k];
      c[k] = pft_depth_camera_enc{{s.depth, s.depth_step, s.bgr, s.bgr_step, s.width, s.height, s.fx, s.fy, s.cx, s.cy, s.has_pose ? s.pose : nullptr},
                                  pft::depthEncoding(s.depth_encoding), pft::colourEncoding(s.colour_encoding)};
      n += (size_t)s.width * s.height;
      registration = registration || s.has_registration;
    }
    if (!dev_) { ctx_ = ctx; pft::check(pft_cloud_create(ctx_->get(), &dev_)); }
    if (registration) {  // pft_cloud_upload_depth_images_reg(_async): register on the device, then convert
      std::vector<pft_depth_camera_reg> r(cams.size());
      for (size_t k = 0; k < cams.size(); ++k) {
        const pft::DepthCamera& s = cams[k];
        r[k] = pft_depth_camera_reg{c[k], s.has_registration ? s.depth_to_colour : nullptr, s.depth_width, s.depth_height, s.depth_fx, s.depth_fy,
                                    s.depth_cx, s.depth_cy, s.depth_tx, s.depth_ty, s.colour_tx, s.colour_ty, s.fill_upsampling ? 1 : 0};
      }
      pft::check(asynchronous ? pft_cloud_upload_depth_images_reg_async(dev_, r.data(), (int)r.size())
                              : pft_cloud_upload_depth_images_reg(dev_, r.data(), (int)r.size()));
    } else {
      pft::check(asynchronous ? pft_cloud_upload_depth_images_enc_async(dev_, c.data(), (int)c.size())
                              : pft_cloud_upload_depth_images_enc(dev_, c.data(), (int)c.size()));
    }
    points.clear();
    width = (uint32_t)n; height = 1;
    mark_device_written();
  }
  size_t device_size() const { size_t n = 0; pft::check(pft_cloud_size(dev_, &n)); return n; }
  const std::vector<PointT>& host_points() const { const_cast<PointCloud*>(this)->download(); return points; }
  mutable pft_cloud* dev_ = nullptr;
  mutable std::shared_ptr<pft::Context> ctx_;
  mutable bool host_dirty_ = true;
  mutable bool device_only_ = false;
};

// pcl::PassThrough (ref: src/auto_tracking.cpp:539-545)
template <typename PointT>
class PassThrough {
 public:
  void setFilterFieldName(const std::string& f) {
    if (f == "x") field_ = 0; else if (f == "y") field_ = 1; else if (f == "z") field_ = 2;
    else throw pft::Error(PFT_ERR_INVALID, "PassThrough: field must be x, y or z");
  }
  void setFilterLimits(float lo, float hi) { lo_ = lo; hi_ = hi; }
  void setKeepOrganized(bool keep) { if (keep) throw pft::Error(PFT_ERR_INVALID, "setKeepOrganized(true) is not supported (ref :542 passes false)"); }
  void setInputCloud(const typename PointCloud<PointT>::ConstPtr& c) { in_ = c; }
  void filter(PointCloud<PointT>& out) {
    auto& ctx = pft::Context::Default();
    pft::check(pft_passthrough(ctx->get(), in_->device(ctx), out.device(ctx), field_, lo_, hi_));
    out.mark_device_written();
  }
 private:
  typename PointCloud<PointT>::ConstPtr in_;
  int field_ = 2;
  float lo_ = -3.4028235e38f, hi_ = 3.4028235e38f;
};

// pcl::VoxelGrid / pcl::ApproximateVoxelGrid (ref: src/auto_tracking.cpp:553-557, :568-571)
template <typename PointT>
class VoxelGrid {
 public:
  void setLeafSize(float lx, float ly, float lz) {
    if (lx != ly || lx != lz) throw pft::Error(PFT_ERR_INVALID, "anisotropic leaf sizes are not supported (ref :555, :569 pass one size)");
    leaf_ = lx;
  }
  void setInputCloud(const typename PointCloud<PointT>::ConstPtr& c) { in_ = c; }
  void filter(PointCloud<PointT>& out) {
    auto& ctx = pft::Context::Default();
    pft::check(pft_passthrough_voxel_grid(ctx->get(), in_->device(ctx), out.device(ctx), leaf_, -1, 0.f, 0.f));
    out.mark_device_written();
  }
 private:
  typename PointCloud<PointT>::ConstPtr in_;
  float leaf_ = 0.01f;
};
template <typename PointT> using ApproximateVoxelGrid = VoxelGrid<PointT>;

// pcl::io::loadPCDFile / savePCDFile* / pcl::PCDWriter::write for PointXYZRGBA clouds (PCD v0.7, DATA ascii | binary):
// the model builder writes one models/<time>/<k>.pcd per cluster with writer.write(path, cloud, false)
// (ref: src/create_model.cpp:209-230); offline runs replay frames stored as PCD files.  Fields x, y, z (float32)
// plus rgba (uint32) or rgb (the same bytes as a float32); other fields are skipped.  Host-side only.
namespace io {
namespace detail {
struct PcdField { std::string name; int size = 4; char type = 'F'; int count = 1; };
inline double pcd_number(const std::string& tok) { return std::strtod(tok.c_str(), nullptr); }  // accepts nan / inf
}  // namespace detail

template <typename PointT>
int loadPCDFile(const std::string& path, PointCloud<PointT>& cloud) {
  std::ifstream f(path, std::ios::binary);
  if (!f) return -1;
  std::vector<detail::PcdField> fields;
  uint32_t width = 0, height = 1;
  size_t points = 0;
  std::string data, line;
  bool have_points = false;
  while (std::getline(f, line)) {
    if (!line.empty() && line.back() == '\r') line.pop_back();
    if (line.empty() || line[0] == '#') continue;
    std::istringstream ls(line);
    std::string key;
    ls >> key;
    std::vector<std::string> vals;
    for (std::string v; ls >> v;) vals.push_back(v);
    if (key == "FIELDS") { fields.resize(vals.size()); for (size_t i = 0; i < vals.size(); ++i) fields[i].name = vals[i]; }
    else if (key == "SIZE") { for (size_t i = 0; i < vals.size() && i < fields.size(); ++i) fields[i].size = std::atoi(vals[i].c_str()); }
    else if (key == "TYPE") { for (size_t i = 0; i < vals.size() && i < fields.size(); ++i) fields[i].type = vals[i][0]; }
    else if (key == "COUNT") { for (size_t i = 0; i < vals.size() && i < fields.size(); ++i) fields[i].count = std::atoi(vals[i].c_str()); }
    else if (key == "WIDTH" && !vals.empty()) width = (uint32_t)std::strtoul(vals[0].c_str(), nullptr, 10);
    else if (key == "HEIGHT" && !vals.empty()) height = (uint32_t)std::strtoul(vals[0].c_str(), nullptr, 10);
    else if (key == "POINTS" && !vals.empty()) { points = (size_t)std::strtoull(vals[0].c_str(), nullptr, 10); have_points = true; }
    else if (key == "DATA" && !vals.empty()) { data = vals[0]; break; }
  }
  const size_t n = (size_t)width * height;
  if (data.empty() || fields.empty() || (have_points && points != n)) return -1;
  int ix = -1, iy = -1, iz = -1, ic = -1;
  size_t stride = 0;
  std::vector<size_t> offs(fields.size());
  size_t cols = 0;
  std::vector<size_t> col0(fields.size());
  for (size_t i = 0; i < fields.size(); ++i) {
    offs[i] = stride; col0[i] = cols;
    stride += (size_t)fields[i].size * fields[i].count; cols += (size_t)fields[i].count;
    if (fields[i].count != 1 || fields[i].size != 4) continue;
    if (fields[i].name == "x") ix = (int)i; else if (fields[i].name == "y") iy = (int)i; else if (fields[i].name == "z") iz = (int)i;
    else if (fields[i].name == "rgba" || (fields[i].name == "rgb" && ic < 0)) ic = (int)i;
  }
  if (ix < 0 || iy < 0 || iz < 0) return -1;
  cloud.points.assign(n, PointT());
  if (data == "binary") {
    std::vector<char> rec(stride);
    for (size_t p = 0; p < n; ++p) {
      if (!f.read(rec.data(), (std::streamsize)stride)) return -1;
      PointT& q = cloud.points[p];
      std::memcpy(&q.x, rec.data() + offs[ix], 4); std::memcpy(&q.y, rec.data() + offs[iy], 4); std::memcpy(&q.z, rec.data() + offs[iz], 4);
      if (ic >= 0) std::memcpy(&q.rgba, rec.data() + offs[ic], 4);
    }
  } else if (data == "ascii") {
    for (size_t p = 0; p < n; ++p) {
      do { if (!std::getline(f, line)) return -1; } while (line.empty());
      std::istringstream ls(line);
      std::vector<std::string> tok;
      for (std::string v; ls >> v;) tok.push_back(v);
      if (tok.size() < cols) return -1;
      PointT& q = cloud.points[p];
      q.x = (float)detail::pcd_number(tok[col0[ix]]); q.y = (float)detail::pcd_number(tok[col0[iy]]); q.z = (float)detail::pcd_number(tok[col0[iz]]);
      if (ic >= 0) {
        if (fields[ic].type == 'F') { const float c = (float)detail::pcd_number(tok[col0[ic]]); std::memcpy(&q.rgba, &c, 4); }  // packed colour printed as a float
        else q.rgba = (uint32_t)std::strtoul(tok[col0[ic]].c_str(), nullptr, 10);
      }
    }
  } else {
    return -1;  // binary_compressed is not supported
  }
  cloud.width = width; cloud.height = height;
  cloud.touch();
  return 0;
}

template <typename PointT>
int savePCDFile(const std::string& path, const PointCloud<PointT>& cloud_in, bool binary_mode = false) {
  PointCloud<PointT> cloud(cloud_in);  // (downloads a device-only cloud)
  std::ofstream f(path, std::ios::binary);
  if (!f) return -1;
  const size_t n = cloud.points.size();
  const bool organised = (size_t)cloud.width * cloud.height == n && cloud.height > 1;
  f << "# .PCD v0.7 - Point Cloud Data file format\nVERSION 0.7\nFIELDS x y z rgba\nSIZE 4 4 4 4\nTYPE F F F U\nCOUNT 1 1 1 1\n"
    << "WIDTH " << (organised ? cloud.width : (uint32_t)n) << "\nHEIGHT " << (organised ? cloud.height : 1u) << "\nVIEWPOINT 0 0 0 1 0 0 0\nPOINTS " << n
    << "\nDATA " << (binary_mode ? "binary" : "ascii") << "\n";
  for (size_t p = 0; p < n; ++p) {
    const PointT& q = cloud.points[p];
    if (binary_mode) {
      f.write(reinterpret_cast<const char*>(&q.x), 4); f.write(reinterpret_cast<const char*>(&q.y), 4); f.write(reinterpret_cast<const char*>(&q.z), 4);
      f.write(reinterpret_cast<const char*>(&q.rgba), 4);
    } else {
      char buf[128];
      auto num = [](float v, char* out) { if (std::isnan(v)) std::strcpy(out, "nan"); else if (std::isinf(v)) std::strcpy(out, v > 0 ? "inf" : "-inf"); else std::snprintf(out, 32, "%.9g", (double)v); };
      char a[32], b[32], c[32];
      num(q.x, a); num(q.y, b); num(q.z, c);
      std::snprintf(buf, sizeof(buf), "%s %s %s %u\n", a, b, c, (unsigned)q.rgba);
      f << buf;
    }
  }
  return f ? 0 : -1;
}
template <typename PointT> int savePCDFileASCII(const std::string& path, const PointCloud<PointT>& c) { return savePCDFile(path, c, false); }
template <typename PointT> int savePCDFileBinary(const std::string& path, const PointCloud<PointT>& c) { return savePCDFile(path, c, true); }
}  // namespace io

// pcl::PCDWriter (ref: src/create_model.cpp:209-223: writer.write<PointType>(path, *cloud_cluster, false))
struct PCDWriter {
  template <typename PointT> int write(const std::string& path, const PointCloud<PointT>& cloud, bool binary = false) { return io::savePCDFile(path, cloud, binary); }
};

// pcl::PointIndices + pcl::EuclideanClusterExtraction as the model builder uses them (ref: src/create_model.cpp:169-179)
struct PointIndices { std::vector<int> indices; };
template <typename PointT>
class EuclideanClusterExtraction {
 public:
  void setClusterTolerance(double t) { tol_ = t; }
  void setMinClusterSize(int n) { min_ = n; }
  void setMaxClusterSize(int n) { max_ = n; }
  template <typename TreePtr> void setSearchMethod(const TreePtr&) {}  // the KdTree (ref :169-173) is replaced by a uniform grid
  void setInputCloud(const typename PointCloud<PointT>::ConstPtr& c) { in_ = c; }
  // clusters ranked by size descending, indices sorted (as upstream); cluster k as a device cloud: clusterCloud(k, out)
  void extract(std::vector<PointIndices>& clusters) {
    auto& ctx = pft::Context::Default();
    const size_t n = in_->size();
    std::vector<int32_t> labels(n ? n : 1), sizes(4096);
    size_t k = 0;
    pft::check(pft_euclidean_clusters(ctx->get(), in_->device(ctx), tol_, min_, max_, n ? labels.data() : nullptr, n, sizes.data(), sizes.size(), &k));
    clusters.assign(k, PointIndices());
    for (size_t c = 0; c < k; ++c) clusters[c].indices.reserve((size_t)sizes[c]);
    for (size_t i = 0; i < n; ++i) if (labels[i] >= 0) clusters[(size_t)labels[i]].indices.push_back((int)i);
  }
  void clusterCloud(int k, PointCloud<PointT>& out) {  // ref: src/create_model.cpp:209-230 (one cloud per cluster)
    auto& ctx = pft::Context::Default();
    pft::check(pft_cloud_select_cluster(ctx->get(), in_->device(ctx), k, out.device(ctx)));
    out.mark_device_written();
  }
 private:
  typename PointCloud<PointT>::ConstPtr in_;
  double tol_ = 0.0;
  int min_ = 1, max_ = 2147483647;
};

// pcl::getTime (pcl/common/time.h; ref: src/auto_tracking.cpp:552, :559): seconds, wall clock
inline double getTime() {
  struct timespec ts;
  clock_gettime(CLOCK_REALTIME, &ts);
  return (double)ts.tv_sec + 1.0e-9 * (double)ts.tv_nsec;
}

namespace search {
// pcl::search::Octree(resolution) (ref :250): the cell size of the uniform-grid index
template <typename PointT> struct Octree {
  typedef pft::sp::shared_ptr<Octree<PointT>> Ptr;
  explicit Octree(double r) : resolution(r) {}
  double resolution;
};
// pcl::search::KdTree (ref :155-156, :183): only constructed by the reference (normals are off, ref :233)
template <typename PointT> struct KdTree {
  typedef pft::sp::shared_ptr<KdTree<PointT>> Ptr;
  explicit KdTree(bool sorted = true) : sorted_results(sorted) {}
  bool sorted_results;
};
}  // namespace search

namespace tracking {

// pcl::tracking::ParticleXYZRPY (ref :142): same 32-byte record as pft_particle
struct ParticleXYZRPY {
  float x = 0.f, y = 0.f, z = 0.f, one = 1.f, roll = 0.f, pitch = 0.f, yaw = 0.f, weight = 0.f;
  // ParticleXYZRPY::toEigenMatrix (ref :310), evaluated by the same device routine weight() uses
  pft::AffineResult toEigenMatrix() const {
    float m12[12];
    pft::check(pft_particle_to_matrix(pft::Context::Default()->get(), reinterpret_cast<const pft_particle*>(this), m12));
    pft::AffineResult a = pft::AffineResult::Identity();
    for (int r = 0; r < 3; ++r) for (int c = 0; c < 4; ++c) a(r, c) = m12[r * 4 + c];
    return a;
  }
};
static_assert(sizeof(ParticleXYZRPY) == sizeof(pft_particle), "particle layout");

template <typename PointT> struct PointCoherence {
  typedef pft::sp::shared_ptr<PointCoherence<PointT>> Ptr;
  virtual ~PointCoherence() {}
};
// pcl::tracking::DistanceCoherence (ref :240-242)
template <typename PointT> struct DistanceCoherence : PointCoherence<PointT> {
  typedef pft::sp::shared_ptr<DistanceCoherence<PointT>> Ptr;
  void setWeight(double w) { weight = w; }
  double weight = 1.0;
};
// pcl::tracking::HSVColorCoherence (ref :244-247)
template <typename PointT> struct HSVColorCoherence : PointCoherence<PointT> {
  typedef pft::sp::shared_ptr<HSVColorCoherence<PointT>> Ptr;
  void setWeight(double w) { weight = w; }
  void setHWeight(double w) { h_weight = w; }
  void setSWeight(double w) { s_weight = w; }
  void setVWeight(double w) { v_weight = w; }
  double weight = 1.0, h_weight = 1.0, s_weight = 1.0, v_weight = 0.0;
};
// pcl::tracking::PointCloudCoherence: what ParticleFilterTracker::setCloudCoherence takes (CoherencePtr, ref :154, :254)
template <typename PointT> struct PointCloudCoherence {
  typedef pft::sp::shared_ptr<PointCloudCoherence<PointT>> Ptr;
  typedef typename PointCoherence<PointT>::Ptr PointCoherencePtr;
  virtual ~PointCloudCoherence() {}
  void addPointCoherence(const PointCoherencePtr& c) { point_coherences.push_back(c); }          // ref :242, :247
  std::vector<PointCoherencePtr> point_coherences;
  double resolution = 0.01, maximum_distance = 1.79769313486231570815e308;
  bool pcl_approximate_search = false;
};
// pcl::tracking::NearestPairPointCloudCoherence / ApproxNearestPairPointCloudCoherence (ref :235-238)
template <typename PointT> struct NearestPairPointCloudCoherence : PointCloudCoherence<PointT> {
  typedef pft::sp::shared_ptr<NearestPairPointCloudCoherence<PointT>> Ptr;
  void setSearchMethod(const typename pcl::search::Octree<PointT>::Ptr& s) { this->resolution = s->resolution; }  // ref :252
  void setMaximumDistance(double d) { this->maximum_distance = d; }                                              // ref :253
};
// Both classes run the exact search unless setPclApproximateSearch(true) asks for the parity mode that reproduces
// upstream's greedy approxNearestSearch (PFT_NN_PCL_APPROX: same misses as PCL, far slower).
template <typename PointT> struct ApproxNearestPairPointCloudCoherence : NearestPairPointCloudCoherence<PointT> {
  typedef pft::sp::shared_ptr<ApproxNearestPairPointCloudCoherence<PointT>> Ptr;
  void setPclApproximateSearch(bool on) { this->pcl_approximate_search = on; }
};

// pcl::tracking::ParticleFilterTracker: the type the reference declares its trackers with
// (`typedef ParticleFilterTracker<RefPointType, ParticleT> ParticleFilter`, `boost::shared_ptr<ParticleFilter> tracker_`,
// ref: src/auto_tracking.cpp:153, :199) -- everything it calls through that pointer lives here (ref :225-254, :673-693,
// :270, :309).  Constructed directly it is the fixed-size tracker (as upstream's base class is).
template <typename PointT, typename StateT>
class ParticleFilterTracker {
 public:
  typedef typename PointCloud<PointT>::Ptr PointCloudInPtr;
  typedef typename PointCloud<PointT>::ConstPtr PointCloudInConstPtr;
  typedef pft::sp::shared_ptr<PointCloud<StateT>> PointCloudStatePtr;
  typedef PointCloudCoherence<PointT> CloudCoherence;
  typedef typename CloudCoherence::Ptr CloudCoherencePtr;
  typedef CloudCoherencePtr CoherencePtr;                                                         // ref :154
  ParticleFilterTracker() : ParticleFilterTracker(0, 0) {}
  virtual ~ParticleFilterTracker() { pft_tracker_destroy(h_); }  // (before ctx_ lets go of the context)
  ParticleFilterTracker(const ParticleFilterTracker&) = delete;
  ParticleFilterTracker& operator=(const ParticleFilterTracker&) = delete;
  // any affine type with operator()(row, col): Eigen::Affine3f (ref :225, :674), pft::Affine3f
  template <typename AffineT> void setTrans(const AffineT& t) {
    float m12[12];
    for (int r = 0; r < 3; ++r) for (int c = 0; c < 4; ++c) m12[r * 4 + c] = t(r, c);
    pft::check(pft_tracker_set_trans(h_, m12));
  }
  void setStepNoiseCovariance(const std::vector<double>& v) { sv(PFT_STEP_NOISE_COV, v); }        // ref :226
  void setInitialNoiseCovariance(const std::vector<double>& v) { sv(PFT_INIT_NOISE_COV, v); }     // ref :227
  void setInitialNoiseMean(const std::vector<double>& v) { sv(PFT_INIT_NOISE_MEAN, v); }          // ref :228
  void setIterationNum(int n) { si(PFT_ITERATION_NUM, n); }                                       // ref :229
  void setParticleNum(int n) { si(PFT_PARTICLE_NUM, n); }                                         // ref :231
  void setResampleLikelihoodThr(double v) { sd(PFT_RESAMPLE_LIKELIHOOD_THR, v); }                 // ref :232
  void setUseNormal(bool u) { si(PFT_USE_NORMAL, u ? 1 : 0); }                                    // ref :233
  void setMinIndices(int n) { si(PFT_MIN_INDICES, n); }                                           // ref :676
  // change detector (pcl::tracking::ParticleFilterTracker; off by default, never enabled by the reference)
  void setUseChangeDetector(bool u) { si(PFT_USE_CHANGE_DETECTOR, u ? 1 : 0); }
  void setIntervalOfChangeDetection(unsigned int n) { si(PFT_CHANGE_DETECTOR_INTERVAL, (int)n); }
  void setMinPointsOfChangeDetection(unsigned int n) { si(PFT_CHANGE_DETECTOR_MIN_POINTS, (int)n); }
  void setResolutionOfChangeDetection(double r) { sd(PFT_CHANGE_DETECTOR_RESOLUTION, r); }
  void setAlpha(double a) { sd(PFT_ALPHA, a); }
  void setMotionRatio(double r) { sd(PFT_MOTION_RATIO, r); }
  void setCloudCoherence(const CloudCoherencePtr& c) {                                            // ref :254
    int use_d = 0, use_h = 0;
    for (auto& pc : c->point_coherences) {
      if (auto* d = dynamic_cast<DistanceCoherence<PointT>*>(pc.get())) { use_d = 1; sd(PFT_DIST_WEIGHT, d->weight); }
      else if (auto* hsv = dynamic_cast<HSVColorCoherence<PointT>*>(pc.get())) {
        use_h = 1; sd(PFT_HSV_WEIGHT, hsv->weight); sd(PFT_H_WEIGHT, hsv->h_weight); sd(PFT_S_WEIGHT, hsv->s_weight); sd(PFT_V_WEIGHT, hsv->v_weight);
      } else throw pft::Error(PFT_ERR_INVALID, "unsupported point coherence");
    }
    si(PFT_USE_DISTANCE, use_d); si(PFT_USE_HSV, use_h); si(PFT_NN_MODE, c->pcl_approximate_search ? PFT_NN_PCL_APPROX : PFT_NN_EXACT);
    sd(PFT_MAX_DIST, c->maximum_distance); sd(PFT_SEARCH_RESOLUTION, c->resolution);
    coherence_ = c;
  }
  CloudCoherencePtr getCloudCoherence() const { return coherence_; }
  void setReferenceCloud(const PointCloudInConstPtr& c) {                                         // ref :673
    ref_ = c;
    pft::check(pft_tracker_set_reference_cloud(h_, c->device()));
  }
  PointCloudInConstPtr getReferenceCloud() const { return ref_; }
  void setInputCloud(const PointCloudInConstPtr& c) {                                             // ref :691
    input_ = c;
    pft::check(pft_tracker_set_input_cloud(h_, c ? c->device() : nullptr));
  }
  void compute() { pft::check(pft_tracker_compute(h_)); }                                        // ref :693
  StateT getResult() const {                                                                      // ref :309
    StateT s;
    pft::check(pft_tracker_get_result(h_, reinterpret_cast<pft_particle*>(&s)));
    return s;
  }
  PointCloudStatePtr getParticles() const {                                                       // ref :270
    PointCloudStatePtr out = pft::sp::make_shared<PointCloud<StateT>>();
    size_t n = 0;
    int rc = pft_tracker_get_particles(h_, nullptr, 0, &n);
    if (rc != PFT_OK && rc != PFT_ERR_CAPACITY) pft::check(rc);
    out->points.resize(n);
    if (n) pft::check(pft_tracker_get_particles(h_, reinterpret_cast<pft_particle*>(out->points.data()), n, &n));
    return out;
  }
  pft::AffineResult toEigenMatrix(const StateT& particle) { return particle.toEigenMatrix(); }    // ref :310
  // what viz_cb derives from getResult() per object (ref :309-316, :432-466, :481-515): published centroid + PCA box
  pft_result_box getResultBox(float z_offset = -0.005f) const {
    pft_result_box b;
    pft::check(pft_tracker_get_result_box(h_, z_offset, &b));
    return b;
  }
  void resetTracking() { pft::check(pft_tracker_reset(h_)); }
  double getFitRatio() const { double v = 0; pft::check(pft_tracker_get_fit_ratio(h_, &v)); return v; }
  pft_tracker* handle() const { return h_; }

 protected:
  ParticleFilterTracker(unsigned int nr_threads, int kld) : ctx_(pft::nextTrackerContext()) {
    pft::check(pft_tracker_create(ctx_->get(), kld, &h_));
    // single-process multi-device mode: the reference's constructor call (ref :201, :215) cannot name GPUs, so the
    // list comes from pft::setTrackerDevices({0, 1, ...}) or the environment (PFT_DEVICES=0,1,...); first = device 0
    const std::vector<int>& devs = pft::trackerDevices();
    if (devs.size() > 1) pft::check(pft_tracker_set_devices(h_, (int)devs.size(), devs.data()));
    si(PFT_THREADS, (int)nr_threads);
  }
  void si(int k, int v) { pft::check(pft_tracker_set_i(h_, k, v)); }
  void sd(int k, double v) { pft::check(pft_tracker_set_d(h_, k, v)); }
  void sv(int k, const std::vector<double>& v) {
    if (v.size() != 6) throw pft::Error(PFT_ERR_INVALID, "expected 6 values");
    pft::check(pft_tracker_set_vec6(h_, k, v.data()));
  }
  std::shared_ptr<pft::Context> ctx_;
  pft_tracker* h_ = nullptr;
  PointCloudInConstPtr ref_, input_;
  CloudCoherencePtr coherence_;
};

// pcl::tracking::ParticleFilterOMPTracker (ref :201-206)
template <typename PointT, typename StateT>
class ParticleFilterOMPTracker : public ParticleFilterTracker<PointT, StateT> {
 public:
  explicit ParticleFilterOMPTracker(unsigned int nr_threads = 0) : ParticleFilterTracker<PointT, StateT>(nr_threads, 0) {}
  void setNumberOfThreads(unsigned int n) { this->si(PFT_THREADS, (int)n); }

 protected:
  ParticleFilterOMPTracker(unsigned int nr_threads, int kld) : ParticleFilterTracker<PointT, StateT>(nr_threads, kld) {}
};

// pcl::tracking::KLDAdaptiveParticleFilterTracker / KLDAdaptiveParticleFilterOMPTracker (ref :209-222; :150-151 commented)
template <typename PointT, typename StateT>
class KLDAdaptiveParticleFilterTracker : public ParticleFilterTracker<PointT, StateT> {
 public:
  KLDAdaptiveParticleFilterTracker() : ParticleFilterTracker<PointT, StateT>(0, 1) {}
  void setMaximumParticleNum(unsigned int n) { this->si(PFT_MAX_PARTICLE_NUM, (int)n); }          // ref :211
  void setDelta(double d) { this->sd(PFT_DELTA, d); }                                            // ref :212
  void setEpsilon(double e) { this->sd(PFT_EPSILON, e); }                                        // ref :213
  void setBinSize(const StateT& b) {                                                              // ref :214-221
    this->sv(PFT_BIN_SIZE, {b.x, b.y, b.z, b.roll, b.pitch, b.yaw});
  }

 protected:
  explicit KLDAdaptiveParticleFilterTracker(unsigned int nr_threads) : ParticleFilterTracker<PointT, StateT>(nr_threads, 1) {}
};
template <typename PointT, typename StateT>
class KLDAdaptiveParticleFilterOMPTracker : public KLDAdaptiveParticleFilterTracker<PointT, StateT> {
 public:
  explicit KLDAdaptiveParticleFilterOMPTracker(unsigned int nr_threads = 0) : KLDAdaptiveParticleFilterTracker<PointT, StateT>(nr_threads) {}
  void setNumberOfThreads(unsigned int n) { this->si(PFT_THREADS, (int)n); }
};

}  // namespace tracking

// pcl::NormalEstimationOMP (ref :168, :183-185): constructed and configured by the reference, never run (setUseNormal(false), ref :233)
template <typename PointInT, typename PointOutT>
class NormalEstimationOMP {
 public:
  explicit NormalEstimationOMP(unsigned int nr_threads = 0) : threads_(nr_threads) {}
  template <typename TreePtr> void setSearchMethod(const TreePtr&) {}
  void setRadiusSearch(double r) { radius_ = r; }
 private:
  unsigned int threads_;
  double radius_ = 0.0;
};
struct Normal { float normal_x = 0.f, normal_y = 0.f, normal_z = 0.f, curvature = 0.f; };
}  // namespace pcl
#endif  // PFT_SHIM_USE_PCL_TYPES

#endif  // PFT_PCL_SHIM_HPP_
