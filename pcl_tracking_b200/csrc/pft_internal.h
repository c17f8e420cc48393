// pft_internal.h -- host-side objects behind the opaque C handles and the kernel launchers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <vector>

#include "../../include/pft/pft.h"
#include "pft_common.cuh"

namespace pft {

// Grow-only device buffer.
struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  int reserve(size_t need);
  void release();
  template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

}  // namespace pft

struct pft_context {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  // K1 scratch
  pft::DevBuf k1_keys, k1_first, k1_vid, k1_slot_of, k1_acc_xyz, k1_acc_rgbc, k1_blk, staging, tmp_cloud_pts, tmp_hdr, tmp_f;
  void* pinned = nullptr;  // small pinned buffer for scalar read-backs
  size_t pinned_bytes = 0;
  // NCCL communicator shared by the clouds and trackers of this context (one process per GPU)
  void* comm = nullptr;
  int nranks = 1, rank = 0;
  // captured downsample sequences (pft_filters.cu: run_voxel_grid), keyed by every pointer / size / parameter they use
  struct K1Key { const void* p[11]; size_t cap, H; float leaf, lo, hi; int field; };
  static constexpr int kK1Graphs = 8;
  K1Key k1_key[kK1Graphs];
  cudaGraphExec_t k1_exec[kK1Graphs] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  int k1_next = 0;
  // Euclidean clustering scratch (pft_cluster.cu); the labels of the last call stay on the device for pft_cloud_select_cluster
  pft::DevBuf cl_grid, cl_cells, cl_work, cl_sel;
  size_t cl_n = 0;
  int cl_count = 0;
  const pft_cloud* cl_src = nullptr;
  cudaEvent_t batch_fork = nullptr;  // pft_compute_batch: the point of the context stream the trackers' streams fork from
  // frame ingest overlapped with compute (pft_cloud_upload_async): copies and unpack kernels run on a stream of their own
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t copy_fence = nullptr;  // "everything enqueued on `stream` so far": the copy must not overtake earlier readers
};

struct pft_cloud {
  pft_context* ctx = nullptr;
  pft::DevBuf pts;              // float4[capacity]
  pft::DevBuf hdr;              // CloudHeader
  size_t capacity = 0;          // host-known upper bound on n
  long long host_n = -1;        // exact n if known on the host, else -1
  // identity of the contents for the replicas that other contexts read (pft_tracker.cu): `serial` is never reused in the
  // process, `version` changes with every library call that writes the cloud (written())
  unsigned long long serial = 0, version = 1;
  void written(long long n) { host_n = n; ++version; }
  // pft_cloud_upload_async: `ready` fires on the copy stream once the points are in place; the first consumer on the
  // context stream waits for it (join_upload)
  pft::DevBuf raw_staging;      // raw PointCloud2 / 32-byte records / depth + colour images of an asynchronous upload
  cudaEvent_t ready = nullptr;
  mutable bool upload_pending = false;
  int join_upload() const;
  // scene distribution by peer stores (pft_cloud_peer_*): once exported the storage never moves
  bool peer_exported = false, peer_attached = false;
  size_t peer_capacity = 0;
  int peer_nranks = 0, peer_rank = 0;
  pft::DevBuf peer_sync;         // {flag, blocks done}
  void* peer_pts[16] = {nullptr}; void* peer_hdr[16] = {nullptr}; void* peer_flag[16] = {nullptr};
  unsigned int* peer_error = nullptr;  // host-mapped
  unsigned int peer_epoch = 0;
  float4* d_pts() const { return pts.as<float4>(); }
  pft::CloudHeader* d_hdr() const { return hdr.as<pft::CloudHeader>(); }
  int ensure(size_t cap);
};

namespace pft {

// ---- filters (pft_filters.cu)
int launch_unpack_pcl32(cudaStream_t s, const void* src32, float4* dst, size_t n);
int launch_pack_pcl32(cudaStream_t s, const float4* src, void* dst32, size_t n);
int launch_unpack_pointcloud2(cudaStream_t s, const void* src, float4* dst, unsigned int width, unsigned int height, unsigned int point_step,
                              unsigned int row_step, int off_x, int off_y, int off_z, int off_rgb);
// One camera of a depth-image ingest, as depth_image_kernel reads it (by value, one launch for every camera): its two
// images at byte offsets of the staging buffer, their encodings (pft_depth_encoding, pft_colour_encoding), its first
// point in the output cloud, cx, cy, kx = unit / fx, ky as the fp32 constants of the conversion (unit = 0.001f for
// 16UC1, 1 for 32FC1), and the optional camera -> common frame matrix (3x4 row-major).
struct DepthCamera {
  size_t depth_off, bgr_off, out_off;
  unsigned int width, height, depth_step, bgr_step;
  int depth_enc, colour_enc;
  float cx, cy, kx, ky;
  int has_m;
  float m[12];
};
struct DepthCameras { DepthCamera cam[PFT_MAX_DEPTH_CAMERAS]; };
// cameras 0 .. n-1 of `cams`, none of them empty, converted by one launch (blockIdx.z = camera)
int launch_depth_image(cudaStream_t s, const void* src, float4* dst, const DepthCameras& cams, int n);
// The registration of camera k of a depth-image ingest (depth_image_proc::RegisterNodelet::convert<T>), as the three
// register kernels read it: its raw depth image (depth_width x depth_height, rows depth_step bytes apart) and its
// z-buffer (reset: uint32, key: uint64 per colour pixel) at byte offsets of the staging buffer, and the registered
// image (width x height colour pixels, packed rows of pft_depth_encoding `depth_enc`) they write at `reg_off`, where
// depth_image_kernel reads the camera's depth.  The camera intrinsics are pinhole P entries; m = depth -> colour.
struct RegCamera {
  size_t raw_off, reg_off, key_off, reset_off;
  unsigned int depth_width, depth_height, depth_step, width, height;
  int registered, depth_enc, fill;
  double inv_fx, inv_fy, cx, cy, tx, ty;              // depth camera (1 / fx, 1 / fy as upstream computes them)
  double rgb_fx, rgb_fy, rgb_cx, rgb_cy, rgb_tx, rgb_ty;
  double m[12];
};
struct RegCameras { RegCamera cam[PFT_MAX_DEPTH_CAMERAS]; };
// The cameras of `cams` with `registered` set, of cameras 0 .. n-1, registered by three launches (blockIdx.z = camera)
// into `staging`; their z-buffers must be zero.
int launch_register_depth(cudaStream_t s, void* staging, const RegCameras& cams, int n);
int launch_set_header(cudaStream_t s, CloudHeader* hdr, int n);
int run_passthrough(pft_context* ctx, const pft_cloud* in, pft_cloud* out, int field, float lo, float hi, int drop_zero);
int run_voxel_grid(pft_context* ctx, const pft_cloud* in, pft_cloud* out, float leaf, int field, float lo, float hi);
int run_approx_voxel_grid_pcl(pft_context* ctx, const pft_cloud* in, pft_cloud* out, float leaf, int field, float lo, float hi);
int run_centre_on_centroid(pft_context* ctx, pft_cloud* cloud, float* d_centroid3);

// ---- scene replicas (pft_tracker.cu): every replica of a cloud goes with it, every replica a context holds goes with it
void release_replicas_of(const pft_cloud* src);
void release_replicas_in(const pft_context* dst);

}  // namespace pft
