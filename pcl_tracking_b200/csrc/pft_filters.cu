// pft_filters.cu -- kernel K1: PassThrough + voxel-grid downsampling as a sort-free voxel-hash
// reduction, plus the order-preserving PassThrough compaction and the model preparation helpers.
//
// Replaces pcl::PassThrough::filter and pcl::(Approximate)VoxelGrid::filter as called from
// ref: src/auto_tracking.cpp:536-575 (SURVEY.md 8a rows a1-a4, Appendix A.1/A.2).
//
// Data layout: clouds are float4 {x,y,z,rgba} arrays in HBM with a 16-byte device header holding the
// point count (no host round trip between stages).  The voxel hash is an open-addressing table of
// 16-byte slots holding the voxel's three int32 lattice indices (exact: no two voxels share a key);
// per-voxel sums are kept in double (coordinates) and uint32 (colour bytes), which makes the centroid
// independent of the order the atomics land in wherever the fp64 sums are exact (k1_accum_kernel).
// Output order = order of first appearance.
#include <stdlib.h>
#include <string.h>

#include <type_traits>
#include <utility>

#include "pft_internal.h"

namespace pft {

namespace {

constexpr int kFirstInit = 0x7f7f7f7f;

__device__ __forceinline__ bool finite3(const float4& p) { return isfinite(p.x) && isfinite(p.y) && isfinite(p.z); }

__device__ __forceinline__ bool passes(const float4& p, int field, float lo, float hi) {
  if (!finite3(p)) return false;
  if (field < 0) return true;
  const float v = field == 0 ? p.x : (field == 1 ? p.y : p.z);
  return !(v < lo || v > hi);
}

// Lattice index of upstream (Approximate)VoxelGrid: floor(coord * inverse_leaf_size), the product rounded to fp32.
// Outside the int32 range it saturates (cvt.rmi.s32.f32): |coord * inv| >= 2^31 is index INT_MAX or INT_MIN.
__device__ __forceinline__ int voxel_index(float v, float inv) { return __float2int_rd(v * inv); }
// Hash of a voxel's three indices (all 96 bits feed the 64-bit finaliser of MurmurHash3).
__device__ __forceinline__ unsigned int voxel_hash(int ix, int iy, int iz) {
  unsigned long long k = (((unsigned long long)(unsigned int)ix << 32) | (unsigned int)iy) ^ ((unsigned long long)(unsigned int)iz * 0x9e3779b97f4a7c15ull);
  k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
  return (unsigned int)k;
}

__global__ void unpack_pcl32_kernel(const uint4* __restrict__ src, float4* __restrict__ dst, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const uint4 a = src[2 * i];      // x y z w
    const uint4 b = src[2 * i + 1];  // rgba pad pad pad
    dst[i] = make_float4(__uint_as_float(a.x), __uint_as_float(a.y), __uint_as_float(a.z), __uint_as_float(b.x));
  }
}
__global__ void pack_pcl32_kernel(const float4* __restrict__ src, uint4* __restrict__ dst, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float4 p = src[i];
    dst[2 * i] = make_uint4(__float_as_uint(p.x), __float_as_uint(p.y), __float_as_uint(p.z), __float_as_uint(1.0f));
    dst[2 * i + 1] = make_uint4(__float_as_uint(p.w), 0u, 0u, 0u);
  }
}
// sensor_msgs/PointCloud2 -> float4 {x,y,z,rgba}: replaces pcl_conversions::toPCL + pcl::fromPCLPointCloud2
// (ref: src/auto_tracking.cpp:619-622).  Rows of `row_step` bytes hold `width` records of `point_step` bytes; the
// float32 fields x, y, z and the 4 colour bytes sit at arbitrary (4-byte aligned) offsets inside a record.  Organised
// clouds keep their row-major order, as fromPCLPointCloud2 does.  A warp reads whole 4-byte words of consecutive
// records, so the loads of a row are as coalesced as the record stride allows.
__global__ void unpack_pointcloud2_kernel(const unsigned int* __restrict__ src, float4* __restrict__ dst, unsigned int width, unsigned int height,
                                          unsigned int point_words, unsigned int row_words, int wx, int wy, int wz, int wrgb) {
  const size_t n = (size_t)width * height;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const size_t row = i / width, col = i - row * width;
    const unsigned int* rec = src + row * row_words + col * point_words;
    const unsigned int rgba = wrgb >= 0 ? rec[wrgb] : 0u;
    dst[i] = make_float4(__uint_as_float(rec[wx]), __uint_as_float(rec[wy]), __uint_as_float(rec[wz]), __uint_as_float(rgba));
  }
}
// Pixel u of a colour row in encoding C (pft_colour_encoding) as the nodelet packs it, rgba = b | g << 8 | r << 16 |
// 255 << 24, with r, g, b read at the encoding's byte offsets: 2, 1, 0 of 3 (bgr8) or 4 (bgra8) bytes, 0, 1, 2 of 3
// (rgb8) or 4 (rgba8), 0, 0, 0 of 1 (mono8).  Alpha is ignored.  No colour image: 0, and nothing is read.
template <int C>
__device__ __forceinline__ unsigned int colour_rgba(const unsigned char* __restrict__ row, unsigned int u) {
  if constexpr (C == PFT_COLOUR_NONE) {
    return 0u;
  } else {
    constexpr bool mono = C == PFT_COLOUR_MONO8, bgr = C == PFT_COLOUR_BGR8 || C == PFT_COLOUR_BGRA8;
    constexpr int bpp = mono ? 1 : (C == PFT_COLOUR_BGRA8 || C == PFT_COLOUR_RGBA8) ? 4 : 3;
    constexpr int r = mono ? 0 : bgr ? 2 : 0, g = mono ? 0 : 1, b = mono ? 0 : bgr ? 0 : 2;
    const unsigned char* c = row + bpp * (size_t)u;
    return (unsigned int)c[b] | ((unsigned int)c[g] << 8) | ((unsigned int)c[r] << 16) | 0xff000000u;
  }
}

// Registered depth + colour images -> float4 {x,y,z,rgba}: replaces the depth_image_proc point_cloud_xyzrgb nodelet
// that computes the /kinect2/<res>/points topic the reference subscribes to (ref: src/auto_tracking.cpp:775), i.e.
// depth_image_proc::convert<T> + its colour copy, or point_cloud_xyz (no colour image, rgba = 0).  Every fp32
// operation is rounded on its own (-fmad=false), in the nodelet's order: x = ((u - cx) * d) * kx with kx = unit / fx.
// D = unsigned short (16UC1, mm): z = d * 0.001f, d == 0 is invalid; D = float (32FC1, m): z = d, a non-finite d is
// invalid (0 and negative depths are kept, as upstream).  An invalid pixel is a quiet-NaN point (colour still
// written).  C is the colour encoding (colour_rgba).  Camera blockIdx.z of `cams` has its depth rows (`depth_step`
// bytes apart, a multiple of sizeof(D)) at byte `depth_off` of `src`, its colour rows at byte `bgr_off`, and its
// organised row-major points from point `out_off` of `dst`: several calibrated cameras fused into one cloud (`scene
// += cloud_k`) in one launch.  A camera with a matrix (camera -> common frame) then moves each finite point as
// pcl::transformPointCloud does (PCL 1.8.0, not dense: non-finite points are copied untouched), x' = ((m00 x + m01 y)
// + m02 z) + m03.  The encodings and the matrix are per camera, so every branch on them is uniform per block.  Thread
// = pixel along a row: the warp's 2- or 4-byte depth loads, 1-, 3- or 4-byte colour loads and 16-byte stores each
// cover one contiguous span.  One camera without a matrix is the single-image ingest.
template <typename D, int C>
__device__ __forceinline__ void depth_image_camera(const unsigned char* __restrict__ src, float4* __restrict__ dst, const DepthCamera& k) {
  constexpr bool metres = sizeof(D) == 4;
  const float nan = __uint_as_float(0x7fc00000u);
  const unsigned int width = k.width, height = k.height;
  for (unsigned int v = blockIdx.y; v < height; v += gridDim.y) {
    const D* drow = reinterpret_cast<const D*>(src + k.depth_off + (size_t)v * k.depth_step);
    const unsigned char* crow = src + k.bgr_off + (size_t)v * k.bgr_step;
    float4* orow = dst + k.out_off + (size_t)v * width;
    const float fy = (float)v - k.cy;
    for (unsigned int u = blockIdx.x * blockDim.x + threadIdx.x; u < width; u += gridDim.x * blockDim.x) {
      const D d = drow[u];
      float4 p = make_float4(nan, nan, nan, __uint_as_float(colour_rgba<C>(crow, u)));
      if (metres ? isfinite((float)d) : d != 0) {
        const float fd = (float)d;
        p.x = (((float)u - k.cx) * fd) * k.kx;
        p.y = (fy * fd) * k.ky;
        p.z = metres ? fd : fd * 0.001f;
        if (k.has_m && finite3(p)) xform(k.m, p.x, p.y, p.z, p.x, p.y, p.z);  // pcl::transformPointCloud, not dense
      }
      orow[u] = p;
    }
  }
}
template <typename D>
__device__ __forceinline__ void depth_image_colour(const unsigned char* __restrict__ src, float4* __restrict__ dst, const DepthCamera& k) {
  switch (k.colour_enc) {
    case PFT_COLOUR_BGR8: depth_image_camera<D, PFT_COLOUR_BGR8>(src, dst, k); break;
    case PFT_COLOUR_RGB8: depth_image_camera<D, PFT_COLOUR_RGB8>(src, dst, k); break;
    case PFT_COLOUR_BGRA8: depth_image_camera<D, PFT_COLOUR_BGRA8>(src, dst, k); break;
    case PFT_COLOUR_RGBA8: depth_image_camera<D, PFT_COLOUR_RGBA8>(src, dst, k); break;
    case PFT_COLOUR_MONO8: depth_image_camera<D, PFT_COLOUR_MONO8>(src, dst, k); break;
    default: depth_image_camera<D, PFT_COLOUR_NONE>(src, dst, k); break;
  }
}
// Pair = depth_enc * kColourEncodings + colour_enc when every camera of the frame has that pair of encodings: the
// block runs that pair's loop alone.  Pair = kMixedPairs: cameras with different pairs, each block dispatches on its
// camera's pair.  A block converts one row of 128 pixels, so the dispatch's dependent constant loads are a visible
// share of its time: +0.4 us (sd) and +0.6 us (qhd) per 16UC1 + bgr8 frame on a B200 at 1000 W, about 14 %.  Frames of
// one pair, the common case, skip it; the 16UC1 + bgr8 instance is the single-encoding kernel it replaces.  The mixed
// instance inlines all 12 loops: each alone needs at most 30 registers, together ptxas takes 38 unless bounded.  16
// blocks of 128 threads (32 registers, no spills) keep the SM at full occupancy.
constexpr int kColourEncodings = PFT_COLOUR_NONE + 1, kMixedPairs = 2 * kColourEncodings;
template <int Pair>
__global__ void __launch_bounds__(128, 16)
    depth_image_kernel(const unsigned char* __restrict__ src, float4* __restrict__ dst, const __grid_constant__ DepthCameras cams) {
  const DepthCamera& k = cams.cam[blockIdx.z];
  if constexpr (Pair == kMixedPairs) {
    if (k.depth_enc == PFT_DEPTH_32FC1) depth_image_colour<float>(src, dst, k);
    else depth_image_colour<unsigned short>(src, dst, k);
  } else {
    using D = std::conditional_t<Pair / kColourEncodings == PFT_DEPTH_32FC1, float, unsigned short>;
    depth_image_camera<D, Pair % kColourEncodings>(src, dst, k);
  }
}
using DepthImageKernel = void (*)(const unsigned char*, float4*, const DepthCameras);
template <int... Pair>
DepthImageKernel depth_image_instance(int pair, std::integer_sequence<int, Pair...>) {
  static constexpr DepthImageKernel instances[] = {&depth_image_kernel<Pair>...};
  return instances[pair];
}

// Depth image of a depth camera -> depth image registered into its colour camera: replaces the depth_image_proc/register
// nodelet (RegisterNodelet::convert<T>) in front of point_cloud_xyzrgb.  Depth pixel (u, v), visited in raster order
// upstream, back-projects in double (fill_upsampling: its two corners (u -/+ 0.5f, v -/+ 0.5f)), moves by the 3x4
// depth -> colour matrix, projects to colour pixel (int)(((fx x + Tx) / z + cx) + 0.5) (a rectangle between the two
// corners' pixels) and offers its z there as a T: the z-buffer keeps it `if (!valid(reg) || reg > new)`.  A candidate
// that is itself invalid (16UC1 0, 32FC1 -inf: a reset) replaces anything, so the result depends on the order of the
// candidates through the resets alone; at each colour pixel it is the smallest valid (or +inf) candidate after the last
// reset, the earliest of equal ones, else the reset value, else the initial one.  The GPU scatters twice: the reset
// kernel keeps each pixel's last reset (atomicMax of raster index + 1), the z-buffer kernel the least key (value in
// order-preserving bits, raster index, sign of a zero) of the later candidates, as atomicMax of its complement so that
// a zero-filled z-buffer is empty.  The finalise kernel writes the T image.  Thread = depth (colour) pixel along a row.
// Where upstream is undefined (a double -> int cast of NaN or outside int, a 16UC1 fromMeters outside 0 .. 65535), or
// a 32FC1 candidate is NaN, the candidate is dropped.
__device__ __forceinline__ bool to_int(double x, int& i) {
  if (!(x > -2147483649.0 && x < 2147483648.0)) return false;
  i = (int)x;  // truncation toward zero: (-1, 0) -> 0, as upstream
  return true;
}
__device__ __forceinline__ bool reg_project(const RegCamera& r, double pu, double pv, double depth, int& cu, int& cv, double& z) {
  const double X = ((pu - r.cx) * depth - r.tx) * r.inv_fx;
  const double Y = ((pv - r.cy) * depth - r.ty) * r.inv_fy;
  const double* m = r.m;
  const double x = ((m[0] * X + m[1] * Y) + m[2] * depth) + m[3];
  const double y = ((m[4] * X + m[5] * Y) + m[6] * depth) + m[7];
  z = ((m[8] * X + m[9] * Y) + m[10] * depth) + m[11];
  const double inv_z = __drcp_rn(z);  // = 1.0 / z, correctly rounded
  return to_int(((r.rgb_fx * x + r.rgb_tx) * inv_z + r.rgb_cx) + 0.5, cu) && to_int(((r.rgb_fy * y + r.rgb_ty) * inv_z + r.rgb_cy) + 0.5, cv);
}
// z-buffer key of a valid candidate (16UC1: the uint16, 32FC1: the float's bits): the value in order-preserving bits
// (+0 and -0 alike, +inf above every finite value), then the raster index, then the sign bit that tells -0 from +0
__device__ __forceinline__ unsigned long long reg_key(bool metres, unsigned int b, unsigned int idx) {
  const unsigned int o = !metres ? b : (b << 1) == 0 ? 0x80000000u : (b & 0x80000000u) ? ~b : (b | 0x80000000u);
  return ((unsigned long long)o << 32) | (idx << 1) | (metres ? b >> 31 : 0u);
}
__device__ __forceinline__ void reg_value(unsigned long long k, unsigned short& d) { d = (unsigned short)(k >> 32); }
__device__ __forceinline__ void reg_value(unsigned long long k, float& d) {
  const unsigned int o = (unsigned int)(k >> 32);
  d = __uint_as_float(o == 0x80000000u ? (unsigned int)(k & 1u) << 31 : (o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}

// The candidate of depth pixel (u, v): the colour rectangle [u1, u2] x [v1, v2] and the value's bits (16UC1: the
// uint16, 32FC1: the float).  Both encodings and both modes share one projection (one call site of the reciprocal's
// slow path, so nothing is spilled around it).
__device__ __forceinline__ bool reg_candidate(const RegCamera& r, const unsigned char* drow, unsigned int u, unsigned int v, int& u1, int& v1, int& u2,
                                              int& v2, unsigned int& val) {
  const bool metres = r.depth_enc == PFT_DEPTH_32FC1;
  const unsigned int d = metres ? reinterpret_cast<const unsigned int*>(drow)[u] : reinterpret_cast<const unsigned short*>(drow)[u];
  if (metres ? !isfinite(__uint_as_float(d)) : d == 0) return false;
  const double depth = metres ? (double)__uint_as_float(d) : (double)((float)d * 0.001f);  // DepthTraits<T>::toMeters
  double z1 = 0.0, z2 = 0.0;
  // fill_upsampling: corner (u - 0.5f, v - 0.5f), then (u + 0.5f, v + 0.5f), each a float sum upstream; else (u, v)
#pragma unroll 1
  for (int c = r.fill ? 0 : 1; c < 2; ++c) {
    const float off = c ? 0.5f : -0.5f;
    u1 = u2; v1 = v2; z1 = z2;
    if (!reg_project(r, r.fill ? (double)((float)u + off) : (double)u, r.fill ? (double)((float)v + off) : (double)v, depth, u2, v2, z2)) return false;
  }
  if (!r.fill) { u1 = u2; v1 = v2; }
  if (u1 < 0 || u2 >= (int)r.width || v1 < 0 || v2 >= (int)r.height) return false;
  const float m = r.fill ? (float)(0.5 * (z1 + z2)) : (float)z2;
  if (metres) {  // DepthTraits<float>::fromMeters
    val = __float_as_uint(m);
    return !isnan(m);
  }
  const float t = m * 1000.0f + 0.5f;  // DepthTraits<uint16_t>::fromMeters, undefined outside 0 .. 65535
  val = (unsigned int)(int)t;
  return t > -1.0f && t < 65536.0f;
}
// Pass 0: resets, pass 1: the other candidates after the last reset of their pixel.
template <int Pass>
__device__ __forceinline__ void register_camera(unsigned char* base, const RegCamera& r) {
  unsigned int* reset = reinterpret_cast<unsigned int*>(base + r.reset_off);
  unsigned long long* key = reinterpret_cast<unsigned long long*>(base + r.key_off);
  const bool metres = r.depth_enc == PFT_DEPTH_32FC1;
  for (unsigned int v = blockIdx.y; v < r.depth_height; v += gridDim.y) {
    const unsigned char* drow = base + r.raw_off + (size_t)v * r.depth_step;
    for (unsigned int u = blockIdx.x * blockDim.x + threadIdx.x; u < r.depth_width; u += gridDim.x * blockDim.x) {
      int u1 = 0, v1 = 0, u2 = 0, v2 = 0;
      unsigned int val;
      if (!reg_candidate(r, drow, u, v, u1, v1, u2, v2, val)) continue;
      if ((val == (metres ? 0xff800000u : 0u)) != (Pass == 0)) continue;  // 16UC1 0, 32FC1 -inf: a reset
      const unsigned int idx = v * r.depth_width + u;
      const unsigned long long k = ~reg_key(metres, val, idx);
      for (int cv = v1; cv <= v2; ++cv) {
        for (int cu = u1; cu <= u2; ++cu) {
          const size_t t = (size_t)cv * r.width + cu;
          if (Pass == 0) atomicMax(&reset[t], idx + 1);
          else if (idx >= reset[t]) atomicMax(&key[t], k);
        }
      }
    }
  }
}
template <typename D>
__device__ __forceinline__ void register_finalise_camera(unsigned char* base, const RegCamera& r) {
  const unsigned int* reset = reinterpret_cast<const unsigned int*>(base + r.reset_off);
  const unsigned long long* key = reinterpret_cast<const unsigned long long*>(base + r.key_off);
  D* reg = reinterpret_cast<D*>(base + r.reg_off);
  D initial = 0, reset_value = 0;  // 16UC1: 0 and 0
  if constexpr (sizeof(D) == 4) { initial = __uint_as_float(0x7fc00000u); reset_value = -INFINITY; }
  for (unsigned int v = blockIdx.y; v < r.height; v += gridDim.y) {
    for (unsigned int u = blockIdx.x * blockDim.x + threadIdx.x; u < r.width; u += gridDim.x * blockDim.x) {
      const size_t t = (size_t)v * r.width + u;
      const unsigned long long k = key[t];
      D d = reset[t] ? reset_value : initial;
      if (k) reg_value(~k, d);
      reg[t] = d;
    }
  }
}
// The reciprocal's slow path is a subroutine call, and ptxas spills a few bytes around it unless bounded: these bounds
// give 48 and 40 registers, no stack and no spills (-Xptxas -v).
__global__ void __launch_bounds__(128, 10) register_reset_kernel(unsigned char* base, const __grid_constant__ RegCameras cams) {
  register_camera<0>(base, cams.cam[blockIdx.z]);
}
__global__ void __launch_bounds__(128, 12) register_zbuffer_kernel(unsigned char* base, const __grid_constant__ RegCameras cams) {
  register_camera<1>(base, cams.cam[blockIdx.z]);
}
__global__ void __launch_bounds__(128) register_finalise_kernel(unsigned char* base, const __grid_constant__ RegCameras cams) {
  const RegCamera& r = cams.cam[blockIdx.z];
  if (!r.registered) return;
  if (r.depth_enc == PFT_DEPTH_32FC1) register_finalise_camera<float>(base, r);
  else register_finalise_camera<unsigned short>(base, r);
}

__global__ void set_header_kernel(CloudHeader* h, int n) { h->n = n; }

// ---- pcl::transformPointCloud (PCL 1.8.0, not dense): every point in input order, finite ones moved by the 3x4
// matrix, the others copied as they are, rgba kept.  The count is read from the input's header (no host round trip
// after a filter).  In place (in == out, out_hdr NULL) each thread reads its point before it writes it back.
struct Matrix12 { float m[12]; };
__global__ void __launch_bounds__(256) transform_cloud_kernel(const float4* in, const CloudHeader* __restrict__ in_hdr, float4* out,
                                                              CloudHeader* out_hdr, const Matrix12 m) {
  const int n = in_hdr->n;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) out[i] = transform_point(m.m, in[i]);
  if (out_hdr && blockIdx.x == 0 && threadIdx.x == 0) out_hdr->n = n;
}

// ---- PassThrough (order-preserving compaction), one thread block: flags -> exclusive scan -> scatter.
__global__ void __launch_bounds__(1024) passthrough_kernel(const float4* __restrict__ in, const CloudHeader* __restrict__ in_hdr,
                                                           float4* __restrict__ out, CloudHeader* out_hdr, int field, float lo,
                                                           float hi, int drop_zero) {
  __shared__ int smem[34];
  const int n = in_hdr->n;
  auto keep = [&](int i) -> int {
    const float4 p = in[i];
    if (!passes(p, field, lo, hi)) return 0;
    // removeZeroPoints (ref: src/auto_tracking.cpp:577-595): the comparison is made in double upstream
    if (drop_zero && fabs((double)p.x) < 0.01 && fabs((double)p.y) < 0.01 && fabs((double)p.z) < 0.01) return 0;
    return 1;
  };
  const int total = block_exclusive_scan<int>(
      n, keep, [&](int i, int ex) { const float4 p = in[i]; if (keep(i)) out[ex] = p; }, smem);
  if (threadIdx.x == 0) out_hdr->n = total;
}

// ---- K1a: insert every surviving point's voxel key; remember the lowest point index per voxel.
// A slot is {ix, iy, iz, 1} once claimed, all zero while empty; one 16-byte compare-and-swap claims it or returns its key.
__global__ void k1_insert_kernel(const float4* __restrict__ in, const CloudHeader* __restrict__ in_hdr, int4* keys, int* first,
                                 int* __restrict__ slot_of, unsigned int mask, float inv, int field, float lo, float hi) {
  const int n = in_hdr->n;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = in[i];
    int slot = -1;
    if (passes(p, field, lo, hi)) {
      const int4 key = make_int4(voxel_index(p.x, inv), voxel_index(p.y, inv), voxel_index(p.z, inv), 1);
      unsigned int s = voxel_hash(key.x, key.y, key.z) & mask;
      while (true) {
        const int4 prev = atomicCAS(&keys[s], make_int4(0, 0, 0, 0), key);
        if (prev.w == 0 || (prev.x == key.x && prev.y == key.y && prev.z == key.z)) break;
        s = (s + 1) & mask;
      }
      slot = (int)s;
      atomicMin(&first[s], i);
    }
    slot_of[i] = slot;
  }
}
// ---- K1b: voxel id = rank of the voxel's first point among all first points (output order = order of first
// appearance).  Three small kernels: per-tile counts, one-block scan of the tile counts, per-tile assignment.
constexpr int kTile = 4096;  // points per block (1024 threads x 4)

__device__ __forceinline__ int k1_is_first(int i, int n, const int* __restrict__ slot_of, const int* __restrict__ first) {
  if (i >= n) return 0;
  const int s = slot_of[i];
  return (s >= 0 && first[s] == i) ? 1 : 0;
}
__global__ void __launch_bounds__(1024) k1_tile_count_kernel(const CloudHeader* __restrict__ in_hdr, const int* __restrict__ slot_of,
                                                             const int* __restrict__ first, int* __restrict__ tile_count) {
  __shared__ int red[32];
  const int n = in_hdr->n;
  const int base = blockIdx.x * kTile + threadIdx.x * 4;
  int c = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) c += k1_is_first(base + k, n, slot_of, first);
  c = warp_sum(c);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x < 32) {
    int v = red[threadIdx.x];
    v = warp_sum(v);
    if (threadIdx.x == 0) tile_count[blockIdx.x] = v;
  }
}
__global__ void __launch_bounds__(1024) k1_tile_scan_kernel(int n_tiles, int* tile_count, CloudHeader* out_hdr) {
  __shared__ int smem[34];
  const int total = block_exclusive_scan<int>(
      n_tiles, [&](int i) { return tile_count[i]; }, [&](int i, int ex) { tile_count[i] = ex; }, smem);
  if (threadIdx.x == 0) out_hdr->n = total;
}
__global__ void __launch_bounds__(1024) k1_tile_assign_kernel(const CloudHeader* __restrict__ in_hdr, const int* __restrict__ slot_of,
                                                              const int* __restrict__ first, const int* __restrict__ tile_offset,
                                                              int* __restrict__ vid, double* acc_xyz, unsigned int* acc_rgbc) {
  __shared__ int wsum[32];
  const int n = in_hdr->n;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int base = blockIdx.x * kTile + threadIdx.x * 4;
  int f[4], sum = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) { f[k] = k1_is_first(base + k, n, slot_of, first); sum += f[k]; }
  int inc = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(kFull, inc, o); if (lane >= o) inc += t; }
  if (lane == 31) wsum[wid] = inc;
  __syncthreads();
  if (wid == 0) {
    const int w = wsum[lane];
    int winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(kFull, winc, o); if (lane >= o) winc += t; }
    wsum[lane] = winc - w;
  }
  __syncthreads();
  int ex = tile_offset[blockIdx.x] + wsum[wid] + (inc - sum);
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (f[k]) {
      vid[slot_of[base + k]] = ex;  // (the accumulators were cleared by two contiguous memsets before the pass)
      ++ex;
    }
  }
}
// ---- K1c: accumulate in fp64.  Every fp32 coordinate is a multiple of its own ulp, so a voxel's sums are exact, and
// the centroid does not depend on the order the atomics land in, while they stay below 2^53 times the smallest ulp among
// the voxel's coordinates.  That holds in every voxel whose index is neither 0 nor -1 on an axis: its coordinates on
// that axis are within a factor of about 2 of each other (2^25 ulps), so up to 2^28 points sum exactly.  A voxel on a
// coordinate plane can also hold coordinates far below the leaf size; next to leaf-sized ones (below about 2^-36 m
// with centimetre-scale ones at a 1 cm leaf) the sum rounds, and its last bit can depend on the order.
__global__ void k1_accum_kernel(const float4* __restrict__ in, const CloudHeader* __restrict__ in_hdr, const int* __restrict__ slot_of,
                                const int* __restrict__ vid, double* acc_xyz, unsigned int* acc_rgbc) {
  const int n = in_hdr->n;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int s = slot_of[i];
    if (s < 0) continue;
    const int v = vid[s];
    const float4 p = in[i];
    const unsigned int rgba = __float_as_uint(p.w);
    atomicAdd(&acc_xyz[3 * v], (double)p.x);
    atomicAdd(&acc_xyz[3 * v + 1], (double)p.y);
    atomicAdd(&acc_xyz[3 * v + 2], (double)p.z);
    atomicAdd(&acc_rgbc[4 * v], (rgba >> 16) & 0xffu);
    atomicAdd(&acc_rgbc[4 * v + 1], (rgba >> 8) & 0xffu);
    atomicAdd(&acc_rgbc[4 * v + 2], rgba & 0xffu);
    atomicAdd(&acc_rgbc[4 * v + 3], 1u);
  }
}
// ---- K1d: centroid = fp64 quotient rounded to fp32; colour = (int)(float_sum / float_count), alpha 0
__global__ void k1_final_kernel(const CloudHeader* __restrict__ out_hdr, const double* __restrict__ acc_xyz,
                                const unsigned int* __restrict__ acc_rgbc, float4* __restrict__ out) {
  const int n = out_hdr->n;
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < n; v += gridDim.x * blockDim.x) {
    const uint4 c = reinterpret_cast<const uint4*>(acc_rgbc)[v];
    const double cnt = (double)c.w;
    const float fc = (float)c.w;
    const unsigned int r = (unsigned int)(int)((float)c.x / fc), g = (unsigned int)(int)((float)c.y / fc), b = (unsigned int)(int)((float)c.z / fc);
    out[v] = make_float4((float)(acc_xyz[3 * v] / cnt), (float)(acc_xyz[3 * v + 1] / cnt), (float)(acc_xyz[3 * v + 2] / cnt),
                         __uint_as_float((r << 16) | (g << 8) | b));
  }
}

// ---- pcl::ApproximateVoxelGrid<PointXYZRGBA>::applyFilter reproduced exactly (PCL-1.8.0 filters/impl/approximate_voxel_grid.hpp,
// SURVEY A.1; ref: src/auto_tracking.cpp:563-575): a 512-entry direct-mapped cache of voxel accumulators walked in input
// order, an entry flushed (a partial centroid emitted) whenever another voxel hashes onto it, the rest flushed at the end
// in slot order.  Output order, duplicate partial centroids and the sequential fp32 sums all depend on the input order:
// the algorithm is a sequential scan, run here by ONE thread.  Parity mode (pft_approx_voxel_grid_pcl); the product
// path is the exact one-centroid-per-voxel reduction above.
__global__ void approx_voxel_grid_pcl_kernel(const float4* __restrict__ in, const CloudHeader* __restrict__ in_hdr, float inv, int field, float lo,
                                             float hi, float4* __restrict__ out, CloudHeader* out_hdr) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  constexpr int kHist = 512;
  __shared__ int s_key[kHist][4];   // ix, iy, iz, count
  __shared__ float s_acc[kHist][6]; // x, y, z, r, g, b  (upstream's 7-vector also carries the constant 1 of the padding lane)
  for (int k = 0; k < kHist; ++k) { s_key[k][3] = 0; for (int q = 0; q < 6; ++q) s_acc[k][q] = 0.f; }
  const int n = in_hdr->n;
  int op = 0;
  auto flush = [&](int k) {
    const float cnt = (float)s_key[k][3];
    const unsigned int r = (unsigned int)(int)(s_acc[k][3] / cnt), g = (unsigned int)(int)(s_acc[k][4] / cnt), b = (unsigned int)(int)(s_acc[k][5] / cnt);
    out[op++] = make_float4(s_acc[k][0] / cnt, s_acc[k][1] / cnt, s_acc[k][2] / cnt, __uint_as_float((r << 16) | (g << 8) | b));
  };
  for (int i = 0; i < n; ++i) {
    const float4 p = in[i];
    if (!passes(p, field, lo, hi)) continue;  // the PassThrough that precedes the grid (ref :637), order preserving
    const int ix = voxel_index(p.x, inv), iy = voxel_index(p.y, inv), iz = voxel_index(p.z, inv);
    // upstream's int hash in unsigned arithmetic: the same bits, without signed overflow
    const int k = (int)(((unsigned int)ix * 7171u + (unsigned int)iy * 3079u + (unsigned int)iz * 4231u) & (unsigned int)(kHist - 1));
    if (s_key[k][3] && (ix != s_key[k][0] || iy != s_key[k][1] || iz != s_key[k][2])) {
      flush(k);
      s_key[k][3] = 0;
      for (int q = 0; q < 6; ++q) s_acc[k][q] = 0.f;
    }
    s_key[k][0] = ix; s_key[k][1] = iy; s_key[k][2] = iz; s_key[k][3]++;
    const unsigned int rgba = __float_as_uint(p.w);
    s_acc[k][0] += p.x; s_acc[k][1] += p.y; s_acc[k][2] += p.z;
    s_acc[k][3] += (float)((rgba >> 16) & 0xffu); s_acc[k][4] += (float)((rgba >> 8) & 0xffu); s_acc[k][5] += (float)(rgba & 0xffu);
  }
  for (int k = 0; k < kHist; ++k) if (s_key[k][3]) flush(k);
  out_hdr->n = op;
}

// ---- centroid (fp64 sums, exact) and in-place translation by -centroid; one block.
__global__ void __launch_bounds__(1024) centre_kernel(float4* pts, const CloudHeader* __restrict__ hdr, float* centroid3) {
  __shared__ double red[32];
  __shared__ float c[3];
  const int n = hdr->n;
  double sx = 0, sy = 0, sz = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) { const float4 p = pts[i]; sx += (double)p.x; sy += (double)p.y; sz += (double)p.z; }
  sx = block_sum(sx, red); sy = block_sum(sy, red); sz = block_sum(sz, red);
  if (threadIdx.x == 0) {
    const double dn = n > 0 ? (double)n : 1.0;
    c[0] = (float)(sx / dn); c[1] = (float)(sy / dn); c[2] = (float)(sz / dn);
    centroid3[0] = c[0]; centroid3[1] = c[1]; centroid3[2] = c[2];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) { float4 p = pts[i]; p.x = p.x - c[0]; p.y = p.y - c[1]; p.z = p.z - c[2]; pts[i] = p; }
}

inline int grid_for(size_t n, int block, int sm_count) {
  size_t g = (n + block - 1) / block;
  size_t cap = (size_t)sm_count * 8;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace

int launch_unpack_pcl32(cudaStream_t s, const void* src32, float4* dst, size_t n) {
  if (n == 0) return PFT_OK;
  unpack_pcl32_kernel<<<grid_for(n, 256, 148), 256, 0, s>>>(reinterpret_cast<const uint4*>(src32), dst, n);
  PFT_LAUNCH_CHECK();
  return PFT_OK;
}
int launch_unpack_pointcloud2(cudaStream_t s, const void* src, float4* dst, unsigned int width, unsigned int height, unsigned int point_step,
                              unsigned int row_step, int off_x, int off_y, int off_z, int off_rgb) {
  const size_t n = (size_t)width * height;
  if (n == 0) return PFT_OK;
  unpack_pointcloud2_kernel<<<grid_for(n, 256, 148), 256, 0, s>>>(reinterpret_cast<const unsigned int*>(src), dst, width, height, point_step / 4, row_step / 4,
                                                                 off_x / 4, off_y / 4, off_z / 4, off_rgb >= 0 ? off_rgb / 4 : -1);
  PFT_LAUNCH_CHECK();
  return PFT_OK;
}
int launch_depth_image(cudaStream_t s, const void* src, float4* dst, const DepthCameras& cams, int n) {
  if (n < 1) return PFT_OK;
  // blocks past a smaller camera's width or height find no pixel and return
  unsigned int width = 0, height = 0;
  int pair = cams.cam[0].depth_enc * kColourEncodings + cams.cam[0].colour_enc;
  for (int k = 0; k < n; ++k) {
    width = cams.cam[k].width > width ? cams.cam[k].width : width;
    height = cams.cam[k].height > height ? cams.cam[k].height : height;
    if (cams.cam[k].depth_enc * kColourEncodings + cams.cam[k].colour_enc != pair) pair = kMixedPairs;
  }
  const dim3 grid((width + 127) / 128, height < 65535u ? height : 65535u, (unsigned int)n);
  const DepthImageKernel kernel = depth_image_instance(pair, std::make_integer_sequence<int, kMixedPairs + 1>());
  kernel<<<grid, 128, 0, s>>>(reinterpret_cast<const unsigned char*>(src), dst, cams);
  PFT_LAUNCH_CHECK();
  return PFT_OK;
}
int launch_register_depth(cudaStream_t s, void* staging, const RegCameras& cams, int n) {
  // three launches whatever the cameras: a grid without a pixel to visit still runs
  unsigned int dw = 1, dh = 1, w = 1, h = 1;
  for (int k = 0; k < n; ++k) {
    const RegCamera& r = cams.cam[k];
    if (!r.registered) continue;
    dw = r.depth_width > dw ? r.depth_width : dw;
    dh = r.depth_height > dh ? r.depth_height : dh;
    w = r.width > w ? r.width : w;
    h = r.height > h ? r.height : h;
  }
  unsigned char* base = reinterpret_cast<unsigned char*>(staging);
  const dim3 scatter((dw + 127) / 128, dh < 65535u ? dh : 65535u, (unsigned int)n), finalise((w + 127) / 128, h < 65535u ? h : 65535u, (unsigned int)n);
  register_reset_kernel<<<scatter, 128, 0, s>>>(base, cams);
  PFT_LAUNCH_CHECK();
  register_zbuffer_kernel<<<scatter, 128, 0, s>>>(base, cams);
  PFT_LAUNCH_CHECK();
  register_finalise_kernel<<<finalise, 128, 0, s>>>(base, cams);
  PFT_LAUNCH_CHECK();
  return PFT_OK;
}
int launch_pack_pcl32(cudaStream_t s, const float4* src, void* dst32, size_t n) {
  if (n == 0) return PFT_OK;
  pack_pcl32_kernel<<<grid_for(n, 256, 148), 256, 0, s>>>(src, reinterpret_cast<uint4*>(dst32), n);
  PFT_LAUNCH_CHECK();
  return PFT_OK;
}
int launch_set_header(cudaStream_t s, CloudHeader* hdr, int n) {
  set_header_kernel<<<1, 1, 0, s>>>(hdr, n);
  PFT_LAUNCH_CHECK();
  return PFT_OK;
}

int run_passthrough(pft_context* ctx, const pft_cloud* in, pft_cloud* out, int field, float lo, float hi, int drop_zero) {
  int rc = out->ensure(in->capacity);
  if (rc) return rc;
  passthrough_kernel<<<1, 1024, 0, ctx->stream>>>(in->d_pts(), in->d_hdr(), out->d_pts(), out->d_hdr(), field, lo, hi, drop_zero);
  PFT_LAUNCH_CHECK();
  out->written(-1);
  return PFT_OK;
}

int run_transform_cloud(pft_context* ctx, const pft_cloud* in, pft_cloud* out, const float* m12) {
  const bool in_place = in == out;
  if (!in_place) {
    int rc = out->ensure(in->capacity);
    if (rc) return rc;
  }
  Matrix12 m;
  memcpy(m.m, m12, sizeof(m.m));
  transform_cloud_kernel<<<grid_for(in->capacity, 256, ctx->sm_count), 256, 0, ctx->stream>>>(in->d_pts(), in->d_hdr(), out->d_pts(),
                                                                                           in_place ? nullptr : out->d_hdr(), m);
  PFT_LAUNCH_CHECK();
  out->written(in->host_n);
  return PFT_OK;
}

// The ten stream operations of one downsample (4 memsets + 6 kernels).
static int enqueue_voxel_grid(pft_context* ctx, const pft_cloud* in, pft_cloud* out, float leaf, int field, float lo, float hi, size_t cap, size_t H,
                              int n_tiles) {
  cudaStream_t s = ctx->stream;
  PFT_CUDA_TRY(cudaMemsetAsync(ctx->k1_keys.p, 0, H * sizeof(int4), s));
  PFT_CUDA_TRY(cudaMemsetAsync(ctx->k1_first.p, 0x7f, H * sizeof(int), s));
  PFT_CUDA_TRY(cudaMemsetAsync(ctx->k1_acc_xyz.p, 0, cap * 3 * sizeof(double), s));
  PFT_CUDA_TRY(cudaMemsetAsync(ctx->k1_acc_rgbc.p, 0, cap * 4 * sizeof(unsigned int), s));
  const float inv = 1.0f / leaf;
  const int grid = grid_for(cap, 256, ctx->sm_count);
  k1_insert_kernel<<<grid, 256, 0, s>>>(in->d_pts(), in->d_hdr(), ctx->k1_keys.as<int4>(), ctx->k1_first.as<int>(),
                                        ctx->k1_slot_of.as<int>(), (unsigned int)(H - 1), inv, field, lo, hi);
  PFT_LAUNCH_CHECK();
  k1_tile_count_kernel<<<n_tiles, 1024, 0, s>>>(in->d_hdr(), ctx->k1_slot_of.as<int>(), ctx->k1_first.as<int>(), ctx->k1_blk.as<int>());
  PFT_LAUNCH_CHECK();
  k1_tile_scan_kernel<<<1, 1024, 0, s>>>(n_tiles, ctx->k1_blk.as<int>(), out->d_hdr());
  PFT_LAUNCH_CHECK();
  k1_tile_assign_kernel<<<n_tiles, 1024, 0, s>>>(in->d_hdr(), ctx->k1_slot_of.as<int>(), ctx->k1_first.as<int>(), ctx->k1_blk.as<int>(),
                                                 ctx->k1_vid.as<int>(), ctx->k1_acc_xyz.as<double>(), ctx->k1_acc_rgbc.as<unsigned int>());
  PFT_LAUNCH_CHECK();
  k1_accum_kernel<<<grid, 256, 0, s>>>(in->d_pts(), in->d_hdr(), ctx->k1_slot_of.as<int>(), ctx->k1_vid.as<int>(),
                                       ctx->k1_acc_xyz.as<double>(), ctx->k1_acc_rgbc.as<unsigned int>());
  PFT_LAUNCH_CHECK();
  k1_final_kernel<<<grid, 256, 0, s>>>(out->d_hdr(), ctx->k1_acc_xyz.as<double>(), ctx->k1_acc_rgbc.as<unsigned int>(), out->d_pts());
  PFT_LAUNCH_CHECK();
  return PFT_OK;
}

int run_voxel_grid(pft_context* ctx, const pft_cloud* in, pft_cloud* out, float leaf, int field, float lo, float hi) {
  if (!(leaf > 0.f)) { set_last_error("leaf size must be positive"); return PFT_ERR_INVALID; }
  const size_t cap = in->capacity;
  int rc = out->ensure(cap);
  if (rc) return rc;
  if (cap == 0) return launch_set_header(ctx->stream, out->d_hdr(), 0);
  size_t H = 1024;
  while (H < 2 * cap) H <<= 1;
  if ((rc = ctx->k1_keys.reserve(H * sizeof(int4)))) return rc;
  if ((rc = ctx->k1_first.reserve(H * sizeof(int)))) return rc;
  if ((rc = ctx->k1_vid.reserve(H * sizeof(int)))) return rc;
  if ((rc = ctx->k1_slot_of.reserve(cap * sizeof(int)))) return rc;
  if ((rc = ctx->k1_acc_xyz.reserve(cap * 3 * sizeof(double)))) return rc;
  if ((rc = ctx->k1_acc_rgbc.reserve(cap * 4 * sizeof(unsigned int)))) return rc;
  const int n_tiles = (int)((cap + kTile - 1) / kTile);
  if ((rc = ctx->k1_blk.reserve((size_t)n_tiles * sizeof(int)))) return rc;
  out->written(-1);
  (void)kFirstInit;
  // A camera stream downsamples frame after frame between the same buffers: the ten operations are captured once
  // into a CUDA graph and replayed (one launch per frame instead of ten).  Everything the sequence touches is in the key.
  static const bool use_graph = [] { const char* e = getenv("PFT_NO_GRAPH"); return !(e && e[0] == '1'); }();
  if (!use_graph) return enqueue_voxel_grid(ctx, in, out, leaf, field, lo, hi, cap, H, n_tiles);
  pft_context::K1Key key;
  memset(&key, 0, sizeof(key));
  key.p[0] = in->d_pts(); key.p[1] = in->d_hdr(); key.p[2] = out->d_pts(); key.p[3] = out->d_hdr();
  key.p[4] = ctx->k1_keys.p; key.p[5] = ctx->k1_first.p; key.p[6] = ctx->k1_vid.p; key.p[7] = ctx->k1_slot_of.p;
  key.p[8] = ctx->k1_acc_xyz.p; key.p[9] = ctx->k1_acc_rgbc.p; key.p[10] = ctx->k1_blk.p;
  key.cap = cap; key.H = H; key.leaf = leaf; key.lo = lo; key.hi = hi; key.field = field;
  // a few alternating (in, out) pairs are common (double-buffered frames): keep a small set of graphs
  int slot = -1;
  for (int k = 0; k < pft_context::kK1Graphs; ++k)
    if (ctx->k1_exec[k] && memcmp(&ctx->k1_key[k], &key, sizeof(key)) == 0) { slot = k; break; }
  if (slot < 0) {
    slot = ctx->k1_next;
    ctx->k1_next = (ctx->k1_next + 1) % pft_context::kK1Graphs;
    if (ctx->k1_exec[slot]) { cudaGraphExecDestroy(ctx->k1_exec[slot]); ctx->k1_exec[slot] = nullptr; }
    cudaGraph_t graph = nullptr;
    const unsigned long long before = g_launch_count.load();
    PFT_CUDA_TRY(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
    rc = enqueue_voxel_grid(ctx, in, out, leaf, field, lo, hi, cap, H, n_tiles);
    cudaError_t ce = cudaStreamEndCapture(ctx->stream, &graph);
    g_launch_count -= g_launch_count.load() - before;  // captured, not launched
    if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
    if (ce != cudaSuccess) { set_last_error("downsample graph capture failed: %s", cudaGetErrorString(ce)); cudaGetLastError(); return PFT_ERR_CUDA; }
    cudaError_t ie = cudaGraphInstantiate(&ctx->k1_exec[slot], graph, 0);
    cudaGraphDestroy(graph);
    if (ie != cudaSuccess) { set_last_error("downsample graph instantiate failed: %s", cudaGetErrorString(ie)); cudaGetLastError(); ctx->k1_exec[slot] = nullptr; return PFT_ERR_CUDA; }
    ctx->k1_key[slot] = key;
  }
  PFT_CUDA_TRY(cudaGraphLaunch(ctx->k1_exec[slot], ctx->stream));
  g_launch_count += 6;  // the six kernels of the sequence
  return PFT_OK;
}

int run_approx_voxel_grid_pcl(pft_context* ctx, const pft_cloud* in, pft_cloud* out, float leaf, int field, float lo, float hi) {
  if (!(leaf > 0.f)) { set_last_error("leaf size must be positive"); return PFT_ERR_INVALID; }
  int rc = out->ensure(in->capacity);
  if (rc) return rc;
  approx_voxel_grid_pcl_kernel<<<1, 32, 0, ctx->stream>>>(in->d_pts(), in->d_hdr(), 1.0f / leaf, field, lo, hi, out->d_pts(), out->d_hdr());
  PFT_LAUNCH_CHECK();
  out->written(-1);
  return PFT_OK;
}

int run_centre_on_centroid(pft_context* ctx, pft_cloud* cloud, float* d_centroid3) {
  centre_kernel<<<1, 1024, 0, ctx->stream>>>(cloud->d_pts(), cloud->d_hdr(), d_centroid3);
  PFT_LAUNCH_CHECK();
  return PFT_OK;
}

}  // namespace pft
