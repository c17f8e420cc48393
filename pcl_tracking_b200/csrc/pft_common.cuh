// pft_common.cuh -- internal helpers shared by the sm_100a kernels of the tracker.
//
// Arithmetic contract (DESIGN.md "Arithmetic contract"): this library is compiled with
// -fmad=false, so every fp32/fp64 add and multiply is rounded on its own exactly as the x86-64
// default-march build of PCL does it; sin/cos/atan2/asin/exp are evaluated in double and rounded
// to float where PCL calls the float overloads.  That is what makes nearest-neighbour indices
// comparable bit-for-bit with the CPU oracle.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <float.h>
#include <string.h>

#include <atomic>

namespace pft {

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;

// ------------------------------------------------------------------ error plumbing (host)
void set_last_error(const char* fmt, ...);
extern std::atomic<unsigned long long> g_launch_count;  // (trackers of distinct contexts may be driven from distinct threads)
#define PFT_CUDA_TRY(expr)                                                                         \
  do {                                                                                             \
    cudaError_t _e = (expr);                                                                       \
    if (_e != cudaSuccess) {                                                                       \
      ::pft::set_last_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return PFT_ERR_CUDA;                                                                         \
    }                                                                                              \
  } while (0)
#define PFT_LAUNCH_CHECK()                                                                         \
  do {                                                                                             \
    ++::pft::g_launch_count;                                                                       \
    cudaError_t _e = cudaGetLastError();                                                           \
    if (_e != cudaSuccess) {                                                                       \
      ::pft::set_last_error("%s:%d: kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
      return PFT_ERR_CUDA;                                                                         \
    }                                                                                              \
  } while (0)

// ------------------------------------------------------------------ device structs
// Device point: float4 {x, y, z, bits}.  bits = rgba for clouds, packed HSV (h | s<<8 | v<<16) for
// the model and the sorted scene index.
struct __align__(16) DevParticle { float x, y, z, one, roll, pitch, yaw, weight; };  // = pcl ParticleXYZRPY

// Device-resident cloud header: the point count lives on the device so that no stage needs a host
// round trip (cloud sizes after K1, particle counts after the KLD resample).
struct CloudHeader { int n; int pad[3]; };

// Scene index header, recomputed by every weight() call from the crop AABB.
struct IndexHeader {
  float aabb[6];      // crop box: minx,miny,minz,maxx,maxy,maxz (inclusive, fp32)
  int origin[3];      // lattice coordinate (at `level`) of cell (0,0,0)
  int dim[3];         // cells per axis
  int level;          // cell edge = resolution * 2^level
  int n_cells;        // dim[0] * dim[1] * dim[2]
  int n_cropped;      // scene points inside the crop box (= indexed points)
  float cell;         // cell edge in metres
  float inv_leaf;     // 1 / resolution  (lattice = floor((coord * inv_leaf) * 2^-level))
  float level_scale;  // 2^-level
  int valid;          // 0: empty AABB (no model / no particles)
  // candidate lists: one list of index slots per cell of the FINE lattice (edge = resolution) over the crop box
  int f_origin[3];    // fine lattice coordinate of fine cell (0,0,0)
  int f_dim[3];
  int f_cells;        // f_dim[0] * f_dim[1] * f_dim[2]
  int use_lists;      // lists are built and used by this weight() (enough queries to amortise the build)
  // One index per frame: with the lists on, the index covers the crop box DILATED by a margin (`built`), so that the
  // later weight() calls of the same compute() -- whose crop boxes differ by the step noise of one resample -- find
  // their points in it and only build the lists of the cells their queries newly reach.  Exactness: a nearest
  // neighbour found among the points of `built` that lies inside the crop box IS the nearest neighbour among the
  // cropped points.  The list build keeps that true for every query: cells whose lists can only depend on points well
  // inside the crop box are built from all points and reused; cells near the faces are built from the cropped points
  // only and rebuilt by the next weight().  (Safety net: a winner outside the crop box -- flag in bit 31 of the staged
  // point's fourth word -- would send the query to the brute-force search over the cropped points.)
  float built[6];     // box the indexed points were taken from (= aabb when the lists are off)
  float core[6];      // hull of the crop boxes of the frame so far, each shrunk by `dilate`: the lists marked reusable only
                      // depend on points inside it, so a later crop box must contain it (and lie inside `built`)
  float dilate;       // the margin (0: the index holds the crop box only and nothing is reused)
  int reuse;          // this weight() reuses the index of an earlier weight() of the frame (its crop box lies in `built`)
  int n_in_crop;      // indexed points inside the crop box of THIS weight() (what cropInputPointCloud would return)
  unsigned int epoch; // weight() calls so far (diagnostics)
};

// ------------------------------------------------------------------ device helpers
__device__ __forceinline__ void atomic_min_float(float* addr, float v) {
  if (v >= 0.f) atomicMin(reinterpret_cast<int*>(addr), __float_as_int(v));
  else atomicMax(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}
__device__ __forceinline__ void atomic_max_float(float* addr, float v) {
  if (v >= 0.f) atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));
  else atomicMin(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}

__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(kFull, v, o));
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(kFull, v, o));
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}
__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}

// ------------------------------------------------------------------ pcl::transformPointCloud (PCL 1.8.0, common/impl/transforms.hpp)
// m = 3x4 row-major [R|t].  Dense branch: x' = ((m00 x + m01 y) + m02 z) + m03, y' and z' likewise, every fp32
// operation rounded on its own (-fmad=false).
__device__ __forceinline__ void xform(const float* m, float x, float y, float z, float& ox, float& oy, float& oz) {
  ox = ((m[0] * x + m[1] * y) + m[2] * z) + m[3];
  oy = ((m[4] * x + m[5] * y) + m[6] * z) + m[7];
  oz = ((m[8] * x + m[9] * y) + m[10] * z) + m[11];
}
// Non-dense branch: a point with a non-finite coordinate is copied as it is; the fourth word (rgba) is kept.
__device__ __forceinline__ float4 transform_point(const float* m, float4 p) {
  if (isfinite(p.x) && isfinite(p.y) && isfinite(p.z)) xform(m, p.x, p.y, p.z, p.x, p.y, p.z);
  return p;
}

// ------------------------------------------------------------------ bulk async copy (TMA, 1-D) + mbarrier
// One thread arms the barrier with the byte count and issues the copies; every consumer waits on the phase bit.
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// global -> shared, `bytes` a multiple of 16, both addresses 16-byte aligned; completion is counted on `bar`
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes),
               "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, uint32_t parity) {
  asm volatile(
      "{\n .reg .pred p;\n WAIT_%=:\n mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n @p bra DONE_%=;\n bra WAIT_%=;\n DONE_%=:\n}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

// ------------------------------------------------------------------ packed fp32 pairs (FADD2 / FMUL2: IEEE round-to-nearest per half, no contraction)
__device__ __forceinline__ float2 sub2_rn(float2 a, float2 b) {
  unsigned long long ra, rb, rc;
  memcpy(&ra, &a, 8); memcpy(&rb, &b, 8);
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(rc) : "l"(ra), "l"(rb));
  float2 c; memcpy(&c, &rc, 8);
  return c;
}
__device__ __forceinline__ float2 mul2_rn(float2 a, float2 b) {
  unsigned long long ra, rb, rc;
  memcpy(&ra, &a, 8); memcpy(&rb, &b, 8);
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(rc) : "l"(ra), "l"(rb));
  float2 c; memcpy(&c, &rc, 8);
  return c;
}
__device__ __forceinline__ float2 add2_rn(float2 a, float2 b) {
  unsigned long long ra, rb, rc;
  memcpy(&ra, &a, 8); memcpy(&rb, &b, 8);
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(rc) : "l"(ra), "l"(rb));
  float2 c; memcpy(&c, &rc, 8);
  return c;
}

// 1 / x for a finite double x >= 1: hardware seed (20 bits) + two Newton steps (explicit fused multiply-adds: the
// error of the result is below one ulp; it is not the correctly rounded quotient, see DESIGN "Arithmetic contract")
__device__ __forceinline__ double rcp_f64(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  double e = __fma_rn(-x, r, 1.0);
  r = __fma_rn(r, e, r);
  e = __fma_rn(-x, r, 1.0);
  r = __fma_rn(r, e, r);
  return r;
}

// Block-wide sum of doubles; result valid in thread 0.  `red` holds >= 32 doubles.
__device__ __forceinline__ double block_sum(double v, double* red) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) red[wid] = v;
  __syncthreads();
  if (wid == 0) {
    double t = lane < nw ? red[lane] : 0.0;
    t = warp_sum(t);
    v = t;
  }
  return v;
}

// Six block-wide sums at once (same association order as six block_sum calls, two barriers instead of twelve);
// results valid in thread 0.  `red6` holds >= 192 doubles.
__device__ __forceinline__ void block_sum6(double* v, double* red6) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int d = 0; d < 6; ++d) v[d] = warp_sum(v[d]);
  __syncthreads();
  if (lane == 0) {
#pragma unroll
    for (int d = 0; d < 6; ++d) red6[wid * 6 + d] = v[d];
  }
  __syncthreads();
  if (wid == 0) {
#pragma unroll
    for (int d = 0; d < 6; ++d) {
      double t = lane < nw ? red6[lane * 6 + d] : 0.0;
      v[d] = warp_sum(t);
    }
  }
}

// Exclusive scan over n values produced by `load(i)`, written through `store(i, exclusive_prefix)`,
// executed by ONE thread block (any size that is a multiple of 32, <= 1024).  Returns the grand
// total to every thread.  Integer types only: the result is independent of the association order,
// which is what makes cumulative tables bit-identical to a sequential CPU loop.
template <typename T, typename Load, typename Store>
__device__ T block_exclusive_scan(int n, Load load, Store store, T* smem /* >= 33 entries */) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  constexpr int ITEMS = 4;
  T carry = 0;
  const int tile = blockDim.x * ITEMS;
  for (int base = 0; base < n; base += tile) {
    T v[ITEMS];
    T sum = 0;
    const int i0 = base + threadIdx.x * ITEMS;
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) { v[k] = (i0 + k < n) ? load(i0 + k) : T(0); sum += v[k]; }
    T inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { T t = __shfl_up_sync(kFull, inc, o); if (lane >= o) inc += t; }
    __syncthreads();
    if (lane == 31) smem[wid] = inc;
    __syncthreads();
    if (wid == 0) {
      T w = lane < nw ? smem[lane] : T(0);
      T winc = w;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { T t = __shfl_up_sync(kFull, winc, o); if (lane >= o) winc += t; }
      smem[lane] = winc - w;            // exclusive prefix of warp totals
      if (lane == 31) smem[32] = winc;  // tile total
    }
    __syncthreads();
    T ex = carry + smem[wid] + (inc - sum);
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) { if (i0 + k < n) store(i0 + k, ex); ex += v[k]; }
    carry += smem[32];
  }
  __syncthreads();
  return carry;
}

}  // namespace pft
