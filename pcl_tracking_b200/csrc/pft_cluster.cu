// pft_cluster.cu -- model acquisition (SURVEY 8 f-2): Euclidean cluster extraction on the GPU.
//
// Replaces pcl::EuclideanClusterExtraction as used by the model builder (ref: src/create_model.cpp:169-179:
// KdTree + setClusterTolerance(0.02) + setMinClusterSize(500) + setMaxClusterSize(25000) + extract), whose clusters
// become the reference clouds of the trackers (ref: src/create_model.cpp:209-230, src/auto_tracking.cpp:749-765).
// Upstream (PCL-1.8.0 segmentation/impl/extract_clusters.hpp, extractEuclideanClusters) grows every cluster
// breadth first with KdTree radius searches (FLANN: squared distance < (float)(tolerance^2), distance accumulated as
// (dx^2 + dy^2) + dz^2 in fp32): a cluster is a connected component of the graph "closer than the tolerance".
// Here: counting sort into a uniform grid (cell >= tolerance), lock-free union-find over the 27-cell neighbourhoods
// (the larger root is always hooked under the smaller one, so a component's root is its lowest point index = the seed
// upstream starts it from), component sizes, then the components inside [min, max] ordered by size descending
// (upstream: std::sort over reverse iterators; ties are unspecified there, here the lower seed index goes first).
#include <float.h>
#include <string.h>

#include <algorithm>

#include "pft_internal.h"

namespace pft {
namespace {

struct ClusterGrid {
  float origin[3];
  float inv_cell;
  int dim[3];
  int n_cells;
  int valid;
};

constexpr int kMaxClusterCells = 1 << 22;
constexpr int kMaxClusters = 4096;  // clusters that can pass the size filter (each holds >= min_size points)

__device__ __forceinline__ bool finite3(const float4& p) { return isfinite(p.x) && isfinite(p.y) && isfinite(p.z); }

// bounding box of the finite points -> grid header (one block)
__global__ void __launch_bounds__(1024) cl_grid_kernel(const float4* __restrict__ pts, const CloudHeader* __restrict__ hdr, float cell, ClusterGrid* g) {
  __shared__ float s_mn[32][3], s_mx[32][3];
  const int n = hdr->n;
  float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float4 p = pts[i];
    if (!finite3(p)) continue;
    mn[0] = fminf(mn[0], p.x); mn[1] = fminf(mn[1], p.y); mn[2] = fminf(mn[2], p.z);
    mx[0] = fmaxf(mx[0], p.x); mx[1] = fmaxf(mx[1], p.y); mx[2] = fmaxf(mx[2], p.z);
  }
  for (int d = 0; d < 3; ++d) { mn[d] = warp_min(mn[d]); mx[d] = warp_max(mx[d]); }
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) for (int d = 0; d < 3; ++d) { s_mn[wid][d] = mn[d]; s_mx[wid][d] = mx[d]; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) for (int d = 0; d < 3; ++d) { mn[d] = fminf(mn[d], s_mn[w][d]); mx[d] = fmaxf(mx[d], s_mx[w][d]); }
    ClusterGrid h;
    h.valid = mn[0] <= mx[0] ? 1 : 0;
    // cell edge: the tolerance, doubled until the grid fits (a larger cell only means more candidates per neighbourhood)
    float c = cell;
    for (int it = 0; it < 40; ++it) {
      long long cells = 1;
      for (int d = 0; d < 3; ++d) {
        h.dim[d] = h.valid ? (int)fminf(floorf((mx[d] - mn[d]) / c), 2.0e9f) + 1 : 1;
        cells *= (long long)h.dim[d];
        if (cells > (1ll << 40)) cells = 1ll << 40;
      }
      if (cells <= (long long)kMaxClusterCells) { h.n_cells = (int)cells; break; }
      c *= 2.0f;
    }
    for (int d = 0; d < 3; ++d) h.origin[d] = h.valid ? mn[d] : 0.f;
    h.inv_cell = 1.0f / c;
    *g = h;
  }
}

__device__ __forceinline__ void cl_cell_of(const ClusterGrid& g, const float4& p, int& cx, int& cy, int& cz) {
  cx = min(max((int)floorf((p.x - g.origin[0]) * g.inv_cell), 0), g.dim[0] - 1);
  cy = min(max((int)floorf((p.y - g.origin[1]) * g.inv_cell), 0), g.dim[1] - 1);
  cz = min(max((int)floorf((p.z - g.origin[2]) * g.inv_cell), 0), g.dim[2] - 1);
}

__global__ void cl_count_kernel(const float4* __restrict__ pts, const CloudHeader* __restrict__ hdr, const ClusterGrid* __restrict__ gp, int* cell_count,
                                int* __restrict__ parent, int* __restrict__ comp_size) {
  const ClusterGrid g = *gp;
  const int n = hdr->n;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = pts[i];
    comp_size[i] = 0;
    if (!finite3(p)) { parent[i] = -1; continue; }  // never part of a cluster (the model builder drops NaNs first, ref: src/create_model.cpp:59-77)
    parent[i] = i;
    int cx, cy, cz;
    cl_cell_of(g, p, cx, cy, cz);
    atomicAdd(&cell_count[(cz * g.dim[1] + cy) * g.dim[0] + cx], 1);
  }
}

__global__ void __launch_bounds__(1024) cl_scan_kernel(const ClusterGrid* __restrict__ gp, int* cell_count, int* __restrict__ cell_start) {
  __shared__ int smem[34];
  const int nc = gp->n_cells;
  const int total = block_exclusive_scan<int>(
      nc, [&](int i) { return cell_count[i]; }, [&](int i, int ex) { cell_start[i] = ex; cell_count[i] = 0; }, smem);
  if (threadIdx.x == 0) cell_start[nc] = total;
}

__global__ void cl_scatter_kernel(const float4* __restrict__ pts, const CloudHeader* __restrict__ hdr, const ClusterGrid* __restrict__ gp,
                                  const int* __restrict__ cell_start, int* cell_count, int* __restrict__ order) {
  const ClusterGrid g = *gp;
  const int n = hdr->n;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = pts[i];
    if (!finite3(p)) continue;
    int cx, cy, cz;
    cl_cell_of(g, p, cx, cy, cz);
    const int c = (cz * g.dim[1] + cy) * g.dim[0] + cx;
    order[cell_start[c] + atomicAdd(&cell_count[c], 1)] = i;
  }
}

__device__ __forceinline__ int cl_find(int* parent, int i) {
  // path halving; parent links only ever point to lower indices, so concurrent hooks keep this loop finite
  int p = parent[i];
  while (p != i) {
    const int gp = parent[p];
    if (gp != p) parent[i] = gp;
    i = p; p = gp;
  }
  return i;
}
__device__ __forceinline__ void cl_unite(int* parent, int a, int b) {
  while (true) {
    a = cl_find(parent, a); b = cl_find(parent, b);
    if (a == b) return;
    if (a < b) { const int t = a; a = b; b = t; }   // hook the larger root under the smaller one
    const int old = atomicCAS(&parent[a], a, b);
    if (old == a) return;
    a = old;
  }
}

// every point against the points of its 27 neighbouring cells with a lower index (each pair once)
__global__ void cl_union_kernel(const float4* __restrict__ pts, const CloudHeader* __restrict__ hdr, const ClusterGrid* __restrict__ gp,
                                const int* __restrict__ cell_start, const int* __restrict__ order, int* parent, float tol2) {
  const ClusterGrid g = *gp;
  const int n = hdr->n;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = pts[i];
    if (!finite3(p)) continue;
    int cx, cy, cz;
    cl_cell_of(g, p, cx, cy, cz);
    for (int z = max(cz - 1, 0); z <= min(cz + 1, g.dim[2] - 1); ++z)
      for (int y = max(cy - 1, 0); y <= min(cy + 1, g.dim[1] - 1); ++y) {
        const int x0 = max(cx - 1, 0), x1 = min(cx + 1, g.dim[0] - 1);
        const int base = (z * g.dim[1] + y) * g.dim[0];
        const int s1 = cell_start[base + x1 + 1];
        for (int s = cell_start[base + x0]; s < s1; ++s) {  // cells are x-fastest: the three cells of a row are one slot range
          const int j = order[s];
          if (j >= i) continue;
          const float4 q = pts[j];
          const float dx = p.x - q.x, dy = p.y - q.y, dz = p.z - q.z;
          const float d2 = (dx * dx + dy * dy) + dz * dz;
          if (d2 < tol2) cl_unite(parent, i, j);
        }
      }
  }
}

__global__ void cl_flatten_kernel(const CloudHeader* __restrict__ hdr, int* parent, int* comp_size) {
  const int n = hdr->n;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    if (parent[i] < 0) continue;
    int r = i;
    while (parent[r] != r) r = parent[r];
    atomicAdd(&comp_size[r], 1);
    // (roots are final: all hooks happened in the previous kernel; writing the root back here would race with the
    //  walks of other threads only benignly, but labels are taken from a fresh walk in cl_label_kernel anyway)
  }
}

// the components inside [min, max], ordered by size descending then seed ascending (one block)
__global__ void __launch_bounds__(1024) cl_select_kernel(const CloudHeader* __restrict__ hdr, const int* __restrict__ parent, const int* __restrict__ comp_size,
                                                         int min_size, int max_size, unsigned long long* keys /* [kMaxClusters] */, int* __restrict__ rank_of_root,
                                                         int* __restrict__ out_sizes, int* out_count /* [0] clusters kept, [1] clusters that passed (may exceed the cap) */) {
  __shared__ int smem[34];
  __shared__ unsigned long long s_key[kMaxClusters];
  const int n = hdr->n;
  auto is_kept = [&](int i) -> int { return (parent[i] == i && comp_size[i] >= min_size && comp_size[i] <= max_size) ? 1 : 0; };
  for (int k = threadIdx.x; k < kMaxClusters; k += blockDim.x) s_key[k] = ~0ull;
  __syncthreads();
  const int total = block_exclusive_scan<int>(
      n, is_kept,
      [&](int i, int ex) {
        if (is_kept(i) && ex < kMaxClusters) s_key[ex] = ((unsigned long long)(0xffffffffu - (unsigned int)comp_size[i]) << 32) | (unsigned int)i;
      },
      smem);
  __syncthreads();
  const int kept = min(total, kMaxClusters);
  // bitonic sort of the (padded) key array in shared memory
  for (int k = 2; k <= kMaxClusters; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = threadIdx.x; t < kMaxClusters; t += blockDim.x) {
        const int ixj = t ^ j;
        if (ixj > t) {
          const unsigned long long a = s_key[t], b = s_key[ixj];
          const bool up = (t & k) == 0;
          if ((a > b) == up) { s_key[t] = b; s_key[ixj] = a; }
        }
      }
      __syncthreads();
    }
  for (int k = threadIdx.x; k < kept; k += blockDim.x) {
    const unsigned long long key = s_key[k];
    const int root = (int)(key & 0xffffffffu);
    keys[k] = key;
    rank_of_root[root] = k;
    out_sizes[k] = (int)(0xffffffffu - (unsigned int)(key >> 32));
  }
  if (threadIdx.x == 0) { out_count[0] = kept; out_count[1] = total; }
}

__global__ void cl_label_kernel(const CloudHeader* __restrict__ hdr, const int* __restrict__ parent, const int* __restrict__ comp_size, int min_size,
                                int max_size, const int* __restrict__ rank_of_root, int* __restrict__ labels) {
  const int n = hdr->n;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    int lab = -1;
    if (parent[i] >= 0) {
      int r = i;
      while (parent[r] != r) r = parent[r];
      if (comp_size[r] >= min_size && comp_size[r] <= max_size) lab = rank_of_root[r];
    }
    labels[i] = lab;
  }
}

// the points carrying one label, in input order (= the cluster's sorted indices upstream): one block
__global__ void __launch_bounds__(1024) cl_extract_kernel(const float4* __restrict__ in, const CloudHeader* __restrict__ in_hdr, const int* __restrict__ labels,
                                                          int label, float4* __restrict__ out, CloudHeader* out_hdr) {
  __shared__ int smem[34];
  const int n = in_hdr->n;
  const int total = block_exclusive_scan<int>(
      n, [&](int i) { return labels[i] == label ? 1 : 0; }, [&](int i, int ex) { if (labels[i] == label) out[ex] = in[i]; }, smem);
  if (threadIdx.x == 0) out_hdr->n = total;
}

inline int cl_grid_for(size_t n, int sm) {
  size_t g = (n + 255) / 256;
  if (g > (size_t)sm * 8) g = (size_t)sm * 8;
  return (int)std::max<size_t>(g, 1);
}

}  // namespace
}  // namespace pft

using namespace pft;

extern "C" {

int pft_euclidean_clusters(pft_context* ctx, const pft_cloud* in, double tolerance, int min_size, int max_size, int32_t* labels, size_t labels_capacity,
                           int32_t* sizes, size_t sizes_capacity, size_t* n_clusters) {
  if (!ctx || !in || !n_clusters) { set_last_error("pft_euclidean_clusters: null argument"); return PFT_ERR_INVALID; }
  if (in->ctx != ctx) { set_last_error("pft_euclidean_clusters: cloud belongs to another context"); return PFT_ERR_INVALID; }
  if (!(tolerance > 0.0) || min_size < 1 || max_size < min_size) { set_last_error("pft_euclidean_clusters: need tolerance > 0 and 1 <= min_size <= max_size"); return PFT_ERR_INVALID; }
  PFT_CUDA_TRY(cudaSetDevice(ctx->device));
  size_t n = 0;
  int rc = pft_cloud_size(const_cast<pft_cloud*>(in), &n);
  if (rc) return rc;
  *n_clusters = 0;
  ctx->cl_n = n;
  ctx->cl_src = in;
  if (n == 0) return PFT_OK;
  if (labels && labels_capacity < n) { set_last_error("pft_euclidean_clusters: labels capacity %zu < %zu points", labels_capacity, n); return PFT_ERR_CAPACITY; }
  cudaStream_t s = ctx->stream;
  if ((rc = ctx->cl_grid.reserve(sizeof(ClusterGrid)))) return rc;
  if ((rc = ctx->cl_cells.reserve(((size_t)kMaxClusterCells + 16) * sizeof(int) * 2))) return rc;
  if ((rc = ctx->cl_work.reserve(n * sizeof(int) * 5 + 64))) return rc;
  if ((rc = ctx->cl_sel.reserve((size_t)kMaxClusters * (sizeof(unsigned long long) + sizeof(int)) + 64))) return rc;
  int* cell_count = ctx->cl_cells.as<int>();
  int* cell_start = cell_count + kMaxClusterCells + 16;
  int* parent = ctx->cl_work.as<int>();
  int* comp_size = parent + n;
  int* order = comp_size + n;
  int* rank_of_root = order + n;
  int* dlabels = rank_of_root + n;
  unsigned long long* keys = ctx->cl_sel.as<unsigned long long>();
  int* out_sizes = reinterpret_cast<int*>(keys + kMaxClusters);
  int* out_count = out_sizes + kMaxClusters;
  ClusterGrid* g = ctx->cl_grid.as<ClusterGrid>();
  const float tol2 = (float)(tolerance * tolerance);  // KdTreeFLANN::radiusSearch passes (float)(radius * radius)
  const int grid = cl_grid_for(n, ctx->sm_count);
  cl_grid_kernel<<<1, 1024, 0, s>>>(in->d_pts(), in->d_hdr(), (float)tolerance * 1.0001f, g);
  PFT_LAUNCH_CHECK();
  PFT_CUDA_TRY(cudaMemsetAsync(cell_count, 0, ((size_t)kMaxClusterCells + 16) * sizeof(int), s));
  cl_count_kernel<<<grid, 256, 0, s>>>(in->d_pts(), in->d_hdr(), g, cell_count, parent, comp_size);
  PFT_LAUNCH_CHECK();
  cl_scan_kernel<<<1, 1024, 0, s>>>(g, cell_count, cell_start);
  PFT_LAUNCH_CHECK();
  cl_scatter_kernel<<<grid, 256, 0, s>>>(in->d_pts(), in->d_hdr(), g, cell_start, cell_count, order);
  PFT_LAUNCH_CHECK();
  cl_union_kernel<<<grid, 256, 0, s>>>(in->d_pts(), in->d_hdr(), g, cell_start, order, parent, tol2);
  PFT_LAUNCH_CHECK();
  cl_flatten_kernel<<<grid, 256, 0, s>>>(in->d_hdr(), parent, comp_size);
  PFT_LAUNCH_CHECK();
  cl_select_kernel<<<1, 1024, 0, s>>>(in->d_hdr(), parent, comp_size, min_size, max_size, keys, rank_of_root, out_sizes, out_count);
  PFT_LAUNCH_CHECK();
  cl_label_kernel<<<grid, 256, 0, s>>>(in->d_hdr(), parent, comp_size, min_size, max_size, rank_of_root, dlabels);
  PFT_LAUNCH_CHECK();
  int counts[2] = {0, 0};
  PFT_CUDA_TRY(cudaMemcpyAsync(counts, out_count, sizeof(counts), cudaMemcpyDeviceToHost, s));
  PFT_CUDA_TRY(cudaStreamSynchronize(s));
  if (counts[1] > kMaxClusters) { set_last_error("pft_euclidean_clusters: %d clusters pass the size filter, at most %d are supported", counts[1], kMaxClusters); return PFT_ERR_CAPACITY; }
  *n_clusters = (size_t)counts[0];
  ctx->cl_count = counts[0];
  if (sizes) {
    if (sizes_capacity < (size_t)counts[0]) { set_last_error("pft_euclidean_clusters: sizes capacity %zu < %d clusters", sizes_capacity, counts[0]); return PFT_ERR_CAPACITY; }
    if (counts[0]) PFT_CUDA_TRY(cudaMemcpy(sizes, out_sizes, (size_t)counts[0] * sizeof(int), cudaMemcpyDeviceToHost));
  }
  if (labels) PFT_CUDA_TRY(cudaMemcpy(labels, dlabels, n * sizeof(int), cudaMemcpyDeviceToHost));
  return PFT_OK;
}

int pft_cloud_select_cluster(pft_context* ctx, const pft_cloud* in, int k, pft_cloud* out) {
  if (!ctx || !in || !out) { set_last_error("pft_cloud_select_cluster: null argument"); return PFT_ERR_INVALID; }
  if (in->ctx != ctx || out->ctx != ctx || in == out) { set_last_error("pft_cloud_select_cluster: clouds must be distinct and belong to the context"); return PFT_ERR_INVALID; }
  size_t n_now = 0;
  int rc0 = pft_cloud_size(const_cast<pft_cloud*>(in), &n_now);
  if (rc0) return rc0;
  if (ctx->cl_src != in || !ctx->cl_work.p || n_now != ctx->cl_n) {
    set_last_error("pft_cloud_select_cluster: call pft_euclidean_clusters on this cloud first (the labels on the device belong to another cloud)");
    return PFT_ERR_STATE;
  }
  if (k < 0 || k >= ctx->cl_count) { set_last_error("pft_cloud_select_cluster: cluster %d of %d", k, ctx->cl_count); return PFT_ERR_INVALID; }
  PFT_CUDA_TRY(cudaSetDevice(ctx->device));
  int rc = out->ensure(in->capacity);
  if (rc) return rc;
  const int* dlabels = ctx->cl_work.as<int>() + 4 * ctx->cl_n;
  cl_extract_kernel<<<1, 1024, 0, ctx->stream>>>(in->d_pts(), in->d_hdr(), dlabels, k, out->d_pts(), out->d_hdr());
  PFT_LAUNCH_CHECK();
  out->written(-1);
  return PFT_OK;
}

}  // extern "C"

// =====================================================================================================================
// Plane segmentation of the model builder's second variant (ref: src/create_model_planar_segmentation.cpp:157-174):
// pcl::SACSegmentation<PointT>(SACMODEL_PLANE, SAC_RANSAC, setMaxIterations(1000), setDistanceThreshold(0.015))::segment
// followed by pcl::ExtractIndices (setNegative(false) -> the plane, setNegative(true) -> everything else).
// Upstream (PCL-1.8.0 sample_consensus/impl/ransac.hpp, sac_model_plane.hpp, segmentation/impl/sac_segmentation.hpp):
//   loop: draw 3 point indices -> plane through them (computeModelCoefficients) -> countWithinDistance -> keep the
//   best, k = log(1 - probability) / log(1 - w^3) with w = best inlier ratio; stop at iterations >= k or > max;
//   selectWithinDistance(best); optimizeModelCoefficients = least-squares plane of the inliers (smallest eigenvector of
//   their covariance, d = -n . centroid); selectWithinDistance(refined).
// Here every drawn hypothesis is scored at once (one thread block per hypothesis over all points), then ONE thread
// replays the sequential accept / adapt-k / stop logic over the scores in draw order: the same plane as the sequential
// loop for the same draws.  The draws are injected (upstream uses rand(): not reproducible) or generated with Philox.
// A collinear sample is skipped without counting as an iteration (upstream redraws inside getSamples).
namespace pft {
namespace {

struct PlaneResult {
  float coeff[4];        // after the optional refinement
  float ransac_coeff[4]; // the winning hypothesis
  int best;              // index of the winning hypothesis (-1: none)
  int iterations;        // RANSAC iterations performed
  int n_inliers;         // final inlier count
  int pad;
};

__device__ __forceinline__ bool plane_from_sample(const float4& p0, const float4& p1, const float4& p2, float* c) {
  // SampleConsensusModelPlane::computeModelCoefficients
  const float ax = p1.x - p0.x, ay = p1.y - p0.y, az = p1.z - p0.z;
  const float bx = p2.x - p0.x, by = p2.y - p0.y, bz = p2.z - p0.z;
  const float rx = ax / bx, ry = ay / by, rz = az / bz;      // dy1dy2 = p1p0 / p2p0
  if (rx == ry && rz == ry) return false;                    // collinear
  float nx = ay * bz - az * by, ny = az * bx - ax * bz, nz = ax * by - ay * bx;
  // Eigen's 4-float reductions (normalize, dot) add lanes as (0 + 2) + (1 + 3) on SSE; lane 3 of the normal is 0
  const float len = sqrtf((nx * nx + nz * nz) + (ny * ny + 0.0f));
  nx = nx / len; ny = ny / len; nz = nz / len;
  c[0] = nx; c[1] = ny; c[2] = nz;
  c[3] = -1.0f * ((nx * p0.x + nz * p0.z) + (ny * p0.y + 0.0f));
  return isfinite(c[0]) && isfinite(c[1]) && isfinite(c[2]) && isfinite(c[3]);
}
__device__ __forceinline__ bool plane_inlier(const float* c, const float4& p, double thr) {
  // fabs(model_coefficients.dot(Vector4f(x, y, z, 1))) < threshold  (float dot in Eigen's (0 + 2) + (1 + 3) lane order,
  // double compare)
  const float d = (c[0] * p.x + c[2] * p.z) + (c[1] * p.y + c[3]);
  return (double)fabsf(d) < thr;   // (NaN points fail the comparison)
}

// one block per hypothesis: coefficients + inlier count
__global__ void __launch_bounds__(256) plane_score_kernel(const float4* __restrict__ pts, const CloudHeader* __restrict__ hdr, const int* __restrict__ samples3,
                                                          int n_samples, double thr, float* __restrict__ coeffs, int* __restrict__ counts) {
  __shared__ float c[4];
  __shared__ int ok;
  __shared__ int red[8];
  const int n = hdr->n;
  for (int s = blockIdx.x; s < n_samples; s += gridDim.x) {
    if (threadIdx.x == 0) {
      const int i0 = samples3[3 * s], i1 = samples3[3 * s + 1], i2 = samples3[3 * s + 2];
      ok = 0;
      if ((unsigned)i0 < (unsigned)n && (unsigned)i1 < (unsigned)n && (unsigned)i2 < (unsigned)n && i0 != i1 && i0 != i2 && i1 != i2)
        ok = plane_from_sample(pts[i0], pts[i1], pts[i2], c) ? 1 : 0;
      for (int k = 0; k < 4; ++k) coeffs[4 * s + k] = ok ? c[k] : 0.f;
    }
    __syncthreads();
    int cnt = 0;
    if (ok) {
      const float cc[4] = {c[0], c[1], c[2], c[3]};
      for (int i = threadIdx.x; i < n; i += blockDim.x) cnt += plane_inlier(cc, pts[i], thr) ? 1 : 0;
    }
    cnt = warp_sum(cnt);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
      int t = 0;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
      counts[s] = ok ? t : -1;
    }
    __syncthreads();
  }
}

// RandomSampleConsensus::computeModel replayed over the scores (one thread)
__global__ void plane_pick_kernel(const CloudHeader* __restrict__ hdr, const float* __restrict__ coeffs, const int* __restrict__ counts, int n_samples,
                                  int max_iterations, double probability, PlaneResult* out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const int n = hdr->n;
  int iterations = 0, best = -1, best_count = -2147483647, skipped = 0;
  double k = 1.0;
  const double log_probability = log(1.0 - probability);
  const double one_over_indices = n > 0 ? 1.0 / (double)n : 0.0;
  const int max_skip = max_iterations * 10;
  for (int s = 0; s < n_samples && (double)iterations < k && skipped < max_skip; ++s) {
    if (counts[s] < 0) { ++skipped; continue; }   // bad sample: no model
    if (counts[s] > best_count) {
      best_count = counts[s]; best = s;
      const double w = (double)best_count * one_over_indices;
      double p_no_outliers = 1.0 - w * w * w;     // pow(w, 3 samples)
      p_no_outliers = fmax(2.220446049250313e-16, p_no_outliers);
      p_no_outliers = fmin(1.0 - 2.220446049250313e-16, p_no_outliers);
      k = log_probability / log(p_no_outliers);
    }
    ++iterations;
    if (iterations > max_iterations) break;
  }
  PlaneResult r;
  for (int q = 0; q < 4; ++q) { r.ransac_coeff[q] = best >= 0 ? coeffs[4 * best + q] : 0.f; r.coeff[q] = r.ransac_coeff[q]; }
  r.best = best; r.iterations = iterations; r.n_inliers = best >= 0 ? best_count : 0; r.pad = 0;
  *out = r;
}

// optimizeModelCoefficients: least-squares plane of the inliers of the winning hypothesis (one block; fp64 sums of
// fp32 terms: order independent -- upstream accumulates in fp32 sequentially)
__global__ void __launch_bounds__(1024) plane_refine_kernel(const float4* __restrict__ pts, const CloudHeader* __restrict__ hdr, double thr, PlaneResult* res) {
  __shared__ double red[32];
  __shared__ double s_sum[9];
  const int n = hdr->n;
  if (res->best < 0) return;
  const float c[4] = {res->ransac_coeff[0], res->ransac_coeff[1], res->ransac_coeff[2], res->ransac_coeff[3]};
  double acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  double cnt = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float4 p = pts[i];
    if (!plane_inlier(c, p, thr)) continue;
    cnt += 1.0;
    acc[0] += (double)(p.x * p.x); acc[1] += (double)(p.x * p.y); acc[2] += (double)(p.x * p.z);
    acc[3] += (double)(p.y * p.y); acc[4] += (double)(p.y * p.z); acc[5] += (double)(p.z * p.z);
    acc[6] += (double)p.x; acc[7] += (double)p.y; acc[8] += (double)p.z;
  }
  for (int k = 0; k < 9; ++k) { const double v = block_sum(acc[k], red); if (threadIdx.x == 0) s_sum[k] = v; }
  cnt = block_sum(cnt, red);
  if (threadIdx.x != 0 || cnt < 3.0) return;   // upstream needs >= 3 inliers to refine
  // computeMeanAndCovarianceMatrix: accu /= n; cov = E[xx^T] - mean mean^T
  double a[9];
  for (int k = 0; k < 9; ++k) a[k] = s_sum[k] / cnt;
  const double mx = a[6], my = a[7], mz = a[8];
  double A[3][3] = {{a[0] - mx * mx, a[1] - mx * my, a[2] - mx * mz}, {a[1] - mx * my, a[3] - my * my, a[4] - my * mz}, {a[2] - mx * mz, a[4] - my * mz, a[5] - mz * mz}};
  // smallest eigenvector by Jacobi sweeps
  double V[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
  for (int sweep = 0; sweep < 32; ++sweep) {
    const double off = fabs(A[0][1]) + fabs(A[0][2]) + fabs(A[1][2]);
    if (off <= 1.0e-300 || off <= 1.0e-18 * (fabs(A[0][0]) + fabs(A[1][1]) + fabs(A[2][2]))) break;
    for (int p = 0; p < 2; ++p) for (int q = p + 1; q < 3; ++q) {
      if (fabs(A[p][q]) <= 1.0e-300) continue;
      const double theta = (A[q][q] - A[p][p]) / (2.0 * A[p][q]);
      const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
      const double cs = 1.0 / sqrt(t * t + 1.0), sn = t * cs;
      for (int k = 0; k < 3; ++k) { const double akp = A[k][p], akq = A[k][q]; A[k][p] = cs * akp - sn * akq; A[k][q] = sn * akp + cs * akq; }
      for (int k = 0; k < 3; ++k) { const double apk = A[p][k], aqk = A[q][k]; A[p][k] = cs * apk - sn * aqk; A[q][k] = sn * apk + cs * aqk; }
      for (int k = 0; k < 3; ++k) { const double vkp = V[k][p], vkq = V[k][q]; V[k][p] = cs * vkp - sn * vkq; V[k][q] = sn * vkp + cs * vkq; }
    }
  }
  int m = 0;
  if (A[1][1] < A[m][m]) m = 1;
  if (A[2][2] < A[m][m]) m = 2;
  double nx = V[0][m], ny = V[1][m], nz = V[2][m];
  // Eigen leaves the sign of the eigenvector open: keep the side of the RANSAC normal
  if (nx * (double)c[0] + ny * (double)c[1] + nz * (double)c[2] < 0.0) { nx = -nx; ny = -ny; nz = -nz; }
  res->coeff[0] = (float)nx; res->coeff[1] = (float)ny; res->coeff[2] = (float)nz;
  res->coeff[3] = -1.0f * (((float)nx * (float)mx + (float)ny * (float)my) + (float)nz * (float)mz);
}

// ExtractIndices: inliers (setNegative(false)) and the rest (setNegative(true)), both in input order (one block)
__global__ void __launch_bounds__(1024) plane_extract_kernel(const float4* __restrict__ pts, const CloudHeader* __restrict__ hdr, double thr, PlaneResult* res,
                                                             float4* out_in, CloudHeader* out_in_hdr, float4* out_rest, CloudHeader* out_rest_hdr) {
  __shared__ int smem[34];
  const int n = hdr->n;
  const bool have = res->best >= 0;
  const float c[4] = {res->coeff[0], res->coeff[1], res->coeff[2], res->coeff[3]};
  auto is_in = [&](int i) -> int { return (have && plane_inlier(c, pts[i], thr)) ? 1 : 0; };
  const int total = block_exclusive_scan<int>(
      n, is_in,
      [&](int i, int ex) {
        const float4 p = pts[i];
        if (is_in(i)) { if (out_in) out_in[ex] = p; }
        else if (out_rest) out_rest[i - ex] = p;
      },
      smem);
  if (threadIdx.x == 0) {
    res->n_inliers = total;
    if (out_in_hdr) out_in_hdr->n = total;
    if (out_rest_hdr) out_rest_hdr->n = n - total;
  }
}

// RANSAC draws when none are injected: 3 distinct indices per hypothesis from Philox-style integer hashing
__global__ void plane_draw_kernel(const CloudHeader* __restrict__ hdr, int n_samples, unsigned long long seed, int* __restrict__ samples3) {
  const int n = hdr->n;
  for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < n_samples; s += gridDim.x * blockDim.x) {
    unsigned long long x = seed + 0x9E3779B97F4A7C15ull * (unsigned long long)(s + 1);
    int idx[3];
    for (int k = 0; k < 3; ++k) {
      for (int tries = 0; tries < 64; ++tries) {
        x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 27; x *= 0x94D049BB133111EBull; x ^= x >> 31;  // splitmix64
        idx[k] = n > 0 ? (int)(x % (unsigned long long)n) : 0;
        bool dup = false;
        for (int q = 0; q < k; ++q) dup = dup || idx[q] == idx[k];
        if (!dup) break;
      }
      samples3[3 * s + k] = idx[k];
    }
  }
}

}  // namespace
}  // namespace pft

extern "C" {

int pft_segment_plane(pft_context* ctx, const pft_cloud* in, double distance_threshold, int max_iterations, double probability, const int32_t* samples3,
                      int n_samples, uint64_t seed, int optimize_coefficients, float* coefficients4, int32_t* iterations, pft_cloud* plane_out,
                      pft_cloud* rest_out, size_t* n_inliers) {
  if (!ctx || !in) { set_last_error("pft_segment_plane: null argument"); return PFT_ERR_INVALID; }
  if (in->ctx != ctx || (plane_out && plane_out->ctx != ctx) || (rest_out && rest_out->ctx != ctx) || plane_out == in || rest_out == in ||
      (plane_out && plane_out == rest_out)) {
    set_last_error("pft_segment_plane: clouds must be distinct and belong to the context");
    return PFT_ERR_INVALID;
  }
  if (!(distance_threshold > 0.0) || max_iterations < 1 || !(probability > 0.0 && probability < 1.0)) {
    set_last_error("pft_segment_plane: need distance_threshold > 0, max_iterations >= 1, 0 < probability < 1");
    return PFT_ERR_INVALID;
  }
  if (samples3 && n_samples < 1) { set_last_error("pft_segment_plane: injected samples need n_samples >= 1"); return PFT_ERR_INVALID; }
  PFT_CUDA_TRY(cudaSetDevice(ctx->device));
  size_t n = 0;
  int rc = pft_cloud_size(const_cast<pft_cloud*>(in), &n);
  if (rc) return rc;
  cudaStream_t s = ctx->stream;
  if (plane_out && (rc = plane_out->ensure(in->capacity))) return rc;
  if (rest_out && (rc = rest_out->ensure(in->capacity))) return rc;
  // upstream draws until `iterations >= k`; every draw it can ever need is at most max_iterations + the skipped ones
  const int S = samples3 ? n_samples : max_iterations + 1 + max_iterations / 8;
  if ((rc = ctx->cl_sel.reserve((size_t)S * (3 * sizeof(int) + 4 * sizeof(float) + sizeof(int)) + sizeof(PlaneResult) + 256))) return rc;
  PlaneResult* res = ctx->cl_sel.as<PlaneResult>();
  int* d_samples = reinterpret_cast<int*>(res + 1);
  float* d_coeffs = reinterpret_cast<float*>(d_samples + 3 * (size_t)S);
  int* d_counts = reinterpret_cast<int*>(d_coeffs + 4 * (size_t)S);
  if (samples3) PFT_CUDA_TRY(cudaMemcpyAsync(d_samples, samples3, (size_t)S * 3 * sizeof(int), cudaMemcpyHostToDevice, s));
  else {
    plane_draw_kernel<<<(S + 255) / 256, 256, 0, s>>>(in->d_hdr(), S, seed, d_samples);
    PFT_LAUNCH_CHECK();
  }
  plane_score_kernel<<<std::min(S, ctx->sm_count * 8), 256, 0, s>>>(in->d_pts(), in->d_hdr(), d_samples, S, distance_threshold, d_coeffs, d_counts);
  PFT_LAUNCH_CHECK();
  plane_pick_kernel<<<1, 32, 0, s>>>(in->d_hdr(), d_coeffs, d_counts, S, max_iterations, probability, res);
  PFT_LAUNCH_CHECK();
  if (optimize_coefficients) {
    plane_refine_kernel<<<1, 1024, 0, s>>>(in->d_pts(), in->d_hdr(), distance_threshold, res);
    PFT_LAUNCH_CHECK();
  }
  plane_extract_kernel<<<1, 1024, 0, s>>>(in->d_pts(), in->d_hdr(), distance_threshold, res, plane_out ? plane_out->d_pts() : nullptr,
                                          plane_out ? plane_out->d_hdr() : nullptr, rest_out ? rest_out->d_pts() : nullptr, rest_out ? rest_out->d_hdr() : nullptr);
  PFT_LAUNCH_CHECK();
  if (plane_out) plane_out->written(-1);
  if (rest_out) rest_out->written(-1);
  PlaneResult h;
  PFT_CUDA_TRY(cudaMemcpyAsync(&h, res, sizeof(h), cudaMemcpyDeviceToHost, s));
  PFT_CUDA_TRY(cudaStreamSynchronize(s));
  if (coefficients4) memcpy(coefficients4, h.coeff, sizeof(h.coeff));
  if (iterations) *iterations = h.iterations;
  if (n_inliers) *n_inliers = (size_t)h.n_inliers;
  ctx->cl_src = nullptr;  // (the clustering scratch was reused)
  if (h.best < 0) { set_last_error("pft_segment_plane: no valid plane hypothesis among the %d samples", S); return PFT_ERR_STATE; }
  return PFT_OK;
}

}  // extern "C"
