// pft_tracker_kernels.cuh -- device code of kernels K2 (scene index), K3 (weight) and K4
// (normalise / resample / update).  Included by pft_tracker.cu only.
//
// What each kernel replaces (PCL-1.8.0 upstream, SURVEY.md Appendix A; call sites in
// ref: src/auto_tracking.cpp:198-258, :688-697):
//   matrices_kernel      ParticleXYZRPY::toEigenMatrix = pcl::getTransformation          (A.6)
//   aabb_kernel          transformPointCloud per particle + calcBoundingBox               (A.3)
//   index_*_kernel       cropInputPointCloud + search::Octree::setInputCloud              (A.3, A.5)
//   weight_lists_kernel  NearestPairPointCloudCoherence::computeCoherence + Distance/HSV  (A.4)
//   normalize_kernel     ParticleFilterTracker::normalizeWeight                           (A.6)
//   update_kernel        ParticleFilterTracker::update                                    (A.6)
//   cdf/resample/kld_*   (KLDAdaptive)ParticleFilterTracker::resample                     (A.7)
//   init_particles_kernel ParticleFilterTracker::initParticles                            (A.8)
#pragma once
#include <cooperative_groups.h>

#include "pft_common.cuh"

namespace pft {

// tuning builds only (-DPFT_TRACE): nanosecond stamps of key points of the frame, min / max over the CTAs that pass them
#ifdef PFT_TRACE
__device__ unsigned long long g_trace[64];
__device__ __forceinline__ unsigned long long trace_now() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#define PFT_TRACE_MIN(i) do { if ((threadIdx.x & 31) == 0) atomicMin(&g_trace[i], trace_now()); } while (0)
#define PFT_TRACE_MAX(i) do { if ((threadIdx.x & 31) == 0) atomicMax(&g_trace[i], trace_now()); } while (0)
#else
#define PFT_TRACE_MIN(i)
#define PFT_TRACE_MAX(i)
#endif
// ------------------------------------------------------------------ device-resident tracker state
struct TrackerState {
  int particle_num;       // live particle count (changes on the device in KLD mode)
  int has_particles;
  float aabb[6];          // crop box being accumulated by aabb_kernel (atomic min/max)
  DevParticle rep;        // representative_state_
  DevParticle motion;     // motion_
  double fit_ratio;
  double weight_sum;
  unsigned long long draw_call;  // Philox stream position (advanced on the device: graph replays stay distinct)
  // nearest-neighbour distance statistics of the last weight() (micrometres, matched pairs only): they steer the
  // cell size of the next index build.  Integer sums: independent of the order the atomics land in.
  unsigned long long nn_sum_um, nn_count;
  unsigned int peer_epoch;       // weight() calls so far in peer (NVLink P2P) exchange mode
  unsigned int peer_error;       // a wait on a peer's flag timed out (sticky)
  int resample_n_old;            // particle count the running resample draws FROM (cdf_kernel publishes the new count for fixed-N trackers)
  unsigned int work_counter;     // next (particle, model chunk) item of the running weight kernel (reset by index_begin_kernel)
  unsigned long long evals;      // likelihood evaluations so far: sum over weight() calls of particles x model points (whole job)
  unsigned int aabb_blocks_done; // blocks of the running aabb_kernel that have added their boxes (peer mode: the last one exchanges the box)
};

// ------------------------------------------------------------------ NVLink peer exchange (one process per GPU)
// Every rank owns one PeerWindow in its HBM, mapped into all peers with CUDA IPC.  The two exchange steps of weight()
// are plain peer stores issued by the producing kernels themselves, followed by a flag barrier:
//   crop box    the last block of aabb_kernel stores this rank's six values into slot [rank] of every window, signals,
//               waits, reduces locally;
//   raw weights normalize_kernel sums this rank's raw weights, stores every value into every window, signals, waits.
// Flags only ever grow (epoch numbered), so nothing has to be reset between frames or graph replays.  The box slots
// are double-buffered by epoch parity; the raw-weight area needs no second buffer: a rank can only push the weights of
// epoch e+1 after it has passed the box barrier of e+1, which every rank enters after its normalize of epoch e.
constexpr int kMaxPeers = 16;
struct PeerWindow {
  float box[2][kMaxPeers][8];  // [epoch parity][source rank][minx,miny,minz,maxx,maxy,maxz,-,-]
  unsigned int flag_box;       // += 1 by every rank per epoch
  unsigned int flag_raw;       // += 1 by every rank per epoch
  unsigned int pad[30];
  float raw[1];                // [nranks][slice_cap] gathered raw weights (the allocation is larger)
};
struct PeerSet {
  PeerWindow* win[kMaxPeers];  // win[r] = rank r's window as mapped here (win[rank] = the local one)
  int nranks, rank;
};

__device__ __forceinline__ bool peer_wait(volatile unsigned int* flag, unsigned int target, unsigned int* error) {
  const long long t0 = clock64();
  while ((int)(*flag - target) < 0) {
    if (clock64() - t0 > 8000000000ll) { *error = 1u; return false; }  // ~4 s: a peer is gone; give up instead of hanging the GPU
    __nanosleep(64);
  }
  __threadfence_system();
  return true;
}

// Crop-box exchange by one warp: every rank stores its six values into slot [rank] of every window, raises every rank's
// flag, waits for its own to show all ranks of this epoch, reduces locally (an all-reduce(min/max) without a collective).
__device__ __forceinline__ void peer_box_exchange(TrackerState* st, const PeerSet& ps) {
  const int lane = threadIdx.x & 31;
  PeerWindow* me = ps.win[ps.rank];
  unsigned int e = 0;
  if (lane == 0) { e = st->peer_epoch + 1u; st->peer_epoch = e; }
  e = __shfl_sync(kFull, e, 0);
  const int cur = e & 1u;
  // lane = (destination rank, component): 8 floats to each of up to 4 ranks per pass
  for (int r0 = 0; r0 < ps.nranks; r0 += 4) {
    const int r = r0 + (lane >> 3), d = lane & 7;
    if (r < ps.nranks && d < 6) ps.win[r]->box[cur][ps.rank][d] = __ldcg(&st->aabb[d]);  // (L2: the other blocks of aabb_kernel wrote it with atomics)
  }
  // (the pattern NCCL's primitives use: the writers synchronise, ONE thread issues the system-scope fence -- it is
  //  cumulative over what the barrier ordered before it -- and only then are the flags raised)
  __syncwarp();
  if (lane == 0) __threadfence_system();
  __syncwarp();
  if (lane < ps.nranks) atomicAdd_system(&ps.win[lane]->flag_box, 1u);
  bool ok = true;
  if (lane == 0) ok = peer_wait(&me->flag_box, e * (unsigned int)ps.nranks, &st->peer_error);
  ok = __shfl_sync(kFull, ok, 0);
  if (!ok) return;
  if (lane < 6) {
    float v = __ldcg(&me->box[cur][0][lane]);
    for (int r = 1; r < ps.nranks; ++r) {
      const float o = __ldcg(&me->box[cur][r][lane]);
      v = lane < 3 ? fminf(v, o) : fmaxf(v, o);
    }
    st->aabb[lane] = v;
  }
}

// ---- scene distribution by peer stores: ONE rank owns the sensor (upload + downsample), its kernel stores the
// downsampled cloud straight into the cloud of every other rank over NVLink (CUDA IPC mappings) and raises their
// flags; the other ranks' streams wait on the flag.  No collective, no host round trip, one H2D copy per frame for
// the whole job.
struct CloudPeerSet {
  float4* pts[kMaxPeers];
  CloudHeader* hdr[kMaxPeers];
  unsigned int* sync[kMaxPeers];  // [0] flag = number of the last scene that has fully arrived, [1] blocks done (root only)
  int nranks, rank;
};
// Stores the header and the n points of `src` (n read from its header) into every cloud of `ps` but ps.rank's, with
// 16-byte loads and stores.  n > capacity stores an empty cloud and raises *error (if given).
__device__ __forceinline__ void push_cloud(const float4* __restrict__ src, const CloudHeader* __restrict__ src_hdr, const CloudPeerSet& ps, int capacity,
                                           unsigned int* error) {
  int n = src_hdr->n;
  if (n > capacity) { if (error && blockIdx.x == 0 && threadIdx.x == 0) *error = 1u; n = 0; }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = src[i];
    for (int r = 0; r < ps.nranks; ++r) if (r != ps.rank) ps.pts[r][i] = p;
  }
  if (blockIdx.x == 0 && threadIdx.x < ps.nranks && (int)threadIdx.x != ps.rank) { CloudHeader h = *src_hdr; h.n = n; *ps.hdr[threadIdx.x] = h; }
}
__global__ void __launch_bounds__(256) cloud_push_kernel(const float4* __restrict__ src, const CloudHeader* __restrict__ src_hdr, CloudPeerSet ps,
                                                         unsigned int epoch, int capacity, unsigned int* error /* host-mapped */) {
  push_cloud(src, src_hdr, ps, capacity, error);  // (an overflow is loud on the host at the next call; the peers see an empty scene)
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();  // one system-scope fence per block, after the barrier (cumulative over the block's stores)
    unsigned int* mine = ps.sync[ps.rank];
    if (atomicAdd(&mine[1], 1u) + 1u == gridDim.x) {  // every block has pushed its part
      mine[1] = 0u;
      __threadfence_system();
      for (int r = 0; r < ps.nranks; ++r) if (r != ps.rank) atomicExch_system(&ps.sync[r][0], epoch);
    }
  }
}
__global__ void cloud_wait_kernel(unsigned int* sync, unsigned int epoch, unsigned int* error /* host-mapped */) {
  peer_wait(&sync[0], epoch, error);
}
// The scene replicas of other contexts in one process (pft_tracker.cu): the same stores into every cloud of `ps`
// (ps.rank = -1), ordered by stream events instead of flags.  The replicas are sized for the source's capacity.
__global__ void __launch_bounds__(256) cloud_fanout_kernel(const float4* __restrict__ src, const CloudHeader* __restrict__ src_hdr, CloudPeerSet ps,
                                                           int capacity) {
  push_cloud(src, src_hdr, ps, capacity, nullptr);
}

struct NoiseParams {      // host-precomputed square roots (IEEE, identical to the oracle's)
  double mean[6];
  double sigma[6];        // sqrt(cov[d])
  double sigma_q[3];      // sqrt((double)0.2862f * cov[3+d])
  int quat_mode;
};

struct CoherenceParams {
  double max_d2;          // maximum_distance_^2 (double compare, as upstream)
  double dist_w, hsv_w;
  float h_w, s_w, v_w;
  float r_max;            // min(maximum_distance_, 1e18)
  int use_dist, use_hsv;
};


// ------------------------------------------------------------------ small math (arithmetic contract)
__device__ __forceinline__ void sincos_c(float a, float& s, float& c) {
  double ds, dc;
  sincos((double)a, &ds, &dc);
  s = (float)ds; c = (float)dc;
}

// pcl::getTransformation (common/impl/eigen.hpp): row-major 3x4
__device__ __forceinline__ void particle_to_matrix(float x, float y, float z, float roll, float pitch, float yaw, float* m) {
  float A, B, C, D, E, F;
  sincos_c(yaw, B, A); sincos_c(pitch, D, C); sincos_c(roll, F, E);
  const float DE = D * E, DF = D * F;
  m[0] = A * C; m[1] = A * DF - B * E; m[2] = B * F + A * DE;  m[3] = x;
  m[4] = B * C; m[5] = A * E + B * DF; m[6] = B * DE - A * F;  m[7] = y;
  m[8] = -D;    m[9] = C * F;          m[10] = C * E;          m[11] = z;
}
__device__ __forceinline__ void matrix_to_rpy(const float* m, float& roll, float& pitch, float& yaw) {
  roll = (float)atan2((double)m[9], (double)m[10]);
  pitch = (float)asin((double)(-m[8]));
  yaw = (float)atan2((double)m[4], (double)m[0]);
}
// pcl::transformPointCloud, dense branch
__device__ __forceinline__ void xform(const float* m, float x, float y, float z, float& ox, float& oy, float& oz) {
  ox = ((m[0] * x + m[1] * y) + m[2] * z) + m[3];
  oy = ((m[4] * x + m[5] * y) + m[6] * z) + m[7];
  oz = ((m[8] * x + m[9] * y) + m[10] * z) + m[11];
}

struct Quat { float w, x, y, z; };
// Eigen::Quaternionf(Matrix3f)
__device__ inline Quat quat_from_matrix(const float* m) {
  Quat q;
  float t = (m[0] + m[5]) + m[10];
  if (t > 0.f) {
    t = sqrtf(t + 1.0f);
    q.w = 0.5f * t;
    t = 0.5f / t;
    q.x = (m[9] - m[6]) * t; q.y = (m[2] - m[8]) * t; q.z = (m[4] - m[1]) * t;
  } else {
    int i = 0;
    if (m[5] > m[0]) i = 1;
    if (m[10] > m[i * 5]) i = 2;
    const int j = (i + 1) % 3, k = (j + 1) % 3;
    t = sqrtf(((m[i * 5] - m[j * 5]) - m[k * 5]) + 1.0f);
    float v[3];
    v[i] = 0.5f * t;
    t = 0.5f / t;
    q.w = (m[k * 4 + j] - m[j * 4 + k]) * t;
    v[j] = (m[j * 4 + i] + m[i * 4 + j]) * t;
    v[k] = (m[k * 4 + i] + m[i * 4 + k]) * t;
    q.x = v[0]; q.y = v[1]; q.z = v[2];
  }
  return q;
}
__device__ __forceinline__ Quat quat_mul(const Quat& a, const Quat& b) {
  Quat r;
  r.w = ((a.w * b.w - a.x * b.x) - a.y * b.y) - a.z * b.z;
  r.x = ((a.w * b.x + a.x * b.w) + a.y * b.z) - a.z * b.y;
  r.y = ((a.w * b.y + a.y * b.w) + a.z * b.x) - a.x * b.z;
  r.z = ((a.w * b.z + a.z * b.w) + a.x * b.y) - a.y * b.x;
  return r;
}
// ParticleXYZRPY::sample with injected standard normals z[6] (SURVEY A.9)
__device__ inline void particle_sample(DevParticle& p, const NoiseParams& np, const float* z) {
  p.x += (float)(np.mean[0] + np.sigma[0] * (double)z[0]);
  p.y += (float)(np.mean[1] + np.sigma[1] * (double)z[1]);
  p.z += (float)(np.mean[2] + np.sigma[2] * (double)z[2]);
  if (!np.quat_mode) {
    p.roll += (float)(np.mean[3] + np.sigma[3] * (double)z[3]);
    p.pitch += (float)(np.mean[4] + np.sigma[4] * (double)z[4]);
    p.yaw += (float)(np.mean[5] + np.sigma[5] * (double)z[5]);
    return;
  }
  float cur[12], mr[12];
  particle_to_matrix(p.x, p.y, p.z, p.roll, p.pitch, p.yaw, cur);
  const Quat q_cur = quat_from_matrix(cur);
  particle_to_matrix((float)np.mean[0], (float)np.mean[1], (float)np.mean[2], (float)np.mean[3], (float)np.mean[4], (float)np.mean[5], mr);
  const Quat q_mean = quat_from_matrix(mr);
  const float a = (float)(np.sigma_q[0] * (double)z[3]);
  const float b = (float)(np.sigma_q[1] * (double)z[4]);
  const float c = (float)(np.sigma_q[2] * (double)z[5]);
  const float n2 = ((a * a + b * b) + c * c) + 1.0f;  // Quaternionf(Vector4f(a,b,c,1)): x,y,z,w
  const float n = sqrtf(n2);
  const Quat qs{1.0f / n, a / n, b / n, c / n};
  const Quat q = quat_mul(quat_mul(qs, q_mean), q_cur);
  const float tx = 2.f * q.x, ty = 2.f * q.y, tz = 2.f * q.z;
  const float twx = tx * q.w, twy = ty * q.w, twz = tz * q.w;
  const float txx = tx * q.x, txy = ty * q.x, txz = tz * q.x;
  const float tyy = ty * q.y, tyz = tz * q.y, tzz = tz * q.z;
  float R[12];
  R[0] = 1.f - (tyy + tzz); R[1] = txy - twz;         R[2] = txz + twy;
  R[4] = txy + twz;         R[5] = 1.f - (txx + tzz); R[6] = tyz - twx;
  R[8] = txz - twy;         R[9] = tyz + twx;         R[10] = 1.f - (txx + tyy);
  matrix_to_rpy(R, p.roll, p.pitch, p.yaw);
}

// HSVColorCoherence::RGB2HSV (integer, OpenCV style).  Upstream calls it with (Red, Blue, Green).
__device__ __forceinline__ int div_table(int i) { return i == 0 ? 0 : (2088960 + i) / (2 * i); }  // round(1044480/i)
__device__ inline unsigned int rgba_to_hsv_packed(unsigned int rgba) {
  const int B = rgba & 0xff, G = (rgba >> 8) & 0xff, R = (rgba >> 16) & 0xff;
  const int r = R, g = B, b = G;  // upstream quirk: G and B swapped at the call site
  const int v = max(r, max(g, b)), vmin = min(r, min(g, b));
  const int diff = v - vmin;
  const int vr = (v == r) ? -1 : 0, vg = (v == g) ? -1 : 0;
  const int s = (diff * div_table(v)) >> 12;
  int h = (vr & (g - b)) + (~vr & ((vg & (b - r + 2 * diff)) + ((~vg) & (r - g + 4 * diff))));
  h = (h * div_table(diff) * 15 + (1 << 18)) >> 19;
  h += h < 0 ? 180 : 0;
  return (unsigned int)h | ((unsigned int)s << 8) | ((unsigned int)v << 16);
}

// ------------------------------------------------------------------ K: init / matrices / AABB
__global__ void init_particles_kernel(TrackerState* st, DevParticle* parts, int n, const float* __restrict__ trans12,
                                      NoiseParams np, const float* __restrict__ normals /* slot 0: [stride][6] */) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  DevParticle rep{trans12[3], trans12[7], trans12[11], 1.f, 0.f, 0.f, 0.f, 0.f};
  matrix_to_rpy(trans12, rep.roll, rep.pitch, rep.yaw);
  rep.weight = 1.0f / (float)n;
  if (i == 0) {
    st->rep = rep;
    // (motion_ is NOT touched: upstream's initParticles leaves it alone, so after resetTracking() the next resample
    // still applies the motion of the frames before; it starts as zero with the tracker)
    st->particle_num = n;
    st->has_particles = 1;
    st->draw_call += 1ull;
  }
  if (i >= n) return;
  DevParticle p{0.f, 0.f, 0.f, 1.f, 0.f, 0.f, 0.f, 0.f};
  float z[6];
#pragma unroll
  for (int d = 0; d < 6; ++d) z[d] = normals[(size_t)i * 6 + d];
  particle_sample(p, np, z);
  p.x += rep.x; p.y += rep.y; p.z += rep.z; p.roll += rep.roll; p.pitch += rep.pitch; p.yaw += rep.yaw;
  p.weight = 1.0f / (float)n;
  parts[i] = p;
}

__global__ void matrices_kernel(TrackerState* st, const DevParticle* __restrict__ parts, float* __restrict__ mats) {
  const int n = st->particle_num;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) {
    st->aabb[0] = st->aabb[1] = st->aabb[2] = FLT_MAX;
    st->aabb[3] = st->aabb[4] = st->aabb[5] = -FLT_MAX;
  }
  for (int k = i; k < n; k += gridDim.x * blockDim.x) {
    const DevParticle p = parts[k];
    float m[12];
    particle_to_matrix(p.x, p.y, p.z, p.roll, p.pitch, p.yaw, m);
#pragma unroll
    for (int d = 0; d < 3; ++d) reinterpret_cast<float4*>(mats)[(size_t)k * 3 + d] = make_float4(m[4 * d], m[4 * d + 1], m[4 * d + 2], m[4 * d + 3]);
  }
}

// Per-slot boxes + their union.  Live slots of this rank's slice are recomputed; slots >= particle_num keep the box
// of the last particle that occupied them (upstream's stale transed_reference_vector_ entries).  A group of
// WARPS warps (= one block) works on one slot at a time; the union is accumulated per block in registers and
// reaches st->aabb through six atomics per block.  WARPS = 4 for small particle sets (more parallelism per slot),
// 1 for large ones (no block barrier).
template <int WARPS>
__global__ void __launch_bounds__(WARPS * 32) aabb_kernel(TrackerState* st, const float4* __restrict__ model, int M, const float* __restrict__ mats,
                                                          float* __restrict__ slot_aabb, int n_slots, int nranks, int rank,
                                                          PeerSet ps, int peer_exchange /* NVLink peer mode: the last block to finish exchanges the box with the other ranks */) {
  __shared__ float s_red[WARPS][6];
  const int n = st->particle_num;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  float un[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, ux[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};  // union over this block's slots (valid in every lane of warp 0)
  for (int s = blockIdx.x; s < n_slots; s += gridDim.x) {
    float mn[3], mx[3];
    if (s >= n) {
      // stale slot: its stored box still takes part in the union (never used slots hold an inverted box)
#pragma unroll
      for (int d = 0; d < 3; ++d) { mn[d] = slot_aabb[(size_t)s * 6 + d]; mx[d] = slot_aabb[(size_t)s * 6 + 3 + d]; }
      if (mn[0] > mx[0]) continue;
    } else {
      if (s % nranks != rank) continue;  // another rank's live slot (particle i belongs to rank i % nranks)
      float m[12];
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        const float4 r = reinterpret_cast<const float4*>(mats)[(size_t)s * 3 + d];
        m[4 * d] = r.x; m[4 * d + 1] = r.y; m[4 * d + 2] = r.z; m[4 * d + 3] = r.w;
      }
      mn[0] = mn[1] = mn[2] = FLT_MAX; mx[0] = mx[1] = mx[2] = -FLT_MAX;
      for (int j = threadIdx.x; j < M; j += WARPS * 32) {
        const float4 p = model[j];
        float x, y, z;
        xform(m, p.x, p.y, p.z, x, y, z);
        mn[0] = fminf(mn[0], x); mn[1] = fminf(mn[1], y); mn[2] = fminf(mn[2], z);
        mx[0] = fmaxf(mx[0], x); mx[1] = fmaxf(mx[1], y); mx[2] = fmaxf(mx[2], z);
      }
#pragma unroll
      for (int d = 0; d < 3; ++d) { mn[d] = warp_min(mn[d]); mx[d] = warp_max(mx[d]); }
      if (WARPS > 1) {
        __syncthreads();  // (s_red of the previous slot has been consumed)
        if (lane == 0) {
#pragma unroll
          for (int d = 0; d < 3; ++d) { s_red[wid][d] = mn[d]; s_red[wid][3 + d] = mx[d]; }
        }
        __syncthreads();
#pragma unroll
        for (int w = 0; w < WARPS; ++w) {
#pragma unroll
          for (int d = 0; d < 3; ++d) { mn[d] = fminf(mn[d], s_red[w][d]); mx[d] = fmaxf(mx[d], s_red[w][3 + d]); }
        }
      }
      if (wid == 0) {
        if (lane < 3) slot_aabb[(size_t)s * 6 + lane] = mn[lane];
        else if (lane < 6) slot_aabb[(size_t)s * 6 + lane] = mx[lane - 3];
      }
    }
#pragma unroll
    for (int d = 0; d < 3; ++d) { un[d] = fminf(un[d], mn[d]); ux[d] = fmaxf(ux[d], mx[d]); }
  }
  if (wid == 0 && un[0] <= ux[0]) {
    if (lane < 3) atomic_min_float(&st->aabb[lane], un[lane]);
    else if (lane < 6) atomic_max_float(&st->aabb[lane], ux[lane - 3]);
  }
  if (peer_exchange && wid == 0) {
    // the block that finishes last holds this rank's complete box: its first warp runs the exchange (no extra launch)
    unsigned int done = 0;
    __syncwarp();
    if (lane == 0) { __threadfence(); done = atomicAdd(&st->aabb_blocks_done, 1u) + 1u; }
    done = __shfl_sync(kFull, done, 0);
    if (done == gridDim.x) {
      if (lane == 0) { st->aabb_blocks_done = 0u; __threadfence(); }
      __syncwarp();
      peer_box_exchange(st, ps);
    }
  }
}

// ------------------------------------------------------------------ K2: scene index build
// The index is a dense uniform grid over the crop box in CSR form: cell_start[c] .. cell_start[c+1] are the slots
// of the points of cell c (cells x-fastest, so the points of any x-window of a row are ONE contiguous slot range).
// It replaces pcl::search::Octree::setInputCloud (a pointer octree rebuilt by every weight(), SURVEY A.5); the cell
// edge is an internal choice (base resolution x 2^level) that never changes results: the search below is exact.
__device__ inline void compute_index_header(const float* crop, const float* aabb /* box to index: the crop box, possibly dilated */, float inv_leaf,
                                            int base_level, int max_cells, IndexHeader& h) {
#pragma unroll
  for (int d = 0; d < 6; ++d) { h.aabb[d] = crop[d]; h.built[d] = aabb[d]; h.core[d] = crop[d]; }
  h.reuse = 0; h.n_in_crop = 0; h.dilate = 0.f;
  h.inv_leaf = inv_leaf;
  h.n_cropped = 0;
  h.valid = (crop[0] <= crop[3] && crop[1] <= crop[4] && crop[2] <= crop[5]) ? 1 : 0;
  h.level = base_level; h.level_scale = 1.0f; h.n_cells = 0;
  h.dim[0] = h.dim[1] = h.dim[2] = 0; h.origin[0] = h.origin[1] = h.origin[2] = 0;
  h.cell = 1.0f / inv_leaf;
  h.f_cells = 0; h.use_lists = 0;
  h.f_origin[0] = h.f_origin[1] = h.f_origin[2] = 0; h.f_dim[0] = h.f_dim[1] = h.f_dim[2] = 0;
  if (!h.valid) return;
  float lo[3], hi[3];
#pragma unroll
  for (int d = 0; d < 3; ++d) { lo[d] = aabb[d] * inv_leaf; hi[d] = aabb[3 + d] * inv_leaf; }
  {
    long long fc = 1;
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      h.f_origin[d] = (int)floorf(lo[d]);
      h.f_dim[d] = (int)floorf(hi[d]) - h.f_origin[d] + 1;
      fc *= (long long)h.f_dim[d];
      if (fc > (1ll << 30)) fc = 1ll << 30;
    }
    h.f_cells = (int)fc;
  }
  for (int level = base_level; level < 24; ++level) {
    const float ls = 1.0f / (float)(1 << level);
    int dim[3], org[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      org[d] = (int)floorf(lo[d] * ls);
      dim[d] = (int)floorf(hi[d] * ls) - org[d] + 1;
    }
    const long long cells = (long long)dim[0] * dim[1] * dim[2];
    if (cells <= (long long)max_cells || level == 23) {
      h.level = level; h.level_scale = ls; h.n_cells = (int)min(cells, (long long)max_cells);
#pragma unroll
      for (int d = 0; d < 3; ++d) { h.dim[d] = dim[d]; h.origin[d] = org[d]; }
      h.cell = (float)(1 << level) / inv_leaf;
      break;
    }
  }
}

// Every block derives the header from the crop box (a pure function of it), block 0 publishes it, and all
// blocks clear the per-cell counters.
// The cell edge follows the mean nearest-neighbour distance of the previous weight() (a query that is d away from the
// surface walks ~pi (d/cell + 1)^2 rows and ~(d + cell)^2 candidates: cell ~ d balances them).
__global__ void index_begin_kernel(TrackerState* st, IndexHeader* hdr, int* cell_count, float inv_leaf, int max_cells,
                                   int list_max_cells, int M, int nranks, int rank, unsigned int* needed_words,
                                   int* list_counters /* [0] extended lists handed out, [1] needed blocks, [2] cells queued for the far pass, [3] pool groups handed out, [4] cells queued for the octant pass */,
                                   unsigned int* built_bits /* one bit per fine cell: its lists exist (this frame) */, int reuse_allowed, float dilate,
                                   int list_ratio /* the lists are built when this rank's queries outnumber the fine cells of the crop box by this factor */,
                                   const IndexHeader* __restrict__ hdr_prev /* header of the previous weight() (snapshot taken by index_scan_kernel:
                                                                               nothing writes it while this kernel runs, so every block derives the same header) */) {
  __shared__ IndexHeader h;
  PFT_TRACE_MIN(0);
  if (threadIdx.x == 0) {
    const IndexHeader old = *hdr_prev;
    bool reuse = reuse_allowed && old.valid && old.use_lists && old.n_cropped < 65535;
    if (reuse) {
      // the new crop box must lie inside the box the index was built from (an empty crop box reuses nothing)
      reuse = st->aabb[0] <= st->aabb[3] && st->aabb[1] <= st->aabb[4] && st->aabb[2] <= st->aabb[5];
#pragma unroll
      for (int d = 0; d < 3; ++d) reuse = reuse && st->aabb[d] >= old.built[d] && st->aabb[3 + d] <= old.built[3 + d];
      // ... and contain the core the reusable lists depend on (an inverted core = nothing was reusable: no constraint)
      if (old.core[0] <= old.core[3] && old.core[1] <= old.core[4] && old.core[2] <= old.core[5]) {
#pragma unroll
        for (int d = 0; d < 3; ++d) reuse = reuse && st->aabb[d] <= old.core[d] && st->aabb[3 + d] >= old.core[3 + d];
      }
    }
    if (reuse) {
      h = old;
#pragma unroll
      for (int d = 0; d < 6; ++d) h.aabb[d] = st->aabb[d];
      h.reuse = 1; h.n_in_crop = 0; h.epoch = old.epoch + 1u;
#pragma unroll
      for (int d = 0; d < 3; ++d) { h.core[d] = fminf(old.core[d], st->aabb[d] + old.dilate); h.core[3 + d] = fmaxf(old.core[3 + d], st->aabb[3 + d] - old.dilate); }
    } else {
      int base_level = 1;
      if (st->nn_count > 0) {
        const float mean_d = (float)((double)st->nn_sum_um / (double)st->nn_count) * 1.0e-6f;
        const float want = mean_d * 1.15f * inv_leaf;  // cell edge in units of the resolution
        base_level = want <= 1.5f ? 1 : (want <= 3.0f ? 1 : (want <= 6.0f ? 2 : (want <= 12.0f ? 3 : 4)));
      }
      // candidate lists pay off when this rank's queries outnumber the fine cells they are built for
      const int n = st->particle_num;
      const long long n_local = n > rank ? (n - rank + nranks - 1) / nranks : 0;
      float box[6];
#pragma unroll
      for (int d = 0; d < 6; ++d) box[d] = st->aabb[d];
      compute_index_header(st->aabb, box, inv_leaf, base_level, max_cells, h);
      // (M == 0: the caller forces the lists on)
      bool lists = h.valid && h.f_cells > 0 && h.f_cells <= list_max_cells && (M == 0 || n_local * (long long)M >= (long long)list_ratio * h.f_cells);
      if (lists && dilate > 0.f) {
        // lists on: index the dilated box, so that the next weight() of the frame can reuse the index (when the dilated
        // box does not fit the list tables, the plain crop box is indexed and the next weight() rebuilds)
        IndexHeader hd;
#pragma unroll
        for (int d = 0; d < 3; ++d) { box[d] = st->aabb[d] - dilate; box[3 + d] = st->aabb[3 + d] + dilate; }
        compute_index_header(st->aabb, box, inv_leaf, base_level, max_cells, hd);
        if (hd.f_cells > 0 && hd.f_cells <= list_max_cells) {
          h = hd;
          h.dilate = dilate;
#pragma unroll
          for (int d = 0; d < 3; ++d) { h.core[d] = st->aabb[d] + dilate; h.core[3 + d] = st->aabb[3 + d] - dilate; }
        }
      }
      h.use_lists = lists ? 1 : 0;
      h.epoch = old.epoch + 1u;
    }
    if (blockIdx.x == 0) *hdr = h;
  }
  __syncthreads();
  if (!h.reuse) {
    const int nc = h.n_cells + 1;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nc; i += gridDim.x * blockDim.x) cell_count[i] = 0;
  }
  if (h.use_lists) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < h.f_cells; i += gridDim.x * blockDim.x) needed_words[i] = 0u;
    if (!h.reuse) {
      const int words = (h.f_cells + 31) >> 5;
      for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < words; i += gridDim.x * blockDim.x) built_bits[i] = 0u;
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    // (a reusing weight() keeps handing out extended lists and pool groups where the earlier ones stopped)
    if (!h.reuse) { list_counters[0] = 0; list_counters[3] = 0; }
    list_counters[1] = 0; list_counters[2] = 0; list_counters[4] = 0;
    st->work_counter = 0u;
  }
}

// the points the index holds: finite and inside the box it was built from (the crop box, or the crop box dilated)
__device__ __forceinline__ bool in_built(const float4& p, const IndexHeader& h) {
  return isfinite(p.x) && isfinite(p.y) && isfinite(p.z) && p.x >= h.built[0] && p.x <= h.built[3] && p.y >= h.built[1] &&
         p.y <= h.built[4] && p.z >= h.built[2] && p.z <= h.built[5];
}
constexpr unsigned int kInCropBit = 0x80000000u;  // fourth word of a staged point: packed HSV | this bit when the point lies in the crop box of the running weight()
__device__ __forceinline__ bool in_crop(const float4& p, const IndexHeader& h) {
  // three inclusive PassThrough passes (x, y, z) on finite points
  return isfinite(p.x) && isfinite(p.y) && isfinite(p.z) && p.x >= h.aabb[0] && p.x <= h.aabb[3] && p.y >= h.aabb[1] &&
         p.y <= h.aabb[4] && p.z >= h.aabb[2] && p.z <= h.aabb[5];
}
__device__ __forceinline__ int cell_of(const float4& p, const IndexHeader& h) {
  const int cx = (int)floorf((p.x * h.inv_leaf) * h.level_scale) - h.origin[0];
  const int cy = (int)floorf((p.y * h.inv_leaf) * h.level_scale) - h.origin[1];
  const int cz = (int)floorf((p.z * h.inv_leaf) * h.level_scale) - h.origin[2];
  return (cz * h.dim[1] + cy) * h.dim[0] + cx;
}

__global__ void index_count_kernel(const float4* __restrict__ scene, const CloudHeader* __restrict__ scene_hdr, IndexHeader* hdr, int* cell_count,
                                   float4* __restrict__ pts2) {
  __shared__ IndexHeader h;
  if (threadIdx.x == 0) h = *hdr;
  __syncthreads();
  if (!h.valid) return;
  if (h.reuse) {
    // the index stays: only the crop box has changed -- refresh the in-crop flag of every indexed point and count them
    int local = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < h.n_cropped; i += gridDim.x * blockDim.x) {
      float4 p = pts2[i];
      const bool in = in_crop(p, h);
      const unsigned int w = (__float_as_uint(p.w) & ~kInCropBit) | (in ? kInCropBit : 0u);
      if (w != __float_as_uint(p.w)) pts2[i].w = __uint_as_float(w);
      local += in ? 1 : 0;
    }
    local = warp_sum(local);
    if ((threadIdx.x & 31) == 0 && local) atomicAdd(&hdr->n_in_crop, local);
    return;
  }
  const int ns = scene_hdr->n;
  int local = 0, local_in = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < ns; i += gridDim.x * blockDim.x) {
    const float4 p = scene[i];
    if (!in_built(p, h)) continue;
    atomicAdd(&cell_count[cell_of(p, h)], 1);
    ++local;
    local_in += in_crop(p, h) ? 1 : 0;
  }
  local = warp_sum(local);
  local_in = warp_sum(local_in);
  if ((threadIdx.x & 31) == 0 && local) { atomicAdd(&hdr->n_cropped, local); atomicAdd(&hdr->n_in_crop, local_in); }
}

// exclusive prefix of the cell counts -> cell_start; the counters are cleared again (they become the fill cursors)
__global__ void __launch_bounds__(1024) index_scan_kernel(const IndexHeader* __restrict__ hdr, int* cell_count, int* __restrict__ cell_start,
                                                          TrackerState* st, float4* __restrict__ pts, float4* __restrict__ pts2, IndexHeader* hdr_prev) {
  __shared__ int smem[34];
  const int nc = hdr->n_cells;
  if (threadIdx.x == 0) {
    st->nn_sum_um = 0ull; st->nn_count = 0ull;  // consumed by index_begin; refilled by the weight kernel
    *hdr_prev = *hdr;  // what the next weight() of the frame tests its crop box against (the point counts are final by now)
  }
  if (hdr->reuse) return;
  const int total = block_exclusive_scan<int>(
      nc, [&](int i) { return cell_count[i]; }, [&](int i, int ex) { cell_start[i] = ex; cell_count[i] = 0; }, smem);
  if (threadIdx.x == 0) {
    cell_start[nc] = total;
    // slot `total` is a dummy point infinitely far away: candidate lists are padded with it to a multiple of 8 entries
    pts[total] = make_float4(3.0e38f, 3.0e38f, 3.0e38f, __int_as_float(0x7fffffff));
    pts2[total] = make_float4(3.0e38f, 3.0e38f, 3.0e38f, 0.f);
  }
}

__global__ void index_scatter_kernel(const float4* __restrict__ scene, const CloudHeader* __restrict__ scene_hdr, const IndexHeader* __restrict__ hdr,
                                     const int* __restrict__ cell_start, int* cell_count, float4* __restrict__ pts, unsigned int* __restrict__ hsv,
                                     float4* __restrict__ pts2 /* {x, y, z, packed HSV}: what weight_lists_kernel stages into shared memory */) {
  __shared__ IndexHeader h;
  if (threadIdx.x == 0) h = *hdr;
  __syncthreads();
  if (!h.valid || h.reuse) return;
  const int ns = scene_hdr->n;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < ns; i += gridDim.x * blockDim.x) {
    const float4 p = scene[i];
    if (!in_built(p, h)) continue;
    const int c = cell_of(p, h);
    const int pos = cell_start[c] + atomicAdd(&cell_count[c], 1);
    pts[pos] = make_float4(p.x, p.y, p.z, __int_as_float(i));  // .w = index in the input cloud (tie-break key)
    const unsigned int packed = rgba_to_hsv_packed(__float_as_uint(p.w));
    hsv[pos] = packed;
    pts2[pos] = make_float4(p.x, p.y, p.z, __uint_as_float(packed | (in_crop(p, h) ? kInCropBit : 0u)));
  }
}

// ------------------------------------------------------------------ K3: weight
// Exact nearest neighbour over the CSR grid.  One lane = one query.  The (dy,dz) rows of cells around the query cell
// are visited in order of a precomputed lower bound of their distance (RowTable); a row is skipped when its exact
// lower bound exceeds the best distance so far, the traversal stops at the first table entry whose bound does, and
// inside a row only the x-window that can still hold a closer point is read: one contiguous slot range.
// Ties go to the lower input index.  The radius is capped at maximum_distance_ (points farther than that never
// contribute to the coherence); beyond the table's reach the search continues shell by shell.
//
// The index of a typical crop (a few thousand points: ~100 KB of points + ~50 KB of cell starts) is staged into
// shared memory once per CTA by a persistent one-CTA-per-SM launch; larger indices are read through L1/L2.
#ifdef PFT_STATS
__device__ unsigned long long g_stats[48];
#define PFT_STAT(i, v) atomicAdd(&g_stats[i], (unsigned long long)(v))
#else
#define PFT_STAT(i, v)
#endif
constexpr int kRT = 11;                         // table reach in cells (Chebyshev)
constexpr int kRows = (2 * kRT + 1) * (2 * kRT + 1);
struct RowEntry { signed char dy, dz; unsigned short lb2; };  // lb2 = gap(dy)^2 + gap(dz)^2, gap(d) = max(|d|-1, 0)

// Best candidate so far.  Ties in distance go to the lower input index.
struct NNResult {
  float dist2;
  int orig_idx;
  int slot;
  __device__ __forceinline__ float d2() const { return dist2; }
  __device__ __forceinline__ int orig() const { return orig_idx; }
};
__device__ __forceinline__ NNResult nn_none(float lim2) { return NNResult{lim2, (int)0x80000000, -1}; }  // only d2 < lim2 can beat it

__device__ __forceinline__ void nn_eval(const IndexHeader& h, const float4* __restrict__ pts, int slot, float qx, float qy, float qz, NNResult& best) {
  const float4 p = pts[slot];
  // (the index may hold points beyond the crop box of this weight(), see IndexHeader::built: they are not candidates)
  if (!(p.x >= h.aabb[0] && p.x <= h.aabb[3] && p.y >= h.aabb[1] && p.y <= h.aabb[4] && p.z >= h.aabb[2] && p.z <= h.aabb[5])) return;
  const float dx = qx - p.x, dy = qy - p.y, dz = qz - p.z;
  const float d2 = (dx * dx + dy * dy) + dz * dz;
  const int orig = __float_as_int(p.w);
  if (d2 < best.dist2 || (d2 == best.dist2 && orig < best.orig_idx)) { best.dist2 = d2; best.orig_idx = orig; best.slot = slot; }
}

// distance (cell units) from the query at fractional position t of its cell to the cell at offset d, minus a
// safety margin that covers the fp32 rounding of the lattice coordinates (so it is a true lower bound)
__device__ __forceinline__ float axis_gap(int d, float t) {
  const float g = d > 0 ? (float)d - t : (d < 0 ? t - (float)(d + 1) : 0.f);
  return fmaxf(g - 2.5e-4f, 0.f);
}

// Shell-by-shell continuation beyond the row table (large maximum distances / very fine cells): rare path.
template <typename CS>
__device__ __noinline__ NNResult nn_search_shells(const CS* __restrict__ cs, const float4* __restrict__ pts, const IndexHeader& h, float qx, float qy,
                                                  float qz, int cx, int cy, int cz, float tx, float ty, float tz, float lim2, NNResult best) {
  const float tmin = fminf(fminf(fminf(tx, 1.f - tx), fminf(ty, 1.f - ty)), fminf(tz, 1.f - tz));
  const float cell2 = h.cell * h.cell;
  int r_prev = kRT, r = kRT + 1;
  while (true) {
    const float done = ((float)r_prev + tmin - 2.5e-4f) * h.cell;  // everything unscanned is farther than this
    const bool covered = (cx - r_prev <= 0) && (cx + r_prev >= h.dim[0] - 1) && (cy - r_prev <= 0) && (cy + r_prev >= h.dim[1] - 1) &&
                         (cz - r_prev <= 0) && (cz + r_prev >= h.dim[2] - 1);
    if (covered || done * done * 0.9999f > fminf(best.d2(), lim2)) return best;
    const int z0 = max(cz - r, 0), z1 = min(cz + r, h.dim[2] - 1);
    const int y0 = max(cy - r, 0), y1 = min(cy + r, h.dim[1] - 1);
    for (int z = z0; z <= z1; ++z) {
      const int dz = z - cz;
      const float az = axis_gap(dz, tz);
      for (int y = y0; y <= y1; ++y) {
        const int dy = y - cy;
        const float ay = axis_gap(dy, ty);
        if ((az * az + ay * ay) * cell2 * 0.9999f > best.d2()) continue;
        const int base = (z * h.dim[1] + y) * h.dim[0];
        const bool inner = max(abs(dy), abs(dz)) <= r_prev;
        for (int seg = 0; seg < 2; ++seg) {
          int xa, xb;
          if (!inner) { if (seg) break; xa = cx - r; xb = cx + r; }
          else if (seg == 0) { xa = cx - r; xb = cx - r_prev - 1; }
          else { xa = cx + r_prev + 1; xb = cx + r; }
          xa = max(xa, 0); xb = min(xb, h.dim[0] - 1);
          if (xa > xb) continue;
          const int s1 = (int)cs[base + xb + 1];
          for (int s = (int)cs[base + xa]; s < s1; ++s) nn_eval(h, pts, s, qx, qy, qz, best);
        }
      }
    }
    r_prev = r;
    int need = 2 * r;
    if (best.slot >= 0) need = max(r + 1, (int)ceilf(sqrtf(best.d2()) / h.cell - tmin + 0.004f));
    const int rcap = max(r + 1, (int)ceilf(sqrtf(lim2) / h.cell - tmin + 0.004f));
    r = min(need, rcap);
  }
}

template <typename CS>
__device__ __forceinline__ NNResult nn_search(const CS* __restrict__ cs, const float4* __restrict__ pts, const IndexHeader& h,
                                              const RowEntry* __restrict__ table, float qx, float qy, float qz, float lim2) {
  NNResult best = nn_none(lim2);
  const float sx = (qx * h.inv_leaf) * h.level_scale, sy = (qy * h.inv_leaf) * h.level_scale, sz = (qz * h.inv_leaf) * h.level_scale;
  const float fx = floorf(sx), fy = floorf(sy), fz = floorf(sz);
  // (int) of a huge float is undefined: clamp first; such queries are far outside the grid anyway
  const float big = 1.0e9f;
  const int cx = (int)fminf(fmaxf(fx, -big), big) - h.origin[0], cy = (int)fminf(fmaxf(fy, -big), big) - h.origin[1],
            cz = (int)fminf(fmaxf(fz, -big), big) - h.origin[2];
  const float tx = sx - fx, ty = sy - fy, tz = sz - fz;
  const float cell2 = h.cell * h.cell;
  const float inv_cell = 1.0f / h.cell;
  const int dimx = h.dim[0], dimy = h.dim[1], dimz = h.dim[2];
  PFT_STAT(6, 1);
  for (int k = 0; k < kRows; ++k) {
    const RowEntry e = table[k];
    if ((float)e.lb2 * cell2 * 0.9999f > best.d2()) break;  // every later row is at least this far
    PFT_STAT(7, 1);
    const int y = cy + e.dy, z = cz + e.dz;
    if ((unsigned)y >= (unsigned)dimy || (unsigned)z >= (unsigned)dimz) continue;
    const float ay = axis_gap(e.dy, ty), az = axis_gap(e.dz, tz);
    const float row2 = (ay * ay + az * az) * cell2 * 0.9999f;
    if (row2 > best.d2()) continue;
    // cells of this row that can still hold a point at distance <= best: |x gap| <= hw (cell units)
    const float hw = fminf(sqrtf(best.d2() - row2) * inv_cell + 5.0e-4f, (float)kRT);
    int xa = cx + (int)ceilf(tx - 1.0f - hw), xb = cx + (int)floorf(tx + hw);
    xa = max(xa, 0); xb = min(xb, dimx - 1);
    if (xa > xb) continue;
    PFT_STAT(8, 1);
    const int base = (z * dimy + y) * dimx;
    const int s1 = (int)cs[base + xb + 1];
    for (int s = (int)cs[base + xa]; s < s1; ++s) { PFT_STAT(9, 1); nn_eval(h, pts, s, qx, qy, qz, best); }
  }
  // rows outside the table start at a distance of kRT cells: only then can the search have missed something
  if (best.d2() > (float)(kRT * kRT) * cell2 * 0.99f) best = nn_search_shells<CS>(cs, pts, h, qx, qy, qz, cx, cy, cz, tx, ty, tz, lim2, best);
  return best;
}

// ---- candidate lists: the exact nearest neighbour as a table lookup.
// For every cell c of the fine lattice (edge = resolution) the build finds the slots of ALL points that can be the
// nearest neighbour of SOME query inside c: with p0 the point minimising maxdist(c, .) and U = maxdist(c, p0), any
// query q in c has |q - NN(q)| <= |q - p0| <= U, hence mindist(c, NN(q)) <= U, and q lies on NN(q)'s side of the
// bisector plane of (NN(q), p0) (can_win); the list is every point passing both tests (ties included), cut at
// maximum_distance_.  The same two tests are then applied to each of the cell's eight OCTANTS (edge = resolution / 2),
// which is what a query reads: one 32-byte record = header + seven entries, enough for 99.7 % of the queries (mean
// length 3.1); an octant that still holds more than seven points after the p0 tests is pruned pairwise (a point that
// some other candidate beats everywhere in the octant can never win) and what remains beyond seven goes to groups of
// eight taken from a pool.  Every sub-list is in ascending order of the input index, so that the lookup
// resolves distance ties by position (strict <: the first of equals wins = the lower index, the parity contract).
//
// Octant record = 8 words of 32 bits (one 32-byte sector, read by ONE 256-bit load):
//   word 0      header: 0..7 = entry count | count (8..71) + (g << 8) = entries beyond the seventh are in pool groups
//               g, g+1, .. (eight entries each) | kListExtended = word 1 holds the index of an extended list (cells far
//               from the surface whose list pairwise pruning cannot shorten: up to kListKX entries in input-index order),
//               word 2 its length | kListOverflow = no list (the query is answered by brute force)
//   words 1..7  entries as BYTE offsets of the points in the staged array (slot << 4), padded with the dummy slot
constexpr int kL1Cap = 64;                         // a cell's own list is split into octants up to this length; longer ones become extended lists
constexpr int kListKX = 1024;                      // entries of an extended list (cells far from the surface)
constexpr int kListXCells = 8192;                  // extended lists available per build
constexpr int kPoolGroups = 1 << 18;               // groups of eight entries for octant lists longer than seven
constexpr unsigned int kListOverflow = 0xffffffffu;  // no list
constexpr unsigned int kListExtended = 0xfffffffeu;  // extended list
// the build passes carry 16-bit slots: larger crops use the row-table search only
__device__ __forceinline__ bool lists_on(const IndexHeader& h) { return h.use_lists && h.n_cropped < 65535; }

__device__ __forceinline__ float box_mindist2(const float* lo, const float* hi, const float4& p) {
  const float dx = fmaxf(fmaxf(lo[0] - p.x, p.x - hi[0]), 0.f), dy = fmaxf(fmaxf(lo[1] - p.y, p.y - hi[1]), 0.f),
              dz = fmaxf(fmaxf(lo[2] - p.z, p.z - hi[2]), 0.f);
  return (dx * dx + dy * dy) + dz * dz;
}
__device__ __forceinline__ float box_maxdist2(const float* lo, const float* hi, const float4& p) {
  const float dx = fmaxf(fabsf(p.x - lo[0]), fabsf(p.x - hi[0])), dy = fmaxf(fabsf(p.y - lo[1]), fabsf(p.y - hi[1])),
              dz = fmaxf(fabsf(p.z - lo[2]), fabsf(p.z - hi[2]));
  return (dx * dx + dy * dy) + dz * dz;
}

// marks the fine cells that this rank's queries fall into (the lists of the others are never read).
// COUNT (small query sets): needed[c] = number of queries of the cell, one L2 reduction per query -- cells with fewer
// than kCoarseBelow queries get one list for the whole cell instead of eight octant lists (half of the cells hold a few
// per cent of the queries: those of the outlying particles).  Otherwise (large sets: every cell is busy) no global
// atomics and no global loads: a cell is flagged with a plain store (duplicates are harmless); cand_collect_kernel
// then queues the blocks.  (Reading a flag back here costs a round trip between the two L2 partitions whenever
// another SM has just stored to the line: measured 2.5x slower.)
// The particle set is concentrated, so the same model points of different particles fall into the same cells: a
// thread block therefore handles ONE group of kMarkUnroll x 32 consecutive model points for many particles and
// remembers the cells it has flagged in a bitmap of the fine grid in shared memory (f_cells bits, dynamic): every
// block stores every cell at most once.
constexpr int kMarkUnroll = 4;
constexpr unsigned int kCoarseBelow = 24u;               // queries of a cell below which its list is not split into octants
constexpr unsigned int kLightBelow = 256u;               // ... below which a list that fits one record is not split either
template <bool COUNT>
__global__ void __launch_bounds__(256) cand_mark_kernel(const TrackerState* __restrict__ st, const IndexHeader* __restrict__ hdr, const float4* __restrict__ model, int M,
                                                        const float* __restrict__ mats, unsigned int* __restrict__ needed, int nranks, int rank,
                                                        const unsigned int* __restrict__ built_bits) {
  extern __shared__ unsigned int s_bits[];  // (f_cells + 31) / 32 words
  __shared__ IndexHeader h;
  if (threadIdx.x == 0) h = *hdr;
  __syncthreads();
  if (!h.valid || !h.use_lists) return;  // (not lists_on(): the indexed points are being counted beside this kernel)
  // one bit per fine cell: "nothing to do for this cell" -- its lists exist already (a weight() that reuses the index of
  // the frame), or (flag mode) this block has flagged it
  const bool use_bits = !COUNT || h.reuse;
  if (use_bits) {
    const int words = (h.f_cells + 31) >> 5;
    for (int i = threadIdx.x; i < words; i += blockDim.x) s_bits[i] = h.reuse ? built_bits[i] : 0u;
    __syncthreads();
  }
  const int n = st->particle_num;
  const int n_local = n > rank ? (n - rank + nranks - 1) / nranks : 0;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  const int groups = (M + 32 * kMarkUnroll - 1) / (32 * kMarkUnroll);
  const int per_group = max(1, (int)gridDim.x / groups);  // blocks that share one group of model points
  const float inv_leaf = h.inv_leaf;
  const int ox = h.f_origin[0], oy = h.f_origin[1], oz = h.f_origin[2];
  const int fdx = h.f_dim[0], fdy = h.f_dim[1], fdz = h.f_dim[2];
  for (int vb = blockIdx.x; vb < groups * per_group; vb += gridDim.x) {
    const int g = vb % groups, pb = vb / groups;
    const int j0 = g * (32 * kMarkUnroll) + lane;
    float4 mp[kMarkUnroll];
#pragma unroll
    for (int u = 0; u < kMarkUnroll; ++u) mp[u] = (j0 + 32 * u < M) ? model[j0 + 32 * u] : make_float4(0.f, 0.f, 0.f, 0.f);
    for (int l = pb * wpb + wid; l < n_local; l += per_group * wpb) {
      const int i = rank + l * nranks;
      const float4* mr = reinterpret_cast<const float4*>(mats) + (size_t)i * 3;
      const float4 r0 = mr[0], r1 = mr[1], r2 = mr[2];
      const float m[12] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w, r2.x, r2.y, r2.z, r2.w};
#pragma unroll
      for (int u = 0; u < kMarkUnroll; ++u) {
        if (j0 + 32 * u < M) {
          float qx, qy, qz;
          xform(m, mp[u].x, mp[u].y, mp[u].z, qx, qy, qz);
          const float big = 1.0e9f;
          const int ix = (int)fminf(fmaxf(floorf(qx * inv_leaf), -big), big) - ox, iy = (int)fminf(fmaxf(floorf(qy * inv_leaf), -big), big) - oy,
                    iz = (int)fminf(fmaxf(floorf(qz * inv_leaf), -big), big) - oz;
          if ((unsigned)ix < (unsigned)fdx && (unsigned)iy < (unsigned)fdy && (unsigned)iz < (unsigned)fdz) {
            const int c = (iz * fdy + iy) * fdx + ix;
            if (COUNT) {
              if (!use_bits || !((s_bits[c >> 5] >> (c & 31)) & 1u)) atomicAdd(&needed[c], 1u);  // (no return value: a reduction at the L2, nothing comes back)
            } else {
              const unsigned int bit = 1u << (c & 31);
              if (!(s_bits[c >> 5] & bit)) {  // (cheap pre-test; the atomic decides)
                if (!(atomicOr(&s_bits[c >> 5], bit) & bit)) needed[c] = 0x40000000u;  // (a flag: a busy cell)
              }
            }
          }
        }
      }
    }
    // (the bitmap stays valid across the groups of one block: it only records which flags this block has stored)
  }
}

// queues every block of 2x2x2 fine cells that holds a marked cell (one thread per block, warp-aggregated append)
__global__ void __launch_bounds__(256) cand_collect_kernel(const IndexHeader* __restrict__ hdr, const unsigned int* __restrict__ needed,
                                                           int* __restrict__ needed_list, int* __restrict__ list_counters) {
  __shared__ IndexHeader h;
  if (threadIdx.x == 0) h = *hdr;
  __syncthreads();
  if (!h.valid || !h.use_lists) return;
  const int fdx = h.f_dim[0], fdy = h.f_dim[1], fdz = h.f_dim[2];
  const int bdx = (fdx + 1) >> 1, bdy = (fdy + 1) >> 1, bdz = (fdz + 1) >> 1;
  const int nb = bdx * bdy * bdz;
  const int lane = threadIdx.x & 31;
  for (int b0 = (blockIdx.x * blockDim.x + threadIdx.x) & ~31; b0 < nb; b0 += gridDim.x * blockDim.x) {
    const int blk = b0 + lane;
    bool any = false;
    if (blk < nb) {
      const int bz = blk / (bdx * bdy), br = blk - bz * bdx * bdy, by = br / bdx, bx = br - by * bdx;
#pragma unroll
      for (int sub = 0; sub < 8; ++sub) {
        const int fx = 2 * bx + (sub & 1), fy = 2 * by + ((sub >> 1) & 1), fz = 2 * bz + (sub >> 2);
        if (fx < fdx && fy < fdy && fz < fdz) {
          const int c = (fz * fdy + fy) * fdx + fx;
          if (needed[c] != 0u) any = true;
#ifdef PFT_STATS
          { const unsigned int q = needed[c]; if (q) { const int b = min(31 - __clz(q), 9); PFT_STAT(16 + b, 1); PFT_STAT(26 + b, q); } }
#endif
        }
      }
    }
    const unsigned int bal = __ballot_sync(kFull, any);
    PFT_STAT(36, any ? 1 : 0);
    if (bal) {
      int base = 0;
      if (lane == 0) base = atomicAdd(&list_counters[1], __popc(bal));
      base = __shfl_sync(kFull, base, 0);
      if (any) needed_list[base + __popc(bal & ((1u << lane) - 1u))] = blk;
    }
  }
}

// One warp builds the list of one needed cell.
// (1) U = min over nearby points p of maxdist(cell, p): an upper bound of the nearest-neighbour distance of every
//     query of the cell (the tightest one when the minimiser lies in the probed block, a valid one always).
// (2) every point whose distance to the cell does not exceed U is appended (the ball is walked row by row).
// Both steps run over "the points of a set of rows" flattened across the warp: each lane fetches the slot range of
// one row, a warp scan turns the counts into offsets, and the 32 lanes then take consecutive points of the
// concatenation (binary search of the offsets in shared memory), so every lane is busy whatever the row lengths.
struct RowSpan { int s0, cnt; };

template <typename RowFn, typename PointFn>
__device__ __forceinline__ void warp_points_of_rows(int nrows, int* s_pref, int* s_start, RowFn row_span, PointFn fn) {
  const int lane = threadIdx.x & 31;
  for (int rbase = 0; rbase < nrows; rbase += 32) {
    RowSpan sp{0, 0};
    if (rbase + lane < nrows) sp = row_span(rbase + lane);
    int inc = sp.cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(kFull, inc, o); if (lane >= o) inc += t; }
    const int total = __shfl_sync(kFull, inc, 31);
    s_pref[lane] = inc - sp.cnt;
    s_start[lane] = sp.s0;
    __syncwarp();
    for (int t = lane; t < total; t += 32) {
      int r = 0;
#pragma unroll
      for (int step = 16; step > 0; step >>= 1) if (s_pref[r + step] <= t) r += step;  // last row whose offset is <= t
      fn(s_start[r] + (t - s_pref[r]));
    }
    __syncwarp();
  }
}

constexpr int kSuperCap = 256;  // points a block's superset can hold in shared memory

// bisector test: can p be at least as near as p0 for SOME q of the box (centre bc, half extents bh)?
// min over the box of |q-p|^2 - |q-p0|^2 is linear in q and attained at a corner; coordinates relative to the box
// centre keep the fp32 error ~1e-9.
__device__ __forceinline__ bool can_win(const float4& p, const float4& p0, const float* bc, const float* bh) {
  const float px = p.x - bc[0], py = p.y - bc[1], pz = p.z - bc[2];
  const float qx = p0.x - bc[0], qy = p0.y - bc[1], qz = p0.z - bc[2];
  const float pn = (px * px + py * py) + pz * pz, p0n = (qx * qx + qy * qy) + qz * qz;
  const float fmin = (pn - p0n) - 2.0f * ((bh[0] * fabsf(px - qx) + bh[1] * fabsf(py - qy)) + bh[2] * fabsf(pz - qz));
  return fmin <= 1.0e-6f * (pn + p0n) + 1.0e-9f;
}

// index (in records of 8 words) of octant (ox, oy, oz) of fine cell (fx, fy, fz): the octants form one dense lattice of
// edge resolution / 2 over the crop box, x fastest -- what a query computes directly from floor(q * 2 / resolution)
__device__ __forceinline__ size_t octant_record(const IndexHeader& h, int fx, int fy, int fz, int o) {
  return ((size_t)(2 * fz + (o >> 2)) * (size_t)(2 * h.f_dim[1]) + (size_t)(2 * fy + ((o >> 1) & 1))) * (size_t)(2 * h.f_dim[0]) + (size_t)(2 * fx + (o & 1));
}

// All eight octant records of a cell get the same code (lanes 0..7 of the calling warp):
// kListOverflow / 0 (empty list) / kListExtended with the index and length of the extended list.
__device__ __forceinline__ void write_octant_codes(const IndexHeader& h, unsigned int* __restrict__ flists, int fx, int fy, int fz, unsigned int code, int xi, int n) {
  const int lane = threadIdx.x & 31;
  if (lane < 8) {
    const unsigned int dd = (unsigned int)h.n_cropped << 4;
    uint4* r = reinterpret_cast<uint4*>(flists + octant_record(h, fx, fy, fz, lane) * 8);
    r[0] = make_uint4(code, code == kListExtended ? (unsigned int)xi : dd, code == kListExtended ? (unsigned int)n : dd, dd);
    r[1] = make_uint4(dd, dd, dd, dd);
  }
}

// The points of a set of rows, flattened across a whole thread block (the block-wide sibling of warp_points_of_rows):
// warp 0 fetches the slot ranges of 32 rows and scans their lengths, then all threads take consecutive points of the
// concatenation.  Every thread of the block must call it.
template <typename RowFn, typename PointFn>
// (no __restrict__ on the shared arrays: they carry data between threads across the barriers)
__device__ __forceinline__ void block_points_of_rows(int nrows, int* s_pref /* [34]: [32] = sentinel, [33] = total */, int* s_start, RowFn row_span,
                                                     PointFn fn) {
  const int lane = threadIdx.x & 31;
  for (int rbase = 0; rbase < nrows; rbase += 32) {
    if (threadIdx.x < 32) {
      RowSpan sp{0, 0};
      if (rbase + lane < nrows) sp = row_span(rbase + lane);
      int inc = sp.cnt;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(kFull, inc, o); if (lane >= o) inc += t; }
      s_pref[lane] = inc - sp.cnt;
      s_start[lane] = sp.s0;
      if (lane == 31) s_pref[33] = inc;
    }
    __syncthreads();
    const int total = s_pref[33];
    for (int t = threadIdx.x; t < total; t += blockDim.x) {
      int r = 0;
#pragma unroll
      for (int step = 16; step > 0; step >>= 1) if (s_pref[r + step] <= t) r += step;  // last row whose offset is <= t
      fn(s_start[r] + (t - s_pref[r]));
    }
    __syncthreads();
  }
}

// ascending bitonic sort of m2 (a power of two) 64-bit keys in shared memory by the whole thread block
__device__ __forceinline__ void block_bitonic_sort(unsigned long long* keys, int m2) {
  for (int k = 2; k <= m2; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = threadIdx.x; t < m2; t += blockDim.x) {
        const int u = t ^ j;
        if (u > t) {
          const unsigned long long x = keys[t], y = keys[u];
          if (((t & k) == 0) == (x > y)) { keys[t] = y; keys[u] = x; }
        }
      }
      __syncthreads();
    }
  }
}

// One thread BLOCK builds the list of ONE fine cell straight from the grid (no shared-memory superset): used for the
// cells of blocks whose superset does not fit, i.e. far from the surface, where lists are long (extended lists up to
// kListKX) and a single warp would walk ~1000 points on its own while the rest of the GPU waits.
__device__ __forceinline__ void build_cell_direct(const IndexHeader& h, const int* __restrict__ cs, const float4* __restrict__ pts, int cell,
                                                  float leaf, float margin, float r_max,
                                                  unsigned int* __restrict__ flists, unsigned int* __restrict__ xlists,
                                                  int* __restrict__ list_counters, int* pref, int* start, int* s_cnt, float* s_m2, int* s_ms, int* s_xi,
                                                  unsigned short* s_list /* [kListKX] shared */, float4* s_pt4 /* [kListKX] shared */,
                                                  unsigned long long* s_key /* [kListKX] shared */, unsigned long long* s_key2 /* [kListKX] shared */,
                                                  const unsigned int* __restrict__ needed,
                                                  int2* __restrict__ cell_items, unsigned short* __restrict__ l1_slots, unsigned int* __restrict__ built_bits) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int fdx = h.f_dim[0], fdy = h.f_dim[1];
  const float cell_m = h.cell;
  const int dimx = h.dim[0], dimy = h.dim[1];
  const int fz = cell / (fdx * fdy), r2 = cell - fz * fdx * fdy, fy = r2 / fdx, fx = r2 - fy * fdx;
  // the cell in metric space, widened by the rounding of q * inv_leaf near its faces
  float lo[3], hi[3];
  lo[0] = (float)(h.f_origin[0] + fx) * leaf - margin; hi[0] = (float)(h.f_origin[0] + fx + 1) * leaf + margin;
  lo[1] = (float)(h.f_origin[1] + fy) * leaf - margin; hi[1] = (float)(h.f_origin[1] + fy + 1) * leaf + margin;
  lo[2] = (float)(h.f_origin[2] + fz) * leaf - margin; hi[2] = (float)(h.f_origin[2] + fz + 1) * leaf + margin;
  // coarse cells overlapping the box dilated by r.  floor((p * inv_leaf) * 2^-level) is monotone in p, so every point
  // with lo - r <= p <= hi + r (per axis) lies in cells [c0, c1]: no padding is needed.
  auto coarse_range = [&](int d, float r, int& a, int& b) {
    a = max((int)floorf(((lo[d] - r) * h.inv_leaf) * h.level_scale) - h.origin[d], 0);
    b = min((int)floorf(((hi[d] + r) * h.inv_leaf) * h.level_scale) - h.origin[d], h.dim[d] - 1);
  };
  // (one index per frame: see cand_build_kernel) far from the faces of the crop box the list is built from all points
  // and serves every weight() of the frame; near them it is built from the cropped points, for this weight() only
  const bool dilated = h.dilate > 0.f;
  bool crop_only = false, indep = true;
retry:
  // ---- (1) U: probe the box dilated by a growing radius until it holds a point
  float U2 = 3.0e38f;
  int p0_slot = -1;
  bool no_match = false;
  float pr = fmaxf(2.0f * leaf, 0.5f * cell_m);
  for (int round = 0; round < 8; ++round, pr *= 2.0f) {
    int x0, x1, y0, y1, z0, z1;
    coarse_range(0, pr, x0, x1); coarse_range(1, pr, y0, y1); coarse_range(2, pr, z0, z1);
    float m2 = 3.0e38f;
    int ms = -1;
    if (x0 <= x1 && y0 <= y1 && z0 <= z1) {
      const int ny = y1 - y0 + 1;
      block_points_of_rows(
          ny * (z1 - z0 + 1), pref, start,
          [&](int r) { const int zz = r / ny; const int base = ((z0 + zz) * dimy + (y0 + r - zz * ny)) * dimx; const int a = cs[base + x0]; return RowSpan{a, cs[base + x1 + 1] - a}; },
          [&](int s) { const float4 p = pts[s]; if (crop_only && !in_crop(p, h)) return; const float v = box_maxdist2(lo, hi, p); if (v < m2 || (v == m2 && s > ms)) { m2 = v; ms = s; } });
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float om = __shfl_xor_sync(kFull, m2, o);
        const int os = __shfl_xor_sync(kFull, ms, o);
        if (om < m2 || (om == m2 && os > ms)) { m2 = om; ms = os; }  // any deterministic choice among equals
      }
      if (lane == 0) { s_m2[wid] = m2; s_ms[wid] = ms; }
      __syncthreads();
      m2 = s_m2[0]; ms = s_ms[0];
      for (int w = 1; w < nw; ++w) { const float om = s_m2[w]; const int os = s_ms[w]; if (om < m2 || (om == m2 && os > ms)) { m2 = om; ms = os; } }
      __syncthreads();
    }
    if (m2 < 3.0e38f) { U2 = m2 * 1.00002f; p0_slot = ms; break; }
    if (pr > r_max) { no_match = true; break; }  // nothing within pr (> maximum_distance_) of the box: no query of the cell can match
  }
  if (U2 >= 3.0e38f) {
    // provably no point within maximum_distance_ of any query of the cell (empty lists), or the probe gave up (the
    // queries of this cell are answered by brute force)
    if (threadIdx.x < 32) write_octant_codes(h, flists, fx, fy, fz, no_match ? 0u : kListOverflow, 0, 0);
    if (!crop_only && threadIdx.x == 0) atomicOr(&built_bits[cell >> 5], 1u << (cell & 31));  // (found among all points: holds for every crop box)
    return;
  }
  U2 = fminf(U2, r_max * r_max);
  const float reach = sqrtf(U2) * 1.00001f;
  if (dilated && !crop_only) {
#pragma unroll
    for (int d = 0; d < 3; ++d)
      indep = indep && lo[d] - reach >= h.aabb[d] + h.dilate && hi[d] + reach <= h.aabb[3 + d] - h.dilate;
    if (!indep) { crop_only = true; __syncthreads(); goto retry; }
  }
  // Second, sharper filter: the nearest neighbour p* of a query q of the cell satisfies |q - p*| <= |q - p0| for the
  // reference point p0 found above, i.e. q lies on p*'s side of the bisector plane of (p*, p0) (see can_win).
  float bc[3], bh[3];
#pragma unroll
  for (int d = 0; d < 3; ++d) { bc[d] = 0.5f * (lo[d] + hi[d]); bh[d] = 0.5f * (hi[d] - lo[d]); }
  const float4 p0 = pts[p0_slot];
  // ---- (2) gather: rows of coarse cells that intersect the ball-dilated box
  int c0[3], c1[3];
  coarse_range(1, reach, c0[1], c1[1]); coarse_range(2, reach, c0[2], c1[2]);
  const int ny = c1[1] - c0[1] + 1, nrows = max(ny, 0) * max(c1[2] - c0[2] + 1, 0);
  // one gather into shared memory (up to the capacity of an extended list), then the list goes where its length says
  if (threadIdx.x == 0) *s_cnt = 0;
  __syncthreads();
  block_points_of_rows(
      nrows, pref, start,
      [&](int r) {
        const int zz = r / ny, y = c0[1] + (r - zz * ny), z = c0[2] + zz;
        const float zlo = (float)(z + h.origin[2]) * cell_m - 2.0f * margin, zhi = (float)(z + 1 + h.origin[2]) * cell_m + 2.0f * margin;
        const float gz = fmaxf(fmaxf(lo[2] - zhi, zlo - hi[2]), 0.f);
        const float ylo = (float)(y + h.origin[1]) * cell_m - 2.0f * margin, yhi = (float)(y + 1 + h.origin[1]) * cell_m + 2.0f * margin;
        const float gy = fmaxf(fmaxf(lo[1] - yhi, ylo - hi[1]), 0.f);
        const float rem = U2 - (gy * gy + gz * gz) * 0.9999f;
        if (rem < 0.f) return RowSpan{0, 0};
        const float xr = sqrtf(rem) * 1.00001f + 2.0f * margin;
        const int xa = max((int)floorf(((lo[0] - xr) * h.inv_leaf) * h.level_scale) - h.origin[0], 0);
        const int xb = min((int)floorf(((hi[0] + xr) * h.inv_leaf) * h.level_scale) - h.origin[0], dimx - 1);
        if (xa > xb) return RowSpan{0, 0};
        const int base = (z * dimy + y) * dimx;
        const int a = cs[base + xa];
        return RowSpan{a, cs[base + xb + 1] - a};
      },
      [&](int s) {
        const float4 p = pts[s];
        if (crop_only && !in_crop(p, h)) return;
        if (box_mindist2(lo, hi, p) <= U2 && can_win(p, p0, bc, bh)) {
          const int pos = atomicAdd(s_cnt, 1);
          if (pos < kListKX) s_list[pos] = (unsigned short)s;
        }
      });
  const int n = *s_cnt;
  __syncthreads();  // every thread holds the count before thread 0 reuses the counter for the survivors below (without
                    // this barrier a warp that is scheduled late -- other kernels share the SM when several trackers
                    // run side by side -- read 0 and left the block's barriers out of step: an intermittent fault of
                    // the multi-object batch)
  if (n > kListKX) { if (threadIdx.x < 32) write_octant_codes(h, flists, fx, fy, fz, kListOverflow, 0, 0); return; }
  // ---- (3) pairwise pruning.  Far from the surface the two tests above keep hundreds of points (they only compare
  // with ONE competitor, p0); nearly all of them are beaten everywhere in the cell by some other candidate (a point
  // of the same face that lies nearer to the cell).  Every thread scans the competitors of its candidate and stops at
  // the first that dominates it (domination is transitive: whatever dominated the dominator dominates the candidate
  // too, so testing against every candidate, kept or not, is valid); the survivors are the cell's list.
  const float ch = 0.5f * (hi[0] - lo[0]) + 1.0e-6f;  // half extent of the (cubic) cell box
  // candidates in ascending order of their distance from the cell centre: only a nearer candidate can dominate, and the
  // dominators of a far candidate are found within a few steps, so every scan is short
  int n2 = 1;
  while (n2 < n) n2 <<= 1;
  for (int t = threadIdx.x; t < n2; t += blockDim.x) {
    unsigned long long key = ~0ull;
    if (t < n) {
      const float4 p = pts[s_list[t]];
      const float x = p.x - bc[0], y = p.y - bc[1], z = p.z - bc[2];
      s_pt4[t] = make_float4(x, y, z, p.w);
      key = ((unsigned long long)__float_as_uint((x * x + y * y) + z * z) << 32) | (unsigned long long)t;
    }
    s_key[t] = key;
  }
  if (threadIdx.x == 0) *s_cnt = 0;
  __syncthreads();
  unsigned long long* s_sorted = s_key;   // the keys in ascending order
  unsigned long long* s_out = s_key2;     // the survivors' keys
  if (n <= 512) {
    // rank by counting (the keys are distinct): no barrier per step, cheaper than the bitonic network at these sizes
    for (int t = threadIdx.x; t < n; t += blockDim.x) {
      const unsigned long long my = s_key[t];
      int r = 0;
      for (int k = 0; k < n; ++k) r += s_key[k] < my ? 1 : 0;
      s_key2[r] = my;
    }
    __syncthreads();
    s_sorted = s_key2; s_out = s_key;
  } else {
    block_bitonic_sort(s_key, n2);
  }
  for (int r0 = 0; r0 < n; r0 += blockDim.x) {
    const int r = r0 + threadIdx.x;
    if (r < n) {
      const int t = (int)(s_sorted[r] & 0xffffffffull);
      const float4 p = s_pt4[t];
      const float pn = (p.x * p.x + p.y * p.y) + p.z * p.z;
      bool alive = true;
      for (int k = 0; k < r; ++k) {
        const float4 c = s_pt4[(int)(s_sorted[k] & 0xffffffffull)];
        const float cn = (c.x * c.x + c.y * c.y) + c.z * c.z;
        // min over the cube of |q-p|^2 - |q-c|^2: positive (beyond the rounding slack) = c is nearer everywhere
        const float fmin = (pn - cn) - 2.0f * (ch * ((fabsf(p.x - c.x) + fabsf(p.y - c.y)) + fabsf(p.z - c.z)));
        if (fmin > 1.0e-6f * (pn + cn) + 1.0e-9f) { alive = false; break; }
      }
      // key = input index (upper half: the order of the extended list) | position in s_list
      if (alive) s_out[atomicAdd(s_cnt, 1)] = ((unsigned long long)(unsigned int)__float_as_int(p.w) << 32) | (unsigned long long)t;
    }
  }
  __syncthreads();
  const int m = *s_cnt;
  PFT_STAT(11, threadIdx.x == 0 ? 1 : 0);
  if (indep && threadIdx.x == 0) atomicOr(&built_bits[cell >> 5], 1u << (cell & 31));  // (the next weight() of the frame need not build it again)
  if (m <= kL1Cap) {
    // a normal cell after all: its list goes to cand_octant_kernel like those of cand_build_kernel
    if ((int)threadIdx.x < m) l1_slots[(size_t)cell * kL1Cap + threadIdx.x] = s_list[(int)(s_out[threadIdx.x] & 0xffffffffull)];
    if (threadIdx.x == 0) {
      const int item = cell | (m << 24) | (needed[cell] < kCoarseBelow ? (int)0x80000000 : 0);
      const int xyz = (fx < 1024 && fy < 1024 && fz < 1024) ? (fx | (fy << 10) | (fz << 20) | (needed[cell] < kLightBelow ? (1 << 30) : 0)) : -1;
      cell_items[atomicAdd(&list_counters[4], 1)] = make_int2(item, xyz);
    }
    return;
  }
  // still long: an extended list in ascending order of the input index, scanned entry by entry by the queries of the cell
  int m2 = 1;
  while (m2 < m) m2 <<= 1;
  for (int t = m + threadIdx.x; t < m2; t += blockDim.x) s_out[t] = ~0ull;
  __syncthreads();
  block_bitonic_sort(s_out, m2);
  s_key = s_out;
  if (threadIdx.x == 0) *s_xi = atomicAdd(&list_counters[0], 1);
  __syncthreads();
  const int xi = *s_xi;
  if (xi >= kListXCells) { if (threadIdx.x < 32) write_octant_codes(h, flists, fx, fy, fz, kListOverflow, 0, 0); return; }
  unsigned int* dst = xlists + (size_t)xi * kListKX;
  const unsigned int dummy = (unsigned int)h.n_cropped << 4;
  const int m4 = (m + 3) & ~3;  // the lookup reads four entries at a time
  for (int t = threadIdx.x; t < m4; t += blockDim.x) dst[t] = t < m ? ((unsigned int)s_list[(int)(s_key[t] & 0xffffffffull)] << 4) : dummy;
  if (threadIdx.x < 32) write_octant_codes(h, flists, fx, fy, fz, kListExtended, xi, m);
  PFT_STAT(15, threadIdx.x == 0 ? 1 : 0);
}

// One warp builds the lists of one block of 2x2x2 fine cells: the points that can be the nearest neighbour of some
// query of the BLOCK are gathered once into shared memory (a superset of every cell's list), then each needed cell
// of the block filters that superset with its own bound and bisector test.
__global__ void __launch_bounds__(256) cand_build_kernel(const IndexHeader* __restrict__ hdr, const int* __restrict__ cs,
                                                         const float4* __restrict__ pts, double max_d2,
                                                         unsigned int* __restrict__ flists,
                                                         const unsigned int* __restrict__ needed, const int* __restrict__ needed_list,
                                                         int* __restrict__ list_counters,
                                                         int* __restrict__ far_list, int2* __restrict__ cell_items,
                                                         unsigned short* __restrict__ l1_slots, unsigned int* __restrict__ built_bits) {
  __shared__ IndexHeader h;
  __shared__ int s_cnt[8];
  __shared__ int s_pref[8][33], s_start[8][32];
  __shared__ float4 s_pt[8][kSuperCap];
  __shared__ unsigned short s_slot[8][kSuperCap];
  if (threadIdx.x == 0) h = *hdr;
  __syncthreads();
  if (!h.valid || !lists_on(h)) return;
  const int n_needed = list_counters[1];
  const float leaf = 1.0f / h.inv_leaf;
  const float margin = 1.0e-5f + 4.0e-6f * leaf * (float)(abs(h.f_origin[0]) + abs(h.f_origin[1]) + abs(h.f_origin[2]) + h.f_dim[0] + h.f_dim[1] + h.f_dim[2]);
  const float r_max = max_d2 >= 1.0e30 ? 1.0e15f : (float)sqrt(max_d2) * 1.00001f;
  const int fdx = h.f_dim[0], fdy = h.f_dim[1], fdz = h.f_dim[2];
  const int bdx = (fdx + 1) >> 1, bdy = (fdy + 1) >> 1;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  const float cell_m = h.cell;
  const int dimx = h.dim[0], dimy = h.dim[1];
  int* pref = s_pref[wib];
  int* start = s_start[wib];
  float4* spt = s_pt[wib];
  unsigned short* sslot = s_slot[wib];
  if (lane == 0) pref[32] = 0x7fffffff;  // sentinel for the binary search
  for (int idx = warp; idx < n_needed; idx += nwarps) {
    const int blk = needed_list[idx];
    const int bz = blk / (bdx * bdy), br = blk - bz * bdx * bdy, by = br / bdx, bx = br - by * bdx;
    // the block (2x2x2 fine cells) in metric space, widened by the rounding of q * inv_leaf near its faces
    float lo[3], hi[3];
    lo[0] = (float)(h.f_origin[0] + 2 * bx) * leaf - margin; hi[0] = (float)(h.f_origin[0] + 2 * bx + 2) * leaf + margin;
    lo[1] = (float)(h.f_origin[1] + 2 * by) * leaf - margin; hi[1] = (float)(h.f_origin[1] + 2 * by + 2) * leaf + margin;
    lo[2] = (float)(h.f_origin[2] + 2 * bz) * leaf - margin; hi[2] = (float)(h.f_origin[2] + 2 * bz + 2) * leaf + margin;
    // every fine cell of the block gets `value` (used when the whole block is decided at once)
    auto set_all = [&](unsigned int value, bool reusable) {
      for (int sub = 0; sub < 8; ++sub) {
        const int fx = 2 * bx + (sub & 1), fy = 2 * by + ((sub >> 1) & 1), fz = 2 * bz + (sub >> 2);
        if (fx < fdx && fy < fdy && fz < fdz) {
          const int c = (fz * fdy + fy) * fdx + fx;
          // every octant: header + dummy slots (value 0 = empty list: nothing within maximum_distance_)
          if (needed[c]) {
            write_octant_codes(h, flists, fx, fy, fz, value, 0, 0);
            if (reusable && lane == 0) atomicOr(&built_bits[c >> 5], 1u << (c & 31));
          }
        }
      }
    };
    // coarse cells overlapping the box dilated by r.  floor((p * inv_leaf) * 2^-level) is monotone in p, so every point
    // with lo - r <= p <= hi + r (per axis) lies in cells [c0, c1]: no padding is needed.
    auto coarse_range = [&](int d, float r, int& a, int& b) {
      a = max((int)floorf(((lo[d] - r) * h.inv_leaf) * h.level_scale) - h.origin[d], 0);
      b = min((int)floorf(((hi[d] + r) * h.inv_leaf) * h.level_scale) - h.origin[d], h.dim[d] - 1);
    };
    // One index per frame (IndexHeader::built): when the index holds more than the crop box, a block whose lists cannot
    // depend on where the faces of the crop box are -- every point that matters lies well inside it -- is built from all
    // points and marked as built for the later weight() calls of the frame; a block near the faces is built from the
    // cropped points only (exact for THIS weight(), rebuilt by the next).
    const bool dilated = h.dilate > 0.f;
    bool crop_only = false, indep = true;
  retry:
    // ---- (1) U_B = min over points of maxdist(block, p): probe the block dilated by a growing radius until it holds a point
    float U2 = 3.0e38f;
    int p0_slot = -1;
    bool no_match = false;
    float pr = fmaxf(2.0f * leaf, 0.5f * cell_m);
    for (int round = 0; round < 8; ++round, pr *= 2.0f) {
      int x0, x1, y0, y1, z0, z1;
      coarse_range(0, pr, x0, x1); coarse_range(1, pr, y0, y1); coarse_range(2, pr, z0, z1);
      float m2 = 3.0e38f;
      int ms = -1;
      if (x0 <= x1 && y0 <= y1 && z0 <= z1) {
        const int ny = y1 - y0 + 1;
        warp_points_of_rows(
            ny * (z1 - z0 + 1), pref, start,
            [&](int r) { const int zz = r / ny; const int base = ((z0 + zz) * dimy + (y0 + r - zz * ny)) * dimx; const int a = cs[base + x0]; return RowSpan{a, cs[base + x1 + 1] - a}; },
            [&](int s) { const float4 p = pts[s]; if (crop_only && !in_crop(p, h)) return; const float v = box_maxdist2(lo, hi, p); if (v < m2) { m2 = v; ms = s; } });
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const float om = __shfl_xor_sync(kFull, m2, o);
          const int os = __shfl_xor_sync(kFull, ms, o);
          if (om < m2 || (om == m2 && os > ms)) { m2 = om; ms = os; }  // any deterministic choice among equals
        }
      }
      if (m2 < 3.0e38f) { U2 = m2 * 1.00002f; p0_slot = ms; break; }
      if (pr > r_max) { no_match = true; break; }  // nothing within pr (> maximum_distance_) of the block: none of its queries can match
    }
    if (U2 >= 3.0e38f) {
      // provably no point within maximum_distance_ of any query of the block (empty lists), or the probe gave up
      // (the queries of the block are answered by brute force).  Found among ALL points, it holds for every crop box.
      set_all(no_match ? 0u : kListOverflow, !crop_only);
      continue;
    }
    U2 = fminf(U2, r_max * r_max);
    const float reach = sqrtf(U2) * 1.00001f;
    if (dilated && !crop_only) {
      // every point the lists of this block can depend on lies within `reach` of it: inside the crop box shrunk by the
      // dilation margin on every side, they are the same whatever the next crop box of the frame is
#pragma unroll
      for (int d = 0; d < 3; ++d)
        indep = indep && lo[d] - reach >= h.aabb[d] + h.dilate && hi[d] + reach <= h.aabb[3 + d] - h.dilate;
      if (!indep) { crop_only = true; goto retry; }
    }
    float bc[3], bh[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) { bc[d] = 0.5f * (lo[d] + hi[d]); bh[d] = 0.5f * (hi[d] - lo[d]); }
    const float4 p0 = pts[p0_slot];
    // ---- (2) superset of the block: { p : mindist(block, p) <= U_B and p can beat p0 somewhere in the block }
    int c0[3], c1[3];
    coarse_range(1, reach, c0[1], c1[1]); coarse_range(2, reach, c0[2], c1[2]);
    const int ny = c1[1] - c0[1] + 1, nrows = max(ny, 0) * max(c1[2] - c0[2] + 1, 0);
    if (lane == 0) s_cnt[wib] = 0;
    __syncwarp();
    warp_points_of_rows(
        nrows, pref, start,
        [&](int r) {
          const int zz = r / ny, y = c0[1] + (r - zz * ny), z = c0[2] + zz;
          const float zlo = (float)(z + h.origin[2]) * cell_m - 2.0f * margin, zhi = (float)(z + 1 + h.origin[2]) * cell_m + 2.0f * margin;
          const float gz = fmaxf(fmaxf(lo[2] - zhi, zlo - hi[2]), 0.f);
          const float ylo = (float)(y + h.origin[1]) * cell_m - 2.0f * margin, yhi = (float)(y + 1 + h.origin[1]) * cell_m + 2.0f * margin;
          const float gy = fmaxf(fmaxf(lo[1] - yhi, ylo - hi[1]), 0.f);
          const float rem = U2 - (gy * gy + gz * gz) * 0.9999f;
          if (rem < 0.f) return RowSpan{0, 0};
          const float xr = sqrtf(rem) * 1.00001f + 2.0f * margin;
          const int xa = max((int)floorf(((lo[0] - xr) * h.inv_leaf) * h.level_scale) - h.origin[0], 0);
          const int xb = min((int)floorf(((hi[0] + xr) * h.inv_leaf) * h.level_scale) - h.origin[0], dimx - 1);
          if (xa > xb) return RowSpan{0, 0};
          const int base = (z * dimy + y) * dimx;
          const int a = cs[base + xa];
          return RowSpan{a, cs[base + xb + 1] - a};
        },
        [&](int s) {
          const float4 p = pts[s];
          if (crop_only && !in_crop(p, h)) return;
          if (box_mindist2(lo, hi, p) <= U2 && can_win(p, p0, bc, bh)) {
            const int pos = atomicAdd(&s_cnt[wib], 1);
            if (pos < kSuperCap) { spt[pos] = p; sslot[pos] = (unsigned short)s; }
          }
        });
    __syncwarp();
    const int ns = s_cnt[wib];
    __syncwarp();
    if (ns > kSuperCap) {
      // far from the surface: long lists.  Their cells are queued for cand_build_far_kernel (one warp per cell, straight
      // from the grid) instead of being built one after the other by this warp.
      if (lane < 8) {
        const int fx = 2 * bx + (lane & 1), fy = 2 * by + ((lane >> 1) & 1), fz = 2 * bz + (lane >> 2);
        if (fx < fdx && fy < fdy && fz < fdz) {
          const int c = (fz * fdy + fy) * fdx + fx;
          if (needed[c]) { far_list[atomicAdd(&list_counters[2], 1)] = c; PFT_STAT(10, 1); }
        }
      }
      continue;
    }
    // ---- (3) each needed fine cell filters the superset with its own bound and bisector test
    unsigned int sub_mask;  // which of the block's 8 cells are needed: one load per lane instead of eight serial ones
    {
      bool mine = false;
      if (lane < 8) {
        const int fx = 2 * bx + (lane & 1), fy = 2 * by + ((lane >> 1) & 1), fz = 2 * bz + (lane >> 2);
        mine = fx < fdx && fy < fdy && fz < fdz && needed[(fz * fdy + fy) * fdx + fx] != 0u;
      }
      sub_mask = __ballot_sync(kFull, mine);
    }
    int my_item = 0, my_xyz = 0;  // lane `sub` remembers the cell it has to queue
    bool my_valid = false;
    for (int sub = 0; sub < 8; ++sub) {
      if (!((sub_mask >> sub) & 1u)) continue;
      const int fx = 2 * bx + (sub & 1), fy = 2 * by + ((sub >> 1) & 1), fz = 2 * bz + (sub >> 2);
      const int cell = (fz * fdy + fy) * fdx + fx;
      float flo[3], fhi[3], fc[3], fh[3];
      flo[0] = (float)(h.f_origin[0] + fx) * leaf - margin; fhi[0] = (float)(h.f_origin[0] + fx + 1) * leaf + margin;
      flo[1] = (float)(h.f_origin[1] + fy) * leaf - margin; fhi[1] = (float)(h.f_origin[1] + fy + 1) * leaf + margin;
      flo[2] = (float)(h.f_origin[2] + fz) * leaf - margin; fhi[2] = (float)(h.f_origin[2] + fz + 1) * leaf + margin;
#pragma unroll
      for (int d = 0; d < 3; ++d) { fc[d] = 0.5f * (flo[d] + fhi[d]); fh[d] = 0.5f * (fhi[d] - flo[d]); }
      // U_f and its reference point: the minimiser of maxdist(cell, .) over all points lies in the superset
      float m2 = 3.0e38f;
      int mi = -1;
      for (int t = lane; t < ns; t += 32) { const float v = box_maxdist2(flo, fhi, spt[t]); if (v < m2) { m2 = v; mi = t; } }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float om = __shfl_xor_sync(kFull, m2, o);
        const int oi = __shfl_xor_sync(kFull, mi, o);
        if (om < m2 || (om == m2 && oi > mi)) { m2 = om; mi = oi; }
      }
      const float Uf2 = fminf(m2 * 1.00002f, r_max * r_max);
      const float4 pf = spt[mi];
      // the cell's own list L1 (every point that can be the nearest neighbour of some query of the 1 cm cell): the keep
      // test is evaluated once; its ballots (ns <= kSuperCap = 8 x 32) give the compaction offsets
      int n = 0;
      unsigned int keep_bal[kSuperCap / 32];
#pragma unroll
      for (int q = 0; q < kSuperCap / 32; ++q) {
        keep_bal[q] = 0u;
        if (q * 32 < ns) {
          const int t = q * 32 + lane;
          const bool keep = t < ns && box_mindist2(flo, fhi, spt[t]) <= Uf2 && can_win(spt[t], pf, fc, fh);
          keep_bal[q] = __ballot_sync(kFull, keep);
          n += __popc(keep_bal[q]);
        }
      }
      if (n > kL1Cap) {
        // long list (far from the surface): the far pass prunes it pairwise
        if (lane == 0) { far_list[atomicAdd(&list_counters[2], 1)] = cell; PFT_STAT(10, 1); }
        continue;
      }
      // ---- (4) hand the cell's list to cand_octant_kernel (slots in superset order; the octant pass sorts them)
      {
        unsigned short* dst = l1_slots + (size_t)cell * kL1Cap;
        int w = 0;
#pragma unroll
        for (int q = 0; q < kSuperCap / 32; ++q) {
          if (q * 32 < ns) {
            const unsigned int bal = keep_bal[q];
            if ((bal >> lane) & 1u) dst[w + __popc(bal & ((1u << lane) - 1u))] = sslot[q * 32 + lane];
            w += __popc(bal);
          }
        }
      }
      if (lane == sub) {
        // item = cell | list length << 24 | (few queries: one list for the whole cell) << 31, and the cell's coordinates
        my_item = cell | (n << 24) | (needed[cell] < kCoarseBelow ? (int)0x80000000 : 0);
        my_xyz = (fx < 1024 && fy < 1024 && fz < 1024) ? (fx | (fy << 10) | (fz << 20) | (needed[cell] < kLightBelow ? (1 << 30) : 0)) : -1;
        my_valid = true;
        if (indep) atomicOr(&built_bits[cell >> 5], 1u << (cell & 31));  // (the next weight() of the frame need not build it again)
      }
      PFT_STAT(15, lane == 0 ? 1 : 0);
    }
    // queue the cells of this block: one atomic per block
    {
      const unsigned int bal = __ballot_sync(kFull, my_valid);
      if (bal) {
        int base = 0;
        if (lane == 0) base = atomicAdd(&list_counters[4], __popc(bal));
        base = __shfl_sync(kFull, base, 0);
        if (my_valid) cell_items[base + __popc(bal & ((1u << lane) - 1u))] = make_int2(my_item, my_xyz);
      }
    }
  }
}

// Third pass of the build: the records of every cell queued by cand_build_kernel, one warp per cell.
// The cell's list is sorted by input index (the lookup resolves distance ties by position: the first of equals wins).
// Cells with few queries (`coarse`) get that list in each of their eight octant records.  Otherwise G lanes work on one
// octant (G = the power of two >= list length, 32 / G octants per pass; lane % G = entry): p0 = the entry minimising
// maxdist(octant, .), keep = mindist <= U and can-win against p0 (both from the entry's offset to the octant centre:
// the octant is a cube); when an octant keeps more than seven, every octant of the pass is pruned pairwise (an entry
// that another kept entry beats everywhere in the octant never wins); ballot compaction keeps the order.  Entries
// beyond the seventh go to groups of eight taken from a pool (the header carries the first group).  The eight records
// are assembled in shared memory and written out together.
__global__ void __launch_bounds__(256) cand_octant_kernel(const IndexHeader* __restrict__ hdr, const float4* __restrict__ pts, double max_d2,
                                                          unsigned int* __restrict__ flists, unsigned int* __restrict__ pool,
                                                          int* __restrict__ list_counters, const int2* __restrict__ cell_items,
                                                          const unsigned short* __restrict__ l1_slots) {
  __shared__ IndexHeader h;
  __shared__ float4 s_pt[8][kL1Cap];
  __shared__ unsigned int s_off[8][kL1Cap];
  __shared__ __align__(16) unsigned int s_rec[8][64];
  if (threadIdx.x == 0) h = *hdr;
  __syncthreads();
  if (!h.valid || !lists_on(h)) return;
  const int n_items = list_counters[4];
  const float leaf = 1.0f / h.inv_leaf;
  const float margin = 1.0e-5f + 4.0e-6f * leaf * (float)(abs(h.f_origin[0]) + abs(h.f_origin[1]) + abs(h.f_origin[2]) + h.f_dim[0] + h.f_dim[1] + h.f_dim[2]);
  const float r_max = max_d2 >= 1.0e30 ? 1.0e15f : (float)sqrt(max_d2) * 1.00001f;
  const float rmax2 = r_max * r_max;
  const float quarter = 0.25f * leaf;
  // half extent of an octant box: the octant itself, the rounding of q * inv_leaf near its faces (margin) and of the
  // centre computed below
  const float oh = quarter + margin + 1.0e-6f;
  const int fdx = h.f_dim[0], fdy = h.f_dim[1];
  const unsigned int d2x = 2u * (unsigned int)h.f_dim[0], d2y = 2u * (unsigned int)h.f_dim[1];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  const unsigned int lt = (1u << lane) - 1u;
  const unsigned int dummy = (unsigned int)h.n_cropped << 4;
  float4* spt = s_pt[wib];
  unsigned int* soff = s_off[wib];
  unsigned int* srec = s_rec[wib];
  // can p (offset x, y, z from the octant centre) be at least as near as the competitor (offset cx, cy, cz) somewhere in
  // the octant?  min over the cube of |q-p|^2 - |q-c|^2 = (|p|^2 - |c|^2) - 2 oh (|px-cx| + |py-cy| + |pz-cz|)
  auto can_win_c = [&](float x, float y, float z, float cx, float cy, float cz) {
    const float pn = (x * x + y * y) + z * z, cn = (cx * cx + cy * cy) + cz * cz;
    const float fmin = (pn - cn) - 2.0f * (oh * ((fabsf(x - cx) + fabsf(y - cy)) + fabsf(z - cz)));
    return fmin <= 1.0e-6f * (pn + cn) + 1.0e-9f;
  };
  auto maxd2 = [&](float x, float y, float z) { const float u = fabsf(x) + oh, v = fabsf(y) + oh, w = fabsf(z) + oh; return (u * u + v * v) + w * w; };
  auto mind2 = [&](float x, float y, float z) {
    const float u = fmaxf(fabsf(x) - oh, 0.f), v = fmaxf(fabsf(y) - oh, 0.f), w = fmaxf(fabsf(z) - oh, 0.f);
    return (u * u + v * v) + w * w;
  };
  for (int it = warp; it < n_items; it += nwarps) {
    const int2 item = cell_items[it];
    const int cell = item.x & 0xffffff;
    int n = (item.x >> 24) & 0x7f;
    const bool coarse = item.x < 0;
    int fx, fy, fz;
    const bool light = item.y >= 0 && ((item.y >> 30) & 1);
    if (item.y >= 0) { fx = item.y & 1023; fy = (item.y >> 10) & 1023; fz = (item.y >> 20) & 1023; }
    else { fz = cell / (fdx * fdy); const int r2 = cell - fz * fdx * fdy; fy = r2 / fdx; fx = r2 - fy * fdx; }
    bool two = n > 32;
    // ---- the list in ascending order of the input index (rank = how many keys are smaller; keys are distinct)
    {
      const unsigned short* src = l1_slots + (size_t)cell * kL1Cap;
      const int s0 = lane < n ? (int)src[lane] : 0;
      const float4 p0 = pts[s0];
      const int k0 = lane < n ? __float_as_int(p0.w) : 0x7fffffff;
      int r0 = 0;
      if (!two) {
        for (int c = 0; c < n; ++c) r0 += __shfl_sync(kFull, k0, c) < k0 ? 1 : 0;
      } else {
        const int s1 = lane + 32 < n ? (int)src[lane + 32] : 0;
        const float4 p1 = pts[s1];
        const int k1 = lane + 32 < n ? __float_as_int(p1.w) : 0x7fffffff;
        int r1 = 0;
        for (int c = 0; c < 32; ++c) { const int k = __shfl_sync(kFull, k0, c); r0 += k < k0 ? 1 : 0; r1 += k < k1 ? 1 : 0; }
        for (int c = 32; c < n; ++c) { const int k = __shfl_sync(kFull, k1, c - 32); r0 += k < k0 ? 1 : 0; r1 += k < k1 ? 1 : 0; }
        if (lane + 32 < n) { spt[r1] = p1; soff[r1] = (unsigned int)s1 << 4; }
      }
      if (lane < n) { spt[r0] = p0; soff[r0] = (unsigned int)s0 << 4; }
    }
    srec[lane] = dummy; srec[lane + 32] = dummy;
    __syncwarp();
    // ---- lists longer than one record: pairwise pruning at the cell level first -- an entry that another entry beats
    // everywhere in the cell never wins (domination is transitive, so testing against every entry, kept or not, is
    // valid); typically 10 entries become 6-7
    if (n > 7) {
      const float chh = 0.5f * leaf + margin + 1.0e-6f;
      const float ccx = (float)(2 * (h.f_origin[0] + fx) + 1) * (0.5f * leaf), ccy = (float)(2 * (h.f_origin[1] + fy) + 1) * (0.5f * leaf),
                  ccz = (float)(2 * (h.f_origin[2] + fz) + 1) * (0.5f * leaf);
      const bool ia = lane < n, ib = two && lane + 32 < n;
      const float4 ea = spt[ia ? lane : 0], eb = spt[ib ? lane + 32 : 0];
      const unsigned int oa = soff[ia ? lane : 0], ob = soff[ib ? lane + 32 : 0];
      const float ax = ea.x - ccx, ay = ea.y - ccy, az = ea.z - ccz, bx = eb.x - ccx, by = eb.y - ccy, bz = eb.z - ccz;
      const float an = (ax * ax + ay * ay) + az * az, bn = (bx * bx + by * by) + bz * bz;
      bool la = ia, lb = ib;
      for (int c = 0; c < n; ++c) {
        const float4 pc = spt[c];
        const float cx = pc.x - ccx, cy = pc.y - ccy, cz = pc.z - ccz;
        const float cn = (cx * cx + cy * cy) + cz * cz;
        // min over the cube of |q-p|^2 - |q-c|^2: positive (beyond the rounding slack) = c is nearer everywhere
        if ((an - cn) - 2.0f * (chh * ((fabsf(ax - cx) + fabsf(ay - cy)) + fabsf(az - cz))) > 1.0e-6f * (an + cn) + 1.0e-9f) la = false;
        if (two && (bn - cn) - 2.0f * (chh * ((fabsf(bx - cx) + fabsf(by - cy)) + fabsf(bz - cz))) > 1.0e-6f * (bn + cn) + 1.0e-9f) lb = false;
      }
      const unsigned int ka = __ballot_sync(kFull, la), kb = __ballot_sync(kFull, lb);
      __syncwarp();
      if (la) { const int pos = __popc(ka & lt); spt[pos] = ea; soff[pos] = oa; }
      if (lb) { const int pos = __popc(ka) + __popc(kb & lt); spt[pos] = eb; soff[pos] = ob; }
      n = __popc(ka) + __popc(kb);
      two = n > 32;
      __syncwarp();
    }
    // records of octant o: word index of its first word (the octants form one dense lattice, x fastest)
    auto rec_word = [&](int o) { return (((unsigned int)(2 * fz + (o >> 2)) * d2y + (unsigned int)(2 * fy + ((o >> 1) & 1))) * d2x + (unsigned int)(2 * fx + (o & 1))) * 8u; };
    if (coarse || (light && n <= 7)) {
      // the cell's own list in every octant record: the cell has few queries (entries beyond the seventh in ONE run of pool
      // groups), or not many and the list fits one record anyway (a lookup evaluates seven slots whatever the length;
      // busy cells are still split: shorter lists mean fewer shared-memory wavefronts per lookup)
      unsigned int hw = (unsigned int)n;
      int pg = 0;
      if (n > 7) {
        const int need = (n - 7 + 7) >> 3;
        if (lane == 0) pg = atomicAdd(&list_counters[3], need);
        pg = __shfl_sync(kFull, pg, 0);
        if (pg + need > kPoolGroups) hw = kListOverflow;
        else {
          hw |= (unsigned int)pg << 8;
          for (int t = 7 + lane; t < 7 + need * 8; t += 32) pool[(size_t)pg * 8 + (size_t)(t - 7)] = t < n ? soff[t] : dummy;
        }
      }
      // lane l: word (l & 7) of octants (l >> 3) and 4 + (l >> 3)
      const int w = lane & 7;
      const unsigned int val = w == 0 ? hw : ((hw != kListOverflow && w - 1 < n) ? soff[w - 1] : dummy);
      flists[rec_word(lane >> 3) + (unsigned int)w] = val;
      flists[rec_word(4 + (lane >> 3)) + (unsigned int)w] = val;
      __syncwarp();
      continue;
    }
    // ---- octants: G lanes each
    const int G = n > 16 ? 32 : (n > 8 ? 16 : (n > 4 ? 8 : 4));
    const int P = 32 / G;
    const int e = lane & (G - 1), gbase = lane & ~(G - 1), sub = lane / G;
    const unsigned int gmask = G == 32 ? kFull : (((1u << G) - 1u) << gbase);
    const bool va = e < n, vb = two && e + 32 < n;
    const float4 far_pt = make_float4(3.0e38f, 3.0e38f, 3.0e38f, 0.f);
    const float4 pa = va ? spt[e] : far_pt, pb = vb ? spt[e + 32] : far_pt;
    const unsigned int sa = soff[va ? e : 0], sb = soff[vb ? e + 32 : 0];
    const int cx4 = 4 * (h.f_origin[0] + fx) + 1, cy4 = 4 * (h.f_origin[1] + fy) + 1, cz4 = 4 * (h.f_origin[2] + fz) + 1;
#pragma unroll 1
    for (int ps = 0; ps < 8 / P; ++ps) {
      const int o = ps * P + sub;
      const float ocx = (float)(cx4 + 2 * (o & 1)) * quarter, ocy = (float)(cy4 + 2 * ((o >> 1) & 1)) * quarter, ocz = (float)(cz4 + 2 * (o >> 2)) * quarter;
      const float ax = pa.x - ocx, ay = pa.y - ocy, az = pa.z - ocz;
      const float bx = pb.x - ocx, by = pb.y - ocy, bz = pb.z - ocz;
      // (non-negative floats order like their bit patterns) minimum over the group: xor butterfly
      const unsigned int mda = va ? __float_as_uint(maxd2(ax, ay, az)) : 0x7f7fffffu;
      const unsigned int mdb = vb ? __float_as_uint(maxd2(bx, by, bz)) : 0x7f7fffffu;
      unsigned int mb = min(mda, mdb);
      for (int x = G >> 1; x > 0; x >>= 1) mb = min(mb, __shfl_xor_sync(kFull, mb, x));
      const unsigned int who_a = __ballot_sync(kFull, mda == mb) & gmask, who_b = __ballot_sync(kFull, mdb == mb) & gmask;
      // p0 relative to the octant centre
      const int src = who_a ? __ffs(who_a) - 1 : __ffs(who_b) - 1;
      const float qx = __shfl_sync(kFull, who_a ? ax : bx, src), qy = __shfl_sync(kFull, who_a ? ay : by, src), qz = __shfl_sync(kFull, who_a ? az : bz, src);
      const float U2 = fminf(__uint_as_float(mb) * 1.00002f, rmax2);
      bool ka = va && mind2(ax, ay, az) <= U2 && can_win_c(ax, ay, az, qx, qy, qz);
      bool kb = vb && mind2(bx, by, bz) <= U2 && can_win_c(bx, by, bz, qx, qy, qz);
      unsigned int ba = __ballot_sync(kFull, ka) & gmask, bb = two ? (__ballot_sync(kFull, kb) & gmask) : 0u;
      int cnt = __popc(ba) + __popc(bb);
      if (__any_sync(kFull, cnt > 7)) {
        // pairwise pruning against every entry the p0 tests kept (valid for every octant: it only shortens lists)
        for (int c = 0; c < G; ++c) {
          const float cx = __shfl_sync(kFull, ax, gbase + c), cy = __shfl_sync(kFull, ay, gbase + c), cz = __shfl_sync(kFull, az, gbase + c);
          if ((ba >> (gbase + c)) & 1u) {
            if (ka && !can_win_c(ax, ay, az, cx, cy, cz)) ka = false;
            if (kb && !can_win_c(bx, by, bz, cx, cy, cz)) kb = false;
          }
          if (two) {
            const float dx = __shfl_sync(kFull, bx, c), dy = __shfl_sync(kFull, by, c), dz = __shfl_sync(kFull, bz, c);
            if ((bb >> c) & 1u) {
              if (ka && !can_win_c(ax, ay, az, dx, dy, dz)) ka = false;
              if (kb && !can_win_c(bx, by, bz, dx, dy, dz)) kb = false;
            }
          }
        }
        ba = __ballot_sync(kFull, ka) & gmask;
        bb = two ? (__ballot_sync(kFull, kb) & gmask) : 0u;
        cnt = __popc(ba) + __popc(bb);
      }
      PFT_STAT(0, e == 0 && cnt > 7 ? 1 : 0); PFT_STAT(1, e == 0 ? cnt : 0); PFT_STAT(2, e == 0 ? 1 : 0);
      unsigned int hw = (unsigned int)cnt;
      int pg = 0;
      if (cnt > 7) {  // (uniform within the group)
        const int need = (cnt - 7 + 7) >> 3;
        if (e == 0) pg = atomicAdd(&list_counters[3], need);
        pg = __shfl_sync(gmask, pg, gbase);
        if (pg + need > kPoolGroups) hw = kListOverflow;
        else {
          hw |= (unsigned int)pg << 8;
          // pad the last group with the dummy slot (the lookup reads whole groups)
          const int tail = need * 8 - (cnt - 7);
          if (e < tail) pool[(size_t)pg * 8 + (size_t)(cnt - 7 + e)] = dummy;
        }
      }
      if (hw != kListOverflow) {
        if (ka) { const int pos = __popc(ba & lt); if (pos < 7) srec[o * 8 + 1 + pos] = sa; else pool[(size_t)pg * 8 + (size_t)(pos - 7)] = sa; }
        if (kb) { const int pos = __popc(ba) + __popc(bb & lt); if (pos < 7) srec[o * 8 + 1 + pos] = sb; else pool[(size_t)pg * 8 + (size_t)(pos - 7)] = sb; }
      }
      if (e == 0) srec[o * 8] = hw;
    }
    __syncwarp();
    // lane l: word (l & 7) of octant (l >> 3), then of octant 4 + (l >> 3)
    flists[rec_word(lane >> 3) + (unsigned int)(lane & 7)] = srec[lane];
    flists[rec_word(4 + (lane >> 3)) + (unsigned int)(lane & 7)] = srec[lane + 32];
    __syncwarp();
  }
  PFT_TRACE_MAX(1);
}

// second pass of the build: the cells queued by cand_build_kernel, one thread block each
__global__ void __launch_bounds__(256) cand_build_far_kernel(const IndexHeader* __restrict__ hdr, const int* __restrict__ cs,
                                                             const float4* __restrict__ pts, double max_d2,
                                                             unsigned int* __restrict__ flists, unsigned int* __restrict__ xlists,
                                                             int* __restrict__ list_counters, const int* __restrict__ far_list,
                                                             const unsigned int* __restrict__ needed, int2* __restrict__ cell_items,
                                                             unsigned short* __restrict__ l1_slots, unsigned int* __restrict__ built_bits) {
  __shared__ IndexHeader h;
  __shared__ int s_cnt, s_xi;
  __shared__ int s_pref[34], s_start[32], s_ms[8];
  __shared__ float s_m2[8];
  __shared__ unsigned short s_list[kListKX];
  __shared__ float4 s_pt4[kListKX];
  __shared__ unsigned long long s_key[kListKX], s_key2[kListKX];
  if (threadIdx.x == 0) { h = *hdr; s_pref[32] = 0x7fffffff; }
  __syncthreads();
  if (!h.valid || !lists_on(h)) return;
  const int n_far = list_counters[2];
  const float leaf = 1.0f / h.inv_leaf;
  const float margin = 1.0e-5f + 4.0e-6f * leaf * (float)(abs(h.f_origin[0]) + abs(h.f_origin[1]) + abs(h.f_origin[2]) + h.f_dim[0] + h.f_dim[1] + h.f_dim[2]);
  const float r_max = max_d2 >= 1.0e30 ? 1.0e15f : (float)sqrt(max_d2) * 1.00001f;
  for (int idx = blockIdx.x; idx < n_far; idx += gridDim.x) {
    build_cell_direct(h, cs, pts, far_list[idx], leaf, margin, r_max, flists, xlists, list_counters, s_pref, s_start, &s_cnt, s_m2, s_ms, &s_xi, s_list, s_pt4, s_key, s_key2,
                      needed, cell_items, l1_slots, built_bits);
    __syncthreads();
  }
  PFT_TRACE_MAX(2);
}

struct WeightArgs {
  TrackerState* st;
  const IndexHeader* hdr;
  const int* cell_start;      // [n_cells + 1]
  const float4* pts;          // {x, y, z, input index} in cell order
  const float4* pts2;         // {x, y, z, packed HSV} in cell order (what weight_lists_kernel stages)
  const unsigned int* hsv;    // packed HSV of every slot
  const RowEntry* table;      // kRows entries sorted by lb2
  const unsigned int* flists;    // candidate lists (see cand_build_kernel): one record of 8 words per octant of the fine lattice
  const unsigned int* pool;      // groups of eight entries for octant lists longer than seven
  const unsigned int* xlists;    // extended lists (byte offsets, ascending input index, padded to a multiple of four)
  const float4* model;        // {x,y,z,hsv} in tile order
  const int* model_perm;      // tile order -> order of the reference cloud as given
  int M;
  const float* mats;
  double* partial;            // [chunks][n_max]
  int chunks, chunk_len, n_max;
  int nranks, rank_id;        // particle i is evaluated by rank i % nranks
  CoherenceParams co;
  int dbg_k; int* dbg_idx; float* dbg_d2;
  int smem_bytes;             // dynamic shared memory available for staging the index
};

// One (particle, model chunk) item by one warp: transform, nearest neighbour, coherence, warp reduction.
template <bool USE_HSV, bool DYN, typename CS>
__device__ __forceinline__ void weight_items(const WeightArgs& a, const IndexHeader& h, const CS* __restrict__ cs, const float4* __restrict__ pts,
                                             const unsigned int* __restrict__ hsv, const RowEntry* __restrict__ table, const float* __restrict__ lut_h,
                                             const float* __restrict__ lut_s) {
  const int n = a.st->particle_num;
  const int n_local = n > a.rank_id ? (n - a.rank_id + a.nranks - 1) / a.nranks : 0;
  const int items = n_local * a.chunks;
  const int lane = threadIdx.x & 31;
  // maximum_distance_^2 as the float just above it: every point with (double)d2 < max_d2 has d2 <= lim2
  const float lim2 = a.co.max_d2 >= 3.0e38 ? FLT_MAX : __double2float_ru(a.co.max_d2);
  // Large particle sets (many items per warp): items are handed out dynamically, one atomic per item with the next
  // one requested before the current one is worked on -- query cost varies with the list lengths (measured -4 % on
  // 100k particles).  Small sets (~4 items per warp): static interleaved assignment; there the atomic's latency costs
  // more than the imbalance.  Which warp evaluates an item never matters: each item owns its output slot.
  const int total_warps = gridDim.x * (blockDim.x >> 5);
  int next = (threadIdx.x >> 5) * gridDim.x + blockIdx.x;  // static: blocks interleaved so that consecutive items spread over the SMs
  if (DYN) {
    if (lane == 0) next = (int)atomicAdd(&a.st->work_counter, 1u);
    next = __shfl_sync(kFull, next, 0);
  }
  while (next < items) {
    const int item = next;
    if (!DYN) next = item + total_warps;
    else if (lane == 0) next = (int)atomicAdd(&a.st->work_counter, 1u);
    const int il = item / a.chunks, c = item - il * a.chunks;
    const int i = a.rank_id + il * a.nranks;
    float m[12];
    {
      const float4* mp = reinterpret_cast<const float4*>(a.mats) + (size_t)i * 3;
      const float4 r0 = mp[0], r1 = mp[1], r2 = mp[2];
      m[0] = r0.x; m[1] = r0.y; m[2] = r0.z; m[3] = r0.w; m[4] = r1.x; m[5] = r1.y; m[6] = r1.z; m[7] = r1.w;
      m[8] = r2.x; m[9] = r2.y; m[10] = r2.z; m[11] = r2.w;
    }
    const int j0 = c * a.chunk_len, j1 = min(a.M, j0 + a.chunk_len);
    double val = 0.0;
    unsigned int sum_um = 0, matched = 0;
    for (int j = j0 + lane; j < j1; j += 32) {
      const float4 mp = a.model[j];
      float qx, qy, qz;
      xform(m, mp.x, mp.y, mp.z, qx, qy, qz);
      NNResult nn = nn_none(lim2);
      if (h.n_cropped > 0) {
        nn = nn_search<CS>(cs, pts, h, table, qx, qy, qz, lim2);
      }
      if (i < a.dbg_k) {
        const size_t o = (size_t)i * a.M + a.model_perm[j];
        a.dbg_idx[o] = nn.slot >= 0 ? nn.orig() : -1;
        a.dbg_d2[o] = nn.slot >= 0 ? nn.d2() : FLT_MAX;
      }
      if (nn.slot >= 0 && (double)nn.d2() < a.co.max_d2) {
        // DistanceCoherence x HSVColorCoherence: 1/(1+d^2 w_d) * 1/(1+w_h diff) evaluated as one fp64 reciprocal of
        // the product of the denominators (differs from the product of reciprocals by ~1 ulp of fp64)
        double den = 1.0;
        const float df = sqrtf(nn.d2());
        sum_um += (unsigned int)fminf(df * 1.0e6f, 1.0e8f);
        ++matched;
        if (a.co.use_dist) {
          const double d = (double)df;
          den = 1.0 + d * d * a.co.dist_w;
        }
        if (USE_HSV) {
          const unsigned int sb = __float_as_uint(mp.w), tb = hsv[nn.slot];
          const float sh = lut_h[sb & 0xff], ss = lut_s[(sb >> 8) & 0xff], sv = lut_s[(sb >> 16) & 0xff];
          const float th = lut_h[tb & 0xff], ts = lut_s[(tb >> 8) & 0xff], tv = lut_s[(tb >> 16) & 0xff];
          const float hd = fabsf(sh - th);
          float hd2;
          if (sh < th) hd2 = fabsf(1.0f + sh - th); else hd2 = fabsf(1.0f + th - sh);
          float h_diff;
          if (hd < hd2) h_diff = a.co.h_w * hd * hd; else h_diff = a.co.h_w * hd2 * hd2;
          const float s_diff = a.co.s_w * (ss - ts) * (ss - ts);
          const float v_diff = a.co.v_w * (sv - tv) * (sv - tv);
          const float diff2 = h_diff + s_diff + v_diff;
          den *= 1.0 + a.co.hsv_w * (double)diff2;
        }
        val += rcp_f64(den);
      }
    }
    val = warp_sum(val);
    sum_um = (unsigned int)warp_sum((int)sum_um);  // <= 32 x chunk_len/32 x 1e8 um would overflow: chunk sums stay far below (d <= maximum distance)
    matched = (unsigned int)warp_sum((int)matched);
    if (lane == 0) {
      a.partial[(size_t)c * a.n_max + i] = val;
      if (matched) { atomicAdd(&a.st->nn_sum_um, (unsigned long long)sum_um); atomicAdd(&a.st->nn_count, (unsigned long long)matched); }
    }
    if (DYN) next = __shfl_sync(kFull, next, 0);
  }
}

// The whole weight() of one CTA of weight_lists_kernel through the row-table search, when the index header says the
// lists are off (PFT_CANDIDATE_LISTS = 0, too few queries, or a crop too large for the tables).  h, the two look-up
// tables and s_table live in the caller's shared memory; the tables are filled here.
template <bool USE_HSV, bool DYN>
__device__ __noinline__ void weight_rowtable_body(const WeightArgs a /* by value: a reference would pull the caller's kernel parameters into local memory */,
                                                  const IndexHeader& h, float* lut_h, float* lut_s, RowEntry* s_table) {
  extern __shared__ uint4 dyn_smem[];
  for (int i = threadIdx.x; i < kRows; i += blockDim.x) s_table[i] = a.table[i];
  if (USE_HSV) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) { lut_h[i] = (float)i / 180.0f; lut_s[i] = (float)i / 255.0f; }
  }
  __syncthreads();
  // ---- stage the scene index into shared memory: the points (float4) whenever they fit, then their packed HSV, then
  // (only when the candidate lists are off: nothing else reads them) the cell starts as 16-bit values
  const int n_pts = h.n_cropped + 1;  // + the dummy point that pads the candidate lists
  const long long need_pts = 16ll * n_pts;
  const long long need_hsv = 4ll * ((n_pts + 3) & ~3);
  const long long need_cs = 2ll * (((long long)h.n_cells + 1 + 7) & ~7ll);
  const bool pts_staged = h.valid && need_pts <= (long long)a.smem_bytes;
  const bool hsv_staged = USE_HSV && pts_staged && need_pts + need_hsv <= (long long)a.smem_bytes;
  const long long used = need_pts + (hsv_staged ? need_hsv : 0);
  const bool cs_staged = pts_staged && n_pts < 65536 && used + need_cs <= (long long)a.smem_bytes;
  uint4* s_pts = dyn_smem;
  unsigned int* s_hsv = reinterpret_cast<unsigned int*>(dyn_smem + n_pts);
  if (pts_staged) {
    const uint4* gp = reinterpret_cast<const uint4*>(a.pts);
    for (int i = threadIdx.x; i < n_pts; i += blockDim.x) s_pts[i] = gp[i];
  }
  if (hsv_staged) {
    for (int i = threadIdx.x; i < h.n_cropped; i += blockDim.x) s_hsv[i] = a.hsv[i];
  }
  // (separate call sites so that the compiler sees which pointers are shared memory: LDS instead of generic loads)
  if (cs_staged) {
    unsigned short* s_cs = reinterpret_cast<unsigned short*>(reinterpret_cast<unsigned char*>(dyn_smem) + used);
    for (int i = threadIdx.x; i <= h.n_cells; i += blockDim.x) s_cs[i] = (unsigned short)a.cell_start[i];
    __syncthreads();
    if (hsv_staged) weight_items<USE_HSV, DYN, unsigned short>(a, h, s_cs, reinterpret_cast<const float4*>(s_pts), s_hsv, s_table, lut_h, lut_s);
    else weight_items<USE_HSV, DYN, unsigned short>(a, h, s_cs, reinterpret_cast<const float4*>(s_pts), a.hsv, s_table, lut_h, lut_s);
  } else if (pts_staged) {
    __syncthreads();
    if (hsv_staged) weight_items<USE_HSV, DYN, int>(a, h, a.cell_start, reinterpret_cast<const float4*>(s_pts), s_hsv, s_table, lut_h, lut_s);
    else weight_items<USE_HSV, DYN, int>(a, h, a.cell_start, reinterpret_cast<const float4*>(s_pts), a.hsv, s_table, lut_h, lut_s);
  } else {
    weight_items<USE_HSV, DYN, int>(a, h, a.cell_start, a.pts, a.hsv, s_table, lut_h, lut_s);
  }
}

// ------------------------------------------------------------------ K3, list path: weight_lists_kernel
// The exact-search weight() (weight_rowtable_body when the lists are off).  Persistent, one CTA per SM; the indexed points
// {x, y, z, packed HSV} travel into shared memory as ONE bulk asynchronous copy (cp.async.bulk + mbarrier, issued by
// one thread while the others set up), each warp takes (particle, model chunk) items, a lane = one model point:
//   transform -> octant of the fine lattice -> ONE 16-byte load (header + seven slots) -> seven candidates from shared
//   memory, straight-line (dx, dy as packed FADD2 / FMUL2; the list is in input-index order, so strict < resolves
//   ties) -> coherence in fp64 -> warp-shuffle sum.
// The few queries whose octant has no short list (extended lists far from the surface, cells without a list) are
// answered one at a time by the whole warp (nn_slow_warp), bit-identical to the brute-force search.
struct SlowNN { float d2; int slot; };

// One query by a whole warp, brute force: every lane scans a 32nd of the indexed points that lie inside the crop box
// (the staged copy carries the flag), lexicographic (distance, input index) minimum across the lanes; the input index
// of a point is only fetched (from the global copy) to settle a tie or to compare the lanes' winners.
__device__ __noinline__ SlowNN nn_slow_warp(const unsigned char* __restrict__ sbase /* staged points {x,y,z,HSV|flag} */,
                                            const float4* __restrict__ pts /* {x,y,z,input index}, global */, int n, float qx, float qy, float qz, float lim2) {
  const int lane = threadIdx.x & 31;
  float bd = lim2;
  int bs = -1;
  for (int slot = lane; slot < n; slot += 32) {
    const float4 p = *reinterpret_cast<const float4*>(sbase + ((size_t)slot << 4));
    if (!(__float_as_uint(p.w) & kInCropBit)) continue;
    const float dx = qx - p.x, dy = qy - p.y, dz = qz - p.z;
    const float d2 = (dx * dx + dy * dy) + dz * dz;
    if (d2 < bd) { bd = d2; bs = slot; }
    else if (d2 == bd && bs >= 0 && __float_as_int(pts[slot].w) < __float_as_int(pts[bs].w)) bs = slot;
  }
  int bo = bs >= 0 ? __float_as_int(pts[bs].w) : 0x7fffffff;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float od = __shfl_xor_sync(kFull, bd, o);
    const int oo = __shfl_xor_sync(kFull, bo, o), os = __shfl_xor_sync(kFull, bs, o);
    if (os >= 0 && (od < bd || (od == bd && (bs < 0 || oo < bo)))) { bd = od; bo = oo; bs = os; }
  }
  return SlowNN{bd, bs};
}

// one 32-byte record (header + seven entries, or a pool group of eight entries) as ONE 256-bit load
struct Rec8 { unsigned int w[8]; };
__device__ __forceinline__ Rec8 load_rec8(const unsigned int* __restrict__ p) {
  Rec8 r;
  asm volatile("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r.w[0]), "=r"(r.w[1]), "=r"(r.w[2]), "=r"(r.w[3]), "=r"(r.w[4]), "=r"(r.w[5]), "=r"(r.w[6]), "=r"(r.w[7])
               : "l"(p));
  return r;
}

// one candidate: OFF = byte offset of the point in the staged array.  d2 follows the arithmetic contract
// ((dx*dx + dy*dy) + dz*dz, every operation rounded on its own); dx, dy as one packed FADD2 / FMUL2 pair.
#define PFT_CAND(OFF)                                                                          \
  {                                                                                            \
    const unsigned int of_ = (OFF);                                                            \
    const float4 p_ = *reinterpret_cast<const float4*>(sbase + of_);                           \
    const float2 d_ = sub2_rn(qxy, make_float2(p_.x, p_.y));                                   \
    const float dz_ = q.z - p_.z;                                                              \
    const float2 dd_ = mul2_rn(d_, d_);                                                        \
    const float d2_ = (dd_.x + dd_.y) + dz_ * dz_;                                             \
    if (d2_ < best) { best = d2_; boff = of_; }                                                \
  }

// a query on its way: the transformed model point, its packed HSV, the octant record
struct ListQuery { float x, y, z; unsigned int hsv; Rec8 r; };

template <bool USE_HSV, bool DYN>
__device__ __forceinline__ void weight_list_items(const WeightArgs& a, const IndexHeader& h, const unsigned char* __restrict__ sbase,
                                                  const float* __restrict__ lut_h, const float* __restrict__ lut_s) {
  const int n = a.st->particle_num;
  const int n_local = n > a.rank_id ? (n - a.rank_id + a.nranks - 1) / a.nranks : 0;
  const int items = n_local * a.chunks;
  const int lane = threadIdx.x & 31;
  // maximum_distance_^2 as the float just above it: (double)d2 < max_d2  <=>  d2 < lim2
  const float lim2 = a.co.max_d2 >= 3.0e38 ? FLT_MAX : __double2float_ru(a.co.max_d2);
  const float inv2 = h.inv_leaf * 2.0f;  // octant lattice: floor(q * 2 / resolution); (q * inv_leaf) * 2 == q * (inv_leaf * 2) exactly
  const int o2x = 2 * h.f_origin[0], o2y = 2 * h.f_origin[1], o2z = 2 * h.f_origin[2];
  const unsigned int d2x = 2u * (unsigned int)h.f_dim[0], d2y = 2u * (unsigned int)h.f_dim[1], d2z = 2u * (unsigned int)h.f_dim[2];
  const bool any_pts = h.n_cropped > 0;
  const bool use_v = a.co.v_w != 0.f;
  const int total_warps = gridDim.x * (blockDim.x >> 5);
  unsigned long long sum_um64 = 0ull;  // distance statistics: per lane, flushed once at the end
  unsigned int matched = 0;
  int next = (threadIdx.x >> 5) * gridDim.x + blockIdx.x;  // static: blocks interleaved so that consecutive items spread over the SMs
  if (DYN) {
    if (lane == 0) next = (int)atomicAdd(&a.st->work_counter, 1u);
    next = __shfl_sync(kFull, next, 0);
  }
  while (next < items) {
    const int item = next;
#ifdef PFT_TRACE
    const unsigned long long t_item0 = trace_now();
#endif
    if (!DYN) next = item + total_warps;
    else if (lane == 0) next = (int)atomicAdd(&a.st->work_counter, 1u);
    const int il = item / a.chunks, c = item - il * a.chunks;
    const int i = a.rank_id + il * a.nranks;
    float m[12];
    {
      const float4* mp = reinterpret_cast<const float4*>(a.mats) + (size_t)i * 3;
      const float4 r0 = mp[0], r1 = mp[1], r2 = mp[2];
      m[0] = r0.x; m[1] = r0.y; m[2] = r0.z; m[3] = r0.w; m[4] = r1.x; m[5] = r1.y; m[6] = r1.z; m[7] = r1.w;
      m[8] = r2.x; m[9] = r2.y; m[10] = r2.z; m[11] = r2.w;
    }
    const int j0 = c * a.chunk_len, j1 = min(a.M, j0 + a.chunk_len);
    // transform + octant + record load of the model point of round jb (inactive lanes repeat the last point)
    auto fetch = [&](int jb) {
      ListQuery q;
      const float4 mp = a.model[min(jb + lane, j1 - 1)];
      xform(m, mp.x, mp.y, mp.z, q.x, q.y, q.z);
      q.hsv = __float_as_uint(mp.w);
      // (cvt.rmi saturates: a far-away or non-finite query fails the range test)
      const int ix = __float2int_rd(q.x * inv2) - o2x, iy = __float2int_rd(q.y * inv2) - o2y, iz = __float2int_rd(q.z * inv2) - o2z;
      q.r.w[0] = kListOverflow;
      if ((unsigned int)ix < d2x && (unsigned int)iy < d2y && (unsigned int)iz < d2z)
        q.r = load_rec8(a.flists + (size_t)(((unsigned int)iz * d2y + (unsigned int)iy) * d2x + (unsigned int)ix) * 8);
      return q;
    };
    double val = 0.0;
    unsigned int sum_um = 0;  // (<= chunk_len / 32 x 1e8 per lane: no overflow for chunks below ~1300 points)
    auto eval = [&](const ListQuery& q, int jb) {
      const bool act = jb + lane < j1;
      const float2 qxy = make_float2(q.x, q.y);
      float best = lim2;
      unsigned int boff = 0xffffffffu;
      const unsigned int hw = q.r.w[0];
      if (hw == kListExtended) {
        // far from the surface (and not prunable to a short list): the lane scans its cell's extended list
        const uint4* xl = reinterpret_cast<const uint4*>(a.xlists + (size_t)q.r.w[1] * kListKX);
        const int n4 = ((int)q.r.w[2] + 3) >> 2;
        PFT_STAT(13, act ? 1 : 0); PFT_STAT(14, act ? (int)q.r.w[2] : 0);
        for (int g = 0; g < n4; ++g) {
          const uint4 w = xl[g];
          PFT_CAND(w.x) PFT_CAND(w.y) PFT_CAND(w.z) PFT_CAND(w.w)
        }
      } else if (hw < kListExtended) {
        PFT_CAND(q.r.w[1]) PFT_CAND(q.r.w[2]) PFT_CAND(q.r.w[3]) PFT_CAND(q.r.w[4]) PFT_CAND(q.r.w[5]) PFT_CAND(q.r.w[6]) PFT_CAND(q.r.w[7])
        const int cnt = (int)(hw & 0xffu);
        PFT_STAT(12, act ? 1 : 0); PFT_STAT(5, act ? cnt : 0);
        if (cnt > 7) {
          PFT_STAT(3, act ? 1 : 0); PFT_STAT(6, act ? cnt : 0);
          const unsigned int* pg = a.pool + (size_t)(hw >> 8) * 8;
          for (int g = 0; g < ((cnt - 7 + 7) >> 3); ++g) {
            const Rec8 w = load_rec8(pg + g * 8);
            PFT_CAND(w.w[0]) PFT_CAND(w.w[1]) PFT_CAND(w.w[2]) PFT_CAND(w.w[3]) PFT_CAND(w.w[4]) PFT_CAND(w.w[5]) PFT_CAND(w.w[6]) PFT_CAND(w.w[7])
          }
        }
      }
      // fourth word of the winner: packed HSV | in-crop flag.  The index may hold points beyond the crop box of this
      // weight() (one index per frame): a winner inside the box is the nearest CROPPED point; one outside is not an answer
      unsigned int tb = kInCropBit;
      if (boff != 0xffffffffu) tb = *reinterpret_cast<const unsigned int*>(sbase + boff + 12);
      // queries whose winner lies outside the crop box (near its faces), or whose cell has no list at all (the build gave
      // up: extremely rare): brute force over the cropped points, one query at a time, by the whole warp
      unsigned int slow = __ballot_sync(kFull, act && any_pts && (hw == kListOverflow || !(tb & kInCropBit)));
      while (slow) {
        const int src = __ffs(slow) - 1;
        slow &= slow - 1u;
        const float sx = __shfl_sync(kFull, q.x, src), sy = __shfl_sync(kFull, q.y, src), sz = __shfl_sync(kFull, q.z, src);
        PFT_STAT(4, lane == 0 ? 1 : 0);
        const SlowNN r = nn_slow_warp(sbase, a.pts, h.n_cropped, sx, sy, sz, lim2);
        if (lane == src) {
          best = r.d2; boff = r.slot >= 0 ? (unsigned int)r.slot << 4 : 0xffffffffu;
          if (r.slot >= 0) tb = *reinterpret_cast<const unsigned int*>(sbase + boff + 12);
        }
      }
      const bool hit = act && boff != 0xffffffffu;
      if (i < a.dbg_k && act) {
        const size_t o = (size_t)i * a.M + a.model_perm[min(jb + lane, j1 - 1)];
        a.dbg_idx[o] = hit ? __float_as_int(a.pts[boff >> 4].w) : -1;
        a.dbg_d2[o] = hit ? best : FLT_MAX;
      }
      if (hit) {
        // DistanceCoherence x HSVColorCoherence: 1/(1+d^2 w_d) * 1/(1+w_h diff) evaluated as one fp64 reciprocal of
        // the product of the denominators (differs from the product of reciprocals by ~1 ulp of fp64)
        double den = 1.0;
        const float df = sqrtf(best);
        sum_um += (unsigned int)fminf(df * 1.0e6f, 1.0e8f);
        ++matched;
        if (a.co.use_dist) {
          const double d = (double)df;
          den = 1.0 + d * d * a.co.dist_w;
        }
        if (USE_HSV) {
          const unsigned int sb = q.hsv;
          const float sh = lut_h[sb & 0xff], ss = lut_s[(sb >> 8) & 0xff];
          const float th = lut_h[tb & 0xff], ts = lut_s[(tb >> 8) & 0xff];
          const float hd = fabsf(sh - th);
          float hd2;
          if (sh < th) hd2 = fabsf(1.0f + sh - th); else hd2 = fabsf(1.0f + th - sh);
          float h_diff;
          if (hd < hd2) h_diff = a.co.h_w * hd * hd; else h_diff = a.co.h_w * hd2 * hd2;
          const float s_diff = a.co.s_w * (ss - ts) * (ss - ts);
          float v_diff = 0.f;  // (v_w == 0, the upstream default: the term is +0 whatever the values)
          if (use_v) { const float sv = lut_s[(sb >> 16) & 0xff], tv = lut_s[(tb >> 16) & 0xff]; v_diff = a.co.v_w * (sv - tv) * (sv - tv); }
          const float diff2 = h_diff + s_diff + v_diff;
          den *= 1.0 + a.co.hsv_w * (double)diff2;
        }
        val += rcp_f64(den);
      }
    };
    for (int jb = j0; jb < j1; jb += 32) eval(fetch(jb), jb);
    val = warp_sum(val);
    sum_um64 += sum_um;
    if (lane == 0) a.partial[(size_t)c * a.n_max + i] = val;
    if (DYN) next = __shfl_sync(kFull, next, 0);
#ifdef PFT_TRACE
    if (lane == 0) {
      const unsigned long long dt = trace_now() - t_item0;
      const unsigned long long old = atomicMax(&g_trace[12], dt);
      if (dt > old) g_trace[13] = (unsigned long long)item;
      if (dt > 8000ull) atomicAdd(&g_trace[14], 1ull);
      if (dt > 16000ull) atomicAdd(&g_trace[15], 1ull);
      atomicAdd(&g_trace[16], dt);
      atomicAdd(&g_trace[17], 1ull);
    }
#endif
  }
  // nearest-neighbour distance statistics (they steer the cell size of the next index build): integer sums, so the
  // totals do not depend on the order the atomics land in
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum_um64 += __shfl_xor_sync(kFull, sum_um64, o);
  matched = (unsigned int)warp_sum((int)matched);
  if (lane == 0 && matched) { atomicAdd(&a.st->nn_sum_um, sum_um64); atomicAdd(&a.st->nn_count, (unsigned long long)matched); }
}
#undef PFT_CAND

template <bool USE_HSV, int THREADS, bool DYN>
__global__ void __launch_bounds__(THREADS, 1) weight_lists_kernel(const WeightArgs a) {
  extern __shared__ uint4 dyn_smem[];
  __shared__ IndexHeader h;
  __shared__ float lut_h[256], lut_s[256];
  __shared__ __align__(8) unsigned long long s_bar;
  __shared__ RowEntry s_table[kRows];
  PFT_TRACE_MIN(3); PFT_TRACE_MAX(4);
  if (threadIdx.x == 0) h = *a.hdr;
  __syncthreads();
  if (!lists_on(h)) {
    // the index header says the lists are off for this crop (too few queries for the fine cells of the box, or a crop
    // too large for the tables): the same launch runs the row-table search instead -- one kernel either way, the
    // host never has to know
    weight_rowtable_body<USE_HSV, DYN>(a, h, lut_h, lut_s, s_table);
    return;
  }
  PFT_TRACE_MAX(5);
  const int n_pts = h.n_cropped + 1;  // + the dummy point that pads the lists
  const bool staged = 16ll * n_pts <= (long long)a.smem_bytes;
  if (staged && threadIdx.x == 0) {
    mbar_init(&s_bar, 1);
    const uint32_t bytes = 16u * (uint32_t)n_pts;
    mbar_expect_tx(&s_bar, bytes);
    for (uint32_t off = 0; off < bytes; off += 65536u)
      bulk_g2s(reinterpret_cast<unsigned char*>(dyn_smem) + off, reinterpret_cast<const unsigned char*>(a.pts2) + off, min(65536u, bytes - off), &s_bar);
  }
  if (USE_HSV) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) { lut_h[i] = (float)i / 180.0f; lut_s[i] = (float)i / 255.0f; }
  }
  __syncthreads();  // (the barrier is initialised, the tables are written)
  if (staged) {
    // (measured and dropped: waiting inside the item loop, after the first transform and record load -- nothing gained on
    // 1000 particles, 13 % lost on 100 000: the extra live register costs more than the ~3 us of overlap)
    mbar_wait(&s_bar, 0);
    PFT_TRACE_MAX(6);
    weight_list_items<USE_HSV, DYN>(a, h, reinterpret_cast<const unsigned char*>(dyn_smem), lut_h, lut_s);
    PFT_TRACE_MIN(7); PFT_TRACE_MAX(8);
  } else {
    weight_list_items<USE_HSV, DYN>(a, h, reinterpret_cast<const unsigned char*>(a.pts2), lut_h, lut_s);
  }
}

// ------------------------------------------------------------------ parity mode: ApproxNearestPairPointCloudCoherence
// The reference's own coherence (ref: src/auto_tracking.cpp:235-238, :250-252) searches with
// pcl::octree::OctreePointCloudSearch::approxNearestSearch: a greedy descent to the child whose voxel centre is
// nearest, then a linear scan of that leaf -- it may miss the true nearest neighbour.  PFT_NN_PCL_APPROX reproduces it
// (PCL-1.8.0 octree/impl/octree_pointcloud.hpp, octree_search.hpp; SURVEY A.5): the pointer octree is rebuilt by
// every weight() exactly as upstream builds it -- point by point in cloud order, the bounding box doubling towards
// each point that falls outside (the resulting keys depend on that order), which is a sequential process and runs on
// ONE thread -- and queried by every (particle, model point) in parallel.  Not the product path: the default
// (PFT_NN_EXACT) finds the true nearest neighbour and is ~100x faster.
struct OctNodeD { int child[8]; int head, tail; };
struct OctHeaderD {
  double mn[3], mx[3];
  double res;
  int depth, root, leaf_count, n_nodes, bbox_defined, overflow, pad0, pad1;
};

// Change detector (SURVEY 8 f-4): the same tree with per-leaf test stamps instead of point lists, kept across tests
struct CdNodeD { int child[8]; int last, count, prev_hit, pad; };
struct CdHeaderD {
  double mn[3], mx[3];
  double res;
  int depth, root, leaf_count, n_nodes, bbox_defined, overflow, test_id, found;
};

__device__ inline void oct_node_init(OctNodeD& n) { n.head = -1; n.tail = -1; }
__device__ inline void oct_node_init(CdNodeD& n) { n.last = 0; n.count = 0; n.prev_hit = 0; n.pad = 0; }

template <typename NodeT, typename HdrT>
__device__ inline int oct_new_node(NodeT* nodes, HdrT& H, int cap) {
  if (H.n_nodes >= cap) { H.overflow = 1; return 0; }
  NodeT& n = nodes[H.n_nodes];
#pragma unroll
  for (int c = 0; c < 8; ++c) n.child[c] = -1;
  oct_node_init(n);
  return H.n_nodes++;
}

// OctreePointCloud::addPointIdx up to the leaf: adoptBoundingBoxToPoint (the box doubles towards a point that falls
// outside: a new root is put on top), then the key from the CURRENT box and the descent, creating what is missing.
// Returns the leaf node (meaningless once H.overflow is set).
template <typename NodeT, typename HdrT>
__device__ inline int oct_insert(HdrT& H, NodeT* nodes, int node_cap, const double v[3]) {
  const double min_value = (double)1.1920928955078125e-07f;  // std::numeric_limits<float>::epsilon()
  while (true) {
    bool up[3], any = false;
    for (int d = 0; d < 3; ++d) { const bool lo = v[d] < H.mn[d]; up[d] = v[d] >= H.mx[d]; any = any || lo || up[d]; }
    if (!(any || !H.bbox_defined)) break;
    if (H.bbox_defined) {
      const int ci = ((!up[0]) << 2) | ((!up[1]) << 1) | (!up[2]);
      const int nr = oct_new_node(nodes, H, node_cap);
      nodes[nr].child[ci] = H.root;
      H.root = nr;
      double side = (double)(1 << H.depth) * H.res;
      for (int d = 0; d < 3; ++d) if (!up[d]) H.mn[d] -= side;
      H.depth++;
      side = (double)(1 << H.depth) * H.res - min_value;
      for (int d = 0; d < 3; ++d) H.mx[d] = H.mn[d] + side;
      if (H.depth > 30 || H.overflow) { H.overflow = 1; return 0; }
    } else {
      for (int d = 0; d < 3; ++d) { H.mn[d] = v[d] - H.res / 2; H.mx[d] = v[d] + H.res / 2; }
      // getKeyBitSize (the tree is empty whenever the box is still undefined)
      unsigned int mk[3];
      for (int d = 0; d < 3; ++d) mk[d] = (unsigned int)ceil((H.mx[d] - H.mn[d]) / H.res);
      const unsigned int max_voxels = max(max(max(mk[0], mk[1]), mk[2]), 2u);
      H.depth = (int)fmax(fmin(30.0, ceil(log2((double)max_voxels) - min_value)), 0.0);
      const double side = (double)(1 << H.depth) * H.res - min_value;
      for (int d = 0; d < 3; ++d) { const double over = (side - (H.mx[d] - H.mn[d])) / 2.0; H.mn[d] -= over; H.mx[d] += over; }
      H.bbox_defined = 1;
    }
  }
  const unsigned int key[3] = {(unsigned int)((v[0] - H.mn[0]) / H.res), (unsigned int)((v[1] - H.mn[1]) / H.res), (unsigned int)((v[2] - H.mn[2]) / H.res)};
  int n = H.root;
  for (int level = H.depth - 1; level >= 0; --level) {
    const unsigned int mask = 1u << level;
    const int ci = ((!!(key[0] & mask)) << 2) | ((!!(key[1] & mask)) << 1) | (!!(key[2] & mask));
    if (nodes[n].child[ci] < 0) { const int c = oct_new_node(nodes, H, node_cap); nodes[n].child[ci] = c; }
    n = nodes[n].child[ci];
  }
  return n;
}

__global__ void octree_build_kernel(const float4* __restrict__ scene, const CloudHeader* __restrict__ scene_hdr, const IndexHeader* __restrict__ ihdr,
                                    double res, OctNodeD* nodes, int node_cap, int* __restrict__ next, OctHeaderD* out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const IndexHeader h = *ihdr;
  OctHeaderD H;
  for (int d = 0; d < 3; ++d) { H.mn[d] = 0.0; H.mx[d] = 0.0; }
  H.res = res; H.depth = 0; H.leaf_count = 0; H.n_nodes = 0; H.bbox_defined = 0; H.overflow = 0; H.pad0 = H.pad1 = 0;
  H.root = oct_new_node(nodes, H, node_cap);
  const int ns = h.valid ? scene_hdr->n : 0;
  for (int i = 0; i < ns; ++i) {
    const float4 p = scene[i];
    if (!in_crop(p, h)) continue;  // cropInputPointCloud: the octree indexes the cropped cloud, in input order
    const double v[3] = {(double)p.x, (double)p.y, (double)p.z};
    const int n = oct_insert(H, nodes, node_cap, v);
    if (H.overflow) break;
    // append to the leaf (insertion order)
    if (nodes[n].head < 0) { nodes[n].head = i; H.leaf_count++; } else next[nodes[n].tail] = i;
    nodes[n].tail = i;
    next[i] = -1;
  }
  *out = H;
}

// ParticleFilterTracker::testChangeDetection: setInputCloud(cropped) + addPointsFromInputCloud +
// getPointIndicesFromNewVoxels(min_points) + switchBuffers of a pcl::octree::OctreePointCloudChangeDetector that lives
// as long as the tracker.  The double-buffered octree reports the leaves the previous buffer did not have: here every
// leaf carries the id of the last test that filled it, its point count in that test and whether it had also been
// filled by the test before.  *found = number of point indices upstream would report (changed_ = found > 0).
// One thread: the keys depend on the order in which the box grew (see octree_build_kernel).
__global__ void change_detect_kernel(const float4* __restrict__ scene, const CloudHeader* __restrict__ scene_hdr, const IndexHeader* __restrict__ ihdr,
                                     double res, CdNodeD* nodes, int node_cap, CdHeaderD* hdr, int min_points, int* __restrict__ out /* found, overflow */) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const IndexHeader h = *ihdr;
  CdHeaderD H = *hdr;
  if (H.n_nodes == 0) {  // first test (the buffer is zero-filled when it is allocated or reset)
    for (int d = 0; d < 3; ++d) { H.mn[d] = 0.0; H.mx[d] = 0.0; }
    H.res = res; H.depth = 0; H.leaf_count = 0; H.bbox_defined = 0; H.overflow = 0; H.test_id = 0; H.found = 0;
    H.root = oct_new_node(nodes, H, node_cap);
  }
  const int test = ++H.test_id;
  int found = 0;
  const int ns = h.valid ? scene_hdr->n : 0;
  for (int i = 0; i < ns; ++i) {
    const float4 p = scene[i];
    if (!in_crop(p, h)) continue;
    const double v[3] = {(double)p.x, (double)p.y, (double)p.z};
    const int n = oct_insert(H, nodes, node_cap, v);
    if (H.overflow) break;
    CdNodeD& leaf = nodes[n];
    if (leaf.last != test) {
      leaf.prev_hit = (leaf.last == test - 1 && test > 1) ? 1 : 0;
      leaf.last = test; leaf.count = 0;
    }
    const int c = ++leaf.count;
    // a new leaf is reported once it holds min_points points: all of them at that moment, one more with each later point
    if (!leaf.prev_hit) {
      const int thr = max(min_points, 1);
      if (c == thr) found += c; else if (c > thr) found += 1;
    }
  }
  H.found = found;
  *hdr = H;
  out[0] = found;
  out[1] = H.overflow;
}

// approxNearestSearch + approxNearestSearchRecursive.  Returns the index IN THE INPUT CLOUD (-1: empty tree).
__device__ inline int octree_approx_nearest(const OctHeaderD& H, const OctNodeD* __restrict__ nodes, const int* __restrict__ next,
                                            const float4* __restrict__ scene, float qx, float qy, float qz, float& d2_out) {
  d2_out = 0.f;
  if (H.leaf_count == 0) return -1;
  int node = H.root;
  unsigned int key[3] = {0u, 0u, 0u};
  for (int tree_depth = 1; tree_depth <= H.depth; ++tree_depth) {
    double best = 1.7976931348623157e308;
    int best_ci = -1;
    unsigned int bk[3] = {0u, 0u, 0u};
    const double cell = H.res * (double)(1 << (H.depth - tree_depth));
    for (int ci = 0; ci < 8; ++ci) {
      if (nodes[node].child[ci] < 0) continue;
      const unsigned int nk[3] = {(key[0] << 1) + (unsigned int)(!!(ci & 4)), (key[1] << 1) + (unsigned int)(!!(ci & 2)), (key[2] << 1) + (unsigned int)(!!(ci & 1))};
      const float cx = (float)(((double)nk[0] + 0.5) * cell + H.mn[0]);
      const float cy = (float)(((double)nk[1] + 0.5) * cell + H.mn[1]);
      const float cz = (float)(((double)nk[2] + 0.5) * cell + H.mn[2]);
      const float dx = cx - qx, dy = cy - qy, dz = cz - qz;
      const double dist = (double)((dx * dx + dy * dy) + dz * dz);
      if (dist >= best) continue;
      best = dist; best_ci = ci; bk[0] = nk[0]; bk[1] = nk[1]; bk[2] = nk[2];
    }
    if (best_ci < 0) return -1;
    node = nodes[node].child[best_ci];
    key[0] = bk[0]; key[1] = bk[1]; key[2] = bk[2];
  }
  // leaf: linear scan in insertion order, the first of equally near points wins
  double smallest = 1.7976931348623157e308;
  int idx = -1;
  for (int i = nodes[node].head; i >= 0; i = next[i]) {
    const float4 c = scene[i];
    const float dx = c.x - qx, dy = c.y - qy, dz = c.z - qz;
    const double sd = (double)((dx * dx + dy * dy) + dz * dz);
    if (sd >= smallest) continue;
    idx = i; smallest = sd; d2_out = (float)sd;
  }
  return idx;
}

struct WeightApproxArgs {
  const TrackerState* st;
  const OctHeaderD* oct; const OctNodeD* nodes; const int* next;
  const float4* scene;        // the input cloud (rgba in .w)
  const float4* model;        // {x,y,z,packed HSV} in tile order
  const int* model_perm;
  int M;
  const float* mats;
  double* partial;            // [chunks][n_max]
  int chunks, chunk_len, n_max, nranks, rank_id;
  CoherenceParams co;
  int dbg_k; int* dbg_idx; float* dbg_d2;
};

__global__ void __launch_bounds__(256) weight_approx_kernel(const WeightApproxArgs a) {
  __shared__ OctHeaderD H;
  if (threadIdx.x == 0) H = *a.oct;
  __syncthreads();
  const int n = a.st->particle_num;
  const int n_local = n > a.rank_id ? (n - a.rank_id + a.nranks - 1) / a.nranks : 0;
  const int items = n_local * a.chunks;
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  for (int item = warp; item < items; item += nwarps) {
    const int il = item / a.chunks, c = item - il * a.chunks;
    const int i = a.rank_id + il * a.nranks;
    float m[12];
    {
      const float4* mp = reinterpret_cast<const float4*>(a.mats) + (size_t)i * 3;
      const float4 r0 = mp[0], r1 = mp[1], r2 = mp[2];
      m[0] = r0.x; m[1] = r0.y; m[2] = r0.z; m[3] = r0.w; m[4] = r1.x; m[5] = r1.y; m[6] = r1.z; m[7] = r1.w;
      m[8] = r2.x; m[9] = r2.y; m[10] = r2.z; m[11] = r2.w;
    }
    const int j0 = c * a.chunk_len, j1 = min(a.M, j0 + a.chunk_len);
    double val = 0.0;
    for (int j = j0 + lane; j < j1; j += 32) {
      const float4 mp = a.model[j];
      float qx, qy, qz, d2 = FLT_MAX;
      xform(m, mp.x, mp.y, mp.z, qx, qy, qz);
      int idx = H.overflow ? -1 : octree_approx_nearest(H, a.nodes, a.next, a.scene, qx, qy, qz, d2);
      if (idx < 0) d2 = FLT_MAX;
      if (i < a.dbg_k) {
        const size_t o = (size_t)i * a.M + a.model_perm[j];
        a.dbg_idx[o] = idx;
        a.dbg_d2[o] = d2;
      }
      if (idx >= 0 && (double)d2 < a.co.max_d2) {
        double den = 1.0;
        if (a.co.use_dist) { const double d = (double)sqrtf(d2); den = 1.0 + d * d * a.co.dist_w; }
        if (a.co.use_hsv) {
          const unsigned int sb = __float_as_uint(mp.w), tb = rgba_to_hsv_packed(__float_as_uint(a.scene[idx].w));
          const float sh = (float)(sb & 0xff) / 180.0f, ss = (float)((sb >> 8) & 0xff) / 255.0f, sv = (float)((sb >> 16) & 0xff) / 255.0f;
          const float th = (float)(tb & 0xff) / 180.0f, ts = (float)((tb >> 8) & 0xff) / 255.0f, tv = (float)((tb >> 16) & 0xff) / 255.0f;
          const float hd = fabsf(sh - th);
          float hd2;
          if (sh < th) hd2 = fabsf(1.0f + sh - th); else hd2 = fabsf(1.0f + th - sh);
          float h_diff;
          if (hd < hd2) h_diff = a.co.h_w * hd * hd; else h_diff = a.co.h_w * hd2 * hd2;
          const float s_diff = a.co.s_w * (ss - ts) * (ss - ts);
          const float v_diff = a.co.v_w * (sv - tv) * (sv - tv);
          den *= 1.0 + a.co.hsv_w * (double)(h_diff + s_diff + v_diff);
        }
        val += 1.0 / den;
      }
    }
    val = warp_sum(val);
    if (lane == 0) a.partial[(size_t)c * a.n_max + i] = val;
  }
}

// Where particle i's raw weight lives in the all-gathered buffer [nranks][slice_cap].
__device__ __forceinline__ int raw_slot(int i, int nranks, int slice_cap) { return (i % nranks) * slice_cap + i / nranks; }

// change detector found nothing new: normalizeWeight() runs on the weights the particles already carry
__global__ void weights_to_raw_kernel(const TrackerState* st, const DevParticle* __restrict__ parts, float* __restrict__ raw, int nranks, int slice_cap) {
  const int n = st->particle_num;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) raw[raw_slot(i, nranks, slice_cap)] = parts[i].weight;
}

// Particle i's raw weight: -(float) of its per-chunk partials summed in the fixed chunk order.  Every path that turns
// partials into raw weights sums here, which is what keeps sharded and unsharded weights bit-identical.
__device__ __forceinline__ float raw_weight(const double* __restrict__ partial, int chunks, int n_max, int i) {
  double v = 0.0;
  for (int c = 0; c < chunks; ++c) v += partial[(size_t)c * n_max + i];
  return -(float)v;
}

// this rank's raw weights into its slice of the gathered buffer [nranks][slice_cap]
__global__ void raw_weights_kernel(const TrackerState* st, const double* __restrict__ partial, int chunks, int n_max,
                                   float* __restrict__ raw, int slice_cap, int nranks, int rank) {
  const int n = st->particle_num;
  for (int l = blockIdx.x * blockDim.x + threadIdx.x; rank + l * nranks < n; l += gridDim.x * blockDim.x)
    raw[rank * slice_cap + l] = raw_weight(partial, chunks, n_max, rank + l * nranks);
}

// ------------------------------------------------------------------ K4a: normalizeWeight
// The O(N) stages between two weight() calls (normalise, update, cumulative table) are replicated on every rank and
// grow with the TOTAL particle count, so they run as ONE thread-block cluster of kClusterCtas CTAs: every CTA reduces
// its slice, the per-CTA partials are exchanged through distributed shared memory and combined in a fixed order
// (identical results on every rank and every run), with cluster.sync() between the phases.  Small particle sets use
// the CTAS = 1 instantiation (no cluster launch overhead).
namespace cg = cooperative_groups;
constexpr int kClusterCtas = 8;

// ParticleFilterTracker::update: rep = the weighted sum of the particles' states, motion = its change.  Every thread
// sums the particles particle(i) of its slice, then the CTA (block_sum6), then the CTAs of the cluster in their fixed
// order.  update_kernel and the update fused into normalize_kernel both run this: the same result bit for bit.
template <int CTAS, typename Particle>
__device__ __forceinline__ void update_state(TrackerState* st, int n, Particle particle, double* red6 /* shared [192] */,
                                             double* s_part /* shared [6] */) {
  cg::cluster_group cluster = cg::this_cluster();
  const unsigned int crank = cluster.block_rank();
  double acc[6] = {0, 0, 0, 0, 0, 0};
  for (int i = crank * blockDim.x + threadIdx.x; i < n; i += CTAS * blockDim.x) {
    const DevParticle p = particle(i);
    const double w = (double)p.weight;
    acc[0] += (double)(float)((double)p.x * w); acc[1] += (double)(float)((double)p.y * w); acc[2] += (double)(float)((double)p.z * w);
    acc[3] += (double)(float)((double)p.roll * w); acc[4] += (double)(float)((double)p.pitch * w); acc[5] += (double)(float)((double)p.yaw * w);
  }
  block_sum6(acc, red6);
  if (threadIdx.x == 0) {
#pragma unroll
    for (int d = 0; d < 6; ++d) s_part[d] = acc[d];
  }
  cluster.sync();
  if (crank == 0 && threadIdx.x == 0) {
    double tot[6] = {0, 0, 0, 0, 0, 0};
    for (int r = 0; r < CTAS; ++r) {  // fixed order
      const double* p = cluster.map_shared_rank(s_part, r);
      for (int d = 0; d < 6; ++d) tot[d] += p[d];
    }
    const DevParticle o = st->rep;
    DevParticle r{(float)tot[0], (float)tot[1], (float)tot[2], 1.f, (float)tot[3], (float)tot[4], (float)tot[5], 1.0f / (float)n};
    st->rep = r;
    st->motion = DevParticle{r.x - o.x, r.y - o.y, r.z - o.z, 1.f, r.roll - o.roll, r.pitch - o.pitch, r.yaw - o.yaw, 0.f};
  }
}

template <int CTAS>
__global__ void __cluster_dims__(CTAS, 1, 1) __launch_bounds__(1024)
normalize_kernel(TrackerState* st, DevParticle* parts, float* raw /* [nranks][slice_cap] gathered raw weights */, double alpha, int nranks,
                 int slice_cap, const CloudHeader* __restrict__ scene_hdr, int M,
                 const double* __restrict__ partial /* non-null: this rank's raw weights are summed here from the weight kernel's
                                                       per-chunk partials; null: `raw` already holds every rank's */,
                 int chunks, int n_max, int fuse_update /* compute(): update() follows every weight(), do it in the same launch */,
                 PeerSet ps /* NVLink peer mode (ps.nranks > 1): this launch is the all-gather of the raw weights */) {
  cg::cluster_group cluster = cg::this_cluster();
  const unsigned int crank = cluster.block_rank();
  PFT_TRACE_MIN(11);
  __shared__ double red[32];
  __shared__ double s_part[3];  // this CTA's partial min, max, sum (read by the other CTAs of the cluster)
  __shared__ double s_upd[6];   // fused update(): this CTA's partial weighted state
  __shared__ double red6[192];
  if (partial && ps.nranks > 1) {
    // this rank's raw weights go straight into EVERY rank's window, then every rank's flag is raised; once the local
    // flag shows all ranks of this epoch, the local window holds them all
    const int np = st->particle_num;
    for (int l = crank * blockDim.x + threadIdx.x; ps.rank + l * nranks < np; l += CTAS * blockDim.x) {
      const float w = raw_weight(partial, chunks, n_max, ps.rank + l * nranks);
      for (int r = 0; r < nranks; ++r) ps.win[r]->raw[ps.rank * slice_cap + l] = w;
    }
    cluster.sync();  // every store of this rank is issued ...
    if (crank == 0 && threadIdx.x == 0) {
      __threadfence_system();  // ... and ordered (cumulatively) before the flags
      for (int r = 0; r < nranks; ++r) atomicAdd_system(&ps.win[r]->flag_raw, 1u);
      peer_wait(&ps.win[ps.rank]->flag_raw, st->peer_epoch * (unsigned int)nranks, &st->peer_error);
    }
    cluster.sync();
    raw = ps.win[ps.rank]->raw;
    partial = nullptr;
  }
  if (scene_hdr->n <= 0) return;  // Tracker::initCompute fails on an empty input cloud: compute() is a no-op
  const int n = st->particle_num;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int first = crank * blockDim.x + threadIdx.x, stride = CTAS * blockDim.x;
  double wmin = DBL_MAX, wmax = -DBL_MAX;
  for (int i = first; i < n; i += stride) {
    double w;
    if (partial) {
      // one rank: raw slot i (every thread re-reads below only the slots it writes here)
      const float wf = raw_weight(partial, chunks, n_max, i);
      raw[i] = wf;
      w = (double)wf;
    } else {
      w = (double)__ldcg(&raw[raw_slot(i, nranks, slice_cap)]);
    }
    if (wmin > w) wmin = w;
    if (w != 0.0 && wmax < w) wmax = w;
  }
  for (int o = 16; o > 0; o >>= 1) { wmin = fmin(wmin, __shfl_xor_sync(kFull, wmin, o)); wmax = fmax(wmax, __shfl_xor_sync(kFull, wmax, o)); }
  if (lane == 0) { red[wid] = wmin; red6[wid] = wmax; }
  __syncthreads();
  if (threadIdx.x < 2) {  // thread 0: minimum, thread 1: maximum of the per-warp values
    double v = threadIdx.x ? -DBL_MAX : DBL_MAX;
    for (int k = 0; k < nw; ++k) v = threadIdx.x ? fmax(v, red6[k]) : fmin(v, red[k]);
    s_part[threadIdx.x] = v;
  }
  cluster.sync();
  wmin = DBL_MAX; wmax = -DBL_MAX;
  for (int r = 0; r < CTAS; ++r) {
    const double* p = cluster.map_shared_rank(s_part, r);
    wmin = fmin(wmin, p[0]); wmax = fmax(wmax, p[1]);
  }
  double sum = 0.0;
  for (int i = first; i < n; i += stride) {
    float w = __ldcg(&raw[raw_slot(i, nranks, slice_cap)]);
    if (wmax != wmin) {
      if (w != 0.0f) w = (float)exp(1.0 - alpha * ((double)w - wmin) / (wmax - wmin));
    } else {
      w = 1.0f / (float)n;
    }
    parts[i].weight = w;
    sum += (double)w;
  }
  sum = block_sum(sum, red);
  if (threadIdx.x == 0) s_part[2] = sum;
  cluster.sync();
  sum = 0.0;
  for (int r = 0; r < CTAS; ++r) sum += cluster.map_shared_rank(s_part, r)[2];  // fixed order
  if (crank == 0 && threadIdx.x == 0) { st->fit_ratio = wmin; st->weight_sum = sum; st->evals += (unsigned long long)n * (unsigned long long)M; }
  const float fs = (float)sum;
  auto normalized = [&](int i) {
    DevParticle p = parts[i];
    if (sum != 0.0) p.weight = p.weight / fs;
    else p.weight = 1.0f / (float)n;
    parts[i].weight = p.weight;
    return p;
  };
  if (fuse_update) update_state<CTAS>(st, n, normalized, red6, s_upd);
  else for (int i = first; i < n; i += stride) normalized(i);
  cluster.sync();  // the partials of this CTA stay readable until every CTA of the cluster is done with them
}

// ------------------------------------------------------------------ K4c: update
template <int CTAS>
__global__ void __cluster_dims__(CTAS, 1, 1) __launch_bounds__(1024)
update_kernel(TrackerState* st, const DevParticle* __restrict__ parts, const CloudHeader* __restrict__ scene_hdr) {
  __shared__ double red6[192];
  __shared__ double s_part[6];
  if (scene_hdr->n <= 0) return;
  update_state<CTAS>(st, st->particle_num, [&](int i) { return parts[i]; }, red6, s_part);
  cg::this_cluster().sync();
}

// ------------------------------------------------------------------ K4b: resample
// Cumulative table in 2^-40 fixed point (order-independent integer prefix sums).  Every CTA of the cluster scans one
// contiguous segment; the segment totals travel through distributed shared memory.
template <int CTAS>
__global__ void __cluster_dims__(CTAS, 1, 1) __launch_bounds__(1024)
cdf_kernel(TrackerState* st, const DevParticle* __restrict__ parts, unsigned long long* __restrict__ cdf, unsigned long long* total_out,
           int* __restrict__ tbl_rep, int* __restrict__ tbl_min, int tbl_size, int n_target /* fixed-N tracker: particle_num_ (setParticleNum may have
           changed it since the last resample); 0: KLD, the stop rule sets the count */, const CloudHeader* __restrict__ scene_hdr) {
  cg::cluster_group cluster = cg::this_cluster();
  const unsigned int crank = cluster.block_rank();
  __shared__ unsigned long long smem[34];
  __shared__ unsigned long long s_total;
  const int n = st->particle_num;
  if (crank == 0 && threadIdx.x == 0) st->draw_call += 1ull;  // the draws of this resample were generated by the previous launch
  for (int i = crank * blockDim.x + threadIdx.x; i < tbl_size; i += CTAS * blockDim.x) { tbl_rep[i] = -1; tbl_min[i] = 0x7fffffff; }
  const int seg = (((n + CTAS - 1) / CTAS) + 3) & ~3;
  const int i0 = min((int)crank * seg, n), i1 = min(i0 + seg, n);
  auto wq = [&](int i) -> unsigned long long {
    const double w = (double)parts[i0 + i].weight;
    return (w > 0.0) ? (unsigned long long)(w * 1099511627776.0) : 0ull;
  };
  const unsigned long long mine = block_exclusive_scan<unsigned long long>(
      i1 - i0, wq, [&](int i, unsigned long long ex) { cdf[i0 + i] = ex + wq(i); }, smem);
  if (threadIdx.x == 0) s_total = mine;
  cluster.sync();
  unsigned long long before = 0ull, total = 0ull;
  for (int r = 0; r < CTAS; ++r) {
    const unsigned long long v = *cluster.map_shared_rank(&s_total, r);
    if (r < (int)crank) before += v;
    total += v;
  }
  if (before) for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x) cdf[i] += before;
  if (crank == 0 && threadIdx.x == 0) {
    *total_out = total;
    st->resample_n_old = n;
  }
  cluster.sync();
  // (every CTA has read the old count by now) fixed-N: the resample that follows produces particle_num_ particles
  if (crank == 0 && threadIdx.x == 0 && n_target > 0 && scene_hdr->n > 0) st->particle_num = n_target;
}

// ------------------------------------------------------------------ on-device draws (Philox4x32-10)
__device__ __forceinline__ void philox_round(unsigned int& c0, unsigned int& c1, unsigned int& c2, unsigned int& c3, unsigned int k0, unsigned int k1) {
  const unsigned int hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
  const unsigned int hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
  c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
}
__device__ inline void philox4(unsigned int c0, unsigned int c1, unsigned int c2, unsigned int c3, unsigned int k0, unsigned int k1, unsigned int* out) {
#pragma unroll
  for (int r = 0; r < 10; ++r) { philox_round(c0, c1, c2, c3, k0, k1); k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
// the draws of candidate n in resample call `call`: one selection uniform, one motion uniform, six standard normals
// (Box-Muller).  A pure function of (seed, call, n): every rank and every graph replay generates the same numbers.
__device__ inline void gen_draws(int n, unsigned long long call, unsigned long long seed, float& u_select, float& u_motion, float* z6) {
  unsigned int r[8];
  philox4((unsigned int)n, (unsigned int)call, (unsigned int)(call >> 32), 0u, (unsigned int)seed, (unsigned int)(seed >> 32), r);
  philox4((unsigned int)n, (unsigned int)call, (unsigned int)(call >> 32), 1u, (unsigned int)seed, (unsigned int)(seed >> 32), r + 4);
  const float k = 1.0f / 16777216.0f;
  u_select = (float)(r[0] >> 8) * k;
  u_motion = (float)(r[1] >> 8) * k;
#pragma unroll
  for (int p = 0; p < 3; ++p) {
    const float u1 = ((float)(r[2 + 2 * p] >> 8) + 1.0f) * k;  // (0,1]
    const float u2 = (float)(r[3 + 2 * p] >> 8) * k;
    const float rad = sqrtf(-2.0f * logf(u1));
    float sn, cs;
    sincosf(6.28318530718f * u2, &sn, &cs);
    z6[2 * p] = rad * cs;
    z6[2 * p + 1] = rad * sn;
  }
}
// draw arrays of one call (initParticles; resample generates its draws inline unless they are injected)
__global__ void draws_kernel(const TrackerState* __restrict__ st, float* u_select, float* normals, float* u_motion, int count,
                             unsigned long long seed) {
  const unsigned long long call = st->draw_call;
  for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < count; n += gridDim.x * blockDim.x) {
    float us, um, z[6];
    gen_draws(n, call, seed, us, um, z);
    u_select[n] = us;
    u_motion[n] = um;
#pragma unroll
    for (int d = 0; d < 6; ++d) normals[(size_t)n * 6 + d] = z[d];
  }
}

struct ResampleArgs {
  const TrackerState* st;
  const DevParticle* old_parts;
  DevParticle* new_parts;
  const unsigned long long* cdf;
  const unsigned long long* cdf_total;
  const float* u_select;   // [stride]      injected draws; all three null: generated inline from (seed, draw call, n)
  const float* normals;    // [stride][6]
  const float* u_motion;   // [stride]
  unsigned long long seed;
  const int* alias_a;      // PFT_SAMPLER_ALIAS_PCL: Walker alias table of the old particle set
  const double* alias_q;
  const CloudHeader* scene_hdr;
  int* ancestors;
  int* bin_keys;           // [n_max][6] (KLD)
  NoiseParams np;
  double motion_ratio;
  float bin_size[6];
  int kld, n_max, sampler;
  int n_target;            // fixed-N tracker: particles to produce (particle_num_)
};

// ParticleFilterTracker::genAliasTable (Walker's alias method, PCL-1.8.0 impl/particle_filter.hpp, SURVEY A.7) exactly
// as upstream runs it: a sequential two-stack construction, here on ONE thread.  Parity mode (PFT_SAMPLER_ALIAS_PCL):
// it reproduces upstream's ancestor choice for the same selection uniforms; the default sampler is the parallel
// cumulative table.
__global__ void alias_table_kernel(const TrackerState* __restrict__ st, const DevParticle* __restrict__ parts, int* __restrict__ a, double* __restrict__ q,
                                   int* __restrict__ HL) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const int N = st->resample_n_old;
  if (N <= 0) return;
  int* H = HL;
  int* L = HL + N - 1;
  for (int i = 0; i < N; ++i) { q[i] = (double)(parts[i].weight * (float)N); a[i] = i; }
  for (int i = 0; i < N; ++i) { if (q[i] >= 1.0) *H++ = i; else *L-- = i; }
  while (H != HL && L != HL + N - 1) {
    const int j = *(L + 1);
    const int k = *(H - 1);
    a[j] = k;
    q[k] += q[j] - 1;
    ++L;
    if (q[k] < 1.0) { *L-- = k; --H; }
  }
}
// sampleWithReplacement
__device__ __forceinline__ int alias_pick(const int* __restrict__ a, const double* __restrict__ q, int n, float u) {
  double rU = (double)u * (double)n;
  int k = (int)rU;
  rU -= k;
  if (k >= n) k = n - 1;
  return rU < q[k] ? k : a[k];
}

__device__ __forceinline__ int cdf_pick(const unsigned long long* __restrict__ cdf, unsigned long long total, int n, double u) {
  if (total == 0ull) { const int k = (int)(u * (double)n); return k >= n ? n - 1 : k; }
  const unsigned long long t = (unsigned long long)(u * (double)total);
  int lo = 0, hi = n - 1;
  while (lo < hi) { const int mid = (lo + hi) >> 1; if (cdf[mid] > t) hi = mid; else lo = mid + 1; }
  return lo;
}

__global__ void resample_kernel(const ResampleArgs a) {
  const int n_old = a.st->resample_n_old;
  const int n_cand = a.kld ? a.n_max : a.n_target;
  const unsigned long long total = *a.cdf_total;
  const bool inline_draws = a.u_select == nullptr;
  const unsigned long long call = a.st->draw_call - 1ull;  // cdf_kernel has already advanced the stream position past this resample
  float u0;
  if (inline_draws) { float um0, z0[6]; gen_draws(0, call, a.seed, u0, um0, z0); }
  else u0 = a.u_select[0];
  const bool skip = a.scene_hdr->n <= 0;  // empty input cloud: compute() is a no-op, particles carried over unchanged
  for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < n_cand; n += gridDim.x * blockDim.x) {
    if (skip) {
      if (n < n_old) a.new_parts[n] = a.old_parts[n];
      if (a.kld) {
#pragma unroll
        for (int d = 0; d < 6; ++d) a.bin_keys[(size_t)n * 6 + d] = 0;
      }
      continue;
    }
    if (!a.kld && n == 0) {  // fixed-N tracker: slot 0 is the representative state
      a.new_parts[0] = a.st->rep;
      a.ancestors[0] = -1;
      continue;
    }
    float us, um, z[6];
    if (inline_draws) {
      gen_draws(n, call, a.seed, us, um, z);
    } else {
      us = a.u_select[n]; um = a.u_motion[n];
#pragma unroll
      for (int d = 0; d < 6; ++d) z[d] = a.normals[(size_t)n * 6 + d];
    }
    double u;
    if (a.sampler == PFT_SAMPLER_CDF_VDC) {
      u = (double)u0 + (double)__brev((unsigned int)n) * (1.0 / 4294967296.0);
      if (u >= 1.0) u -= 1.0;
    } else {
      u = (double)us;
    }
    const int j = a.sampler == PFT_SAMPLER_ALIAS_PCL ? alias_pick(a.alias_a, a.alias_q, n_old, us) : cdf_pick(a.cdf, total, n_old, u);
    DevParticle x = a.old_parts[j];
    particle_sample(x, a.np, z);
    if (a.kld && (double)um < a.motion_ratio) {
      const DevParticle mo = a.st->motion;
      x.x += mo.x; x.y += mo.y; x.z += mo.z; x.roll += mo.roll; x.pitch += mo.pitch; x.yaw += mo.yaw;
    }
    a.new_parts[n] = x;
    a.ancestors[n] = j;
    if (a.kld) {
      const float xs[6] = {x.x, x.y, x.z, x.roll, x.pitch, x.yaw};
#pragma unroll
      for (int d = 0; d < 6; ++d) a.bin_keys[(size_t)n * 6 + d] = (int)(xs[d] / a.bin_size[d]);
    }
  }
}

// KLD: k(n) = number of distinct bins among the first n candidates.  A hash set keyed by the 6-int bin
// records the lowest candidate index of every bin; candidate m is "new" iff it is that lowest index.
__global__ void kld_insert_kernel(const int* __restrict__ bin_keys, int n_max, int* tbl_rep, int* tbl_min, int* __restrict__ slot_of,
                                  unsigned int mask) {
  for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < n_max; n += gridDim.x * blockDim.x) {
    int key[6];
    unsigned int hsh = 2166136261u;
#pragma unroll
    for (int d = 0; d < 6; ++d) { key[d] = bin_keys[(size_t)n * 6 + d]; hsh = (hsh ^ (unsigned int)key[d]) * 16777619u; hsh ^= hsh >> 15; }
    unsigned int s = hsh & mask;
    while (true) {
      int cur = tbl_rep[s];
      if (cur == -1) { const int prev = atomicCAS(&tbl_rep[s], -1, n); cur = (prev == -1) ? n : prev; }
      bool same = true;
#pragma unroll
      for (int d = 0; d < 6; ++d) same = same && (bin_keys[(size_t)cur * 6 + d] == key[d]);
      if (same) { atomicMin(&tbl_min[s], n); slot_of[n] = (int)s; break; }
      s = (s + 1) & mask;
    }
  }
}
// One block: first n >= 1 with !(n < n_max && (k(n) < 2 || n < KLbound(k(n)))) becomes particle_num.
__global__ void __launch_bounds__(1024) kld_stop_kernel(TrackerState* st, const int* __restrict__ tbl_min, const int* __restrict__ slot_of,
                                                        const double* __restrict__ kl_bound, int n_max,
                                                        const CloudHeader* __restrict__ scene_hdr) {
  __shared__ int smem[34];
  __shared__ int stop;
  if (scene_hdr->n <= 0) return;
  if (threadIdx.x == 0) stop = n_max;
  __syncthreads();
  auto is_new = [&](int m) -> int { return tbl_min[slot_of[m]] == m ? 1 : 0; };
  block_exclusive_scan<int>(
      n_max, is_new,
      [&](int m, int ex) {
        const int n = m + 1, k = ex + is_new(m);
        const bool go_on = (n < n_max) && (k < 2 || (double)n < kl_bound[k]);
        if (!go_on) atomicMin(&stop, n);
      },
      smem);
  __syncthreads();
  if (threadIdx.x == 0) st->particle_num = stop;
}

// ------------------------------------------------------------------ model preparation
// HSV packing of the reference cloud + spatial ordering so that a warp's 32 queries are neighbours.
__global__ void model_keys_kernel(const float4* __restrict__ in, int M, unsigned int* __restrict__ keys, int* __restrict__ idx, int M_pad,
                                  const float* __restrict__ bbox6) {
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < M_pad; j += gridDim.x * blockDim.x) {
    unsigned int key = 0xffffffffu;
    if (j < M) {
      const float4 p = in[j];
      const float ext = fmaxf(fmaxf(bbox6[3] - bbox6[0], bbox6[4] - bbox6[1]), fmaxf(bbox6[5] - bbox6[2], 1e-6f));
      auto q = [&](float v, float lo) -> unsigned int { float t = (v - lo) / ext * 1023.0f; t = fminf(fmaxf(t, 0.f), 1023.f); return (unsigned int)t; };
      auto spread = [](unsigned int v) -> unsigned int {
        v = (v | (v << 16)) & 0x030000FFu; v = (v | (v << 8)) & 0x0300F00Fu; v = (v | (v << 4)) & 0x030C30C3u; v = (v | (v << 2)) & 0x09249249u;
        return v;
      };
      key = spread(q(p.x, bbox6[0])) | (spread(q(p.y, bbox6[1])) << 1) | (spread(q(p.z, bbox6[2])) << 2);
    }
    keys[j] = key; idx[j] = j;
  }
}
__global__ void __launch_bounds__(1024) model_bbox_kernel(const float4* __restrict__ in, int M, float* bbox6) {
  __shared__ float red[6][32];
  float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
  for (int j = threadIdx.x; j < M; j += blockDim.x) {
    const float4 p = in[j];
    mn[0] = fminf(mn[0], p.x); mn[1] = fminf(mn[1], p.y); mn[2] = fminf(mn[2], p.z);
    mx[0] = fmaxf(mx[0], p.x); mx[1] = fmaxf(mx[1], p.y); mx[2] = fmaxf(mx[2], p.z);
  }
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int d = 0; d < 3; ++d) { mn[d] = warp_min(mn[d]); mx[d] = warp_max(mx[d]); }
  if (lane == 0) { for (int d = 0; d < 3; ++d) { red[d][wid] = mn[d]; red[3 + d][wid] = mx[d]; } }
  __syncthreads();
  if (threadIdx.x < 6) {
    float v = red[threadIdx.x][0];
    for (int k = 1; k < (int)(blockDim.x >> 5); ++k) v = threadIdx.x < 3 ? fminf(v, red[threadIdx.x][k]) : fmaxf(v, red[threadIdx.x][k]);
    bbox6[threadIdx.x] = v;
  }
}
// Bitonic sort of (key, idx) pairs by (key, idx), one block, data in global memory (init-time only).
__global__ void __launch_bounds__(1024) bitonic_sort_kernel(unsigned int* keys, int* idx, int n_pad) {
  for (int k = 2; k <= n_pad; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < n_pad; i += blockDim.x) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const unsigned int ka = keys[i], kb = keys[ixj];
          const int ia = idx[i], ib = idx[ixj];
          const bool gt = (ka > kb) || (ka == kb && ia > ib);
          const bool up = (i & k) == 0;
          if (gt == up) { keys[i] = kb; keys[ixj] = ka; idx[i] = ib; idx[ixj] = ia; }
        }
      }
      __syncthreads();
    }
  }
}
__global__ void model_gather_kernel(const float4* __restrict__ in, const int* __restrict__ idx, int M, float4* __restrict__ out, int* __restrict__ perm) {
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < M; j += gridDim.x * blockDim.x) {
    const int s = idx[j];
    const float4 p = in[s];
    out[j] = make_float4(p.x, p.y, p.z, __uint_as_float(rgba_to_hsv_packed(__float_as_uint(p.w))));
    perm[j] = s;
  }
}

__global__ void single_matrix_kernel(DevParticle p, float* m12) { particle_to_matrix(p.x, p.y, p.z, p.roll, p.pitch, p.yaw, m12); }

// ------------------------------------------------------------------ result post-processing (SURVEY 8 f-3)
// What viz_cb derives from getResult() for every object (ref: src/auto_tracking.cpp:309-316, :432-466): the model
// moved to the result pose (+ the viewer's z offset), its centroid (compute3DCentroid: the position that is published
// on /visual/cam_frame_obj_pos_vector, ref :481-515), the normalised covariance, its eigenvectors (ascending
// eigenvalues; third axis = first x second as in the reference) and the oriented bounding box in that frame.
// Sums are accumulated in fp64 from fp32 terms (order independent); Eigen's SelfAdjointEigenSolver leaves the sign
// of an eigenvector unspecified, here the largest component of the first two axes is made positive.
struct ResultBox {
  float centroid[3];
  float axes[9];        // row-major 3x3, columns = box axes (eigDx)
  float extent[3];      // max_pt - min_pt in the box frame
  float center[3];      // tfinal = eigDx * 0.5 (max_pt + min_pt) + centroid
  float quat[4];        // qfinal = Quaternionf(eigDx): w, x, y, z
  float eigenvalues[3];
  int n;
};

__device__ inline void jacobi_eigen3(double A[3][3], double V[3][3], double w[3]) {
  for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) V[i][j] = i == j ? 1.0 : 0.0;
  for (int sweep = 0; sweep < 32; ++sweep) {
    const double off = fabs(A[0][1]) + fabs(A[0][2]) + fabs(A[1][2]);
    if (off <= 1.0e-300 || off <= 1.0e-18 * (fabs(A[0][0]) + fabs(A[1][1]) + fabs(A[2][2]))) break;
    for (int p = 0; p < 2; ++p) for (int q = p + 1; q < 3; ++q) {
      if (fabs(A[p][q]) <= 1.0e-300) continue;
      const double theta = (A[q][q] - A[p][p]) / (2.0 * A[p][q]);
      const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
      const double c = 1.0 / sqrt(t * t + 1.0), sn = t * c;
      for (int k = 0; k < 3; ++k) { const double akp = A[k][p], akq = A[k][q]; A[k][p] = c * akp - sn * akq; A[k][q] = sn * akp + c * akq; }
      for (int k = 0; k < 3; ++k) { const double apk = A[p][k], aqk = A[q][k]; A[p][k] = c * apk - sn * aqk; A[q][k] = sn * apk + c * aqk; }
      for (int k = 0; k < 3; ++k) { const double vkp = V[k][p], vkq = V[k][q]; V[k][p] = c * vkp - sn * vkq; V[k][q] = sn * vkp + c * vkq; }
    }
  }
  for (int i = 0; i < 3; ++i) w[i] = A[i][i];
  // ascending eigenvalues (selection sort of three)
  for (int i = 0; i < 2; ++i) for (int j = i + 1; j < 3; ++j) if (w[j] < w[i]) {
    const double tw = w[i]; w[i] = w[j]; w[j] = tw;
    for (int k = 0; k < 3; ++k) { const double tv = V[k][i]; V[k][i] = V[k][j]; V[k][j] = tv; }
  }
}

__global__ void __launch_bounds__(1024) result_box_kernel(const TrackerState* __restrict__ st, const float4* __restrict__ model, int M, float z_offset,
                                                          ResultBox* __restrict__ out) {
  __shared__ double red[32];
  __shared__ double s_sum[9];
  __shared__ float s_c[3], s_E[9], s_t[3];
  __shared__ float s_mn[32][3], s_mx[32][3];
  float m[12];
  const DevParticle rep = st->rep;
  particle_to_matrix(rep.x, rep.y, rep.z, rep.roll, rep.pitch, rep.yaw, m);
  m[11] += z_offset;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  // ---- centroid
  double sx = 0.0, sy = 0.0, sz = 0.0;
  for (int j = threadIdx.x; j < M; j += blockDim.x) {
    const float4 p = model[j];
    float x, y, z;
    xform(m, p.x, p.y, p.z, x, y, z);
    sx += (double)x; sy += (double)y; sz += (double)z;
  }
  sx = block_sum(sx, red); if (threadIdx.x == 0) s_sum[0] = sx;
  sy = block_sum(sy, red); if (threadIdx.x == 0) s_sum[1] = sy;
  sz = block_sum(sz, red); if (threadIdx.x == 0) s_sum[2] = sz;
  __syncthreads();
  if (threadIdx.x < 3) s_c[threadIdx.x] = M > 0 ? (float)(s_sum[threadIdx.x] / (double)M) : 0.f;
  __syncthreads();
  const float cx = s_c[0], cy = s_c[1], cz = s_c[2];
  // ---- normalised covariance about the fp32 centroid (computeCovarianceMatrixNormalized)
  double c6[6] = {0, 0, 0, 0, 0, 0};
  for (int j = threadIdx.x; j < M; j += blockDim.x) {
    const float4 p = model[j];
    float x, y, z;
    xform(m, p.x, p.y, p.z, x, y, z);
    const float dx = x - cx, dy = y - cy, dz = z - cz;
    c6[0] += (double)(dx * dx); c6[1] += (double)(dx * dy); c6[2] += (double)(dx * dz);
    c6[3] += (double)(dy * dy); c6[4] += (double)(dy * dz); c6[5] += (double)(dz * dz);
  }
  for (int k = 0; k < 6; ++k) { const double v = block_sum(c6[k], red); if (threadIdx.x == 0) s_sum[k] = v; }
  __syncthreads();
  if (threadIdx.x == 0) {
    const double inv = M > 0 ? 1.0 / (double)M : 0.0;
    // the reference decomposes the fp32 matrix
    double A[3][3], V[3][3], w[3];
    A[0][0] = (double)(float)(s_sum[0] * inv); A[0][1] = A[1][0] = (double)(float)(s_sum[1] * inv); A[0][2] = A[2][0] = (double)(float)(s_sum[2] * inv);
    A[1][1] = (double)(float)(s_sum[3] * inv); A[1][2] = A[2][1] = (double)(float)(s_sum[4] * inv); A[2][2] = (double)(float)(s_sum[5] * inv);
    jacobi_eigen3(A, V, w);
    for (int col = 0; col < 2; ++col) {  // sign convention: the largest component of an axis is positive
      int big = 0;
      for (int k = 1; k < 3; ++k) if (fabs(V[k][col]) > fabs(V[big][col])) big = k;
      if (V[big][col] < 0.0) for (int k = 0; k < 3; ++k) V[k][col] = -V[k][col];
    }
    float E[9];
    for (int r = 0; r < 3; ++r) for (int col = 0; col < 2; ++col) E[3 * r + col] = (float)V[r][col];
    // eigDx.col(2) = eigDx.col(0).cross(eigDx.col(1))
    E[2] = E[3] * E[7] - E[6] * E[4];
    E[5] = E[6] * E[1] - E[0] * E[7];
    E[8] = E[0] * E[4] - E[3] * E[1];
    for (int k = 0; k < 9; ++k) { s_E[k] = E[k]; out->axes[k] = E[k]; }
    for (int k = 0; k < 3; ++k) out->eigenvalues[k] = (float)w[k];
    // p2w: rotation = eigDx^T, translation = -(eigDx^T * centroid)
    for (int r = 0; r < 3; ++r) s_t[r] = -1.f * ((E[r] * cx + E[3 + r] * cy) + E[6 + r] * cz);
  }
  __syncthreads();
  // ---- extents in the box frame (transformPointCloud with p2w + getMinMax3D)
  float p2w[12];
  for (int r = 0; r < 3; ++r) { p2w[4 * r] = s_E[r]; p2w[4 * r + 1] = s_E[3 + r]; p2w[4 * r + 2] = s_E[6 + r]; p2w[4 * r + 3] = s_t[r]; }
  float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
  for (int j = threadIdx.x; j < M; j += blockDim.x) {
    const float4 p = model[j];
    float x, y, z, u, v, w;
    xform(m, p.x, p.y, p.z, x, y, z);
    xform(p2w, x, y, z, u, v, w);
    mn[0] = fminf(mn[0], u); mn[1] = fminf(mn[1], v); mn[2] = fminf(mn[2], w);
    mx[0] = fmaxf(mx[0], u); mx[1] = fmaxf(mx[1], v); mx[2] = fmaxf(mx[2], w);
  }
  for (int d = 0; d < 3; ++d) { mn[d] = warp_min(mn[d]); mx[d] = warp_max(mx[d]); }
  if (lane == 0) for (int d = 0; d < 3; ++d) { s_mn[wid][d] = mn[d]; s_mx[wid][d] = mx[d]; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < nw; ++w) for (int d = 0; d < 3; ++d) { mn[d] = fminf(mn[d], s_mn[w][d]); mx[d] = fmaxf(mx[d], s_mx[w][d]); }
    if (M <= 0) for (int d = 0; d < 3; ++d) { mn[d] = 0.f; mx[d] = 0.f; }
    float md[3];
    for (int d = 0; d < 3; ++d) { out->extent[d] = mx[d] - mn[d]; md[d] = 0.5f * (mx[d] + mn[d]); out->centroid[d] = s_c[d]; }
    for (int r = 0; r < 3; ++r) out->center[r] = ((s_E[3 * r] * md[0] + s_E[3 * r + 1] * md[1]) + s_E[3 * r + 2] * md[2]) + s_c[r];
    float m34[12];
    for (int r = 0; r < 3; ++r) { m34[4 * r] = s_E[3 * r]; m34[4 * r + 1] = s_E[3 * r + 1]; m34[4 * r + 2] = s_E[3 * r + 2]; m34[4 * r + 3] = 0.f; }
    const Quat q = quat_from_matrix(m34);
    out->quat[0] = q.w; out->quat[1] = q.x; out->quat[2] = q.y; out->quat[3] = q.z;
    out->n = M;
  }
}

}  // namespace pft
