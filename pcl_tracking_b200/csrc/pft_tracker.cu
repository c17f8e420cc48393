// pft_tracker.cu -- C ABI of the tracker object (include/pft/pft.h) and the host-side sequencing of
// kernels K2 (scene index), K3 (weight) and K4 (normalise / resample / update).
//
// Replaces pcl::tracking::KLDAdaptiveParticleFilterOMPTracker / ParticleFilterOMPTracker as configured
// and driven by ref: src/auto_tracking.cpp:198-258 (knobs), :673-676 (reference cloud), :688-697
// (setInputCloud + compute per frame), :270 / :309-310 (read-out).  Upstream control flow restated in
// SURVEY.md Appendix A.3: compute() = initCompute (initParticles on first use) + iteration_num x
// { resample (if changed_) ; weight ; update (if changed_) }.
//
// Everything a frame needs lives on the device (particle set, live particle count, crop box, index
// header, weights, representative state), so one compute() is a fixed kernel sequence without a host
// round trip; in steady state the sequence is replayed from a CUDA graph.  Multi-GPU: particle i is
// weighted by rank i % nranks; the crop box is all-reduced and the raw weights all-gathered either by
// aabb_kernel and normalize_kernel themselves through NVLink peer windows, or over NCCL (loaded with
// dlopen so that the library itself has no link-time NCCL dependency); resample, normalise and update
// run replicated on every rank from identical draws.
#include <dlfcn.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <vector>

#include "pft_internal.h"
#include "pft_tracker_kernels.cuh"

using namespace pft;

// ------------------------------------------------------------------ NCCL through dlopen
namespace {

struct UidByValue { char internal[128]; };  // ncclUniqueId is passed by value
struct NcclApi {
  void* lib = nullptr;
  bool tried = false;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, UidByValue, int) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
  int (*Broadcast)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
NcclApi g_nccl;
constexpr int kNcclFloat = 7;  // ncclFloat32
constexpr int kNcclChar = 0;   // ncclInt8
constexpr int kNcclMax = 2, kNcclMin = 3;

int load_nccl() {
  if (g_nccl.lib) return PFT_OK;
  if (g_nccl.tried) { set_last_error("NCCL is not loadable (libnccl.so.2)"); return PFT_ERR_COMM; }
  g_nccl.tried = true;
  const char* names[] = {getenv("PFT_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
  void* h = nullptr;
  for (const char* n : names) {
    if (!n) continue;
    h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (h) break;
  }
  if (!h) { set_last_error("NCCL is not loadable: %s", dlerror()); return PFT_ERR_COMM; }
  auto sym = [&](const char* n) { return dlsym(h, n); };
  g_nccl.GetUniqueId = (decltype(g_nccl.GetUniqueId))sym("ncclGetUniqueId");
  g_nccl.CommInitRank = (decltype(g_nccl.CommInitRank))sym("ncclCommInitRank");
  g_nccl.CommDestroy = (decltype(g_nccl.CommDestroy))sym("ncclCommDestroy");
  g_nccl.AllGather = (decltype(g_nccl.AllGather))sym("ncclAllGather");
  g_nccl.AllReduce = (decltype(g_nccl.AllReduce))sym("ncclAllReduce");
  g_nccl.Broadcast = (decltype(g_nccl.Broadcast))sym("ncclBroadcast");
  g_nccl.GroupStart = (decltype(g_nccl.GroupStart))sym("ncclGroupStart");
  g_nccl.GroupEnd = (decltype(g_nccl.GroupEnd))sym("ncclGroupEnd");
  g_nccl.GetErrorString = (decltype(g_nccl.GetErrorString))sym("ncclGetErrorString");
  if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.CommDestroy || !g_nccl.AllGather || !g_nccl.AllReduce || !g_nccl.Broadcast || !g_nccl.GroupStart ||
      !g_nccl.GroupEnd) {
    set_last_error("NCCL library lacks a required symbol");
    return PFT_ERR_COMM;
  }
  g_nccl.lib = h;
  return PFT_OK;
}
#define PFT_NCCL_TRY(expr)                                                                                       \
  do {                                                                                                           \
    int _r = (expr);                                                                                             \
    if (_r != 0) {                                                                                               \
      set_last_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, g_nccl.GetErrorString ? g_nccl.GetErrorString(_r) : "nccl error"); \
      return PFT_ERR_COMM;                                                                                       \
    }                                                                                                            \
  } while (0)

inline int blocks_for(long long n, int block, int cap) {
  long long g = (n + block - 1) / block;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace

// The device storage of the candidate lists (format: CandLists), sized for a table of up to `cells` fine cells
struct CandListStore {
  DevBuf records, pool, xlists, cell_items, l1_slots, needed, needed_list, far_list, built_bits, counters;

  // sizes beyond the table: one spare fine cell of records and slots, kSpare entries in the queues and bitmaps, and
  // blocks of 2x2x2 fine cells, at most ceil(d/2)^3 <= (d+1)^3/8, bounded generously by cells/2 + kBlockSlack
  static constexpr size_t kSpare = 16, kBlockSlack = 4096;
  int reserve(int cells) {
    const size_t n = (size_t)cells;
    int rc;
    if ((rc = records.reserve((n + 1) * kCellWords * sizeof(unsigned int)))) return rc;
    if ((rc = pool.reserve((size_t)kPoolGroups * kRecordWords * sizeof(unsigned int)))) return rc;
    if ((rc = xlists.reserve((size_t)kListXCells * kListKX * sizeof(unsigned int)))) return rc;
    if ((rc = cell_items.reserve((n + kSpare) * sizeof(int2)))) return rc;
    if ((rc = l1_slots.reserve((n + 1) * kL1Cap * sizeof(unsigned short)))) return rc;
    if ((rc = needed.reserve((n + kSpare) * sizeof(unsigned int)))) return rc;
    if ((rc = needed_list.reserve((n / 2 + kBlockSlack) * sizeof(int)))) return rc;
    if ((rc = far_list.reserve((n + kSpare) * sizeof(int)))) return rc;
    if ((rc = built_bits.reserve((n / 32 + kSpare) * sizeof(unsigned int)))) return rc;
    return counters.reserve(sizeof(ListCounters));
  }
  CandLists view() const {
    return CandLists{records.as<unsigned int>(), pool.as<unsigned int>(), xlists.as<unsigned int>(), cell_items.as<int2>(), l1_slots.as<unsigned short>(),
                     needed.as<unsigned int>(), needed_list.as<int>(), far_list.as<int>(), built_bits.as<unsigned int>(), counters.as<ListCounters>()};
  }
  void release() {
    for (DevBuf* b : {&records, &pool, &xlists, &cell_items, &l1_slots, &needed, &needed_list, &far_list, &built_bits, &counters}) b->release();
  }
};

// ------------------------------------------------------------------ the tracker object
struct SceneReplica;
struct pft_tracker {
  pft_context* ctx = nullptr;
  bool kld = true;
  // knobs (defaults = PCL constructor defaults, SURVEY A.3; coherence defaults as the CPU oracle)
  int threads = 0, particle_num = 0, max_particle_num = 0, iteration_num = 1, min_indices = 1;
  int nn_mode = PFT_NN_EXACT, use_hsv = 0, use_dist = 1, sampler = PFT_SAMPLER_CDF, quat_sample = 1, debug_nn = 0;
  double delta = 0.99, epsilon = 0.0, alpha = 15.0, motion_ratio = 0.25, max_dist = 1.79769313486231570815e+308;
  double dist_w = 1.0, hsv_w = 1.0, h_w = 1.0, s_w = 1.0, v_w = 0.0, search_res = 0.01, resample_thr = 0.0;
  double step_cov[6] = {0, 0, 0, 0, 0, 0}, init_cov[6] = {0, 0, 0, 0, 0, 0}, init_mean[6] = {0, 0, 0, 0, 0, 0};
  float bin_size[6] = {0, 0, 0, 0, 0, 0};
  float trans[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0};
  unsigned long long seed = 0x5eedull;
  // host mirror of the control state
  bool changed = false, has_particles = false;
  int n_cap = 0;        // allocated particle capacity
  int M = 0;            // model points
  const pft_cloud* input = nullptr;
  // what the kernels read: `input` itself, or this context's replica of an input of another context (resolve_scenes)
  const pft_cloud* scene = nullptr;
  SceneReplica* replica = nullptr;
  size_t scene_cap = 0; // allocated index capacity (scene points)
  int max_cells = 1 << 20;  // cap of the index grid; a larger crop box gets coarser cells
  int list_mode = 1;             // PFT_CANDIDATE_LISTS
  int list_max_cells = kListMaxCells;  // fine cells the candidate lists are sized for; 0 disables the lists
  int cur = 0;          // live particle buffer
  int inj_slots = 0, inj_stride = 0;
  int draw_cap = 0;
  bool timing = false;
  float t_weight_ms = 0.f, t_compute_ms = 0.f;
  std::vector<cudaEvent_t> ev_w;  // pairs around the lookup launches of the last compute
  cudaEvent_t ev_c0 = nullptr, ev_c1 = nullptr;
  int n_ev_used = 0;
  // timing mode: one event after every kernel of the last compute(), for the per-kernel breakdown
  std::vector<cudaEvent_t> ev_k;
  std::vector<const char*> ev_k_name;
  int n_ev_k = 0;
  // sharding (comm = the context's communicator when this tracker exchanges over NCCL)
  void* comm = nullptr;
  int nranks = 1, rank = 0;
  // NVLink peer exchange (pft_tracker_peer_*): the local window + the peers' windows mapped with CUDA IPC
  bool peer_mode = false;
  bool peer_ipc = true;       // the peers' windows were opened with CUDA IPC (false: same process, mapped directly)
  // single-process multi-device mode (pft_tracker_set_devices): this tracker is rank 0; one follower per further device
  struct Follower { pft_context* ctx = nullptr; pft_tracker* t = nullptr; };
  std::vector<Follower> followers;
  bool md_attached = false, md_prepared = false;
  void* peer_local = nullptr;
  size_t peer_bytes = 0;
  PeerSet peers{};
  // graph
  bool graph_enabled = true;
  cudaGraphExec_t graph_exec[2] = {nullptr, nullptr};  // one per value of `cur` at the start of the frame
  const void* graph_scene_pts[2] = {nullptr, nullptr};
  const void* graph_scene_hdr[2] = {nullptr, nullptr};
  unsigned long long config_version = 1, graph_version[2] = {0, 0};
  unsigned long long graph_replays = 0;
  int graph_nodes[2] = {0, 0};
  // device buffers
  DevBuf st, parts[2], mats, slot_aabb, model, model_perm, model_tmp, sort_keys, sort_idx, bbox, raw, partial, cdf, cdf_total, ancestors, bin_keys, tbl_rep,
      tbl_min, slot_of, klb, d_usel, d_normals, d_umot, idx_hdr, idx_hdr_prev, cell_start, ipts, ipts2, ihsv, icount, dbg_idx, dbg_d2, d_trans, row_table, result_box, ref_pts, alias_a, alias_q, alias_hl, oct_hdr, oct_nodes, oct_next, cd_hdr, cd_nodes, cd_out;
  CandListStore lists;
  int oct_node_cap = 0;
  // change detector (SURVEY 8 f-4; PCL ctor defaults, off in the reference): host-driven, one read-back per test
  bool use_cd = false;
  int cd_interval = 10, cd_filter = 10, change_counter = 0, cd_tests = 0, cd_last_found = -1, cd_node_cap = 0, cd_resets = 0;
  double cd_res = 0.01;
  int lists_smem = 0;   // dynamic shared memory of weight_lists_kernel (bytes)
  int tbl_size = 0;
  int n_slots = 0;
  int chunks = 1, chunk_len = 0;

  // pft_compute_batch: every tracker of a batch runs on a stream of its own, forked from / joined to the context stream
  cudaStream_t aux_stream = nullptr;  // mark + collect run beside the point index build
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  cudaStream_t batch_stream = nullptr;
  cudaEvent_t batch_done = nullptr;
  bool batch_active = false;

  int slice_cap() const { return (n_cap + nranks - 1) / nranks; }
  cudaStream_t run_stream() const { return batch_active ? batch_stream : ctx->stream; }
};

namespace {

void invalidate_graph(pft_tracker* t) { t->config_version++; }

// timing mode only: an event on the stream after the kernel just launched
void stage_mark(pft_tracker* t, const char* name) {
  if (!t->timing) return;
  if ((int)t->ev_k.size() <= t->n_ev_k) {
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return;
    t->ev_k.push_back(e);
    t->ev_k_name.push_back(name);
  }
  t->ev_k_name[t->n_ev_k] = name;
  cudaEventRecord(t->ev_k[t->n_ev_k++], t->run_stream());
}

void release_all(pft_tracker* t) {
  DevBuf* bufs[] = {&t->st, &t->parts[0], &t->parts[1], &t->mats, &t->slot_aabb, &t->model, &t->model_perm, &t->model_tmp, &t->sort_keys, &t->sort_idx,
                    &t->bbox, &t->raw, &t->partial, &t->cdf, &t->cdf_total, &t->ancestors, &t->bin_keys, &t->tbl_rep, &t->tbl_min, &t->slot_of, &t->klb,
                    &t->d_usel, &t->d_normals, &t->d_umot, &t->idx_hdr, &t->idx_hdr_prev, &t->cell_start, &t->ipts, &t->ipts2, &t->ihsv, &t->icount, &t->dbg_idx,
                    &t->dbg_d2, &t->d_trans, &t->row_table, &t->result_box, &t->ref_pts, &t->alias_a, &t->alias_q, &t->alias_hl, &t->oct_hdr, &t->oct_nodes, &t->oct_next, &t->cd_hdr, &t->cd_nodes, &t->cd_out};
  for (auto* b : bufs) b->release();
  t->lists.release();
}

NoiseParams make_noise(const pft_tracker* t, const double* mean, const double* cov) {
  NoiseParams np;
  for (int d = 0; d < 6; ++d) { np.mean[d] = mean[d]; np.sigma[d] = sqrt(cov[d]); }
  const float scale_factor = 0.2862f;
  for (int d = 0; d < 3; ++d) np.sigma_q[d] = sqrt((double)scale_factor * cov[3 + d]);
  np.quat_mode = t->quat_sample;
  return np;
}

// KLDAdaptiveParticleFilterTracker::calcKLBound / normalQuantile (SURVEY A.7): evaluated on the host in
// IEEE double once per configuration and tabulated for k = 0..n_max.
double normal_quantile(double u) {
  static const double a[9] = {1.24818987e-4, -1.075204047e-3, 5.198775019e-3, -0.019198292004, 0.059054035642,
                              -0.151968751364, 0.319152932694, -0.5319230073, 0.797884560593};
  static const double b[15] = {-4.5255659e-5, 1.5252929e-4, -1.9538132e-5, -6.76904986e-4, 1.390604284e-3,
                               -7.9462082e-4, -2.034254874e-3, 6.549791214e-3, -0.010557625006, 0.011630447319,
                               -9.279453341e-3, 5.353579108e-3, -2.141268741e-3, 5.35310549e-4, 0.999936657524};
  if (u == 0.) return 0.5;
  double y = u / 2.0, z;
  if (y < -3.) return 0.0;
  if (y > 3.) return 1.0;
  if (y < 0.0) y = -y;
  if (y < 1.0) {
    const double w = y * y;
    z = a[0];
    for (int i = 1; i < 9; i++) z = z * w + a[i];
    z *= (y * 2.0);
  } else {
    y -= 2.0;
    z = b[0];
    for (int i = 1; i < 15; i++) z = z * y + b[i];
  }
  return u < 0.0 ? (1.0 - z) / 2.0 : (1.0 + z) / 2.0;
}
double kl_bound(int k, double delta, double eps) {
  const double z = normal_quantile(delta);
  const double chi = 1.0 - 2.0 / (9.0 * (k - 1)) + sqrt(2.0 / (9.0 * (k - 1))) * z;
  return ((k - 1.0) / (2.0 * eps)) * chi * chi * chi;
}

constexpr long long kMarkCountMaxQueries = 16ll << 20;  // up to this many (particle, model point) pairs cand_mark_kernel counts the queries of every cell
constexpr int kClusterMinParticles = 4096;  // above this capacity the O(N) replicated stages run as a cluster of kClusterCtas CTAs
// CTA size of weight_lists_kernel (one CTA per SM): 96 registers per thread, no spills; large query sets (measured on 100 000
// particles: -4 %) trade 72 registers and a few spilled values for 28 warps per SM
constexpr int kListThreads = 640;
constexpr int kListThreadsBig = 896;
constexpr long long kListBigQueries = 48ll << 20;   // (particle, model point) pairs per weight() from which the large variant runs
constexpr long long kDynItemsPerWarp = 5;           // items per warp from which they are handed out dynamically (measured: 10k-25k particles -7 %)
// choose_chunks: model chunks per particle for ~kItemsPerWarp items per warp of kChunkWarpsPerSm warps per SM (the
// chunking fixes the order of the fp64 sums of a weight)
constexpr int kItemsPerWarp = 6;
constexpr int kChunkWarpsPerSm = 24;
constexpr float kIndexDilate = 0.03f;  // margin (m) of the index around the crop box when the lists are on and a compute() has further weight() calls
constexpr int kListRatio = 2;          // the lists are built when this rank's queries outnumber the fine cells of the crop box by this factor

// The O(N) replicated stages (cdf_kernel, normalize_kernel, update_kernel) run as one CTA, above kClusterMinParticles
// as one cluster of kClusterCtas CTAs
template <typename... P, typename... A>
void launch_replicated(const pft_tracker* t, void (*one)(P...), void (*cluster)(P...), A... args) {
  if (t->n_cap > kClusterMinParticles) cluster<<<kClusterCtas, 1024, 0, t->run_stream()>>>(args...);
  else one<<<1, 1024, 0, t->run_stream()>>>(args...);
}

// Row table of the nearest-neighbour search: the (dy,dz) offsets within kRT cells sorted by the lower bound
// gap(dy)^2 + gap(dz)^2 of their distance (gap(d) = max(|d|-1, 0)), nearer rows first.
int upload_row_table(pft_tracker* t) {
  std::vector<RowEntry> tab;
  tab.reserve(kRows);
  for (int dz = -kRT; dz <= kRT; ++dz)
    for (int dy = -kRT; dy <= kRT; ++dy) {
      const int gy = std::max(std::abs(dy) - 1, 0), gz = std::max(std::abs(dz) - 1, 0);
      tab.push_back(RowEntry{(signed char)dy, (signed char)dz, (unsigned short)(gy * gy + gz * gz)});
    }
  std::stable_sort(tab.begin(), tab.end(), [](const RowEntry& a, const RowEntry& b) {
    if (a.lb2 != b.lb2) return a.lb2 < b.lb2;
    return (a.dy * a.dy + a.dz * a.dz) < (b.dy * b.dy + b.dz * b.dz);  // among equal bounds: the row through the query cell first
  });
  int rc = t->row_table.reserve(tab.size() * sizeof(RowEntry));
  if (rc) return rc;
  PFT_CUDA_TRY(cudaMemcpyAsync(t->row_table.p, tab.data(), tab.size() * sizeof(RowEntry), cudaMemcpyHostToDevice, t->run_stream()));
  PFT_CUDA_TRY(cudaStreamSynchronize(t->run_stream()));
  // the weight kernel stages the scene index in shared memory: ask for everything the SM has
  int dev = t->ctx->device, max_optin = 0;
  PFT_CUDA_TRY(cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  cudaFuncAttributes fa;
  PFT_CUDA_TRY(cudaFuncGetAttributes(&fa, weight_lists_kernel<true, kListThreads, true>));
  int dyn_l = (max_optin - (int)fa.sharedSizeBytes - 1024) & ~15;
  if (dyn_l < 0) dyn_l = 0;
  PFT_CUDA_TRY(cudaFuncSetAttribute(weight_lists_kernel<true, kListThreads, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn_l));
  PFT_CUDA_TRY(cudaFuncSetAttribute(weight_lists_kernel<true, kListThreads, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn_l));
  PFT_CUDA_TRY(cudaFuncSetAttribute(weight_lists_kernel<false, kListThreads, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn_l));
  PFT_CUDA_TRY(cudaFuncSetAttribute(weight_lists_kernel<false, kListThreads, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn_l));
  PFT_CUDA_TRY(cudaFuncSetAttribute(weight_lists_kernel<true, kListThreadsBig, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn_l));
  PFT_CUDA_TRY(cudaFuncSetAttribute(weight_lists_kernel<false, kListThreadsBig, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn_l));
  t->lists_smem = dyn_l;
  if (t->list_max_cells / 8 + 64 > max_optin - 2048) t->list_max_cells = (max_optin - 4096) * 8;  // the mark kernel keeps one bit per fine cell in shared memory
  PFT_CUDA_TRY(cudaFuncSetAttribute(cand_mark_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, t->list_max_cells / 8 + 64));
  PFT_CUDA_TRY(cudaFuncSetAttribute(cand_mark_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, t->list_max_cells / 8 + 64));
  return PFT_OK;
}

int upload_kl_table(pft_tracker* t);

int wanted_cap(const pft_tracker* t) { return t->kld ? std::max(t->max_particle_num, t->particle_num) : t->particle_num; }

// (Re)allocate every particle-count dependent buffer.  Existing particles survive a capacity change.
int ensure_particle_buffers(pft_tracker* t) {
  const int cap = std::max(wanted_cap(t), t->n_cap);  // grow only: a smaller setParticleNum keeps the old set to draw from
  if (cap <= 0) { set_last_error("particle count is zero: call setParticleNum / setMaximumParticleNum first"); return PFT_ERR_STATE; }
  cudaStream_t s = t->run_stream();
  int rc;
  if (!t->st.p) {
    if ((rc = t->st.reserve(sizeof(TrackerState)))) return rc;
    PFT_CUDA_TRY(cudaMemsetAsync(t->st.p, 0, sizeof(TrackerState), s));
    DevParticle one{0.f, 0.f, 0.f, 1.f, 0.f, 0.f, 0.f, 0.f};
    PFT_CUDA_TRY(cudaMemcpyAsync(&t->st.as<TrackerState>()->rep, &one, sizeof(one), cudaMemcpyHostToDevice, s));
    PFT_CUDA_TRY(cudaMemcpyAsync(&t->st.as<TrackerState>()->motion, &one, sizeof(one), cudaMemcpyHostToDevice, s));
    PFT_CUDA_TRY(cudaStreamSynchronize(s));
    if ((rc = t->cdf_total.reserve(sizeof(unsigned long long)))) return rc;
    if ((rc = t->idx_hdr.reserve(sizeof(IndexHeader)))) return rc;
    if ((rc = t->idx_hdr_prev.reserve(sizeof(IndexHeader)))) return rc;
    PFT_CUDA_TRY(cudaMemsetAsync(t->idx_hdr.p, 0, sizeof(IndexHeader), s));
    PFT_CUDA_TRY(cudaMemsetAsync(t->idx_hdr_prev.p, 0, sizeof(IndexHeader), s));
    PFT_CUDA_TRY(cudaStreamSynchronize(s));
    if ((rc = t->d_trans.reserve(12 * sizeof(float)))) return rc;
    if ((rc = t->cell_start.reserve(((size_t)t->max_cells + 16) * sizeof(int)))) return rc;
    if ((rc = t->icount.reserve(((size_t)t->max_cells + 16) * sizeof(int)))) return rc;
    if ((rc = upload_row_table(t))) return rc;
    if (t->list_max_cells > 0 && (rc = t->lists.reserve(t->list_max_cells))) return rc;
  }
  if (cap == t->n_cap) return PFT_OK;
  if (t->peer_local) {
    set_last_error("the particle capacity (%d -> %d) cannot change once the peer window is exported", t->n_cap, cap);
    return PFT_ERR_STATE;
  }
  invalidate_graph(t);
  PFT_CUDA_TRY(cudaStreamSynchronize(s));
  const int old_cap = t->n_cap;
  // particles: keep the live set
  DevBuf np0, np1;
  if ((rc = np0.reserve((size_t)cap * sizeof(DevParticle)))) return rc;
  if ((rc = np1.reserve((size_t)cap * sizeof(DevParticle)))) return rc;
  if (old_cap > 0 && t->has_particles) {
    PFT_CUDA_TRY(cudaMemcpyAsync(np0.p, t->parts[t->cur].p, (size_t)std::min(cap, old_cap) * sizeof(DevParticle), cudaMemcpyDeviceToDevice, s));
    PFT_CUDA_TRY(cudaStreamSynchronize(s));
  }
  t->parts[0].release(); t->parts[1].release();
  t->parts[0] = np0; t->parts[1] = np1; t->cur = 0;
  t->n_cap = cap;
  t->n_slots = cap;
  const int slice = t->slice_cap();
  if ((rc = t->mats.reserve((size_t)cap * 12 * sizeof(float)))) return rc;
  t->slot_aabb.release();
  if ((rc = t->slot_aabb.reserve((size_t)cap * 6 * sizeof(float)))) return rc;
  {
    std::vector<float> init((size_t)cap * 6);
    for (int i = 0; i < cap; ++i) { for (int d = 0; d < 3; ++d) { init[6 * i + d] = FLT_MAX; init[6 * i + 3 + d] = -FLT_MAX; } }
    PFT_CUDA_TRY(cudaMemcpyAsync(t->slot_aabb.p, init.data(), init.size() * sizeof(float), cudaMemcpyHostToDevice, s));
    PFT_CUDA_TRY(cudaStreamSynchronize(s));  // (`init` goes out of scope; the work streams do not synchronise with the legacy default stream)
  }
  if ((rc = t->raw.reserve((size_t)slice * t->nranks * sizeof(float)))) return rc;
  PFT_CUDA_TRY(cudaMemsetAsync(t->raw.p, 0, (size_t)slice * t->nranks * sizeof(float), s));
  if ((rc = t->cdf.reserve((size_t)cap * sizeof(unsigned long long)))) return rc;
  if ((rc = t->ancestors.reserve((size_t)cap * sizeof(int)))) return rc;
  PFT_CUDA_TRY(cudaMemsetAsync(t->ancestors.p, 0xff, (size_t)cap * sizeof(int), s));
  PFT_CUDA_TRY(cudaStreamSynchronize(s));
  if (t->kld) {
    if ((rc = t->bin_keys.reserve((size_t)cap * 6 * sizeof(int)))) return rc;
    int ts = 1024;
    while (ts < 2 * cap) ts <<= 1;
    t->tbl_size = ts;
    if ((rc = t->tbl_rep.reserve((size_t)ts * sizeof(int)))) return rc;
    if ((rc = t->tbl_min.reserve((size_t)ts * sizeof(int)))) return rc;
    if ((rc = t->slot_of.reserve((size_t)cap * sizeof(int)))) return rc;
    if ((rc = t->klb.reserve((size_t)(cap + 2) * sizeof(double)))) return rc;
    if ((rc = upload_kl_table(t))) return rc;  // reserve() dropped the old table: the stop rule reads k up to the new capacity
  }
  return PFT_OK;
}

int upload_kl_table(pft_tracker* t) {
  if (!t->kld) return PFT_OK;
  const int n = t->n_cap + 2;
  std::vector<double> tab(n, 0.0);
  for (int k = 2; k < n; ++k) tab[k] = kl_bound(k, t->delta, t->epsilon);
  PFT_CUDA_TRY(cudaMemcpyAsync(t->klb.p, tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice, t->run_stream()));
  PFT_CUDA_TRY(cudaStreamSynchronize(t->run_stream()));
  return PFT_OK;
}

int ensure_draw_buffers(pft_tracker* t, int slots, int stride) {
  const size_t n = (size_t)slots * stride;
  int rc;
  if ((rc = t->d_usel.reserve(n * sizeof(float)))) return rc;
  if ((rc = t->d_normals.reserve(n * 6 * sizeof(float)))) return rc;
  if ((rc = t->d_umot.reserve(n * sizeof(float)))) return rc;
  return PFT_OK;
}

// Buffers of `count` generated draws (slot 0).
int reserve_generated_draws(pft_tracker* t, int count) {
  if (t->draw_cap >= count) return PFT_OK;
  int rc = ensure_draw_buffers(t, 1, count);
  if (rc) return rc;
  t->draw_cap = count;
  invalidate_graph(t);
  return PFT_OK;
}

// Draw arrays of one resample slot: injected (slot-indexed) or generated on the device into slot 0.
int prepare_draws(pft_tracker* t, int slot, int count, const float** usel, const float** normals, const float** umot) {
  cudaStream_t s = t->run_stream();
  if (t->inj_stride > 0) {
    if (slot >= t->inj_slots || count > t->inj_stride) {
      set_last_error("injected draws cover %d slots x %d, need slot %d x %d", t->inj_slots, t->inj_stride, slot, count);
      return PFT_ERR_STATE;
    }
    *usel = t->d_usel.as<float>() + (size_t)slot * t->inj_stride;
    *normals = t->d_normals.as<float>() + (size_t)slot * t->inj_stride * 6;
    *umot = t->d_umot.as<float>() + (size_t)slot * t->inj_stride;
    return PFT_OK;
  }
  int rc = reserve_generated_draws(t, count);
  if (rc) return rc;
  draws_kernel<<<blocks_for(count, 256, t->ctx->sm_count * 4), 256, 0, s>>>(t->st.as<TrackerState>(), t->d_usel.as<float>(), t->d_normals.as<float>(),
                                                                        t->d_umot.as<float>(), count, t->seed);
  PFT_LAUNCH_CHECK();
  stage_mark(t, "draws_kernel");
  *usel = t->d_usel.as<float>(); *normals = t->d_normals.as<float>(); *umot = t->d_umot.as<float>();
  return PFT_OK;
}

int ensure_index_buffers(pft_tracker* t) {
  const size_t cap = std::max<size_t>(t->scene ? t->scene->capacity : 0, 1);
  if (cap <= t->scene_cap) return PFT_OK;
  invalidate_graph(t);
  PFT_CUDA_TRY(cudaStreamSynchronize(t->run_stream()));
  int rc;
  if ((rc = t->ipts.reserve((cap + 4) * sizeof(float4)))) return rc;
  if ((rc = t->ipts2.reserve((cap + 4) * sizeof(float4)))) return rc;
  if ((rc = t->ihsv.reserve((cap + 4) * sizeof(unsigned int)))) return rc;
  t->scene_cap = cap;
  return PFT_OK;
}

// One work item of the weight kernel = one warp x (particle, chunk of the model).  Enough items for ~6 per
// warp of the persistent grid keeps the tail short; a chunk is a multiple of 32 points (one per lane).
void choose_chunks(pft_tracker* t) {
  const int n_expected = std::max(1, (t->particle_num > 0 ? t->particle_num : t->n_cap) / t->nranks);
  const int total_warps = t->ctx->sm_count * kChunkWarpsPerSm;  // (chunking only matters for small sets: the static split)
  const int target_items = total_warps * kItemsPerWarp;
  const int max_chunks = std::max(1, (t->M + 63) / 64);
  int chunks = (target_items + n_expected - 1) / n_expected;
  chunks = std::min(std::max(chunks, 1), std::min(max_chunks, 256));
  int len = (t->M + chunks - 1) / chunks;
  len = ((len + 31) / 32) * 32;
  if (len < 32) len = 32;
  chunks = std::max(1, (t->M + len - 1) / len);
  if (chunks != t->chunks || len != t->chunk_len) invalidate_graph(t);
  t->chunks = chunks;
  t->chunk_len = len;
}

CoherenceParams make_coherence(const pft_tracker* t) {
  CoherenceParams c;
  c.max_d2 = t->max_dist * t->max_dist;
  c.dist_w = t->dist_w; c.hsv_w = t->hsv_w;
  c.h_w = (float)t->h_w; c.s_w = (float)t->s_w; c.v_w = (float)t->v_w;
  c.r_max = (float)std::min(t->max_dist, 1.0e18);
  c.use_dist = t->use_dist; c.use_hsv = t->use_hsv;
  return c;
}

// ---- stages -------------------------------------------------------------------------------------
int stage_init_particles(pft_tracker* t) {
  int rc = ensure_particle_buffers(t);
  if (rc) return rc;
  if (t->particle_num <= 0) { set_last_error("setParticleNum was not called"); return PFT_ERR_STATE; }
  if ((rc = upload_kl_table(t))) return rc;
  cudaStream_t s = t->run_stream();
  PFT_CUDA_TRY(cudaMemcpyAsync(t->d_trans.p, t->trans, sizeof(t->trans), cudaMemcpyHostToDevice, s));
  const float *usel, *normals, *umot;
  if ((rc = prepare_draws(t, 0, t->particle_num, &usel, &normals, &umot))) return rc;
  const NoiseParams np = make_noise(t, t->init_mean, t->init_cov);
  init_particles_kernel<<<blocks_for(t->particle_num, 128, 1 << 20), 128, 0, s>>>(t->st.as<TrackerState>(), t->parts[t->cur].as<DevParticle>(),
                                                                                   t->particle_num, t->d_trans.as<float>(), np, normals);
  PFT_LAUNCH_CHECK();
  stage_mark(t, "init_particles_kernel");
  t->has_particles = true;
  return PFT_OK;
}

int stage_resample(pft_tracker* t, int slot) {
  if (!t->has_particles) { set_last_error("resample before particles exist"); return PFT_ERR_STATE; }
  if (!t->scene) { set_last_error("resample needs an input cloud (setInputCloud)"); return PFT_ERR_STATE; }
  if (t->kld && t->max_particle_num <= 0) { set_last_error("KLD tracker: setMaximumParticleNum was not called"); return PFT_ERR_STATE; }
  cudaStream_t s = t->run_stream();
  const int count = t->kld ? t->max_particle_num : t->particle_num;
  const float *usel = nullptr, *normals = nullptr, *umot = nullptr;  // null: resample_kernel generates its draws inline (Philox)
  int rc = PFT_OK;
  if (t->inj_stride > 0 && (rc = prepare_draws(t, slot, count, &usel, &normals, &umot))) return rc;
  TrackerState* st = t->st.as<TrackerState>();
  const DevParticle* old_parts = t->parts[t->cur].as<DevParticle>();
  DevParticle* new_parts = t->parts[t->cur ^ 1].as<DevParticle>();
  launch_replicated(t, cdf_kernel<1>, cdf_kernel<kClusterCtas>, st, old_parts, t->cdf.as<unsigned long long>(), t->cdf_total.as<unsigned long long>(),
                    t->tbl_rep.as<int>(), t->tbl_min.as<int>(), t->kld ? t->tbl_size : 0, t->kld ? 0 : t->particle_num, t->scene->d_hdr());
  PFT_LAUNCH_CHECK();
  stage_mark(t, "cdf_kernel");
  if (t->sampler == PFT_SAMPLER_ALIAS_PCL) {  // (buffers sized by prepare_compute: nothing is allocated inside a graph capture)
    alias_table_kernel<<<1, 32, 0, s>>>(st, old_parts, t->alias_a.as<int>(), t->alias_q.as<double>(), t->alias_hl.as<int>());
    PFT_LAUNCH_CHECK();
    stage_mark(t, "alias_table_kernel");
  }
  ResampleArgs a;
  a.alias_a = t->alias_a.as<int>(); a.alias_q = t->alias_q.as<double>();
  a.st = st; a.old_parts = old_parts; a.new_parts = new_parts;
  a.cdf = t->cdf.as<unsigned long long>(); a.cdf_total = t->cdf_total.as<unsigned long long>();
  a.u_select = usel; a.normals = normals; a.u_motion = umot; a.seed = t->seed;
  a.scene_hdr = t->scene->d_hdr();
  a.ancestors = t->ancestors.as<int>(); a.bin_keys = t->bin_keys.as<int>();
  const double zero[6] = {0, 0, 0, 0, 0, 0};
  a.np = make_noise(t, zero, t->step_cov);
  a.motion_ratio = t->motion_ratio;
  for (int d = 0; d < 6; ++d) a.bin_size[d] = t->bin_size[d];
  a.kld = t->kld ? 1 : 0; a.n_max = t->max_particle_num; a.sampler = t->sampler; a.n_target = t->particle_num;
  resample_kernel<<<blocks_for(count, 128, t->ctx->sm_count * 16), 128, 0, s>>>(a);
  PFT_LAUNCH_CHECK();
  stage_mark(t, "resample_kernel");
  if (t->kld) {
    kld_insert_kernel<<<blocks_for(count, 128, t->ctx->sm_count * 16), 128, 0, s>>>(t->bin_keys.as<int>(), t->max_particle_num, t->tbl_rep.as<int>(),
                                                                                    t->tbl_min.as<int>(), t->slot_of.as<int>(), (unsigned)(t->tbl_size - 1));
    PFT_LAUNCH_CHECK();
    stage_mark(t, "kld_insert_kernel");
    kld_stop_kernel<<<1, 1024, 0, s>>>(st, t->tbl_min.as<int>(), t->slot_of.as<int>(), t->klb.as<double>(), t->max_particle_num, t->scene->d_hdr());
    PFT_LAUNCH_CHECK();
    stage_mark(t, "kld_stop_kernel");
  }
  t->cur ^= 1;
  return PFT_OK;
}

int check_weight_ready(pft_tracker* t) {
  if (!t->has_particles) { set_last_error("weight before particles exist"); return PFT_ERR_STATE; }
  if (!t->scene) { set_last_error("weight needs an input cloud (setInputCloud)"); return PFT_ERR_STATE; }
  if (t->M <= 0) { set_last_error("weight needs a reference cloud (setReferenceCloud)"); return PFT_ERR_STATE; }
  return ensure_index_buffers(t);
}

// weight(), part 1: per-particle transforms + this rank's share of the crop box
// (transformPointCloud per slot + calcBoundingBox)
int weight_phase_box(pft_tracker* t) {
  int rc = check_weight_ready(t);
  if (rc) return rc;
  cudaStream_t s = t->run_stream();
  const int sm = t->ctx->sm_count;
  TrackerState* st = t->st.as<TrackerState>();
  DevParticle* parts = t->parts[t->cur].as<DevParticle>();
  matrices_kernel<<<blocks_for(t->n_cap, 128, sm * 8), 128, 0, s>>>(st, parts, t->mats.as<float>());
  PFT_LAUNCH_CHECK();
  stage_mark(t, "matrices_kernel");
  if (t->n_slots <= sm * 32) {
    aabb_kernel<4><<<std::min(t->n_slots, sm * 16), 128, 0, s>>>(st, t->model.as<float4>(), t->M, t->mats.as<float>(), t->slot_aabb.as<float>(), t->n_slots,
                                                                t->nranks, t->rank, t->peers, t->peer_mode ? 1 : 0);
  } else {
    aabb_kernel<1><<<std::min(t->n_slots, sm * 64), 32, 0, s>>>(st, t->model.as<float4>(), t->M, t->mats.as<float>(), t->slot_aabb.as<float>(), t->n_slots,
                                                               t->nranks, t->rank, t->peers, t->peer_mode ? 1 : 0);
  }
  PFT_LAUNCH_CHECK();
  stage_mark(t, "aabb_kernel");
  return PFT_OK;
}

// Who moves the crop box and the raw weights of a sharded weight() between the ranks: in NVLink peer mode the kernels
// themselves (aabb_kernel, normalize_kernel); with a communicator NCCL; with manual shards (pft_tracker_set_shard) the
// caller.  With one rank or in peer mode normalize_kernel sums the raw weights from the partials; otherwise
// raw_weights_kernel first writes this rank's slice of the gathered buffer.
bool nccl_exchange(const pft_tracker* t) { return t->comm && !t->peer_mode; }
bool normalize_sums_partials(const pft_tracker* t) { return t->nranks == 1 || t->peer_mode; }

// crop box exchange over NCCL: union over ranks
int weight_comm_box(pft_tracker* t) {
  cudaStream_t s = t->run_stream();
  TrackerState* st = t->st.as<TrackerState>();
  PFT_NCCL_TRY(g_nccl.GroupStart());
  PFT_NCCL_TRY(g_nccl.AllReduce(st->aabb, st->aabb, 3, kNcclFloat, kNcclMin, t->comm, s));
  PFT_NCCL_TRY(g_nccl.AllReduce(st->aabb + 3, st->aabb + 3, 3, kNcclFloat, kNcclMax, t->comm, s));
  PFT_NCCL_TRY(g_nccl.GroupEnd());
  return PFT_OK;
}

// The launch of the nearest-neighbour lookup, bracketed in timing mode by the pair of events pft_tracker_get_timing reads
template <typename Launch>
int timed_lookup(pft_tracker* t, const char* name, Launch launch) {
  cudaStream_t s = t->run_stream();
  if (t->timing) {
    while ((int)t->ev_w.size() < 2 * (t->n_ev_used + 1)) { cudaEvent_t e; PFT_CUDA_TRY(cudaEventCreate(&e)); t->ev_w.push_back(e); }
    PFT_CUDA_TRY(cudaEventRecord(t->ev_w[2 * t->n_ev_used], s));
  }
  launch();
  PFT_LAUNCH_CHECK();
  stage_mark(t, name);
  if (t->timing) { PFT_CUDA_TRY(cudaEventRecord(t->ev_w[2 * t->n_ev_used + 1], s)); t->n_ev_used++; }
  return PFT_OK;
}

// Per-chunk partials -> this rank's slice of the gathered raw weights
int launch_raw_weights(pft_tracker* t) {
  const int local_cap = t->slice_cap();
  raw_weights_kernel<<<blocks_for(local_cap, 256, t->ctx->sm_count * 4), 256, 0, t->run_stream()>>>(
      t->st.as<TrackerState>(), t->partial.as<double>(), t->chunks, t->n_cap, t->raw.as<float>(), local_cap, t->nranks, t->rank);
  PFT_LAUNCH_CHECK();
  stage_mark(t, "raw_weights_kernel");
  return PFT_OK;
}

// Parity mode PFT_NN_PCL_APPROX (see octree_build_kernel): the octree of the cropped cloud and the greedy search
int weight_eval_pcl_approx(pft_tracker* t) {
  cudaStream_t s = t->run_stream();
  const int sm = t->ctx->sm_count;
  TrackerState* st = t->st.as<TrackerState>();
  const pft_cloud* in = t->scene;
  octree_build_kernel<<<1, 32, 0, s>>>(in->d_pts(), in->d_hdr(), t->idx_hdr.as<IndexHeader>(), t->search_res, t->oct_nodes.as<OctNodeD>(), t->oct_node_cap,
                                       t->oct_next.as<int>(), t->oct_hdr.as<OctHeaderD>());
  PFT_LAUNCH_CHECK();
  stage_mark(t, "octree_build_kernel");
  WeightApproxArgs w;
  w.st = st; w.oct = t->oct_hdr.as<OctHeaderD>(); w.nodes = t->oct_nodes.as<OctNodeD>(); w.next = t->oct_next.as<int>();
  w.scene = in->d_pts(); w.model = t->model.as<float4>(); w.model_perm = t->model_perm.as<int>(); w.M = t->M; w.mats = t->mats.as<float>();
  w.partial = t->partial.as<double>(); w.chunks = t->chunks; w.chunk_len = t->chunk_len; w.n_max = t->n_cap; w.nranks = t->nranks; w.rank_id = t->rank;
  w.co = make_coherence(t);
  w.dbg_k = t->debug_nn; w.dbg_idx = t->dbg_idx.as<int>(); w.dbg_d2 = t->dbg_d2.as<float>();
  return timed_lookup(t, "weight_approx_kernel", [&] { weight_approx_kernel<<<sm * 8, 256, 0, s>>>(w); });
}

// crop box -> index header (also what in_crop() reads) + reset of the per-weight() counters
int launch_index_begin(pft_tracker* t, bool reuse_allowed = false) {
  const int sm = t->ctx->sm_count;
  const float inv_leaf = 1.0f / (float)t->search_res;
  // one index per frame (see IndexHeader): with the lists on, the crop box is dilated by kIndexDilate; the later weight()
  // calls of a compute() reuse the index when their crop box fits
  index_begin_kernel<<<sm, 256, 0, t->run_stream()>>>(t->st.as<TrackerState>(), t->idx_hdr.as<IndexHeader>(), t->icount.as<int>(), inv_leaf, t->max_cells,
                                                      t->list_mode ? t->list_max_cells : 0, t->M, t->nranks, t->rank, t->lists.view(), t->list_mode == 2 ? 1 : 0,
                                                      reuse_allowed ? 1 : 0, t->iteration_num > 1 ? kIndexDilate : 0.f, kListRatio, t->idx_hdr_prev.as<IndexHeader>());
  PFT_LAUNCH_CHECK();
  stage_mark(t, "index_begin_kernel");
  return PFT_OK;
}

// weight(), part 2: cropInputPointCloud + search index rebuild (K2), coherence of this rank's particles (K3)
int weight_phase_eval(pft_tracker* t, bool reuse_allowed = false) {
  int rc = check_weight_ready(t);
  if (rc) return rc;
  cudaStream_t s = t->run_stream();
  const int sm = t->ctx->sm_count;
  TrackerState* st = t->st.as<TrackerState>();
  const pft_cloud* in = t->scene;
  const int ncap_scene = (int)std::max<size_t>(in->capacity, 1);
  IndexHeader* hdr = t->idx_hdr.as<IndexHeader>();
  const float inv_leaf = 1.0f / (float)t->search_res;
  const int gscene = blocks_for(ncap_scene, 256, sm * 4);
  // candidate lists for the exact search (the index header may still turn them off for this crop)
  const bool lists = t->list_max_cells > 0 && t->list_mode && t->nn_mode == PFT_NN_EXACT;
  const CandLists L = t->lists.view();
  if ((rc = launch_index_begin(t, reuse_allowed && lists))) return rc;
  if (lists) {
    // which fine cells the queries fall into (mark + collect) does not depend on the point index being built (count +
    // scan + scatter): the two chains of small kernels run side by side on two streams and join before the list build
    cudaStream_t sa = t->aux_stream;
    PFT_CUDA_TRY(cudaEventRecord(t->ev_fork, s));
    PFT_CUDA_TRY(cudaStreamWaitEvent(sa, t->ev_fork, 0));
    // small query sets: exact query counts per cell (cells with few queries get one list instead of eight octant lists)
    const long long n_queries = (long long)std::max(1, (t->particle_num > 0 ? t->particle_num : t->n_cap) / t->nranks) * t->M;
    const size_t mark_smem = (size_t)(t->list_max_cells / 8 + 64);
    if (n_queries <= kMarkCountMaxQueries) cand_mark_kernel<true><<<sm * 3, 256, mark_smem, sa>>>(st, hdr, t->model.as<float4>(), t->M, t->mats.as<float>(), L, t->nranks, t->rank);
    else cand_mark_kernel<false><<<sm * 3, 256, mark_smem, sa>>>(st, hdr, t->model.as<float4>(), t->M, t->mats.as<float>(), L, t->nranks, t->rank);
    PFT_LAUNCH_CHECK();
    cand_collect_kernel<<<sm * 2, 256, 0, sa>>>(hdr, L);
    PFT_LAUNCH_CHECK();
    PFT_CUDA_TRY(cudaEventRecord(t->ev_join, sa));
  }
  index_count_kernel<<<gscene, 256, 0, s>>>(in->d_pts(), in->d_hdr(), hdr, t->icount.as<int>(), t->ipts2.as<float4>());
  PFT_LAUNCH_CHECK();
  stage_mark(t, "index_count_kernel");
  index_scan_kernel<<<1, 1024, 0, s>>>(hdr, t->icount.as<int>(), t->cell_start.as<int>(), st, t->ipts.as<float4>(), t->ipts2.as<float4>(), t->idx_hdr_prev.as<IndexHeader>());
  PFT_LAUNCH_CHECK();
  stage_mark(t, "index_scan_kernel");
  index_scatter_kernel<<<gscene, 256, 0, s>>>(in->d_pts(), in->d_hdr(), hdr, t->cell_start.as<int>(), t->icount.as<int>(), t->ipts.as<float4>(),
                                              t->ihsv.as<unsigned int>(), t->ipts2.as<float4>());
  PFT_LAUNCH_CHECK();
  stage_mark(t, "index_scatter_kernel");
  if (lists) {
    PFT_CUDA_TRY(cudaStreamWaitEvent(s, t->ev_join, 0));
    stage_mark(t, "cand_mark+collect (beside the index)");
    cand_build_kernel<<<sm * 8, 256, 0, s>>>(hdr, t->cell_start.as<int>(), t->ipts.as<float4>(), t->max_dist * t->max_dist, L);
    PFT_LAUNCH_CHECK();
    stage_mark(t, "cand_build_kernel");
    // cells far from the surface (long lists): pairwise pruning, one thread block each; most of them join the octant pass
    // (measured and dropped: the far pass on a second stream beside the octant pass of the other cells -- it then takes
    // longer than the octant pass it competes with, and the frame does not get shorter)
    cand_build_far_kernel<<<sm * 4, 256, 0, s>>>(hdr, t->cell_start.as<int>(), t->ipts.as<float4>(), t->max_dist * t->max_dist, L);
    PFT_LAUNCH_CHECK();
    stage_mark(t, "cand_build_far_kernel");
    cand_octant_kernel<<<sm * 8, 256, 0, s>>>(hdr, t->ipts.as<float4>(), t->max_dist * t->max_dist, L);
    PFT_LAUNCH_CHECK();
    stage_mark(t, "cand_octant_kernel");
  }
  if (t->nn_mode == PFT_NN_PCL_APPROX) return weight_eval_pcl_approx(t);
  WeightArgs a;
  a.st = st; a.hdr = hdr; a.pts2 = t->ipts2.as<float4>();
  a.records = L.records; a.pool = L.pool; a.xlists = L.xlists;
  a.cell_start = t->cell_start.as<int>(); a.pts = t->ipts.as<float4>();
  a.hsv = t->ihsv.as<unsigned int>(); a.table = t->row_table.as<RowEntry>(); a.smem_bytes = t->lists_smem;
  a.model = t->model.as<float4>(); a.model_perm = t->model_perm.as<int>(); a.M = t->M;
  a.mats = t->mats.as<float>();
  a.partial = t->partial.as<double>(); a.chunks = t->chunks; a.chunk_len = t->chunk_len; a.n_max = t->n_cap;
  a.nranks = t->nranks; a.rank_id = t->rank;
  a.co = make_coherence(t);
  a.dbg_k = t->debug_nn; a.dbg_idx = t->dbg_idx.as<int>(); a.dbg_d2 = t->dbg_d2.as<float>();
  const int wgrid = sm;  // persistent: one CTA per SM
  // many items per warp (large particle sets): dynamic hand-out; few: static interleaved split (see weight_items)
  const long long n_local = std::max(1, (t->particle_num > 0 ? t->particle_num : t->n_cap) / t->nranks);
  const bool dyn = n_local * t->chunks >= kDynItemsPerWarp * sm * (kListThreads / 32);
  // one launch either way: it runs the row-table search itself when the index header says the lists are off
  return timed_lookup(t, "weight_lists_kernel", [&] {
    if (n_local * t->M >= kListBigQueries) {
      if (t->use_hsv) weight_lists_kernel<true, kListThreadsBig, true><<<wgrid, kListThreadsBig, t->lists_smem, s>>>(a);
      else weight_lists_kernel<false, kListThreadsBig, true><<<wgrid, kListThreadsBig, t->lists_smem, s>>>(a);
    } else if (t->use_hsv) {
      if (dyn) weight_lists_kernel<true, kListThreads, true><<<wgrid, kListThreads, t->lists_smem, s>>>(a);
      else weight_lists_kernel<true, kListThreads, false><<<wgrid, kListThreads, t->lists_smem, s>>>(a);
    } else {
      if (dyn) weight_lists_kernel<false, kListThreads, true><<<wgrid, kListThreads, t->lists_smem, s>>>(a);
      else weight_lists_kernel<false, kListThreads, false><<<wgrid, kListThreads, t->lists_smem, s>>>(a);
    }
  });
}

// raw weight exchange over NCCL: every rank ends up with all raw weights
int weight_comm_raw(pft_tracker* t) {
  const int local_cap = t->slice_cap();
  PFT_NCCL_TRY(g_nccl.AllGather(t->raw.as<float>() + (size_t)t->rank * local_cap, t->raw.as<float>(), (size_t)local_cap, kNcclFloat, t->comm,
                                t->run_stream()));
  return PFT_OK;
}

// weight(), part 3: normalizeWeight (replicated)
int weight_phase_normalize(pft_tracker* t, bool fuse_update = false) {
  int rc = check_weight_ready(t);
  if (rc) return rc;
  launch_replicated(t, normalize_kernel<1>, normalize_kernel<kClusterCtas>, t->st.as<TrackerState>(), t->parts[t->cur].as<DevParticle>(), t->raw.as<float>(),
                    t->alpha, t->nranks, t->slice_cap(), t->scene->d_hdr(), t->M, normalize_sums_partials(t) ? t->partial.as<double>() : nullptr,
                    t->chunks, t->n_cap, fuse_update ? 1 : 0, t->peers);
  PFT_LAUNCH_CHECK();
  stage_mark(t, "normalize_kernel");
  t->changed = true;  // change detector is off upstream => changed_ = true after every weight()
  return PFT_OK;
}

// ParticleFilterTracker::testChangeDetection on the cropped cloud (SURVEY 8 f-4): host-driven, the answer is read
// back before weight() goes on.  Every rank of a sharded tracker sees the same crop and takes the same decision.
int change_detection_test(pft_tracker* t, bool* change) {
  int rc = launch_index_begin(t);  // the crop predicate of this weight()
  if (rc) return rc;
  cudaStream_t s = t->run_stream();
  for (int attempt = 0; attempt < 2; ++attempt) {
    change_detect_kernel<<<1, 32, 0, s>>>(t->scene->d_pts(), t->scene->d_hdr(), t->idx_hdr.as<IndexHeader>(), t->cd_res, t->cd_nodes.as<CdNodeD>(), t->cd_node_cap,
                                          t->cd_hdr.as<CdHeaderD>(), t->cd_filter, t->cd_out.as<int>());
    PFT_LAUNCH_CHECK();
    stage_mark(t, "change_detect_kernel");
    int out[2] = {0, 0};
    PFT_CUDA_TRY(cudaMemcpyAsync(out, t->cd_out.p, sizeof(out), cudaMemcpyDeviceToHost, s));
    PFT_CUDA_TRY(cudaStreamSynchronize(s));
    if (!out[1]) { t->cd_last_found = out[0]; t->cd_tests++; *change = out[0] > 0; return PFT_OK; }
    // node pool exhausted (upstream frees what neither buffer uses, this tree only grows): start a new detector --
    // its first test reports every voxel as new
    PFT_CUDA_TRY(cudaMemsetAsync(t->cd_hdr.p, 0, sizeof(CdHeaderD), s));
    t->cd_resets++;
  }
  set_last_error("change detector: the cropped cloud does not fit the node pool");
  return PFT_ERR_CAPACITY;
}

// weight() when the change detector found nothing new: the coherence is not evaluated, the particles keep their
// weights and normalizeWeight() still runs on them (upstream, impl/particle_filter.hpp weight())
int weight_phase_renormalize(pft_tracker* t) {
  cudaStream_t s = t->run_stream();
  TrackerState* st = t->st.as<TrackerState>();
  DevParticle* parts = t->parts[t->cur].as<DevParticle>();
  weights_to_raw_kernel<<<blocks_for(t->n_cap, 256, t->ctx->sm_count * 4), 256, 0, s>>>(st, parts, t->raw.as<float>(), t->nranks, t->slice_cap());
  PFT_LAUNCH_CHECK();
  stage_mark(t, "weights_to_raw_kernel");
  launch_replicated(t, normalize_kernel<1>, normalize_kernel<kClusterCtas>, st, parts, t->raw.as<float>(), t->alpha, t->nranks, t->slice_cap(),
                    t->scene->d_hdr(), 0, nullptr, t->chunks, t->n_cap, 0, t->peers);
  PFT_LAUNCH_CHECK();
  stage_mark(t, "normalize_kernel");
  t->changed = false;
  return PFT_OK;
}

int stage_weight(pft_tracker* t, bool fuse_update = false, bool reuse_allowed = false) {
  int rc;
  if ((rc = weight_phase_box(t))) return rc;
  if (nccl_exchange(t) && (rc = weight_comm_box(t))) return rc;
  if (t->use_cd && t->nranks > 1) { set_last_error("the change detector is not supported on a sharded tracker"); return PFT_ERR_STATE; }
  if (t->use_cd) {
    // change_counter_ (upstream weight()): a test every `interval` calls; nothing new => the weights are not recomputed
    if (t->change_counter == 0) {
      bool change = true;
      if ((rc = change_detection_test(t, &change))) return rc;
      if (!change) return weight_phase_renormalize(t);
      t->change_counter = t->cd_interval;
    } else {
      --t->change_counter;
    }
  }
  if ((rc = weight_phase_eval(t, reuse_allowed))) return rc;
  if (!normalize_sums_partials(t)) {
    if ((rc = launch_raw_weights(t))) return rc;
    if (nccl_exchange(t) && (rc = weight_comm_raw(t))) return rc;
  }
  return weight_phase_normalize(t, fuse_update);
}

int stage_update(pft_tracker* t) {
  if (!t->has_particles || !t->scene) { set_last_error("update before weight"); return PFT_ERR_STATE; }
  launch_replicated(t, update_kernel<1>, update_kernel<kClusterCtas>, t->st.as<TrackerState>(), t->parts[t->cur].as<DevParticle>(), t->scene->d_hdr());
  PFT_LAUNCH_CHECK();
  stage_mark(t, "update_kernel");
  return PFT_OK;
}

int enqueue_tracking(pft_tracker* t) {
  int rc;
  for (int it = 0; it < t->iteration_num; ++it) {
    if (t->changed && (rc = stage_resample(t, it))) return rc;
    // upstream: update() runs when changed_, which every weight() sets (the change detector is off): it is fused into
    // the normalise launch
    // the first weight() of a compute() builds the scene index of the frame; the later ones reuse it when their crop
    // box fits the (dilated) box it was built from (decided on the device, see index_begin_kernel)
    if ((rc = stage_weight(t, true, it > 0 && !t->use_cd))) return rc;
  }
  return PFT_OK;
}

}  // namespace

// ---- scene replicas: a tracker whose input cloud belongs to another context reads a copy of it on its own context.
// One replica per (destination context, source cloud), shared by every tracker of that context; it is refreshed by one
// fan-out launch on the source stream when the source has been written since (pft_cloud::version), and never otherwise.
// Ordering by events: the push waits until the readers of the previous contents have finished (`read`), the destination
// stream waits for the push (`pushed`).  The storage only grows, so that the trackers' graphs stay valid.
struct SceneReplica {
  pft_context* dst = nullptr;
  unsigned long long src_serial = 0, src_version = 0;  // the source (never reused) and the contents held (0: none yet)
  pft_cloud cloud;                                      // on dst
  cudaEvent_t pushed = nullptr;                         // on the source's device
  cudaEvent_t read = nullptr;                           // on dst's device
  bool read_recorded = false;
};

namespace {

std::mutex g_replica_mu;                // guards g_replicas and the replicas' bookkeeping
std::vector<SceneReplica*> g_replicas;

void release_replica(SceneReplica* r) {
  cudaSetDevice(r->dst->device);
  cudaStreamSynchronize(r->dst->stream);  // (the destination stream waited for every push: nothing is left in flight)
  r->cloud.pts.release();
  r->cloud.hdr.release();
  if (r->read) cudaEventDestroy(r->read);
  if (r->pushed) cudaEventDestroy(r->pushed);
  delete r;
}

template <typename Pred> void release_replicas_if(Pred pred) {
  std::vector<SceneReplica*> gone;
  {
    std::lock_guard<std::mutex> lock(g_replica_mu);
    auto keep = std::stable_partition(g_replicas.begin(), g_replicas.end(), [&](SceneReplica* r) { return !pred(r); });
    gone.assign(keep, g_replicas.end());
    g_replicas.erase(keep, g_replicas.end());
  }
  int dev = 0;
  cudaGetDevice(&dev);
  for (SceneReplica* r : gone) release_replica(r);
  cudaSetDevice(dev);
}

// Lets kernels on src_dev store into memory of dst_dev (the fan-out runs on the source's device).
int enable_peer_access(int src_dev, int dst_dev) {
  if (src_dev == dst_dev) return PFT_OK;
  int can = 0;
  PFT_CUDA_TRY(cudaDeviceCanAccessPeer(&can, src_dev, dst_dev));
  if (!can) { set_last_error("device %d cannot map the memory of device %d (needs NVLink/P2P)", src_dev, dst_dev); return PFT_ERR_COMM; }
  PFT_CUDA_TRY(cudaSetDevice(src_dev));
  cudaError_t e = cudaDeviceEnablePeerAccess(dst_dev, 0);
  if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { set_last_error("cudaDeviceEnablePeerAccess(%d -> %d) -> %s", src_dev, dst_dev, cudaGetErrorString(e)); cudaGetLastError(); return PFT_ERR_COMM; }
  cudaGetLastError();
  return PFT_OK;
}

// Refreshes the replicas `rs` of `src` (all stale, at most kMaxPeers) with one fan-out launch.  Caller holds g_replica_mu.
int push_replicas(const pft_cloud* src, SceneReplica* const* rs, int n) {
  const size_t cap = std::max<size_t>(src->capacity, 1);
  int rc;
  for (int k = 0; k < n; ++k) {
    SceneReplica* r = rs[k];
    PFT_CUDA_TRY(cudaSetDevice(r->dst->device));
    if (cap * sizeof(float4) > r->cloud.pts.bytes && r->pushed) PFT_CUDA_TRY(cudaEventSynchronize(r->pushed));  // (the old storage is freed)
    if ((rc = r->cloud.ensure(cap))) return rc;
    if (!r->read) PFT_CUDA_TRY(cudaEventCreateWithFlags(&r->read, cudaEventDisableTiming));
  }
  PFT_CUDA_TRY(cudaSetDevice(src->ctx->device));
  if ((rc = src->join_upload())) return rc;
  cudaStream_t ss = src->ctx->stream;
  CloudPeerSet ps{};
  ps.nranks = n; ps.rank = -1;
  size_t room = SIZE_MAX;
  for (int k = 0; k < n; ++k) {
    SceneReplica* r = rs[k];
    if (!r->pushed) PFT_CUDA_TRY(cudaEventCreateWithFlags(&r->pushed, cudaEventDisableTiming));
    if (r->read_recorded) PFT_CUDA_TRY(cudaStreamWaitEvent(ss, r->read, 0));
    ps.pts[k] = r->cloud.d_pts(); ps.hdr[k] = r->cloud.d_hdr();
    room = std::min(room, r->cloud.pts.bytes / sizeof(float4));
  }
  const int grid = std::max(1, std::min(src->ctx->sm_count, (int)((cap + 255) / 256)));
  cloud_fanout_kernel<<<grid, 256, 0, ss>>>(src->d_pts(), src->d_hdr(), ps, (int)std::min<size_t>(room, 0x7fffffff));
  PFT_LAUNCH_CHECK();
  for (int k = 0; k < n; ++k) PFT_CUDA_TRY(cudaEventRecord(rs[k]->pushed, ss));
  for (int k = 0; k < n; ++k) {
    SceneReplica* r = rs[k];
    PFT_CUDA_TRY(cudaSetDevice(r->dst->device));
    PFT_CUDA_TRY(cudaStreamWaitEvent(r->dst->stream, r->pushed, 0));
    r->cloud.host_n = src->host_n;
    r->src_version = src->version;
  }
  return PFT_OK;
}

// dst's replica of src, created empty when there is none.  Caller holds g_replica_mu.
SceneReplica* replica_for(pft_context* dst, const pft_cloud* src) {
  for (SceneReplica* r : g_replicas) if (r->dst == dst && r->src_serial == src->serial) return r;
  SceneReplica* r = new SceneReplica();
  r->dst = dst; r->src_serial = src->serial; r->cloud.ctx = dst;
  g_replicas.push_back(r);
  return r;
}

// Points every tracker's `scene` at what its kernels read this frame: its input, or its context's replica of the input,
// refreshed first where the input was written since.  The stale replicas of one source are refreshed by one launch.
// Host-side only: nothing here waits for a device.
int resolve_scenes(pft_tracker* const* ts, int n) {
  int dev = 0;
  PFT_CUDA_TRY(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(g_replica_mu);
  std::vector<std::pair<const pft_cloud*, SceneReplica*>> stale;
  int rc = PFT_OK;
  for (int i = 0; i < n && !rc; ++i) {
    pft_tracker* t = ts[i];
    t->replica = nullptr;
    t->scene = t->input;
    if (!t->input) continue;
    if (t->input->ctx == t->ctx) {  // a frame may still be arriving on the copy stream (pft_cloud_upload_async)
      if (cudaSetDevice(t->ctx->device) != cudaSuccess) { set_last_error("cudaSetDevice(%d) failed", t->ctx->device); cudaGetLastError(); rc = PFT_ERR_CUDA; }
      else rc = t->input->join_upload();
      continue;
    }
    SceneReplica* r = replica_for(t->ctx, t->input);
    if (r->src_version != t->input->version && std::find(stale.begin(), stale.end(), std::make_pair(t->input, r)) == stale.end()) stale.push_back({t->input, r});
    t->replica = r;
    t->scene = &r->cloud;
  }
  // one launch per source and up to kMaxPeers destinations
  while (!rc && !stale.empty()) {
    const pft_cloud* src = stale.front().first;
    std::vector<SceneReplica*> rs;
    std::vector<std::pair<const pft_cloud*, SceneReplica*>> rest;
    for (const auto& e : stale) {
      if (e.first == src && (int)rs.size() < kMaxPeers) rs.push_back(e.second);
      else rest.push_back(e);
    }
    stale.swap(rest);
    rc = push_replicas(src, rs.data(), (int)rs.size());
  }
  cudaSetDevice(dev);
  return rc;
}

}  // namespace

void pft::release_replicas_of(const pft_cloud* src) {
  const unsigned long long serial = src->serial;
  release_replicas_if([&](const SceneReplica* r) { return r->src_serial == serial; });
}
void pft::release_replicas_in(const pft_context* dst) {
  release_replicas_if([&](const SceneReplica* r) { return r->dst == dst; });
}

namespace {

// After the trackers that read a replica have been enqueued on (or joined to) its context stream: the next push into it
// waits for them.
int mark_scene_read(pft_tracker* t) {
  if (!t->replica) return PFT_OK;
  std::lock_guard<std::mutex> lock(g_replica_mu);
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  PFT_CUDA_TRY(cudaEventRecord(t->replica->read, t->ctx->stream));
  t->replica->read_recorded = true;
  return PFT_OK;
}

// Every lazy allocation of the frame path happens here, before any stage is enqueued: nothing may be allocated inside a
// graph capture, nor between the enqueues of the ranks of the multi-device mode (see compute_multi_device).
int prepare_compute(pft_tracker* t) {
  int rc = ensure_particle_buffers(t);
  if (rc) return rc;
  if ((rc = resolve_scenes(&t, 1))) return rc;
  if ((rc = ensure_index_buffers(t))) return rc;
  if (t->inj_stride == 0 && (rc = reserve_generated_draws(t, t->n_cap))) return rc;
  if (!t->aux_stream) {  // the candidate-list chain that runs beside the index build (weight_phase_eval)
    PFT_CUDA_TRY(cudaStreamCreateWithFlags(&t->aux_stream, cudaStreamNonBlocking));
    PFT_CUDA_TRY(cudaEventCreateWithFlags(&t->ev_fork, cudaEventDisableTiming));
    PFT_CUDA_TRY(cudaEventCreateWithFlags(&t->ev_join, cudaEventDisableTiming));
  }
  choose_chunks(t);
  const size_t need_partial = (size_t)t->chunks * t->n_cap * sizeof(double);
  if (need_partial > t->partial.bytes) {
    invalidate_graph(t);
    PFT_CUDA_TRY(cudaStreamSynchronize(t->run_stream()));
    if ((rc = t->partial.reserve(need_partial))) return rc;
  }
  if (t->sampler == PFT_SAMPLER_ALIAS_PCL && t->alias_q.bytes < (size_t)t->n_cap * sizeof(double)) {
    invalidate_graph(t);
    PFT_CUDA_TRY(cudaStreamSynchronize(t->run_stream()));
    if ((rc = t->alias_a.reserve((size_t)t->n_cap * sizeof(int)))) return rc;
    if ((rc = t->alias_q.reserve((size_t)t->n_cap * sizeof(double)))) return rc;
    if ((rc = t->alias_hl.reserve((size_t)t->n_cap * sizeof(int)))) return rc;
  }
  if (t->nn_mode == PFT_NN_PCL_APPROX) {
    // parity mode: upstream's pointer octree, rebuilt by every weight() (sized for the whole input cloud: one leaf chain
    // of at most 31 nodes per point plus the roots added while the box grows)
    const size_t cap_pts = std::max<size_t>(t->scene ? t->scene->capacity : 0, 1);
    const size_t want_nodes = cap_pts * 12 + 128;
    if (t->oct_next.bytes < cap_pts * sizeof(int) || (size_t)t->oct_node_cap < want_nodes) {
      invalidate_graph(t);
      PFT_CUDA_TRY(cudaStreamSynchronize(t->run_stream()));
      if ((rc = t->oct_hdr.reserve(sizeof(OctHeaderD)))) return rc;
      if ((rc = t->oct_next.reserve(cap_pts * sizeof(int)))) return rc;
      if ((rc = t->oct_nodes.reserve(want_nodes * sizeof(OctNodeD)))) return rc;
      t->oct_node_cap = (int)want_nodes;
    }
  }
  if (t->use_cd && !t->cd_nodes.p) {
    invalidate_graph(t);
    t->cd_node_cap = 1 << 20;  // the tree lives as long as the tracker; it is rebuilt from scratch if it ever fills up
    if ((rc = t->cd_hdr.reserve(sizeof(CdHeaderD)))) return rc;
    if ((rc = t->cd_out.reserve(2 * sizeof(int)))) return rc;
    if ((rc = t->cd_nodes.reserve((size_t)t->cd_node_cap * sizeof(CdNodeD)))) return rc;
    PFT_CUDA_TRY(cudaMemsetAsync(t->cd_hdr.p, 0, sizeof(CdHeaderD), t->run_stream()));
  }
  if (t->debug_nn > 0) {
    const size_t need = (size_t)t->debug_nn * t->M;
    if (need * sizeof(int) > t->dbg_idx.bytes) {
      invalidate_graph(t);
      PFT_CUDA_TRY(cudaStreamSynchronize(t->run_stream()));
      if ((rc = t->dbg_idx.reserve(need * sizeof(int)))) return rc;
      if ((rc = t->dbg_d2.reserve(need * sizeof(float)))) return rc;
    }
  }
  return PFT_OK;
}

bool is_noop(const pft_tracker* t) {
  // Tracker::initCompute fails silently on an empty input (PCL_ERROR, no exception): compute() does nothing.
  return !t->input || t->M <= 0 || t->input->host_n == 0 || t->input->capacity == 0;
}

}  // namespace

// ------------------------------------------------------------------ C ABI
extern "C" {
static int compute_multi_device(pft_tracker* t);
static void destroy_followers(pft_tracker* t) {
  for (auto& f : t->followers) {
    if (f.t) pft_tracker_destroy(f.t);
    if (f.ctx) pft_context_destroy(f.ctx);
  }
  t->followers.clear();
  t->md_attached = false;
}


int pft_tracker_create(pft_context* ctx, int kld, pft_tracker** out) {
  if (!ctx || !out) { set_last_error("pft_tracker_create: null argument"); return PFT_ERR_INVALID; }
  pft_tracker* t = new pft_tracker();
  t->ctx = ctx;
  t->kld = kld != 0;
  const char* ng = getenv("PFT_NO_GRAPH");
  t->graph_enabled = !(ng && ng[0] == '1');
  *out = t;
  return PFT_OK;
}

void pft_tracker_destroy(pft_tracker* t) {
  if (!t) return;
  // multi-device mode: the followers go first -- they read this tracker's window until their streams are idle
  for (auto& f : t->followers) if (f.t) { cudaSetDevice(f.ctx->device); cudaStreamSynchronize(f.t->run_stream()); }
  destroy_followers(t);
  cudaSetDevice(t->ctx->device);
  cudaStreamSynchronize(t->run_stream());
  for (int g = 0; g < 2; ++g) if (t->graph_exec[g]) cudaGraphExecDestroy(t->graph_exec[g]);
  for (auto e : t->ev_w) cudaEventDestroy(e);
  for (auto e : t->ev_k) cudaEventDestroy(e);
  if (t->ev_c0) cudaEventDestroy(t->ev_c0);
  if (t->ev_c1) cudaEventDestroy(t->ev_c1);
  pft_tracker_peer_detach(t);
  if (t->batch_stream) cudaStreamDestroy(t->batch_stream);
  if (t->aux_stream) { cudaStreamDestroy(t->aux_stream); cudaEventDestroy(t->ev_fork); cudaEventDestroy(t->ev_join); }
  if (t->batch_done) cudaEventDestroy(t->batch_done);
  release_all(t);
  delete t;
}

int pft_tracker_set_i(pft_tracker* t, int key, int v) {
  if (t) for (auto& f_ : t->followers) { int rc_ = pft_tracker_set_i(f_.t, key, v); if (rc_) return rc_; }
  if (!t) { set_last_error("null tracker"); return PFT_ERR_INVALID; }
  switch (key) {
    case PFT_THREADS: t->threads = v; break;  // OpenMP thread count of the CPU tracker: meaningless here
    case PFT_PARTICLE_NUM:
      if (v < 0) { set_last_error("particle number must be >= 0"); return PFT_ERR_INVALID; }
      t->particle_num = v; break;
    case PFT_MAX_PARTICLE_NUM:
      if (v < 0) { set_last_error("maximum particle number must be >= 0"); return PFT_ERR_INVALID; }
      t->max_particle_num = v; break;
    case PFT_ITERATION_NUM:
      if (v < 0) { set_last_error("iteration number must be >= 0"); return PFT_ERR_INVALID; }
      t->iteration_num = v; break;
    case PFT_NN_MODE:
      if (v != PFT_NN_EXACT && v != PFT_NN_PCL_APPROX) { set_last_error("unknown nearest-neighbour mode %d", v); return PFT_ERR_INVALID; }
      if (v != t->nn_mode) invalidate_graph(t);
      t->nn_mode = v; break;
    case PFT_USE_HSV: t->use_hsv = v != 0; break;
    case PFT_USE_DISTANCE: t->use_dist = v != 0; break;
    case PFT_SAMPLER:
      if (v != PFT_SAMPLER_ALIAS_PCL && v != PFT_SAMPLER_CDF && v != PFT_SAMPLER_CDF_VDC) { set_last_error("unknown sampler %d", v); return PFT_ERR_INVALID; }
      t->sampler = v; break;
    case PFT_QUAT_SAMPLE: t->quat_sample = v != 0; break;
    case PFT_USE_NORMAL:
      if (v != 0) { set_last_error("setUseNormal(true) is not supported (the reference runs with false, src/auto_tracking.cpp:233)"); return PFT_ERR_INVALID; }
      break;
    case PFT_MIN_INDICES: t->min_indices = v; break;
    case PFT_CANDIDATE_LISTS:
      if (v < 0 || v > 2) { set_last_error("PFT_CANDIDATE_LISTS must be 0, 1 or 2"); return PFT_ERR_INVALID; }
      t->list_mode = v; break;
    case PFT_DEBUG_NN:
      if (v < 0) { set_last_error("PFT_DEBUG_NN must be >= 0"); return PFT_ERR_INVALID; }
      t->debug_nn = v; break;
    case PFT_USE_CHANGE_DETECTOR: t->use_cd = v != 0; break;
    case PFT_CHANGE_DETECTOR_INTERVAL:
      if (v < 0) { set_last_error("interval of change detection must be >= 0"); return PFT_ERR_INVALID; }
      t->cd_interval = v; break;
    case PFT_CHANGE_DETECTOR_MIN_POINTS: t->cd_filter = v; break;
    default: set_last_error("unknown int key %d", key); return PFT_ERR_INVALID;
  }
  invalidate_graph(t);
  return PFT_OK;
}

int pft_tracker_set_d(pft_tracker* t, int key, double v) {
  if (t) for (auto& f_ : t->followers) { int rc_ = pft_tracker_set_d(f_.t, key, v); if (rc_) return rc_; }
  if (!t) { set_last_error("null tracker"); return PFT_ERR_INVALID; }
  switch (key) {
    case PFT_DELTA: t->delta = v; break;
    case PFT_EPSILON: t->epsilon = v; break;
    case PFT_ALPHA: t->alpha = v; break;
    case PFT_MOTION_RATIO: t->motion_ratio = v; break;
    case PFT_MAX_DIST: t->max_dist = v; break;
    case PFT_DIST_WEIGHT: t->dist_w = v; break;
    case PFT_HSV_WEIGHT: t->hsv_w = v; break;
    case PFT_H_WEIGHT: t->h_w = v; break;
    case PFT_S_WEIGHT: t->s_w = v; break;
    case PFT_V_WEIGHT: t->v_w = v; break;
    case PFT_SEARCH_RESOLUTION:
      if (!(v > 0.0)) { set_last_error("search resolution must be positive"); return PFT_ERR_INVALID; }
      t->search_res = v; break;
    case PFT_RESAMPLE_LIKELIHOOD_THR: t->resample_thr = v; break;
    case PFT_CHANGE_DETECTOR_RESOLUTION:
      if (!(v > 0.0)) { set_last_error("resolution of change detection must be positive"); return PFT_ERR_INVALID; }
      if (v != t->cd_res && t->cd_hdr.p) {  // a new detector: forget the tree of the old one
        PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
        PFT_CUDA_TRY(cudaMemsetAsync(t->cd_hdr.p, 0, sizeof(CdHeaderD), t->run_stream()));
      }
      t->cd_res = v; break;
    default: set_last_error("unknown double key %d", key); return PFT_ERR_INVALID;
  }
  invalidate_graph(t);
  if ((key == PFT_DELTA || key == PFT_EPSILON) && t->klb.p && t->n_cap > 0) return upload_kl_table(t);
  return PFT_OK;
}

int pft_tracker_set_vec6(pft_tracker* t, int key, const double* v) {
  if (t) for (auto& f_ : t->followers) { int rc_ = pft_tracker_set_vec6(f_.t, key, v); if (rc_) return rc_; }
  if (!t || !v) { set_last_error("null argument"); return PFT_ERR_INVALID; }
  switch (key) {
    case PFT_STEP_NOISE_COV: memcpy(t->step_cov, v, sizeof(t->step_cov)); break;
    case PFT_INIT_NOISE_COV: memcpy(t->init_cov, v, sizeof(t->init_cov)); break;
    case PFT_INIT_NOISE_MEAN: memcpy(t->init_mean, v, sizeof(t->init_mean)); break;
    case PFT_BIN_SIZE: for (int d = 0; d < 6; ++d) t->bin_size[d] = (float)v[d]; break;
    default: set_last_error("unknown vec6 key %d", key); return PFT_ERR_INVALID;
  }
  invalidate_graph(t);
  return PFT_OK;
}

int pft_tracker_set_trans(pft_tracker* t, const float* m12) {
  if (t) for (auto& f_ : t->followers) { int rc_ = pft_tracker_set_trans(f_.t, m12); if (rc_) return rc_; }
  if (!t || !m12) { set_last_error("null argument"); return PFT_ERR_INVALID; }
  memcpy(t->trans, m12, sizeof(t->trans));
  return PFT_OK;
}

static int set_reference_device(pft_tracker* t, const float4* d_pts, int n) {
  pft_context* ctx = t->ctx;
  cudaStream_t s = ctx->stream;
  invalidate_graph(t);
  PFT_CUDA_TRY(cudaStreamSynchronize(s));
  t->M = n;
  if (n == 0) return PFT_OK;
  int n_pad = 1;
  while (n_pad < n) n_pad <<= 1;
  int rc;
  if ((rc = t->model.reserve((size_t)n * sizeof(float4)))) return rc;
  if ((rc = t->model_perm.reserve((size_t)n * sizeof(int)))) return rc;
  if ((rc = t->sort_keys.reserve((size_t)n_pad * sizeof(unsigned int)))) return rc;
  if ((rc = t->sort_idx.reserve((size_t)n_pad * sizeof(int)))) return rc;
  if ((rc = t->bbox.reserve(6 * sizeof(float)))) return rc;
  // the reference cloud as given (order, rgba), for pft_tracker_get_result_cloud: `model` is reordered and holds HSV
  if ((rc = t->ref_pts.reserve((size_t)n * sizeof(float4)))) return rc;
  PFT_CUDA_TRY(cudaMemcpyAsync(t->ref_pts.p, d_pts, (size_t)n * sizeof(float4), cudaMemcpyDeviceToDevice, s));
  model_bbox_kernel<<<1, 1024, 0, s>>>(d_pts, n, t->bbox.as<float>());
  PFT_LAUNCH_CHECK();
  model_keys_kernel<<<blocks_for(n_pad, 256, 1024), 256, 0, s>>>(d_pts, n, t->sort_keys.as<unsigned int>(), t->sort_idx.as<int>(), n_pad, t->bbox.as<float>());
  PFT_LAUNCH_CHECK();
  bitonic_sort_kernel<<<1, 1024, 0, s>>>(t->sort_keys.as<unsigned int>(), t->sort_idx.as<int>(), n_pad);
  PFT_LAUNCH_CHECK();
  model_gather_kernel<<<blocks_for(n, 256, 1024), 256, 0, s>>>(d_pts, t->sort_idx.as<int>(), n, t->model.as<float4>(), t->model_perm.as<int>());
  PFT_LAUNCH_CHECK();
  PFT_CUDA_TRY(cudaStreamSynchronize(s));
  choose_chunks(t);
  return PFT_OK;
}

int pft_tracker_set_reference_cloud(pft_tracker* t, const pft_cloud* cloud) {
  if (!t || !cloud) { set_last_error("null argument"); return PFT_ERR_INVALID; }
  for (auto& f_ : t->followers) { int rc_ = pft_tracker_set_reference_cloud(f_.t, cloud); if (rc_) return rc_; }
  size_t n = 0;
  int rc = pft_cloud_size(const_cast<pft_cloud*>(cloud), &n);
  if (rc) return rc;
  const float4* pts = cloud->d_pts();
  if (cloud->ctx != t->ctx) {  // read through this context's replica (set_reference_device synchronises, no reader stays behind)
    if ((rc = enable_peer_access(cloud->ctx->device, t->ctx->device))) return rc;
    std::lock_guard<std::mutex> lock(g_replica_mu);
    SceneReplica* r = replica_for(t->ctx, cloud);
    if (r->src_version != cloud->version && (rc = push_replicas(cloud, &r, 1))) return rc;
    pts = r->cloud.d_pts();
  }
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  return set_reference_device(t, pts, (int)n);
}

int pft_tracker_set_reference_points(pft_tracker* t, const void* host_points, size_t n, int layout) {
  if (t) for (auto& f_ : t->followers) { int rc_ = pft_tracker_set_reference_points(f_.t, host_points, n, layout); if (rc_) return rc_; }
  if (!t || (n && !host_points)) { set_last_error("null argument"); return PFT_ERR_INVALID; }
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  pft_cloud tmp;
  tmp.ctx = t->ctx;
  int rc = tmp.ensure(n);
  if (!rc) rc = pft_cloud_upload(&tmp, host_points, n, layout);
  if (!rc) rc = set_reference_device(t, tmp.d_pts(), (int)n);
  cudaStreamSynchronize(t->run_stream());
  tmp.pts.release(); tmp.hdr.release();
  return rc;
}

int pft_tracker_set_input_cloud(pft_tracker* t, const pft_cloud* cloud) {
  if (!t) { set_last_error("null tracker"); return PFT_ERR_INVALID; }
  if (cloud && cloud->ctx != t->ctx) {
    // sharded trackers (communicator, shard, peer windows) get the scene from their caller; a set_devices tracker is
    // rank 0 of its own ranks and reads like any other tracker
    if ((t->comm || t->nranks > 1 || t->peer_mode) && t->followers.empty()) {
      set_last_error("cloud belongs to another context: a sharded tracker takes its scene from its own context");
      return PFT_ERR_INVALID;
    }
    int dev = 0;
    PFT_CUDA_TRY(cudaGetDevice(&dev));
    int rc = enable_peer_access(cloud->ctx->device, t->ctx->device);
    for (auto& f_ : t->followers) if (!rc) rc = enable_peer_access(cloud->ctx->device, f_.ctx->device);
    cudaSetDevice(dev);
    if (rc) return rc;
  }
  for (auto& f_ : t->followers) { f_.t->input = cloud; f_.t->scene = nullptr; f_.t->replica = nullptr; }
  t->input = cloud;
  t->scene = cloud && cloud->ctx == t->ctx ? cloud : nullptr;  // (a replica is resolved by the next compute())
  t->replica = nullptr;
  return PFT_OK;
}

// ------------------------------------------------------------------ execution
static int compute_one(pft_tracker* t) {
  if (is_noop(t)) { t->replica = nullptr; return PFT_OK; }  // (nothing read)
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  cudaStream_t s = t->run_stream();
  int rc = prepare_compute(t);
  if (rc) return rc;
  if (!t->has_particles && (rc = stage_init_particles(t))) return rc;
  if (t->timing) {
    if (!t->ev_c0) { PFT_CUDA_TRY(cudaEventCreate(&t->ev_c0)); PFT_CUDA_TRY(cudaEventCreate(&t->ev_c1)); }
    t->n_ev_used = 0;
    t->n_ev_k = 0;
    PFT_CUDA_TRY(cudaEventRecord(t->ev_c0, s));
  }
  const bool steady = t->changed && t->graph_enabled && !t->timing && t->debug_nn == 0 && !t->use_cd;  // (the change detector decides on the host)
  if (steady) {
    // The steady-state frame is a fixed launch sequence over fixed buffers: replay it from a graph.  The pointers to
    // the live particle buffer are baked in, and `cur` flips once per resample: one graph per value of `cur` at the
    // start of the frame (an even iteration count always starts from the same one, an odd count -- PCL's default is
    // 1 -- alternates between the two).
    const int g = t->cur;
    const bool valid = t->graph_exec[g] && t->graph_version[g] == t->config_version && t->graph_scene_pts[g] == (const void*)t->scene->d_pts() &&
                       t->graph_scene_hdr[g] == (const void*)t->scene->d_hdr();
    if (!valid) {
      if (t->graph_exec[g]) { cudaGraphExecDestroy(t->graph_exec[g]); t->graph_exec[g] = nullptr; }
      const unsigned long long version = t->config_version;
      const int cur0 = t->cur;
      const bool changed0 = t->changed;
      cudaGraph_t graph = nullptr;
      PFT_CUDA_TRY(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
      const unsigned long long launches_before = g_launch_count.load();
      rc = enqueue_tracking(t);
      cudaError_t ce = cudaStreamEndCapture(s, &graph);
      g_launch_count -= g_launch_count.load() - launches_before;  // captured, not launched (other threads' launches keep counting)
      if (rc || ce != cudaSuccess) {
        // nothing has executed: the host mirror goes back to where the frame started
        t->cur = cur0; t->changed = changed0;
        if (graph) cudaGraphDestroy(graph);
        if (rc) return rc;
        set_last_error("graph capture failed: %s", cudaGetErrorString(ce)); cudaGetLastError(); return PFT_ERR_CUDA;
      }
      size_t n_nodes = 0;
      cudaGraphGetNodes(graph, nullptr, &n_nodes);
      cudaError_t ie = cudaGraphInstantiate(&t->graph_exec[g], graph, 0);
      cudaGraphDestroy(graph);
      if (ie != cudaSuccess) {
        t->cur = cur0; t->changed = changed0;
        set_last_error("graph instantiate failed: %s", cudaGetErrorString(ie)); cudaGetLastError(); t->graph_exec[g] = nullptr; return PFT_ERR_CUDA;
      }
      t->graph_version[g] = version;
      t->config_version = version;  // stages may bump the version while sizing buffers; nothing changed since
      t->graph_scene_pts[g] = t->scene->d_pts();
      t->graph_scene_hdr[g] = t->scene->d_hdr();
      t->graph_nodes[g] = (int)n_nodes;
    } else {
      // replay: the host mirror follows what the captured stages do (one flip of `cur` per resample)
      if (t->iteration_num & 1) t->cur ^= 1;
    }
    PFT_CUDA_TRY(cudaGraphLaunch(t->graph_exec[g], s));
    g_launch_count += (unsigned long long)t->graph_nodes[g];
    t->graph_replays++;
    return PFT_OK;
  }
  rc = enqueue_tracking(t);
  if (rc) return rc;
  if (t->timing) PFT_CUDA_TRY(cudaEventRecord(t->ev_c1, s));
  return PFT_OK;
}

// ---- single-process multi-device mode
static int alloc_peer_window(pft_tracker* t);
// Loads every kernel of the tracker path on the current device (CUDA loads kernels lazily, on first launch, and that
// load may synchronise the context: with several ranks in one process a rank whose kernel spins on a peer flag must
// never be waited for by the host -- see compute_multi_device).
static int preload_kernels() {
  static const void* const kernels[] = {
      (const void*)aabb_kernel<1>,
      (const void*)aabb_kernel<4>,
      (const void*)alias_table_kernel,
      (const void*)bitonic_sort_kernel,
      (const void*)cand_build_far_kernel,
      (const void*)cand_build_kernel,
      (const void*)cand_collect_kernel,
      (const void*)cand_mark_kernel<false>,
      (const void*)cand_mark_kernel<true>,
      (const void*)cand_octant_kernel,
      (const void*)cdf_kernel<1>,
      (const void*)cdf_kernel<kClusterCtas>,
      (const void*)change_detect_kernel,
      (const void*)cloud_fanout_kernel,
      (const void*)cloud_push_kernel,
      (const void*)cloud_wait_kernel,
      (const void*)draws_kernel,
      (const void*)index_begin_kernel,
      (const void*)index_count_kernel,
      (const void*)index_scan_kernel,
      (const void*)index_scatter_kernel,
      (const void*)init_particles_kernel,
      (const void*)kld_insert_kernel,
      (const void*)kld_stop_kernel,
      (const void*)matrices_kernel,
      (const void*)model_bbox_kernel,
      (const void*)model_gather_kernel,
      (const void*)model_keys_kernel,
      (const void*)normalize_kernel<1>,
      (const void*)normalize_kernel<kClusterCtas>,
      (const void*)octree_build_kernel,
      (const void*)raw_weights_kernel,
      (const void*)resample_kernel,
      (const void*)result_box_kernel,
      (const void*)single_matrix_kernel,
      (const void*)update_kernel<1>,
      (const void*)update_kernel<kClusterCtas>,
      (const void*)weight_approx_kernel,
      (const void*)weight_lists_kernel<false, kListThreads, false>,
      (const void*)weight_lists_kernel<false, kListThreads, true>,
      (const void*)weight_lists_kernel<false, kListThreadsBig, true>,
      (const void*)weight_lists_kernel<true, kListThreads, false>,
      (const void*)weight_lists_kernel<true, kListThreads, true>,
      (const void*)weight_lists_kernel<true, kListThreadsBig, true>,
      (const void*)weights_to_raw_kernel};
  for (const void* k : kernels) {
    cudaFuncAttributes a;
    PFT_CUDA_TRY(cudaFuncGetAttributes(&a, k));
  }
  return PFT_OK;
}

// One process, several GPUs: the follower trackers are ordinary sharded trackers whose exchange windows are mapped
// directly (peer access, no IPC).  Per frame: the scene travels to every rank's context (the replicas, one fan-out
// launch), then one frame is enqueued on every device -- nothing here blocks the host, the kernels of the ranks meet through the
// windows exactly as separate processes do.
static int compute_multi_device(pft_tracker* t) {
  if (is_noop(t)) return PFT_OK;
  const int n = (int)t->followers.size() + 1;
  int rc;
  if (!t->md_attached) {
    std::vector<pft_tracker*> all{t};
    for (auto& f : t->followers) all.push_back(f.t);
    for (pft_tracker* x : all) {
      PFT_CUDA_TRY(cudaSetDevice(x->ctx->device));
      if ((rc = alloc_peer_window(x))) return rc;
    }
    for (int r = 0; r < n; ++r) {
      PeerSet ps{};
      ps.nranks = n; ps.rank = r;
      for (int q = 0; q < n; ++q) ps.win[q] = reinterpret_cast<PeerWindow*>(all[q]->peer_local);
      all[r]->peers = ps; all[r]->peer_mode = true; all[r]->peer_ipc = false;
      invalidate_graph(all[r]);
    }
    t->md_attached = true;
  }
  // Everything that may allocate, free or load code happens for EVERY rank before the first frame is enqueued: once a
  // rank's frame is in flight its kernels spin on peer flags until the other ranks' frames arrive, and a host call that
  // waits for the device (cudaFree, a lazy kernel load) in between would stall until their time limit.
  std::vector<pft_tracker*> all{t};
  for (auto& f : t->followers) all.push_back(f.t);
  if ((rc = resolve_scenes(all.data(), n))) return rc;
  for (pft_tracker* x : all) {
    PFT_CUDA_TRY(cudaSetDevice(x->ctx->device));
    if (!x->md_prepared) { if ((rc = preload_kernels())) return rc; }
    if ((rc = prepare_compute(x))) return rc;
    x->md_prepared = true;
  }
  for (int k = 1; k <= n; ++k) {  // rank 0 last
    if ((rc = compute_one(all[k % n]))) return rc;
    if ((rc = mark_scene_read(all[k % n]))) return rc;
  }
  return PFT_OK;
}

int pft_tracker_compute(pft_tracker* t) {
  if (!t) { set_last_error("null tracker"); return PFT_ERR_INVALID; }
  if (!t->followers.empty()) return compute_multi_device(t);
  int rc = compute_one(t);
  return rc ? rc : mark_scene_read(t);
}

// The trackers of one context: each tracker's frame (one graph launch in steady state) runs on a stream of its own,
// forked from the context stream -- which carries the scene that was just downsampled or pushed -- and joined back to
// it, so that the many small latency-bound kernels of the trackers overlap on the GPU.  Trackers that time, exchange
// or drive other devices run one after the other.
static int compute_group(pft_tracker* const* ts, int n) {
  bool concurrent = n > 1;
  for (int i = 0; i < n && concurrent; ++i) concurrent = !ts[i]->timing && !ts[i]->comm && !ts[i]->peer_mode && ts[i]->followers.empty();
  if (!concurrent) {
    for (int i = 0; i < n; ++i) {
      int rc = pft_tracker_compute(ts[i]);
      if (rc) return rc;
    }
    return PFT_OK;
  }
  pft_context* ctx = ts[0]->ctx;
  PFT_CUDA_TRY(cudaSetDevice(ctx->device));
  if (!ctx->batch_fork) PFT_CUDA_TRY(cudaEventCreateWithFlags(&ctx->batch_fork, cudaEventDisableTiming));
  PFT_CUDA_TRY(cudaEventRecord(ctx->batch_fork, ctx->stream));  // (behind the uploads and pushes resolve_scenes joined)
  int rc = PFT_OK;
  int launched = 0;
  for (int i = 0; i < n && rc == PFT_OK; ++i) {
    pft_tracker* t = ts[i];
    if (!t->batch_stream) {
      PFT_CUDA_TRY(cudaStreamCreateWithFlags(&t->batch_stream, cudaStreamNonBlocking));
      PFT_CUDA_TRY(cudaEventCreateWithFlags(&t->batch_done, cudaEventDisableTiming));
    }
    PFT_CUDA_TRY(cudaStreamWaitEvent(t->batch_stream, ctx->batch_fork, 0));
    t->batch_active = true;
    rc = compute_one(t);
    t->batch_active = false;
    cudaEventRecord(t->batch_done, t->batch_stream);
    ++launched;
  }
  for (int i = 0; i < launched; ++i) cudaStreamWaitEvent(ctx->stream, ts[i]->batch_done, 0);
  for (int i = 0; i < launched; ++i) { int mrc = mark_scene_read(ts[i]); if (!rc) rc = mrc; }
  return rc;
}

int pft_compute_batch(pft_tracker** ts, int n) {
  if (n < 0 || (n && !ts)) { set_last_error("pft_compute_batch: bad arguments"); return PFT_ERR_INVALID; }
  // Independent trackers on one scene (ref: src/auto_tracking.cpp:688-697 loops them serially), on one context or on
  // several: the stale scene replicas are refreshed first (one fan-out launch per source), then every context's
  // trackers run as one group on that context's stream.  Nothing here waits for a device.
  for (int i = 0; i < n; ++i) {
    if (!ts[i]) { set_last_error("pft_compute_batch: null tracker %d", i); return PFT_ERR_INVALID; }
  }
  int rc = resolve_scenes(ts, n);
  if (rc) return rc;
  std::vector<pft_context*> ctxs;
  for (int i = 0; i < n; ++i) if (std::find(ctxs.begin(), ctxs.end(), ts[i]->ctx) == ctxs.end()) ctxs.push_back(ts[i]->ctx);
  std::vector<pft_tracker*> group;
  for (pft_context* c : ctxs) {
    group.clear();
    for (int i = 0; i < n; ++i) if (ts[i]->ctx == c) group.push_back(ts[i]);
    if ((rc = compute_group(group.data(), (int)group.size()))) return rc;
  }
  return PFT_OK;
}

static int read_state(pft_tracker* t, TrackerState* host) {
  if (!t->st.p) { memset(host, 0, sizeof(*host)); host->rep.one = 1.f; host->motion.one = 1.f; return PFT_OK; }
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  cudaStream_t s = t->run_stream();
  PFT_CUDA_TRY(cudaMemcpyAsync(t->ctx->pinned, t->st.p, sizeof(TrackerState), cudaMemcpyDeviceToHost, s));
  PFT_CUDA_TRY(cudaStreamSynchronize(s));
  memcpy(host, t->ctx->pinned, sizeof(TrackerState));
  if (host->peer_error) { set_last_error("NVLink peer exchange timed out: a peer rank did not reach the same weight()"); return PFT_ERR_COMM; }
  return PFT_OK;
}

int pft_tracker_get_result(pft_tracker* t, pft_particle* out) {
  if (!t || !out) { set_last_error("null argument"); return PFT_ERR_INVALID; }
  TrackerState h;
  int rc = read_state(t, &h);
  if (rc) return rc;
  memcpy(out, &h.rep, sizeof(pft_particle));
  return PFT_OK;
}

int pft_tracker_get_motion(pft_tracker* t, pft_particle* out) {
  if (!t || !out) { set_last_error("null argument"); return PFT_ERR_INVALID; }
  TrackerState h;
  int rc = read_state(t, &h);
  if (rc) return rc;
  memcpy(out, &h.motion, sizeof(pft_particle));
  return PFT_OK;
}

int pft_tracker_get_eval_count(pft_tracker* t, uint64_t* out) {
  if (!t || !out) { set_last_error("null argument"); return PFT_ERR_INVALID; }
  TrackerState h;
  int rc = read_state(t, &h);
  if (rc) return rc;
  *out = h.evals;
  return PFT_OK;
}

int pft_tracker_get_fit_ratio(pft_tracker* t, double* out) {
  if (!t || !out) { set_last_error("null argument"); return PFT_ERR_INVALID; }
  TrackerState h;
  int rc = read_state(t, &h);
  if (rc) return rc;
  *out = h.fit_ratio;
  return PFT_OK;
}

int pft_tracker_get_particles(pft_tracker* t, pft_particle* out, size_t capacity, size_t* n_out) {
  if (!t) { set_last_error("null tracker"); return PFT_ERR_INVALID; }
  size_t n = 0;
  if (t->has_particles) {
    TrackerState h;
    int rc = read_state(t, &h);
    if (rc) return rc;
    n = (size_t)h.particle_num;
  }
  if (n_out) *n_out = n;
  if (n > capacity) { set_last_error("pft_tracker_get_particles: %zu particles, capacity %zu", n, capacity); return PFT_ERR_CAPACITY; }
  if (n == 0) return PFT_OK;
  if (!out) { set_last_error("null buffer"); return PFT_ERR_INVALID; }
  cudaStream_t s = t->run_stream();
  PFT_CUDA_TRY(cudaMemcpyAsync(out, t->parts[t->cur].p, n * sizeof(pft_particle), cudaMemcpyDeviceToHost, s));
  PFT_CUDA_TRY(cudaStreamSynchronize(s));
  return PFT_OK;
}

int pft_particle_to_matrix(pft_context* ctx, const pft_particle* p, float* m12) {
  if (!ctx || !p || !m12) { set_last_error("null argument"); return PFT_ERR_INVALID; }
  PFT_CUDA_TRY(cudaSetDevice(ctx->device));
  int rc = ctx->tmp_f.reserve(16 * sizeof(float));
  if (rc) return rc;
  DevParticle dp;
  memcpy(&dp, p, sizeof(dp));
  single_matrix_kernel<<<1, 1, 0, ctx->stream>>>(dp, ctx->tmp_f.as<float>() + 4);
  PFT_LAUNCH_CHECK();
  PFT_CUDA_TRY(cudaMemcpyAsync(ctx->pinned, ctx->tmp_f.as<float>() + 4, 12 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  PFT_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  memcpy(m12, ctx->pinned, 12 * sizeof(float));
  return PFT_OK;
}

int pft_tracker_get_result_box(pft_tracker* t, float z_offset, pft_result_box* out) {
  if (!t || !out) { set_last_error("null argument"); return PFT_ERR_INVALID; }
  static_assert(sizeof(pft_result_box) == sizeof(ResultBox), "pft_result_box layout");
  if (!t->st.p || t->M <= 0) { set_last_error("no result yet: setReferenceCloud and compute() first"); return PFT_ERR_STATE; }
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  cudaStream_t s = t->run_stream();
  int rc = t->result_box.reserve(sizeof(ResultBox));
  if (rc) return rc;
  result_box_kernel<<<1, 1024, 0, s>>>(t->st.as<TrackerState>(), t->model.as<float4>(), t->M, z_offset, t->result_box.as<ResultBox>());
  PFT_LAUNCH_CHECK();
  PFT_CUDA_TRY(cudaMemcpyAsync(t->ctx->pinned, t->result_box.p, sizeof(ResultBox), cudaMemcpyDeviceToHost, s));
  PFT_CUDA_TRY(cudaStreamSynchronize(s));
  memcpy(out, t->ctx->pinned, sizeof(ResultBox));
  return PFT_OK;
}

int pft_tracker_get_result_cloud(pft_tracker* t, float z_offset, pft_cloud* out) {
  if (!t || !out) { set_last_error("pft_tracker_get_result_cloud: null argument"); return PFT_ERR_INVALID; }
  if (out->ctx != t->ctx) { set_last_error("pft_tracker_get_result_cloud: the cloud belongs to another context than the tracker"); return PFT_ERR_INVALID; }
  if (!t->st.p || t->M <= 0) { set_last_error("no result yet: setReferenceCloud and compute() first"); return PFT_ERR_STATE; }
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  int rc = out->join_upload();  // an asynchronous upload into the cloud must land before the kernel overwrites it
  if (rc) return rc;
  if ((rc = out->ensure((size_t)t->M))) return rc;
  cudaStream_t s = t->ctx->stream;  // the cloud's stream (a batch has joined it by now)
  result_cloud_kernel<<<blocks_for(t->M, 256, 8 * t->ctx->sm_count), 256, 0, s>>>(t->st.as<TrackerState>(), t->ref_pts.as<float4>(), t->M, z_offset,
                                                                                out->d_pts(), out->d_hdr());
  PFT_LAUNCH_CHECK();
  out->written(t->M);
  return PFT_OK;
}

int pft_tracker_reset(pft_tracker* t) {
  if (t) for (auto& f_ : t->followers) { int rc_ = pft_tracker_reset(f_.t); if (rc_) return rc_; }
  if (!t) { set_last_error("null tracker"); return PFT_ERR_INVALID; }
  // resetTracking: particles are re-drawn around trans_ on the next compute()
  if (t->kld && t->st.p && t->has_particles) {
    // upstream's particle_num_ is whatever the last KLD resample left: that many particles are re-drawn
    TrackerState hs;
    int rc = read_state(t, &hs);
    if (rc) return rc;
    if (hs.particle_num > 0) t->particle_num = hs.particle_num;
  }
  t->has_particles = false;
  // (changed_ is left as it is: upstream's resetTracking() only clears the particle vector, so the compute() that
  // follows re-draws the particles and, when an earlier weight() had set changed_, resamples them in the same frame)
  invalidate_graph(t);
  if (t->st.p) {
    PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
    cudaStream_t s = t->run_stream();
    PFT_CUDA_TRY(cudaMemsetAsync(&t->st.as<TrackerState>()->has_particles, 0, sizeof(int), s));
    // (the per-slot boxes of the transformed model stay: upstream keeps transed_reference_vector_ across resetTracking(),
    // so stale slots go on widening the crop box)
    PFT_CUDA_TRY(cudaStreamSynchronize(s));
  }
  return PFT_OK;
}

// ------------------------------------------------------------------ reproducibility / parity hooks
int pft_tracker_set_particles(pft_tracker* t, const pft_particle* p, size_t n) {
  if (t) for (auto& f_ : t->followers) { int rc_ = pft_tracker_set_particles(f_.t, p, n); if (rc_) return rc_; }
  if (!t || (n && !p)) { set_last_error("null argument"); return PFT_ERR_INVALID; }
  if (n == 0 || n > 0x7fffffffull) { set_last_error("bad particle count %zu", n); return PFT_ERR_INVALID; }
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  t->particle_num = (int)n;  // as PCL: particle_num_ follows the particle set
  int rc = ensure_particle_buffers(t);
  if (rc) return rc;
  if ((rc = upload_kl_table(t))) return rc;
  cudaStream_t s = t->run_stream();
  PFT_CUDA_TRY(cudaMemcpyAsync(t->parts[t->cur].p, p, n * sizeof(pft_particle), cudaMemcpyHostToDevice, s));
  const int nn = (int)n, one = 1;
  PFT_CUDA_TRY(cudaMemcpyAsync(&t->st.as<TrackerState>()->particle_num, &nn, sizeof(int), cudaMemcpyHostToDevice, s));
  PFT_CUDA_TRY(cudaMemcpyAsync(&t->st.as<TrackerState>()->has_particles, &one, sizeof(int), cudaMemcpyHostToDevice, s));
  PFT_CUDA_TRY(cudaStreamSynchronize(s));
  t->has_particles = true;
  invalidate_graph(t);
  return PFT_OK;
}

int pft_tracker_set_result(pft_tracker* t, const pft_particle* rep, const pft_particle* motion) {
  if (t) for (auto& f_ : t->followers) { int rc_ = pft_tracker_set_result(f_.t, rep, motion); if (rc_) return rc_; }
  if (!t) { set_last_error("null tracker"); return PFT_ERR_INVALID; }
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  int rc = ensure_particle_buffers(t);
  if (rc) return rc;
  cudaStream_t s = t->run_stream();
  if (rep) PFT_CUDA_TRY(cudaMemcpyAsync(&t->st.as<TrackerState>()->rep, rep, sizeof(pft_particle), cudaMemcpyHostToDevice, s));
  if (motion) PFT_CUDA_TRY(cudaMemcpyAsync(&t->st.as<TrackerState>()->motion, motion, sizeof(pft_particle), cudaMemcpyHostToDevice, s));
  PFT_CUDA_TRY(cudaStreamSynchronize(s));
  return PFT_OK;
}

int pft_tracker_inject_draws(pft_tracker* t, const float* usel, const float* normals6, const float* umot, int slots, int stride) {
  if (t) for (auto& f_ : t->followers) { int rc_ = pft_tracker_inject_draws(f_.t, usel, normals6, umot, slots, stride); if (rc_) return rc_; }
  if (!t) { set_last_error("null tracker"); return PFT_ERR_INVALID; }
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  invalidate_graph(t);
  PFT_CUDA_TRY(cudaStreamSynchronize(t->run_stream()));
  if (!usel || !normals6 || !umot) {
    t->inj_slots = 0; t->inj_stride = 0; t->draw_cap = 0;
    return PFT_OK;
  }
  if (slots <= 0 || stride <= 0) { set_last_error("bad draw shape %d x %d", slots, stride); return PFT_ERR_INVALID; }
  int rc = ensure_draw_buffers(t, slots, stride);
  if (rc) return rc;
  const size_t n = (size_t)slots * stride;
  cudaStream_t s = t->run_stream();
  PFT_CUDA_TRY(cudaMemcpyAsync(t->d_usel.p, usel, n * sizeof(float), cudaMemcpyHostToDevice, s));
  PFT_CUDA_TRY(cudaMemcpyAsync(t->d_normals.p, normals6, n * 6 * sizeof(float), cudaMemcpyHostToDevice, s));
  PFT_CUDA_TRY(cudaMemcpyAsync(t->d_umot.p, umot, n * sizeof(float), cudaMemcpyHostToDevice, s));
  PFT_CUDA_TRY(cudaStreamSynchronize(s));
  t->inj_slots = slots; t->inj_stride = stride; t->draw_cap = 0;
  return PFT_OK;
}

int pft_tracker_seed(pft_tracker* t, uint64_t seed) {
  if (t) for (auto& f_ : t->followers) { int rc_ = pft_tracker_seed(f_.t, seed); if (rc_) return rc_; }
  if (!t) { set_last_error("null tracker"); return PFT_ERR_INVALID; }
  t->seed = seed;
  invalidate_graph(t);
  if (t->st.p) {
    PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
    PFT_CUDA_TRY(cudaMemsetAsync(&t->st.as<TrackerState>()->draw_call, 0, sizeof(unsigned long long), t->run_stream()));
  }
  return PFT_OK;
}

int pft_tracker_init_particles(pft_tracker* t) {
  if (!t) { set_last_error("null tracker"); return PFT_ERR_INVALID; }
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  return stage_init_particles(t);
}
int pft_tracker_resample(pft_tracker* t, int slot) {
  if (!t) { set_last_error("null tracker"); return PFT_ERR_INVALID; }
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  int rc = prepare_compute(t);
  if (rc) return rc;
  return stage_resample(t, slot);
}
int pft_tracker_weight(pft_tracker* t) {
  if (!t) { set_last_error("null tracker"); return PFT_ERR_INVALID; }
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  int rc = prepare_compute(t);
  if (rc) return rc;
  if (t->timing) t->n_ev_used = 0;
  return stage_weight(t);
}
int pft_tracker_get_change_detector_info(pft_tracker* t, int32_t* out4) {
  if (!t || !out4) { set_last_error("null argument"); return PFT_ERR_INVALID; }
  out4[0] = t->change_counter; out4[1] = t->cd_tests; out4[2] = t->cd_last_found; out4[3] = t->changed ? 1 : 0;
  return PFT_OK;
}
int pft_tracker_update(pft_tracker* t) {
  if (!t) { set_last_error("null tracker"); return PFT_ERR_INVALID; }
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  return stage_update(t);
}
int pft_tracker_set_changed(pft_tracker* t, int changed) {
  if (t) for (auto& f_ : t->followers) { int rc_ = pft_tracker_set_changed(f_.t, changed); if (rc_) return rc_; }
  if (!t) { set_last_error("null tracker"); return PFT_ERR_INVALID; }
  t->changed = changed != 0;
  return PFT_OK;
}

int pft_tracker_get_aabb(pft_tracker* t, float* aabb6) {
  if (!t || !aabb6) { set_last_error("null argument"); return PFT_ERR_INVALID; }
  if (!t->idx_hdr.p) { set_last_error("no weight() has run"); return PFT_ERR_STATE; }
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  cudaStream_t s = t->run_stream();
  PFT_CUDA_TRY(cudaMemcpyAsync(t->ctx->pinned, t->idx_hdr.p, sizeof(IndexHeader), cudaMemcpyDeviceToHost, s));
  PFT_CUDA_TRY(cudaStreamSynchronize(s));
  memcpy(aabb6, reinterpret_cast<IndexHeader*>(t->ctx->pinned)->aabb, 6 * sizeof(float));
  return PFT_OK;
}

int pft_tracker_get_cropped_count(pft_tracker* t, size_t* n) {
  if (!t || !n) { set_last_error("null argument"); return PFT_ERR_INVALID; }
  if (!t->idx_hdr.p) { set_last_error("no weight() has run"); return PFT_ERR_STATE; }
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  cudaStream_t s = t->run_stream();
  PFT_CUDA_TRY(cudaMemcpyAsync(t->ctx->pinned, t->idx_hdr.p, sizeof(IndexHeader), cudaMemcpyDeviceToHost, s));
  PFT_CUDA_TRY(cudaStreamSynchronize(s));
  *n = (size_t)reinterpret_cast<IndexHeader*>(t->ctx->pinned)->n_in_crop;
  return PFT_OK;
}

int pft_tracker_get_index_info(pft_tracker* t, int* info8) {
  if (!t || !info8) { set_last_error("null argument"); return PFT_ERR_INVALID; }
  if (!t->idx_hdr.p) { set_last_error("no weight() has run"); return PFT_ERR_STATE; }
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  cudaStream_t s = t->run_stream();
  PFT_CUDA_TRY(cudaMemcpyAsync(t->ctx->pinned, t->idx_hdr.p, sizeof(IndexHeader), cudaMemcpyDeviceToHost, s));
  PFT_CUDA_TRY(cudaStreamSynchronize(s));
  const IndexHeader* h = reinterpret_cast<IndexHeader*>(t->ctx->pinned);
  info8[0] = h->dim[0]; info8[1] = h->dim[1]; info8[2] = h->dim[2]; info8[3] = h->level;
  info8[4] = h->n_in_crop; info8[5] = h->n_cells; info8[6] = h->use_lists; info8[7] = h->f_cells;
  return PFT_OK;
}

int pft_tracker_get_raw_weights(pft_tracker* t, float* out, size_t capacity, size_t* n_out) {
  if (!t) { set_last_error("null tracker"); return PFT_ERR_INVALID; }
  TrackerState h;
  int rc = read_state(t, &h);
  if (rc) return rc;
  const size_t n = t->has_particles ? (size_t)h.particle_num : 0;
  if (n_out) *n_out = n;
  if (n > capacity) { set_last_error("capacity %zu < %zu", capacity, n); return PFT_ERR_CAPACITY; }
  if (n == 0) return PFT_OK;
  const int slice = t->slice_cap();
  std::vector<float> all((size_t)slice * t->nranks);
  const void* src = t->peer_mode ? (const void*)reinterpret_cast<PeerWindow*>(t->peer_local)->raw : (const void*)t->raw.p;
  PFT_CUDA_TRY(cudaMemcpy(all.data(), src, all.size() * sizeof(float), cudaMemcpyDeviceToHost));
  for (size_t i = 0; i < n; ++i) out[i] = all[(i % t->nranks) * slice + i / t->nranks];
  return PFT_OK;
}

int pft_tracker_get_ancestors(pft_tracker* t, int32_t* out, size_t capacity, size_t* n_out) {
  if (!t) { set_last_error("null tracker"); return PFT_ERR_INVALID; }
  TrackerState h;
  int rc = read_state(t, &h);
  if (rc) return rc;
  const size_t n = t->has_particles ? (size_t)h.particle_num : 0;
  if (n_out) *n_out = n;
  if (n > capacity) { set_last_error("capacity %zu < %zu", capacity, n); return PFT_ERR_CAPACITY; }
  if (n == 0) return PFT_OK;
  PFT_CUDA_TRY(cudaMemcpy(out, t->ancestors.p, n * sizeof(int), cudaMemcpyDeviceToHost));
  return PFT_OK;
}

int pft_tracker_get_nn(pft_tracker* t, int particle, int32_t* idx, float* d2, size_t capacity) {
  if (!t || !idx || !d2) { set_last_error("null argument"); return PFT_ERR_INVALID; }
  if (particle < 0 || particle >= t->debug_nn || !t->dbg_idx.p) { set_last_error("particle %d was not recorded (PFT_DEBUG_NN = %d)", particle, t->debug_nn); return PFT_ERR_STATE; }
  if ((size_t)t->M > capacity) { set_last_error("capacity %zu < %d", capacity, t->M); return PFT_ERR_CAPACITY; }
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  PFT_CUDA_TRY(cudaStreamSynchronize(t->run_stream()));
  PFT_CUDA_TRY(cudaMemcpy(idx, t->dbg_idx.as<int>() + (size_t)particle * t->M, (size_t)t->M * sizeof(int), cudaMemcpyDeviceToHost));
  PFT_CUDA_TRY(cudaMemcpy(d2, t->dbg_d2.as<float>() + (size_t)particle * t->M, (size_t)t->M * sizeof(float), cudaMemcpyDeviceToHost));
  return PFT_OK;
}

int pft_tracker_enable_timing(pft_tracker* t, int on) {
  if (!t) { set_last_error("null tracker"); return PFT_ERR_INVALID; }
  t->timing = on != 0;
  return PFT_OK;
}

int pft_tracker_get_timing(pft_tracker* t, float* weight_ms, float* compute_ms) {
  if (!t) { set_last_error("null tracker"); return PFT_ERR_INVALID; }
  if (!t->timing || !t->ev_c0) { set_last_error("timing is not enabled or no compute() has run"); return PFT_ERR_STATE; }
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  PFT_CUDA_TRY(cudaStreamSynchronize(t->run_stream()));
  float w = 0.f;
  for (int k = 0; k < t->n_ev_used; ++k) {
    float ms = 0.f;
    PFT_CUDA_TRY(cudaEventElapsedTime(&ms, t->ev_w[2 * k], t->ev_w[2 * k + 1]));
    w += ms;
  }
  float c = 0.f;
  if (cudaEventElapsedTime(&c, t->ev_c0, t->ev_c1) != cudaSuccess) { cudaGetLastError(); c = 0.f; }
  if (weight_ms) *weight_ms = w;
  if (compute_ms) *compute_ms = c;
  return PFT_OK;
}

// timing mode: device time of every kernel of the last compute(), in launch order (the time between the event after
// the previous kernel and the event after this one)
int pft_tracker_get_kernel_times(pft_tracker* t, const char** names, float* ms, int capacity, int* n_out) {
  if (!t) { set_last_error("null tracker"); return PFT_ERR_INVALID; }
  if (!t->timing || !t->ev_c0) { set_last_error("timing is not enabled or no compute() has run"); return PFT_ERR_STATE; }
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  PFT_CUDA_TRY(cudaStreamSynchronize(t->run_stream()));
  if (n_out) *n_out = t->n_ev_k;
  if (t->n_ev_k > capacity) { set_last_error("capacity %d < %d", capacity, t->n_ev_k); return PFT_ERR_CAPACITY; }
  for (int k = 0; k < t->n_ev_k; ++k) {
    float v = 0.f;
    if (cudaEventElapsedTime(&v, k ? t->ev_k[k - 1] : t->ev_c0, t->ev_k[k]) != cudaSuccess) { cudaGetLastError(); v = 0.f; }
    if (names) names[k] = t->ev_k_name[k];
    if (ms) ms[k] = v;
  }
  return PFT_OK;
}

// weight() in its three parts, with the two exchange points exposed, so that a sharded run can be
// driven (and tested) without a communicator: 0 = transforms + local crop box, 1 = index + coherence of
// the local particles, 2 = normalise.  A peer-attached tracker exchanges inside its kernels: it refuses.
int pft_tracker_weight_phase(pft_tracker* t, int phase) {
  if (!t) { set_last_error("null tracker"); return PFT_ERR_INVALID; }
  if (t->peer_mode) { set_last_error("the phase API leaves the exchanges to the caller: not on a tracker attached to peer windows"); return PFT_ERR_STATE; }
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  int rc = prepare_compute(t);
  if (rc) return rc;
  switch (phase) {
    case 0: return weight_phase_box(t);
    case 1:  // (raw slices are readable between the phases)
      if (t->timing) t->n_ev_used = 0;
      if ((rc = weight_phase_eval(t))) return rc;
      return launch_raw_weights(t);
    case 2: return weight_phase_normalize(t);
    default: set_last_error("phase must be 0, 1 or 2"); return PFT_ERR_INVALID;
  }
}
int pft_tracker_get_crop_box(pft_tracker* t, float* aabb6) {
  if (!t || !aabb6) { set_last_error("null argument"); return PFT_ERR_INVALID; }
  TrackerState h;
  int rc = read_state(t, &h);
  if (rc) return rc;
  memcpy(aabb6, h.aabb, sizeof(h.aabb));
  return PFT_OK;
}
int pft_tracker_set_crop_box(pft_tracker* t, const float* aabb6) {
  if (!t || !aabb6 || !t->st.p) { set_last_error("null argument / no state"); return PFT_ERR_INVALID; }
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  PFT_CUDA_TRY(cudaMemcpyAsync(t->st.as<TrackerState>()->aabb, aabb6, 6 * sizeof(float), cudaMemcpyHostToDevice, t->run_stream()));
  PFT_CUDA_TRY(cudaStreamSynchronize(t->run_stream()));
  return PFT_OK;
}
int pft_tracker_get_raw_slice(pft_tracker* t, int rank, float* out, size_t capacity, size_t* n_out) {
  if (!t || !t->raw.p) { set_last_error("null argument / no state"); return PFT_ERR_INVALID; }
  if (rank < 0 || rank >= t->nranks) { set_last_error("bad rank"); return PFT_ERR_INVALID; }
  const size_t n = (size_t)t->slice_cap();
  if (n_out) *n_out = n;
  if (n > capacity || !out) { set_last_error("capacity %zu < %zu", capacity, n); return PFT_ERR_CAPACITY; }
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  PFT_CUDA_TRY(cudaStreamSynchronize(t->run_stream()));
  PFT_CUDA_TRY(cudaMemcpy(out, t->raw.as<float>() + (size_t)rank * n, n * sizeof(float), cudaMemcpyDeviceToHost));
  return PFT_OK;
}
int pft_tracker_set_raw_slice(pft_tracker* t, int rank, const float* in, size_t n) {
  if (!t || !in || !t->raw.p) { set_last_error("null argument / no state"); return PFT_ERR_INVALID; }
  if (rank < 0 || rank >= t->nranks || n != (size_t)t->slice_cap()) { set_last_error("bad rank or slice length"); return PFT_ERR_INVALID; }
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  PFT_CUDA_TRY(cudaMemcpyAsync(t->raw.as<float>() + (size_t)rank * n, in, n * sizeof(float), cudaMemcpyHostToDevice, t->run_stream()));
  PFT_CUDA_TRY(cudaStreamSynchronize(t->run_stream()));
  return PFT_OK;
}

// ------------------------------------------------------------------ multi-GPU
int pft_comm_get_unique_id(void* id128) {
  if (!id128) { set_last_error("null id"); return PFT_ERR_INVALID; }
  int rc = load_nccl();
  if (rc) return rc;
  PFT_NCCL_TRY(g_nccl.GetUniqueId(id128));
  return PFT_OK;
}

int pft_context_comm_init(pft_context* ctx, int nranks, int rank, const void* id128) {
  if (!ctx || !id128) { set_last_error("null argument"); return PFT_ERR_INVALID; }
  if (nranks < 1 || rank < 0 || rank >= nranks) { set_last_error("bad rank %d of %d", rank, nranks); return PFT_ERR_INVALID; }
  if (ctx->comm) { set_last_error("context already has a communicator"); return PFT_ERR_STATE; }
  PFT_CUDA_TRY(cudaSetDevice(ctx->device));
  ctx->nranks = nranks; ctx->rank = rank;
  if (nranks == 1) return PFT_OK;
  int rc = load_nccl();
  if (rc) return rc;
  UidByValue uid;
  memcpy(uid.internal, id128, 128);
  PFT_NCCL_TRY(g_nccl.CommInitRank(&ctx->comm, nranks, uid, rank));
  return PFT_OK;
}

int pft_context_comm_destroy(pft_context* ctx) {
  if (!ctx) { set_last_error("null context"); return PFT_ERR_INVALID; }
  if (ctx->comm) {
    PFT_CUDA_TRY(cudaSetDevice(ctx->device));
    PFT_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    g_nccl.CommDestroy(ctx->comm);
    ctx->comm = nullptr;
  }
  ctx->nranks = 1; ctx->rank = 0;
  return PFT_OK;
}

// Replicates a cloud (header + `capacity` points) from `root` to every rank of the context's
// communicator: the NVLink broadcast of the downsampled scene.  The point count stays on the device.
int pft_cloud_broadcast(pft_cloud* cloud, size_t capacity, int root) {
  if (!cloud) { set_last_error("null cloud"); return PFT_ERR_INVALID; }
  pft_context* ctx = cloud->ctx;
  if (root < 0 || root >= ctx->nranks) { set_last_error("bad root %d", root); return PFT_ERR_INVALID; }
  if (ctx->nranks == 1) return PFT_OK;
  if (!ctx->comm) { set_last_error("context has no communicator"); return PFT_ERR_COMM; }
  PFT_CUDA_TRY(cudaSetDevice(ctx->device));
  { int jrc = cloud->join_upload(); if (jrc) return jrc; }
  // every rank posts the SAME count (mismatched counts are undefined in NCCL): the root must hold `capacity` points of
  // storage -- it is never clamped to what the root happens to have
  if (ctx->rank == root) {
    if (cloud->capacity < capacity) { set_last_error("root cloud holds %zu points of storage, the broadcast needs %zu", cloud->capacity, capacity); return PFT_ERR_CAPACITY; }
  } else {
    int rc = cloud->ensure(capacity);
    if (rc) return rc;
  }
  PFT_NCCL_TRY(g_nccl.GroupStart());
  PFT_NCCL_TRY(g_nccl.Broadcast(cloud->hdr.p, cloud->hdr.p, sizeof(CloudHeader), kNcclChar, root, ctx->comm, ctx->stream));
  PFT_NCCL_TRY(g_nccl.Broadcast(cloud->pts.p, cloud->pts.p, capacity * sizeof(float4), kNcclChar, root, ctx->comm, ctx->stream));
  PFT_NCCL_TRY(g_nccl.GroupEnd());
  if (ctx->rank != root) cloud->written(-1);
  return PFT_OK;
}

int pft_tracker_comm_init(pft_tracker* t, int nranks, int rank, const void* id128) {
  if (!t) { set_last_error("null tracker"); return PFT_ERR_INVALID; }
  if (t->n_cap > 0) { set_last_error("pft_tracker_comm_init must precede the first compute()/set_particles()"); return PFT_ERR_STATE; }
  pft_context* ctx = t->ctx;
  if (!ctx->comm && ctx->nranks == 1) {
    int rc = pft_context_comm_init(ctx, nranks, rank, id128);
    if (rc) return rc;
  } else if (ctx->nranks != nranks || ctx->rank != rank) {
    set_last_error("context communicator is rank %d of %d, asked for %d of %d", ctx->rank, ctx->nranks, rank, nranks);
    return PFT_ERR_INVALID;
  }
  t->nranks = ctx->nranks; t->rank = ctx->rank; t->comm = ctx->comm;
  invalidate_graph(t);
  return PFT_OK;
}

int pft_tracker_comm_destroy(pft_tracker* t) {
  if (!t) { set_last_error("null tracker"); return PFT_ERR_INVALID; }
  t->comm = nullptr;
  invalidate_graph(t);
  return PFT_OK;
}

// Set the sharding without a communicator: this rank evaluates particles i % nranks == rank only and the
// caller moves the crop box / raw weights itself.  Used by the world-size-2 CPU (gloo) tests of the host
// logic and by single-GPU emulation of a sharded run.
int pft_tracker_set_shard(pft_tracker* t, int nranks, int rank) {
  if (!t) { set_last_error("null tracker"); return PFT_ERR_INVALID; }
  if (nranks < 1 || rank < 0 || rank >= nranks) { set_last_error("bad rank %d of %d", rank, nranks); return PFT_ERR_INVALID; }
  if (t->n_cap > 0) { set_last_error("pft_tracker_set_shard must precede the first compute()/set_particles()"); return PFT_ERR_STATE; }
  t->nranks = nranks; t->rank = rank;
  invalidate_graph(t);
  return PFT_OK;
}

// ------------------------------------------------------------------ NVLink peer exchange (replaces the NCCL collectives)
// The two exchange steps of weight() become peer stores issued by the producing kernels over NVLink into windows
// that every rank maps with CUDA IPC (see PeerWindow in pft_tracker_kernels.cuh).  Call order on every rank:
//   set_shard / comm_init (rank layout) -> particle numbers -> peer_export -> [host framework all-gathers the
//   64-byte handles] -> peer_attach -> compute ...
static int alloc_peer_window(pft_tracker* t) {
  int rc = ensure_particle_buffers(t);
  if (rc) return rc;
  if (!t->peer_local) {
    const size_t bytes = sizeof(PeerWindow) + (size_t)t->slice_cap() * t->nranks * sizeof(float);
    PFT_CUDA_TRY(cudaMalloc(&t->peer_local, bytes));
    PFT_CUDA_TRY(cudaMemset(t->peer_local, 0, bytes));
    PFT_CUDA_TRY(cudaDeviceSynchronize());
    t->peer_bytes = bytes;
  }
  return PFT_OK;
}

int pft_tracker_peer_export(pft_tracker* t, void* handle64) {
  if (!t || !handle64) { set_last_error("null argument"); return PFT_ERR_INVALID; }
  if (t->nranks < 2) { set_last_error("peer exchange needs a rank layout: call pft_tracker_set_shard / pft_tracker_comm_init first"); return PFT_ERR_STATE; }
  if (t->nranks > kMaxPeers) { set_last_error("peer exchange supports up to %d ranks", kMaxPeers); return PFT_ERR_INVALID; }
  static_assert(sizeof(cudaIpcMemHandle_t) == PFT_PEER_HANDLE_BYTES, "handle size");
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  int rc = alloc_peer_window(t);
  if (rc) return rc;
  cudaIpcMemHandle_t h;
  PFT_CUDA_TRY(cudaIpcGetMemHandle(&h, t->peer_local));
  memcpy(handle64, &h, sizeof(h));
  return PFT_OK;
}

int pft_tracker_peer_attach(pft_tracker* t, const void* handles) {
  if (!t || !handles) { set_last_error("null argument"); return PFT_ERR_INVALID; }
  if (!t->peer_local) { set_last_error("pft_tracker_peer_export must precede pft_tracker_peer_attach"); return PFT_ERR_STATE; }
  if (t->peer_mode) { set_last_error("peer windows are already attached"); return PFT_ERR_STATE; }
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  PeerSet ps{};
  ps.nranks = t->nranks; ps.rank = t->rank;
  for (int r = 0; r < t->nranks; ++r) {
    if (r == t->rank) { ps.win[r] = reinterpret_cast<PeerWindow*>(t->peer_local); continue; }
    cudaIpcMemHandle_t h;
    memcpy(&h, (const char*)handles + (size_t)r * PFT_PEER_HANDLE_BYTES, sizeof(h));
    void* p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      set_last_error("cudaIpcOpenMemHandle(rank %d) -> %s (peer exchange needs NVLink/P2P between the GPUs of one node)", r, cudaGetErrorString(e));
      cudaGetLastError();
      for (int q = 0; q < r; ++q) if (q != t->rank && ps.win[q]) cudaIpcCloseMemHandle(ps.win[q]);
      return PFT_ERR_COMM;
    }
    ps.win[r] = reinterpret_cast<PeerWindow*>(p);
  }
  t->peers = ps;
  t->peer_mode = true;
  invalidate_graph(t);
  return PFT_OK;
}

int pft_tracker_peer_detach(pft_tracker* t) {
  if (!t) { set_last_error("null tracker"); return PFT_ERR_INVALID; }
  if (!t->peer_local && !t->peer_mode) return PFT_OK;
  cudaSetDevice(t->ctx->device);
  cudaStreamSynchronize(t->run_stream());
  if (t->peer_mode && t->peer_ipc) {
    for (int r = 0; r < t->peers.nranks; ++r) if (r != t->peers.rank && t->peers.win[r]) cudaIpcCloseMemHandle(t->peers.win[r]);
  }
  t->peer_ipc = true;
  if (t->peer_local) cudaFree(t->peer_local);
  t->peer_local = nullptr; t->peer_bytes = 0; t->peer_mode = false;
  t->peers = PeerSet{};
  invalidate_graph(t);
  return PFT_OK;
}

// ------------------------------------------------------------------ scene distribution by peer stores
// Call order on every rank: pft_cloud_peer_export (same capacity everywhere) -> the host framework all-gathers the
// PFT_CLOUD_PEER_HANDLE_BYTES handles in rank order -> pft_cloud_peer_attach -> per frame: the root fills the cloud
// (upload + downsample), every rank calls pft_cloud_peer_broadcast.  The root must not refill the cloud before every
// peer has finished reading the previous scene: inside a peer-mode tracker loop that is implied (the root's last
// normalize of a frame waits for every rank's raw weights, which a rank pushes after its last read of the scene);
// elsewhere the caller orders it.
int pft_cloud_peer_export(pft_cloud* c, size_t capacity, void* handles) {
  if (!c || !handles) { set_last_error("null argument"); return PFT_ERR_INVALID; }
  if (c->peer_attached) { set_last_error("the cloud's peer mappings are already attached"); return PFT_ERR_STATE; }
  static_assert(3 * sizeof(cudaIpcMemHandle_t) == PFT_CLOUD_PEER_HANDLE_BYTES, "handle size");
  PFT_CUDA_TRY(cudaSetDevice(c->ctx->device));
  PFT_CUDA_TRY(cudaStreamSynchronize(c->ctx->stream));
  if (!c->peer_exported) {
    const size_t keep = c->capacity;
    int rc = c->ensure(std::max(capacity, c->capacity));
    if (rc) return rc;
    c->capacity = keep;  // (ensure() records its argument as the point bound: the contents did not change)
    if ((rc = c->peer_sync.reserve(2 * sizeof(unsigned int)))) return rc;
    PFT_CUDA_TRY(cudaMemset(c->peer_sync.p, 0, 2 * sizeof(unsigned int)));
    if (!c->peer_error) {
      PFT_CUDA_TRY(cudaHostAlloc((void**)&c->peer_error, sizeof(unsigned int), cudaHostAllocMapped));
      *c->peer_error = 0u;
    }
    PFT_CUDA_TRY(cudaDeviceSynchronize());
    c->peer_capacity = c->pts.bytes / sizeof(float4);
    c->peer_exported = true;
  } else if (capacity > c->peer_capacity) {
    set_last_error("the cloud was exported with room for %zu points", c->peer_capacity);
    return PFT_ERR_CAPACITY;
  }
  cudaIpcMemHandle_t h[3];
  PFT_CUDA_TRY(cudaIpcGetMemHandle(&h[0], c->pts.p));
  PFT_CUDA_TRY(cudaIpcGetMemHandle(&h[1], c->hdr.p));
  PFT_CUDA_TRY(cudaIpcGetMemHandle(&h[2], c->peer_sync.p));
  memcpy(handles, h, sizeof(h));
  return PFT_OK;
}

int pft_cloud_peer_attach(pft_cloud* c, const void* handles, int nranks, int rank) {
  if (!c || !handles) { set_last_error("null argument"); return PFT_ERR_INVALID; }
  if (!c->peer_exported) { set_last_error("pft_cloud_peer_export must precede pft_cloud_peer_attach"); return PFT_ERR_STATE; }
  if (c->peer_attached) { set_last_error("the cloud's peer mappings are already attached"); return PFT_ERR_STATE; }
  if (nranks < 2 || nranks > kMaxPeers || rank < 0 || rank >= nranks) { set_last_error("bad rank %d of %d (at most %d ranks)", rank, nranks, kMaxPeers); return PFT_ERR_INVALID; }
  PFT_CUDA_TRY(cudaSetDevice(c->ctx->device));
  void** maps[3] = {c->peer_pts, c->peer_hdr, c->peer_flag};
  void* local[3] = {c->pts.p, c->hdr.p, c->peer_sync.p};
  for (int r = 0; r < nranks; ++r) {
    for (int k = 0; k < 3; ++k) {
      if (r == rank) { maps[k][r] = local[k]; continue; }
      cudaIpcMemHandle_t h;
      memcpy(&h, (const char*)handles + (size_t)r * PFT_CLOUD_PEER_HANDLE_BYTES + (size_t)k * sizeof(h), sizeof(h));
      void* p = nullptr;
      cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
      if (e != cudaSuccess) {
        set_last_error("cudaIpcOpenMemHandle(rank %d) -> %s (scene distribution by peer stores needs NVLink/P2P between the GPUs of one node)", r, cudaGetErrorString(e));
        cudaGetLastError();
        c->peer_nranks = nranks; c->peer_rank = rank; c->peer_attached = true;
        pft_cloud_peer_detach(c);  // closes what was opened so far
        return PFT_ERR_COMM;
      }
      maps[k][r] = p;
    }
  }
  c->peer_nranks = nranks; c->peer_rank = rank; c->peer_attached = true;
  return PFT_OK;
}

int pft_cloud_peer_broadcast(pft_cloud* c, int root) {
  if (!c) { set_last_error("null cloud"); return PFT_ERR_INVALID; }
  if (!c->peer_attached) { set_last_error("pft_cloud_peer_attach must precede pft_cloud_peer_broadcast"); return PFT_ERR_STATE; }
  if (root < 0 || root >= c->peer_nranks) { set_last_error("bad root %d", root); return PFT_ERR_INVALID; }
  if (*(volatile unsigned int*)c->peer_error) {
    *c->peer_error = 0u;
    set_last_error(c->peer_rank == root ? "an earlier scene held more points than the peers' clouds have room for (%zu)" : "an earlier scene did not arrive within the time limit (rank %d gone?)",
                   c->peer_rank == root ? c->peer_capacity : (size_t)root);
    return c->peer_rank == root ? PFT_ERR_CAPACITY : PFT_ERR_COMM;
  }
  PFT_CUDA_TRY(cudaSetDevice(c->ctx->device));
  cudaStream_t s = c->ctx->stream;
  const unsigned int epoch = ++c->peer_epoch;
  unsigned int* d_err = nullptr;
  PFT_CUDA_TRY(cudaHostGetDevicePointer((void**)&d_err, c->peer_error, 0));
  if (c->peer_rank == root) {
    int jrc = c->join_upload();
    if (jrc) return jrc;
    CloudPeerSet ps{};
    ps.nranks = c->peer_nranks; ps.rank = c->peer_rank;
    for (int r = 0; r < c->peer_nranks; ++r) {
      ps.pts[r] = reinterpret_cast<float4*>(c->peer_pts[r]); ps.hdr[r] = reinterpret_cast<CloudHeader*>(c->peer_hdr[r]);
      ps.sync[r] = reinterpret_cast<unsigned int*>(c->peer_flag[r]);
    }
    const int grid = std::max(1, std::min(c->ctx->sm_count, (int)((std::max<size_t>(c->capacity, 1) + 255) / 256)));
    cloud_push_kernel<<<grid, 256, 0, s>>>(c->d_pts(), c->d_hdr(), ps, epoch, (int)std::min<size_t>(c->peer_capacity, 0x7fffffff), d_err);
    PFT_LAUNCH_CHECK();
  } else {
    cloud_wait_kernel<<<1, 1, 0, s>>>(c->peer_sync.as<unsigned int>(), epoch, d_err);
    PFT_LAUNCH_CHECK();
    c->written(-1);
    c->capacity = c->peer_capacity;  // (the point count stays on the device: this is the host's bound)
  }
  return PFT_OK;
}

int pft_cloud_peer_detach(pft_cloud* c) {
  if (!c) { set_last_error("null cloud"); return PFT_ERR_INVALID; }
  if (!c->peer_exported && !c->peer_attached) return PFT_OK;
  cudaSetDevice(c->ctx->device);
  cudaStreamSynchronize(c->ctx->stream);
  if (c->peer_attached) {
    void** maps[3] = {c->peer_pts, c->peer_hdr, c->peer_flag};
    for (int r = 0; r < c->peer_nranks; ++r)
      for (int k = 0; k < 3; ++k) { if (r != c->peer_rank && maps[k][r]) cudaIpcCloseMemHandle(maps[k][r]); maps[k][r] = nullptr; }
  }
  c->peer_sync.release();
  if (c->peer_error) { cudaFreeHost(c->peer_error); c->peer_error = nullptr; }
  c->peer_exported = false; c->peer_attached = false; c->peer_nranks = 0; c->peer_epoch = 0;
  return PFT_OK;
}

// ------------------------------------------------------------------ single-process multi-device mode
// The reference is ONE process (ref: src/auto_tracking.cpp: one node, one tracker object).  pft_tracker_set_devices lets
// that one tracker object drive n GPUs: rank 0 is the tracker itself (on devices[0] = its context's device), every
// further device gets a follower tracker in a context of its own; the particle set is sharded as in the multi-process
// mode (particle i on rank i % n), the exchange windows of weight() are mapped directly (cudaDeviceEnablePeerAccess),
// the scene and the model reach every device through the followers' replicas of them.  Call it right after pft_tracker_create: the
// setters called afterwards are forwarded to the followers.  compute() and the getters work as before (the replicated
// state is read from rank 0); the stage-by-stage debugging API (resample / weight / update) is not forwarded.
int pft_tracker_set_devices(pft_tracker* t, int n, const int* devices) {
  if (!t || n < 1 || !devices) { set_last_error("pft_tracker_set_devices: bad arguments"); return PFT_ERR_INVALID; }
  if (n > kMaxPeers) { set_last_error("at most %d devices", kMaxPeers); return PFT_ERR_INVALID; }
  if (t->n_cap > 0 || t->comm || t->nranks > 1 || !t->followers.empty()) { set_last_error("pft_tracker_set_devices must be the first call on a new tracker"); return PFT_ERR_STATE; }
  if (devices[0] != t->ctx->device) { set_last_error("devices[0] must be the device of the tracker's context (%d)", t->ctx->device); return PFT_ERR_INVALID; }
  if (n == 1) return PFT_OK;
  int count = 0;
  PFT_CUDA_TRY(cudaGetDeviceCount(&count));
  for (int r = 0; r < n; ++r) if (devices[r] < 0 || devices[r] >= count) { set_last_error("device %d out of range [0,%d)", devices[r], count); return PFT_ERR_INVALID; }
  for (int a = 0; a < n; ++a) {
    for (int b = 0; b < n; ++b) {
      int rc = enable_peer_access(devices[a], devices[b]);
      if (rc) return rc;
    }
  }
  int rc = PFT_OK;
  for (int r = 1; r < n && !rc; ++r) {
    pft_tracker::Follower f;
    if ((rc = pft_context_create(devices[r], &f.ctx))) break;
    if (!rc) rc = pft_tracker_create(f.ctx, t->kld ? 1 : 0, &f.t);
    if (!rc) { f.t->nranks = n; f.t->rank = r; f.t->graph_enabled = t->graph_enabled; }
    t->followers.push_back(f);  // (also on failure: destroy_followers releases what exists)
  }
  if (rc) { destroy_followers(t); return rc; }
  t->nranks = n; t->rank = 0;
  invalidate_graph(t);
  PFT_CUDA_TRY(cudaSetDevice(t->ctx->device));
  return PFT_OK;
}

/* the follower tracker of rank `rank` (1 .. n-1) in multi-device mode: for inspection (getters) only */
int pft_tracker_get_follower(pft_tracker* t, int rank, pft_tracker** out) {
  if (!t || !out) { set_last_error("null argument"); return PFT_ERR_INVALID; }
  if (rank < 1 || rank > (int)t->followers.size()) { set_last_error("no follower of rank %d", rank); return PFT_ERR_INVALID; }
  *out = t->followers[rank - 1].t;
  return PFT_OK;
}

#ifdef PFT_TRACE
// tuning builds only (not declared in pft.h): read and re-arm the stamps (even entries of a pair are minima, see the macros)
__attribute__((visibility("default"))) int pft_debug_trace(unsigned long long* out64, const unsigned long long* init64) {
  cudaDeviceSynchronize();
  if (cudaMemcpyFromSymbol(out64, g_trace, sizeof(unsigned long long) * 64) != cudaSuccess) return -1;
  cudaMemcpyToSymbol(g_trace, init64, sizeof(unsigned long long) * 64);
  return 0;
}
#endif
#ifdef PFT_STATS
// tuning builds only (not declared in pft.h): read and clear the search statistics
__attribute__((visibility("default"))) int pft_debug_stats(unsigned long long* out16) {
  cudaDeviceSynchronize();
  if (cudaMemcpyFromSymbol(out16, g_stats, sizeof(unsigned long long) * 48) != cudaSuccess) return -1;
  unsigned long long z[48] = {0};
  cudaMemcpyToSymbol(g_stats, z, sizeof(z));
  return 0;
}
#endif

int pft_tracker_graph_replays(pft_tracker* t, uint64_t* n) {
  if (!t || !n) { set_last_error("null argument"); return PFT_ERR_INVALID; }
  *n = t->graph_replays;
  return PFT_OK;
}

}  // extern "C"
