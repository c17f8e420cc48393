// =====================================================================================
// pft_oracle.cpp -- CPU ORACLE (TEST INFRASTRUCTURE, NOT PRODUCT CODE)
//
// A plain C++17/OpenMP restatement of the PCL-1.8.0 particle-filter tracking path that
// /root/reference/src/auto_tracking.cpp drives (SURVEY.md section 8a, Appendix A).  Only
// tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
// load this library.  The product path (pcl_tracking_b200/) never links or imports it.
//
// PARITY UNPINNED: the arithmetic of this path lives in PCL 1.8.0 (find_package(PCL 1.8.0
// EXACT), ref: CMakeLists.txt:4), which is NOT vendored under /root/reference, is not
// installed in the build image and cannot be fetched (no network).  The reference ships no
// golden vectors, KATs or PCD fixtures for the tracking path (ref: test/*.cpp never touch
// pcl::tracking; .gitignore:1-4 excludes *.pcd).  This file restates the published
// algorithms; it is pinned only by the derived known-answer vectors of SURVEY.md A.10
// (tests/test_oracle_kat.py) and by internal invariants.
//
// Arithmetic contract shared with the CUDA path (so nearest-neighbour indices can be
// compared bit-for-bit): every fp32/fp64 operation is individually rounded (no FMA
// contraction: this file is built with -ffp-contract=off and default -march), and
// sin/cos/atan2/asin/exp are evaluated in double and rounded to float where PCL calls the
// float overloads.
//
// Each function cites the reference call site (ref: src/auto_tracking.cpp:LINE) and the
// upstream PCL-1.8.0 file it restates.
// =====================================================================================
#include <algorithm>
#include <array>
#include <cfloat>
#include <chrono>
#include <climits>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <memory>
#include <random>
#include <unordered_map>
#include <vector>
#ifdef _OPENMP
#include <omp.h>
#endif

extern "C" {
typedef struct { float x, y, z; uint32_t rgba; } orc_point;
typedef struct { float x, y, z, one, roll, pitch, yaw, weight; } orc_particle;
}

namespace {

using Pt = orc_point;
using Particle = orc_particle;

inline bool finite3(const Pt& p) { return std::isfinite(p.x) && std::isfinite(p.y) && std::isfinite(p.z); }

// ---------------------------------------------------------------------------------
// transcendental helpers: double evaluation rounded to float (arithmetic contract)
// ---------------------------------------------------------------------------------
inline float cosf_c(float a) { return (float)std::cos((double)a); }
inline float sinf_c(float a) { return (float)std::sin((double)a); }
inline float atan2f_c(float y, float x) { return (float)std::atan2((double)y, (double)x); }
inline float asinf_c(float v) { return (float)std::asin((double)v); }

// ---------------------------------------------------------------------------------
// pcl::getTransformation(x,y,z,roll,pitch,yaw)  [PCL-1.8.0 common/impl/eigen.hpp]
// = ParticleXYZRPY::toEigenMatrix (tracking/impl/tracking.hpp); ref: src/auto_tracking.cpp:310
// Row-major 3x4 (R | t).
// ---------------------------------------------------------------------------------
struct Mat34 { float m[12]; };

Mat34 particle_to_matrix(float x, float y, float z, float roll, float pitch, float yaw) {
  float A = cosf_c(yaw), B = sinf_c(yaw), C = cosf_c(pitch), D = sinf_c(pitch);
  float E = cosf_c(roll), F = sinf_c(roll), DE = D * E, DF = D * F;
  Mat34 t;
  t.m[0] = A * C;  t.m[1] = A * DF - B * E;  t.m[2]  = B * F + A * DE;  t.m[3]  = x;
  t.m[4] = B * C;  t.m[5] = A * E + B * DF;  t.m[6]  = B * DE - A * F;  t.m[7]  = y;
  t.m[8] = -D;     t.m[9] = C * F;           t.m[10] = C * E;           t.m[11] = z;
  return t;
}
inline Mat34 particle_to_matrix(const Particle& p) { return particle_to_matrix(p.x, p.y, p.z, p.roll, p.pitch, p.yaw); }

// pcl::getEulerAngles / getTranslationAndEulerAngles [common/impl/eigen.hpp]; = ParticleXYZRPY::toState
void matrix_to_rpy(const float* m /*3x4 row-major*/, float& roll, float& pitch, float& yaw) {
  roll = atan2f_c(m[9], m[10]);
  pitch = asinf_c(-m[8]);
  yaw = atan2f_c(m[4], m[0]);
}

// pcl::transformPointCloud, dense branch [common/impl/transforms.hpp]: ((m0*x + m1*y) + m2*z) + m3
inline void xform(const Mat34& t, float x, float y, float z, float& ox, float& oy, float& oz) {
  ox = ((t.m[0] * x + t.m[1] * y) + t.m[2] * z) + t.m[3];
  oy = ((t.m[4] * x + t.m[5] * y) + t.m[6] * z) + t.m[7];
  oz = ((t.m[8] * x + t.m[9] * y) + t.m[10] * z) + t.m[11];
}

// ---------------------------------------------------------------------------------
// Eigen quaternion helpers (float), evaluation order written out
// ---------------------------------------------------------------------------------
struct Quat { float w, x, y, z; };

// Eigen::Quaternionf(Matrix3f) [Eigen/src/Geometry/Quaternion.h quaternionbase_assign_impl<_,3,3>]
Quat quat_from_matrix(const float* m /*3x4 row-major, rotation part*/) {
  auto M = [&](int r, int c) { return m[r * 4 + c]; };
  Quat q;
  float t = (M(0, 0) + M(1, 1)) + M(2, 2);
  if (t > 0.f) {
    t = std::sqrt(t + 1.0f);
    q.w = 0.5f * t;
    t = 0.5f / t;
    q.x = (M(2, 1) - M(1, 2)) * t;
    q.y = (M(0, 2) - M(2, 0)) * t;
    q.z = (M(1, 0) - M(0, 1)) * t;
  } else {
    int i = 0;
    if (M(1, 1) > M(0, 0)) i = 1;
    if (M(2, 2) > M(i, i)) i = 2;
    int j = (i + 1) % 3, k = (j + 1) % 3;
    t = std::sqrt(((M(i, i) - M(j, j)) - M(k, k)) + 1.0f);
    float v[3];
    v[i] = 0.5f * t;
    t = 0.5f / t;
    q.w = (M(k, j) - M(j, k)) * t;
    v[j] = (M(j, i) + M(i, j)) * t;
    v[k] = (M(k, i) + M(i, k)) * t;
    q.x = v[0]; q.y = v[1]; q.z = v[2];
  }
  return q;
}
inline Quat quat_mul(const Quat& a, const Quat& b) {
  Quat r;
  r.w = ((a.w * b.w - a.x * b.x) - a.y * b.y) - a.z * b.z;
  r.x = ((a.w * b.x + a.x * b.w) + a.y * b.z) - a.z * b.y;
  r.y = ((a.w * b.y + a.y * b.w) + a.z * b.x) - a.x * b.z;
  r.z = ((a.w * b.z + a.z * b.w) + a.x * b.y) - a.y * b.x;
  return r;
}
inline Quat quat_normalize(const Quat& q) {
  float n2 = ((q.x * q.x + q.y * q.y) + q.z * q.z) + q.w * q.w;
  float n = std::sqrt(n2);
  return Quat{q.w / n, q.x / n, q.y / n, q.z / n};
}
// Eigen QuaternionBase::toRotationMatrix
void quat_to_matrix(const Quat& q, float* m /*3x4 row-major; translation untouched*/) {
  float tx = 2.f * q.x, ty = 2.f * q.y, tz = 2.f * q.z;
  float twx = tx * q.w, twy = ty * q.w, twz = tz * q.w;
  float txx = tx * q.x, txy = ty * q.x, txz = tz * q.x;
  float tyy = ty * q.y, tyz = tz * q.y, tzz = tz * q.z;
  m[0] = 1.f - (tyy + tzz); m[1] = txy - twz;         m[2] = txz + twy;
  m[4] = txy + twz;         m[5] = 1.f - (txx + tzz); m[6] = tyz - twx;
  m[8] = txz - twy;         m[9] = tyz + twx;         m[10] = 1.f - (txx + tyy);
}

// ---------------------------------------------------------------------------------
// ParticleXYZRPY::sample(mean, cov) [PCL-1.8.0 tracking/impl/tracking.hpp] with the six
// standard-normal draws z[0..5] injected (sampleNormal(mean,var) = mean + sqrt(var)*z,
// tracking/src/tracking.cpp).  quat_mode=1: PCL>=1.8.0 quaternion-space rotation noise
// (scale 0.2862); quat_mode=0: PCL<=1.7.2 additive RPY noise.  SURVEY A.9.
// Note: upstream takes Affine3f::rotation() (an SVD polar factor) of an exact rotation;
// the oracle uses the linear part directly.
// ---------------------------------------------------------------------------------
void particle_sample(Particle& p, const double* mean, const double* cov, const float* z, int quat_mode) {
  p.x += (float)(mean[0] + std::sqrt(cov[0]) * (double)z[0]);
  p.y += (float)(mean[1] + std::sqrt(cov[1]) * (double)z[1]);
  p.z += (float)(mean[2] + std::sqrt(cov[2]) * (double)z[2]);
  if (!quat_mode) {
    p.roll += (float)(mean[3] + std::sqrt(cov[3]) * (double)z[3]);
    p.pitch += (float)(mean[4] + std::sqrt(cov[4]) * (double)z[4]);
    p.yaw += (float)(mean[5] + std::sqrt(cov[5]) * (double)z[5]);
    return;
  }
  Mat34 cur = particle_to_matrix(p.x, p.y, p.z, p.roll, p.pitch, p.yaw);
  Quat q_cur = quat_from_matrix(cur.m);
  Mat34 mr = particle_to_matrix((float)mean[0], (float)mean[1], (float)mean[2], (float)mean[3], (float)mean[4], (float)mean[5]);
  Quat q_mean = quat_from_matrix(mr.m);
  const float scale_factor = 0.2862f;
  float a = (float)(std::sqrt((double)scale_factor * cov[3]) * (double)z[3]);
  float b = (float)(std::sqrt((double)scale_factor * cov[4]) * (double)z[4]);
  float c = (float)(std::sqrt((double)scale_factor * cov[5]) * (double)z[5]);
  Quat qs = quat_normalize(Quat{1.f, a, b, c});  // Quaternionf(Vector4f(a,b,c,1)): coeffs x,y,z,w
  Quat qr = quat_mul(quat_mul(qs, q_mean), q_cur);
  float R[12];
  quat_to_matrix(qr, R);
  matrix_to_rpy(R, p.roll, p.pitch, p.yaw);
}

// ---------------------------------------------------------------------------------
// HSVColorCoherence [PCL-1.8.0 tracking/impl/hsv_color_coherence.hpp], SURVEY A.4
// ---------------------------------------------------------------------------------
int div_table_entry(int i) {
  if (i == 0) return 0;
  return (int)std::floor(1044480.0 / (double)i + 0.5);  // round((255<<12)/i)
}
struct DivTable { int v[256]; DivTable() { for (int i = 0; i < 256; ++i) v[i] = div_table_entry(i); } };
const DivTable g_div;

void rgb2hsv_int(int r, int g, int b, int& h, int& s, int& v) {
  const int hsv_shift = 12;
  int vmin;
  v = std::max(r, std::max(g, b));
  vmin = std::min(r, std::min(g, b));
  int diff = v - vmin;
  int vr = (v == r) ? -1 : 0;
  int vg = (v == g) ? -1 : 0;
  s = (diff * g_div.v[v]) >> hsv_shift;
  h = (vr & (g - b)) + (~vr & ((vg & (b - r + 2 * diff)) + ((~vg) & (r - g + 4 * diff))));
  h = (h * g_div.v[diff] * 15 + (1 << (hsv_shift + 6))) >> (7 + hsv_shift);
  h += h < 0 ? 180 : 0;
}
inline void rgb2hsv_f(int r, int g, int b, float& fh, float& fs, float& fv) {
  int h, s, v;
  rgb2hsv_int(r, g, b, h, s, v);
  fh = (float)h / 180.0f; fs = (float)s / 255.0f; fv = (float)v / 255.0f;
}
// rgba layout: byte0=b, byte1=g, byte2=r, byte3=a (PointXYZRGBA). Upstream passes (Red, Blue, Green).
inline void rgba_to_hsv_pcl(uint32_t rgba, float& h, float& s, float& v) {
  int B = rgba & 0xff, G = (rgba >> 8) & 0xff, R = (rgba >> 16) & 0xff;
  rgb2hsv_f(R, B, G, h, s, v);  // upstream quirk: G and B swapped
}
double hsv_coherence(uint32_t src, uint32_t tgt, double weight, double hw, double sw, double vw) {
  float sh, ss, sv, th, ts, tv;
  rgba_to_hsv_pcl(src, sh, ss, sv);
  rgba_to_hsv_pcl(tgt, th, ts, tv);
  const float hd = std::fabs(sh - th);
  float hd2;
  if (sh < th) hd2 = std::fabs(1.0f + sh - th); else hd2 = std::fabs(1.0f + th - sh);
  float h_diff;
  if (hd < hd2) h_diff = (float)hw * hd * hd; else h_diff = (float)hw * hd2 * hd2;
  const float s_diff = (float)sw * (ss - ts) * (ss - ts);
  const float v_diff = (float)vw * (sv - tv) * (sv - tv);
  const float diff2 = h_diff + s_diff + v_diff;
  return 1.0 / (1.0 + weight * (double)diff2);
}
// DistanceCoherence [tracking/impl/distance_coherence.hpp]: d = float 4-vector norm, squared in double
inline double distance_coherence_d2(float d2_float, double weight) {
  double d = (double)std::sqrt(d2_float);
  return 1.0 / (1.0 + d * d * weight);
}
inline float sqdist(float ax, float ay, float az, float bx, float by, float bz) {
  float dx = ax - bx, dy = ay - by, dz = az - bz;
  return (dx * dx + dy * dy) + dz * dz;
}

// ---------------------------------------------------------------------------------
// KLD bound [PCL-1.8.0 tracking/kld_adaptive_particle_filter.h], SURVEY A.7
// ---------------------------------------------------------------------------------
double normal_quantile(double u) {
  static const double a[9] = {1.24818987e-4, -1.075204047e-3, 5.198775019e-3, -0.019198292004, 0.059054035642,
                              -0.151968751364, 0.319152932694, -0.5319230073, 0.797884560593};
  static const double b[15] = {-4.5255659e-5, 1.5252929e-4, -1.9538132e-5, -6.76904986e-4, 1.390604284e-3,
                               -7.9462082e-4, -2.034254874e-3, 6.549791214e-3, -0.010557625006, 0.011630447319,
                               -9.279453341e-3, 5.353579108e-3, -2.141268741e-3, 5.35310549e-4, 0.999936657524};
  double w, y, z;
  if (u == 0.) return 0.5;
  y = u / 2.0;
  if (y < -3.) return 0.0;
  if (y > 3.) return 1.0;
  if (y < 0.0) y = -y;
  if (y < 1.0) {
    w = y * y;
    z = a[0];
    for (int i = 1; i < 9; i++) z = z * w + a[i];
    z *= (y * 2.0);
  } else {
    y -= 2.0;
    z = b[0];
    for (int i = 1; i < 15; i++) z = z * y + b[i];
  }
  if (u < 0.0) return (1.0 - z) / 2.0;
  return (1.0 + z) / 2.0;
}
double kl_bound(int k, double delta, double eps) {
  double z = normal_quantile(delta);
  double chi = 1.0 - 2.0 / (9.0 * (k - 1)) + std::sqrt(2.0 / (9.0 * (k - 1))) * z;
  return ((k - 1.0) / (2.0 * eps)) * chi * chi * chi;
}

// ---------------------------------------------------------------------------------
// Filters
// ---------------------------------------------------------------------------------
// pcl::PassThrough::applyFilterIndices, !keep_organized, non-negative
// [filters/impl/passthrough.hpp]; ref: src/auto_tracking.cpp:536-547
int passthrough(const Pt* in, int n, int field, float lo, float hi, Pt* out, int* out_idx) {
  int m = 0;
  for (int i = 0; i < n; ++i) {
    const Pt& p = in[i];
    if (!finite3(p)) continue;
    float v = field == 0 ? p.x : (field == 1 ? p.y : p.z);
    if (!std::isfinite(v)) continue;
    if (v < lo || v > hi) continue;
    if (out) out[m] = p;
    if (out_idx) out_idx[m] = i;
    ++m;
  }
  return m;
}

inline uint32_t pack_rgb_trunc(float r, float g, float b) {
  return ((uint32_t)(int)r << 16) | ((uint32_t)(int)g << 8) | (uint32_t)(int)b;
}

// Lattice index floor(v * inv), the product rounded to float, saturated to the int range (the GPU's conversion; a plain
// cast of a float outside the int range is undefined).
static int voxel_index(float v, float inv) {
  const float f = std::floor(v * inv);
  return f >= 2147483648.0f ? INT_MAX : (f < -2147483648.0f ? INT_MIN : (int)f);
}

// ApproximateVoxelGrid<PointXYZRGBA>::applyFilter [filters/impl/approximate_voxel_grid.hpp],
// SURVEY A.1; ref: src/auto_tracking.cpp:563-575.  Output capacity: n.
int approx_voxel_grid_pcl(const Pt* in, int n, float leaf, Pt* out) {
  const int histsize = 512;
  struct He { int ix, iy, iz, count; float c[7]; };
  std::vector<He> hist(histsize);
  for (auto& h : hist) { h.count = 0; std::fill(h.c, h.c + 7, 0.f); h.ix = h.iy = h.iz = 0; }
  const float inv = 1.0f / leaf;
  int op = 0;
  auto flush = [&](He& h) {
    Pt o;
    float cnt = (float)h.count;
    o.x = h.c[0] / cnt; o.y = h.c[1] / cnt; o.z = h.c[2] / cnt;
    o.rgba = pack_rgb_trunc(h.c[4] / cnt, h.c[5] / cnt, h.c[6] / cnt);
    out[op++] = o;
  };
  for (int i = 0; i < n; ++i) {
    const Pt& p = in[i];
    int ix = voxel_index(p.x, inv), iy = voxel_index(p.y, inv), iz = voxel_index(p.z, inv);
    // upstream's int hash in unsigned arithmetic: the same bits, without signed overflow
    unsigned hash = ((unsigned)ix * 7171u + (unsigned)iy * 3079u + (unsigned)iz * 4231u) & (unsigned)(histsize - 1);
    He& h = hist[hash];
    if (h.count && (ix != h.ix || iy != h.iy || iz != h.iz)) {
      flush(h);
      h.count = 0; std::fill(h.c, h.c + 7, 0.f);
    }
    h.ix = ix; h.iy = iy; h.iz = iz; h.count++;
    h.c[0] += p.x; h.c[1] += p.y; h.c[2] += p.z; h.c[3] += 1.0f;
    h.c[4] += (float)((p.rgba >> 16) & 0xff); h.c[5] += (float)((p.rgba >> 8) & 0xff); h.c[6] += (float)(p.rgba & 0xff);
  }
  for (auto& h : hist) if (h.count) flush(h);
  return op;
}

// VoxelGrid<PointXYZRGBA>::applyFilter [filters/impl/voxel_grid.hpp], SURVEY A.2;
// ref: src/auto_tracking.cpp:549-561.  std::sort order inside a voxel is unspecified upstream;
// here points of one voxel are summed in ascending input index (stable sort).
int voxel_grid_pcl(const Pt* in, int n, float leaf, Pt* out) {
  const float inv = 1.0f / leaf;
  float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
  for (int i = 0; i < n; ++i) {
    if (!finite3(in[i])) continue;
    const float v[3] = {in[i].x, in[i].y, in[i].z};
    for (int d = 0; d < 3; ++d) { mn[d] = std::min(mn[d], v[d]); mx[d] = std::max(mx[d], v[d]); }
  }
  long long minb[3], maxb[3], divb[3];
  for (int d = 0; d < 3; ++d) {
    minb[d] = (long long)std::floor(mn[d] * inv);
    maxb[d] = (long long)std::floor(mx[d] * inv);
    divb[d] = maxb[d] - minb[d] + 1;
  }
  if (mn[0] > mx[0]) return 0;
  if (divb[0] * divb[1] * divb[2] > (long long)INT_MAX) {  // upstream: warn and copy input
    for (int i = 0; i < n; ++i) out[i] = in[i];
    return n;
  }
  long long mul[3] = {1, divb[0], divb[0] * divb[1]};
  std::vector<std::pair<long long, int>> idx;
  idx.reserve(n);
  for (int i = 0; i < n; ++i) {
    if (!finite3(in[i])) continue;
    long long ijk0 = (long long)std::floor(in[i].x * inv) - minb[0];
    long long ijk1 = (long long)std::floor(in[i].y * inv) - minb[1];
    long long ijk2 = (long long)std::floor(in[i].z * inv) - minb[2];
    idx.emplace_back(ijk0 * mul[0] + ijk1 * mul[1] + ijk2 * mul[2], i);
  }
  std::stable_sort(idx.begin(), idx.end(), [](auto& a, auto& b) { return a.first < b.first; });
  int op = 0;
  size_t i = 0;
  while (i < idx.size()) {
    size_t j = i;
    float c[6] = {0, 0, 0, 0, 0, 0};
    int cnt = 0;
    while (j < idx.size() && idx[j].first == idx[i].first) {
      const Pt& p = in[idx[j].second];
      c[0] += p.x; c[1] += p.y; c[2] += p.z;
      c[3] += (float)((p.rgba >> 16) & 0xff); c[4] += (float)((p.rgba >> 8) & 0xff); c[5] += (float)(p.rgba & 0xff);
      ++cnt; ++j;
    }
    float fc = (float)cnt;
    Pt o; o.x = c[0] / fc; o.y = c[1] / fc; o.z = c[2] / fc;
    o.rgba = pack_rgb_trunc(c[3] / fc, c[4] / fc, c[5] / fc);
    out[op++] = o;
    i = j;
  }
  return op;
}

// Exact one-centroid-per-voxel downsample with the PassThrough predicate folded in: the
// specification of the CUDA K1 kernel (SURVEY A.1 "New build").  Same lattice as upstream
// (floor(coord * (1/leaf)), anchored at the origin, saturated to the int range); voxels are
// emitted in order of first appearance in the input; coordinate sums are held in double and
// added in input order (exact, hence equal to the GPU's in any order, except in voxels on a
// coordinate plane that mix coordinates far below the leaf with leaf-sized ones) and the
// centroid is the double quotient rounded to float; colour means follow upstream:
// (int)(float_sum / float_count), alpha = 0.
int voxel_grid_exact(const Pt* in, int n, float leaf, int field, float lo, float hi, Pt* out) {
  const float inv = 1.0f / leaf;
  struct Acc { double sx = 0, sy = 0, sz = 0; uint32_t r = 0, g = 0, b = 0, cnt = 0; };
  struct Key { int x, y, z; bool operator==(const Key& o) const { return x == o.x && y == o.y && z == o.z; } };
  struct KeyHash { size_t operator()(const Key& k) const {
    uint64_t h = (uint64_t)(uint32_t)k.x * 0x9E3779B185EBCA87ull ^ ((uint64_t)(uint32_t)k.y * 0xC2B2AE3D27D4EB4Full) ^ ((uint64_t)(uint32_t)k.z * 0x165667B19E3779F9ull);
    return (size_t)(h ^ (h >> 29)); } };
  std::unordered_map<Key, int, KeyHash> map;
  map.reserve((size_t)n);
  std::vector<Acc> acc;
  for (int i = 0; i < n; ++i) {
    const Pt& p = in[i];
    if (!finite3(p)) continue;
    float v = field == 0 ? p.x : (field == 1 ? p.y : p.z);
    if (field >= 0 && (v < lo || v > hi)) continue;
    Key k{voxel_index(p.x, inv), voxel_index(p.y, inv), voxel_index(p.z, inv)};
    auto it = map.find(k);
    int id;
    if (it == map.end()) { id = (int)acc.size(); map.emplace(k, id); acc.emplace_back(); } else id = it->second;
    Acc& a = acc[id];
    a.sx += (double)p.x; a.sy += (double)p.y; a.sz += (double)p.z;
    a.r += (p.rgba >> 16) & 0xff; a.g += (p.rgba >> 8) & 0xff; a.b += p.rgba & 0xff; a.cnt++;
  }
  for (size_t i = 0; i < acc.size(); ++i) {
    const Acc& a = acc[i];
    double c = (double)a.cnt;
    float fc = (float)a.cnt;
    Pt o; o.x = (float)(a.sx / c); o.y = (float)(a.sy / c); o.z = (float)(a.sz / c);
    o.rgba = pack_rgb_trunc((float)a.r / fc, (float)a.g / fc, (float)a.b / fc);
    out[i] = o;
  }
  return (int)acc.size();
}

// ---------------------------------------------------------------------------------
// pcl::octree::OctreePointCloudSearch restated (pointer tree) for the Approx coherence
// CPU baseline [octree/impl/octree_pointcloud.hpp, octree_search.hpp], SURVEY A.5
// ---------------------------------------------------------------------------------
struct OctNode {
  OctNode* child[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  std::vector<int>* leaf = nullptr;
};
class PclOctree {
 public:
  explicit PclOctree(double res) : res_(res) {}
  ~PclOctree() { clear(); }
  void clear() {
    freeNode(root_); root_ = nullptr; bbox_defined_ = false; depth_ = 0; leaf_count_ = 0;
    min_[0] = min_[1] = min_[2] = max_[0] = max_[1] = max_[2] = 0.0;
  }
  void setInputCloud(const Pt* pts, int n) {
    clear();
    pts_ = pts; n_ = n;
    root_ = new OctNode();
    for (int i = 0; i < n; ++i) if (finite3(pts[i])) addPoint(i);
  }
  // returns false if tree is empty
  bool approxNearest(float qx, float qy, float qz, int& idx, float& d2) const {
    if (!root_ || leaf_count_ == 0) return false;
    idx = -1; d2 = 0.f;
    unsigned key[3] = {0, 0, 0};
    approxRec(qx, qy, qz, root_, key, 1, idx, d2);
    return idx >= 0;
  }
 private:
  void freeNode(OctNode* n) {
    if (!n) return;
    for (auto c : n->child) freeNode(c);
    delete n->leaf;
    delete n;
  }
  void keyBitSize() {
    const float minValue = std::numeric_limits<float>::epsilon();
    unsigned mk[3];
    for (int d = 0; d < 3; ++d) mk[d] = (unsigned)std::ceil((max_[d] - min_[d]) / res_);
    unsigned max_voxels = std::max(std::max(std::max(mk[0], mk[1]), mk[2]), 2u);
    depth_ = std::max(std::min(30.0, std::ceil(std::log2((double)max_voxels) - minValue)), 0.0);
    double side = (double)(1 << depth_) * res_ - minValue;
    if (leaf_count_ == 0) {
      for (int d = 0; d < 3; ++d) { double over = (side - (max_[d] - min_[d])) / 2.0; min_[d] -= over; max_[d] += over; }
    } else {
      for (int d = 0; d < 3; ++d) max_[d] = min_[d] + side;
    }
  }
  void adoptBBox(const Pt& p) {
    const float minValue = std::numeric_limits<float>::epsilon();
    const double v[3] = {p.x, p.y, p.z};
    while (true) {
      bool lo[3], up[3], any = false;
      for (int d = 0; d < 3; ++d) { lo[d] = v[d] < min_[d]; up[d] = v[d] >= max_[d]; any = any || lo[d] || up[d]; }
      if (any || !bbox_defined_) {
        if (bbox_defined_) {
          unsigned char ci = (unsigned char)(((!up[0]) << 2) | ((!up[1]) << 1) | (!up[2]));
          OctNode* nr = new OctNode();
          nr->child[ci] = root_;
          root_ = nr;
          double side = (double)(1 << depth_) * res_;
          for (int d = 0; d < 3; ++d) if (!up[d]) min_[d] -= side;
          depth_++;
          side = (double)(1 << depth_) * res_ - minValue;
          for (int d = 0; d < 3; ++d) max_[d] = min_[d] + side;
        } else {
          for (int d = 0; d < 3; ++d) { min_[d] = v[d] - res_ / 2; max_[d] = v[d] + res_ / 2; }
          keyBitSize();
          bbox_defined_ = true;
        }
      } else break;
    }
  }
  void addPoint(int i) {
    const Pt& p = pts_[i];
    adoptBBox(p);
    unsigned key[3] = {(unsigned)((p.x - min_[0]) / res_), (unsigned)((p.y - min_[1]) / res_), (unsigned)((p.z - min_[2]) / res_)};
    OctNode* n = root_;
    for (int level = depth_ - 1; level >= 0; --level) {
      unsigned mask = 1u << level;
      int ci = ((!!(key[0] & mask)) << 2) | ((!!(key[1] & mask)) << 1) | (!!(key[2] & mask));
      if (!n->child[ci]) n->child[ci] = new OctNode();
      n = n->child[ci];
    }
    if (!n->leaf) { n->leaf = new std::vector<int>(); leaf_count_++; }
    n->leaf->push_back(i);
  }
  void approxRec(float qx, float qy, float qz, const OctNode* node, const unsigned* key, int tree_depth, int& idx, float& d2) const {
    double best = std::numeric_limits<double>::max();
    int best_ci = -1;
    unsigned bk[3] = {0, 0, 0};
    for (int ci = 0; ci < 8; ++ci) {
      if (!node->child[ci]) continue;
      unsigned nk[3] = {(key[0] << 1) + (unsigned)(!!(ci & 4)), (key[1] << 1) + (unsigned)(!!(ci & 2)), (key[2] << 1) + (unsigned)(!!(ci & 1))};
      double cell = res_ * (double)(1 << (depth_ - tree_depth));
      float cx = (float)(((double)nk[0] + 0.5f) * cell + min_[0]);
      float cy = (float)(((double)nk[1] + 0.5f) * cell + min_[1]);
      float cz = (float)(((double)nk[2] + 0.5f) * cell + min_[2]);
      double dist = (double)sqdist(cx, cy, cz, qx, qy, qz);
      if (dist >= best) continue;
      best = dist; best_ci = ci; bk[0] = nk[0]; bk[1] = nk[1]; bk[2] = nk[2];
    }
    if (best_ci < 0) return;
    const OctNode* ch = node->child[best_ci];
    if (tree_depth < depth_) {
      approxRec(qx, qy, qz, ch, bk, tree_depth + 1, idx, d2);
    } else {
      double smallest = std::numeric_limits<double>::max();
      std::vector<int> decoded(*ch->leaf);  // upstream copies the index vector per query
      for (size_t i = 0; i < decoded.size(); ++i) {
        const Pt& c = pts_[decoded[i]];
        double sd = (double)sqdist(c.x, c.y, c.z, qx, qy, qz);
        if (sd >= smallest) continue;
        idx = decoded[i]; smallest = sd; d2 = (float)sd;
      }
    }
  }
  double res_;
  const Pt* pts_ = nullptr;
  int n_ = 0;
  OctNode* root_ = nullptr;
  bool bbox_defined_ = false;
  int depth_ = 0;
  int leaf_count_ = 0;
  double min_[3] = {0, 0, 0}, max_[3] = {0, 0, 0};
};

// ---------------------------------------------------------------------------------
// pcl::octree::OctreePointCloudChangeDetector restated for ParticleFilterTracker::testChangeDetection (SURVEY 8 f-4)
// [octree/octree_pointcloud_changedetector.h, octree/impl/octree2buf_base.hpp, octree/impl/octree_pointcloud.hpp]
// -- recalled, not read from disk.  The detector is a double-buffered octree that lives as long as the tracker: every
// test adds the (cropped) cloud to the current buffer -- same bounding box growth and keys as PclOctree above, the box
// and the depth persist across tests -- collects the points of the leaves that the PREVIOUS buffer did not have
// (leaves with fewer than `min_points` points are ignored) and switches buffers.  Octree2BufBase decides "new" at the
// leaf's parent branch (child present in the current buffer, absent in the previous one); branches are shared by the
// two buffers and growth only adds levels on top, so this is: the voxel was not occupied at the previous test.
// ---------------------------------------------------------------------------------
struct CdNode {
  CdNode* child[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  int last = 0;          // id of the last test that put a point into this leaf
  int count = 0;         // points of that test
  bool prev_hit = false; // the leaf was also occupied at the test before `last`
};
class ChangeDetector {
 public:
  explicit ChangeDetector(double res) : res_(res) {}
  ~ChangeDetector() { freeNode(root_); }
  ChangeDetector(const ChangeDetector&) = delete;
  ChangeDetector& operator=(const ChangeDetector&) = delete;
  // setInputCloud + addPointsFromInputCloud + getPointIndicesFromNewVoxels(min_points) + switchBuffers;
  // returns the number of point indices reported
  int test(const Pt* pts, int n, int min_points) {
    ++test_id_;
    if (!root_) root_ = new CdNode();
    std::vector<CdNode*> touched;
    for (int i = 0; i < n; ++i) {
      if (!finite3(pts[i])) continue;
      CdNode* leaf = insert(pts[i]);
      if (leaf->last != test_id_) {
        leaf->prev_hit = leaf->last == test_id_ - 1 && test_id_ > 1;
        leaf->last = test_id_; leaf->count = 0;
        touched.push_back(leaf);
      }
      leaf->count++;
    }
    int found = 0;
    for (CdNode* leaf : touched) if (!leaf->prev_hit && leaf->count >= min_points) found += leaf->count;
    return found;
  }
 private:
  void freeNode(CdNode* n) { if (!n) return; for (auto c : n->child) freeNode(c); delete n; }
  CdNode* insert(const Pt& p) {
    const float minValue = std::numeric_limits<float>::epsilon();
    const double v[3] = {p.x, p.y, p.z};
    while (true) {  // adoptBoundingBoxToPoint
      bool up[3], any = false;
      for (int d = 0; d < 3; ++d) { const bool lo = v[d] < min_[d]; up[d] = v[d] >= max_[d]; any = any || lo || up[d]; }
      if (!(any || !bbox_defined_)) break;
      if (bbox_defined_) {
        const int ci = ((!up[0]) << 2) | ((!up[1]) << 1) | (!up[2]);
        CdNode* nr = new CdNode();
        nr->child[ci] = root_;
        root_ = nr;
        double side = (double)(1 << depth_) * res_;
        for (int d = 0; d < 3; ++d) if (!up[d]) min_[d] -= side;
        depth_++;
        side = (double)(1 << depth_) * res_ - minValue;
        for (int d = 0; d < 3; ++d) max_[d] = min_[d] + side;
      } else {
        for (int d = 0; d < 3; ++d) { min_[d] = v[d] - res_ / 2; max_[d] = v[d] + res_ / 2; }
        unsigned mk[3];
        for (int d = 0; d < 3; ++d) mk[d] = (unsigned)std::ceil((max_[d] - min_[d]) / res_);
        const unsigned max_voxels = std::max(std::max(std::max(mk[0], mk[1]), mk[2]), 2u);
        depth_ = (int)std::max(std::min(30.0, std::ceil(std::log2((double)max_voxels) - minValue)), 0.0);
        const double side = (double)(1 << depth_) * res_ - minValue;
        for (int d = 0; d < 3; ++d) { const double over = (side - (max_[d] - min_[d])) / 2.0; min_[d] -= over; max_[d] += over; }
        bbox_defined_ = true;
      }
    }
    const unsigned key[3] = {(unsigned)((p.x - min_[0]) / res_), (unsigned)((p.y - min_[1]) / res_), (unsigned)((p.z - min_[2]) / res_)};
    CdNode* n = root_;
    for (int level = depth_ - 1; level >= 0; --level) {
      const unsigned mask = 1u << level;
      const int ci = ((!!(key[0] & mask)) << 2) | ((!!(key[1] & mask)) << 1) | (!!(key[2] & mask));
      if (!n->child[ci]) n->child[ci] = new CdNode();
      n = n->child[ci];
    }
    return n;
  }
  double res_;
  CdNode* root_ = nullptr;
  bool bbox_defined_ = false;
  int depth_ = 0;
  int test_id_ = 0;
  double min_[3] = {0, 0, 0}, max_[3] = {0, 0, 0};
};

// Uniform-grid exact nearest neighbour (oracle-side accelerator; validated against the
// brute-force scan in tests).  Ties resolve to the lowest index, same fp32 distance formula.
class ExactGrid {
 public:
  void build(const Pt* pts, int n, float cell) {
    pts_ = pts; n_ = n; cell_ = cell; inv_ = 1.0f / cell;
    if (n == 0) return;
    for (int d = 0; d < 3; ++d) { lo_[d] = INT_MAX; hi_[d] = INT_MIN; }
    for (int i = 0; i < n; ++i) {
      int c[3]; cellOf(pts[i].x, pts[i].y, pts[i].z, c);
      for (int d = 0; d < 3; ++d) { lo_[d] = std::min(lo_[d], c[d]); hi_[d] = std::max(hi_[d], c[d]); }
    }
    for (int d = 0; d < 3; ++d) dim_[d] = hi_[d] - lo_[d] + 1;
    size_t nc = (size_t)dim_[0] * dim_[1] * dim_[2];
    start_.assign(nc + 1, 0);
    for (int i = 0; i < n; ++i) start_[lin(pts[i]) + 1]++;
    for (size_t c = 0; c < nc; ++c) start_[c + 1] += start_[c];
    order_.resize(n);
    std::vector<int> cur(start_.begin(), start_.end() - 1);
    for (int i = 0; i < n; ++i) order_[cur[lin(pts[i])]++] = i;
  }
  // nearest within sqrt(max_d2) (strictly d2 <= max_d2 examined); returns idx or -1
  int nearest(float qx, float qy, float qz, float max_r, float& d2out) const {
    int best = -1; float bd = FLT_MAX;
    if (n_ == 0) { d2out = bd; return -1; }
    int c[3]; cellOf(qx, qy, qz, c);
    int rmax = (int)std::ceil(max_r * inv_) + 1;
    for (int r = 0; r <= rmax; ++r) {
      // scan shell r
      for (int z = c[2] - r; z <= c[2] + r; ++z) {
        if (z < lo_[2] || z > hi_[2]) continue;
        for (int y = c[1] - r; y <= c[1] + r; ++y) {
          if (y < lo_[1] || y > hi_[1]) continue;
          bool face = (z == c[2] - r || z == c[2] + r || y == c[1] - r || y == c[1] + r);
          int step = face ? 1 : 2 * r;
          if (step == 0) step = 1;
          for (int x = c[0] - r; x <= c[0] + r; x += step) {
            if (x < lo_[0] || x > hi_[0]) continue;
            size_t l = ((size_t)(z - lo_[2]) * dim_[1] + (y - lo_[1])) * dim_[0] + (x - lo_[0]);
            for (int k = start_[l]; k < start_[l + 1]; ++k) {
              int i = order_[k];
              float d = sqdist(qx, qy, qz, pts_[i].x, pts_[i].y, pts_[i].z);
              if (d < bd || (d == bd && i < best)) { bd = d; best = i; }
            }
          }
        }
      }
      // every unscanned point is farther than r*cell (minus rounding slack)
      float guaranteed = (float)r * cell_ * 0.999f;
      if (best >= 0 && bd <= guaranteed * guaranteed) break;
    }
    d2out = bd;
    return best;
  }
 private:
  void cellOf(float x, float y, float z, int* c) const {
    c[0] = (int)std::floor(x * inv_); c[1] = (int)std::floor(y * inv_); c[2] = (int)std::floor(z * inv_);
  }
  size_t lin(const Pt& p) const {
    int c[3]; cellOf(p.x, p.y, p.z, c);
    return ((size_t)(c[2] - lo_[2]) * dim_[1] + (c[1] - lo_[1])) * dim_[0] + (c[0] - lo_[0]);
  }
  const Pt* pts_ = nullptr; int n_ = 0; float cell_ = 0.01f, inv_ = 100.f;
  int lo_[3], hi_[3], dim_[3];
  std::vector<int> start_, order_;
};

// ---------------------------------------------------------------------------------
// Tracker: ParticleFilterTracker / KLDAdaptiveParticleFilter(OMP)Tracker restated
// [PCL-1.8.0 tracking/impl/{tracker,particle_filter,particle_filter_omp,
//  kld_adaptive_particle_filter,kld_adaptive_particle_filter_omp}.hpp], SURVEY A.3-A.9.
// Knobs: ref: src/auto_tracking.cpp:201-254.
// ---------------------------------------------------------------------------------
enum NNMode { NN_EXACT_BRUTE = 0, NN_EXACT_GRID = 1, NN_PCL_APPROX = 2 };
enum SampleMode { SAMPLER_ALIAS_PCL = 0, SAMPLER_CDF = 1, SAMPLER_CDF_VDC = 2 };

struct Tracker {
  // configuration (defaults = PCL ctor defaults, SURVEY A.3)
  bool kld = true;
  int threads = 0;
  int particle_num = 0;
  int max_particle_num = 0;
  double delta = 0.99, epsilon = 0.0;
  float bin_size[6] = {0, 0, 0, 0, 0, 0};
  double step_cov[6] = {0, 0, 0, 0, 0, 0}, init_cov[6] = {0, 0, 0, 0, 0, 0}, init_mean[6] = {0, 0, 0, 0, 0, 0};
  int iteration_num = 1;
  double alpha = 15.0, motion_ratio = 0.25;
  float trans[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0};
  // coherence
  int nn_mode = NN_EXACT_BRUTE;
  double max_dist = DBL_MAX;
  bool use_distance = true; double dist_weight = 1.0;
  bool use_hsv = false; double hsv_weight = 1.0, h_weight = 1.0, s_weight = 1.0, v_weight = 0.0;
  double octree_res = 0.01;
  float grid_cell = 0.01f;
  int sampler = SAMPLER_CDF;
  int quat_sample = 1;
  // change detector (PCL ctor defaults, SURVEY A.3; off in the reference)
  bool use_change_detector = false;
  int cd_interval = 10, cd_filter = 10;
  double cd_resolution = 0.01;
  int change_counter = 0;
  int cd_tests = 0, cd_last_found = -1;   // diagnostics: tests run so far, points reported by the last one
  std::shared_ptr<ChangeDetector> detector;
  // state
  std::vector<Pt> ref, input;
  std::vector<Particle> particles;
  Particle rep{0, 0, 0, 1, 0, 0, 0, 0}, motion{0, 0, 0, 1, 0, 0, 0, 0};
  bool changed = false;
  bool initialised = false;
  double fit_ratio = 0.0;
  // transed_reference_vector_: per-slot AABB is all that crop needs; slot clouds kept for PCL-fidelity timing
  std::vector<std::vector<Pt>> transed;
  std::vector<std::array<float, 6>> slot_aabb;  // minx,miny,minz,maxx,maxy,maxz; empty slot = (+FLT_MAX, -FLT_MAX)
  float aabb[6] = {0, 0, 0, 0, 0, 0};
  float local_aabb[6] = {0, 0, 0, 0, 0, 0};  // union box of this tracker's own slots (before any override)
  bool crop_override = false;       // multi-rank emulation: the crop box is the union over ranks, supplied from outside
  float crop_override_box[6] = {0, 0, 0, 0, 0, 0};
  std::vector<Pt> cropped; std::vector<int> cropped_idx;
  std::vector<float> raw_weights;
  std::vector<int> last_ancestors;
  // injected draws
  std::vector<float> d_usel, d_normals, d_umotion;
  int draw_stride = 0;
  int draw_slot = 0;
  std::mt19937 rng{12345u};
  // timing
  double t_stage[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // transform, crop, index, coherence, normalize, resample, update, total
};

inline double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

Particle zero_particle() { return Particle{0, 0, 0, 1, 0, 0, 0, 0}; }

void get_draw(Tracker& T, int slot, int n, float& usel, float* z6, float& umot) {
  size_t k = (size_t)slot * (size_t)T.draw_stride + (size_t)n;
  if (T.draw_stride > 0 && n < T.draw_stride && k < T.d_usel.size()) {
    usel = T.d_usel[k]; umot = T.d_umotion[k];
    for (int d = 0; d < 6; ++d) z6[d] = T.d_normals[k * 6 + d];
  } else {
    std::uniform_real_distribution<float> U(0.f, 1.f);
    std::normal_distribution<float> Nrm(0.f, 1.f);
    usel = U(T.rng); if (usel >= 1.f) usel = 0.f;
    for (int d = 0; d < 6; ++d) z6[d] = Nrm(T.rng);
    umot = U(T.rng);
  }
}

// ParticleFilterTracker::initParticles [impl/particle_filter.hpp], SURVEY A.8
void init_particles(Tracker& T) {
  T.rep = zero_particle();
  T.rep.x = T.trans[3]; T.rep.y = T.trans[7]; T.rep.z = T.trans[11];
  matrix_to_rpy(T.trans, T.rep.roll, T.rep.pitch, T.rep.yaw);
  T.rep.weight = 1.0f / (float)T.particle_num;
  T.particles.clear();
  for (int i = 0; i < T.particle_num; ++i) {
    Particle p = zero_particle();
    float us, um, z[6];
    get_draw(T, 0, i, us, z, um);
    particle_sample(p, T.init_mean, T.init_cov, z, T.quat_sample);
    p.x += T.rep.x; p.y += T.rep.y; p.z += T.rep.z; p.roll += T.rep.roll; p.pitch += T.rep.pitch; p.yaw += T.rep.yaw;
    p.weight = 1.0f / (float)T.particle_num;
    T.particles.push_back(p);
  }
}

// genAliasTable / sampleWithReplacement [impl/particle_filter.hpp], SURVEY A.7
void gen_alias_table(const std::vector<Particle>& ps, std::vector<int>& a, std::vector<double>& q) {
  const size_t N = ps.size();
  a.resize(N); q.resize(N);
  std::vector<int> HL(N);
  int* H = HL.data();
  int* L = HL.data() + N - 1;
  for (size_t i = 0; i < N; ++i) q[i] = (double)(ps[i].weight * (float)N);
  for (size_t i = 0; i < N; ++i) a[i] = (int)i;
  for (size_t i = 0; i < N; ++i) { if (q[i] >= 1.0) *H++ = (int)i; else *L-- = (int)i; }
  while (H != HL.data() && L != HL.data() + N - 1) {
    int j = *(L + 1);
    int k = *(H - 1);
    a[j] = k;
    q[k] += q[j] - 1;
    ++L;
    if (q[k] < 1.0) { *L-- = k; --H; }
  }
}
inline int sample_alias(const std::vector<int>& a, const std::vector<double>& q, float u) {
  double rU = (double)u * (double)a.size();
  int k = (int)rU;
  rU -= k;
  if (k >= (int)a.size()) k = (int)a.size() - 1;
  return rU < q[k] ? k : a[k];
}
// CDF sampler specification (shared with the CUDA kernels): fixed-point prefix sums make the
// cumulative table independent of summation order.
void build_cdf(const std::vector<Particle>& ps, std::vector<uint64_t>& cdf) {
  cdf.resize(ps.size());
  uint64_t s = 0;
  for (size_t i = 0; i < ps.size(); ++i) {
    double w = (double)ps[i].weight;
    uint64_t wq = (w > 0.0) ? (uint64_t)(w * 1099511627776.0 /*2^40*/) : 0ull;
    s += wq; cdf[i] = s;
  }
}
inline int sample_cdf(const std::vector<uint64_t>& cdf, double u) {
  const uint64_t total = cdf.back();
  const size_t N = cdf.size();
  if (total == 0) { int k = (int)(u * (double)N); return k >= (int)N ? (int)N - 1 : k; }
  uint64_t t = (uint64_t)(u * (double)total);
  size_t lo = 0, hi = N - 1;  // smallest j with cdf[j] > t
  while (lo < hi) { size_t mid = (lo + hi) >> 1; if (cdf[mid] > t) hi = mid; else lo = mid + 1; }
  return (int)lo;
}
inline uint32_t bitrev32(uint32_t v) {
  v = ((v >> 1) & 0x55555555u) | ((v & 0x55555555u) << 1);
  v = ((v >> 2) & 0x33333333u) | ((v & 0x33333333u) << 2);
  v = ((v >> 4) & 0x0F0F0F0Fu) | ((v & 0x0F0F0F0Fu) << 4);
  v = ((v >> 8) & 0x00FF00FFu) | ((v & 0x00FF00FFu) << 8);
  return (v >> 16) | (v << 16);
}
inline double selection_uniform(const Tracker& T, float u_n, float u_0, int n) {
  if (T.sampler == SAMPLER_CDF_VDC) {
    double s = (double)u_0 + (double)bitrev32((uint32_t)n) * (1.0 / 4294967296.0);
    if (s >= 1.0) s -= 1.0;
    return s;
  }
  return (double)u_n;
}

struct Selector {
  std::vector<int> a; std::vector<double> q; std::vector<uint64_t> cdf;
  void build(const Tracker& T) { if (T.sampler == SAMPLER_ALIAS_PCL) gen_alias_table(T.particles, a, q); else build_cdf(T.particles, cdf); }
  int pick(const Tracker& T, float u_n, float u_0, int n) const {
    if (T.sampler == SAMPLER_ALIAS_PCL) return sample_alias(a, q, u_n);
    return sample_cdf(cdf, selection_uniform(T, u_n, u_0, n));
  }
};

// KLDAdaptiveParticleFilterTracker::resample [impl/kld_adaptive_particle_filter.hpp], SURVEY A.7
void resample_kld(Tracker& T, int slot) {
  Selector sel; sel.build(T);
  const double zero_mean[6] = {0, 0, 0, 0, 0, 0};
  std::vector<std::array<int, 6>> bins;
  std::vector<Particle> S;
  T.last_ancestors.clear();
  float u0, um0, z0[6];
  get_draw(T, slot, 0, u0, z0, um0);
  int k = 0, n = 0;
  // insertIntoBins is a linear search upstream (O(n*k)); a hash keeps identical semantics
  struct H6 { size_t operator()(const std::array<int, 6>& b) const { size_t h = 1469598103934665603ull; for (int v : b) { h ^= (uint32_t)v; h *= 1099511628211ull; } return h; } };
  std::unordered_map<std::array<int, 6>, int, H6> seen;
  do {
    float us, um, z[6];
    get_draw(T, slot, n, us, z, um);
    int j = sel.pick(T, us, u0, n);
    Particle x = T.particles[j];
    particle_sample(x, zero_mean, T.step_cov, z, T.quat_sample);
    if ((double)um < T.motion_ratio) {
      x.x += T.motion.x; x.y += T.motion.y; x.z += T.motion.z; x.roll += T.motion.roll; x.pitch += T.motion.pitch; x.yaw += T.motion.yaw;
    }
    S.push_back(x);
    T.last_ancestors.push_back(j);
    const float xs[6] = {x.x, x.y, x.z, x.roll, x.pitch, x.yaw};
    std::array<int, 6> bin;
    for (int d = 0; d < 6; ++d) bin[d] = (int)(xs[d] / T.bin_size[d]);
    if (seen.emplace(bin, 1).second) ++k;
    ++n;
  } while (n < T.max_particle_num && (k < 2 || (double)n < kl_bound(k, T.delta, T.epsilon)));
  T.particles = S;
  T.particle_num = (int)S.size();
}

// ParticleFilterTracker::resampleWithReplacement (fixed N) [impl/particle_filter.hpp].
// Upstream appends to the vector it samples from (aliasing bug, N+1 particles); the oracle
// implements the intended semantics: slot 0 = representative state, slots 1..N-1 sampled from
// the pre-resample set with step noise (motion_num = size*(int)0.25 = 0 => no motion term).
void resample_fixed(Tracker& T, int slot) {
  Selector sel; sel.build(T);
  const double zero_mean[6] = {0, 0, 0, 0, 0, 0};
  std::vector<Particle> S;
  T.last_ancestors.clear();
  S.push_back(T.rep);
  T.last_ancestors.push_back(-1);
  float u0, um0, z0[6];
  get_draw(T, slot, 0, u0, z0, um0);
  for (int i = 1; i < T.particle_num; ++i) {
    float us, um, z[6];
    get_draw(T, slot, i, us, z, um);
    int j = sel.pick(T, us, u0, i);
    Particle x = T.particles[j];
    particle_sample(x, zero_mean, T.step_cov, z, T.quat_sample);
    S.push_back(x);
    T.last_ancestors.push_back(j);
  }
  T.particles = S;
}

// ParticleFilterTracker::normalizeWeight [impl/particle_filter.hpp], SURVEY A.6
void normalize_weight(Tracker& T) {
  double w_min = std::numeric_limits<double>::max(), w_max = -std::numeric_limits<double>::max();
  for (auto& p : T.particles) {
    double w = p.weight;
    if (w_min > w) w_min = w;
    if (w != 0.0 && w_max < w) w_max = w;
  }
  T.fit_ratio = w_min;
  if (w_max != w_min) {
    for (auto& p : T.particles)
      if (p.weight != 0.0f) p.weight = (float)std::exp(1.0 - T.alpha * ((double)p.weight - w_min) / (w_max - w_min));
  } else {
    for (auto& p : T.particles) p.weight = 1.0f / (float)T.particles.size();
  }
  double sum = 0.0;
  for (auto& p : T.particles) sum += p.weight;
  if (sum != 0.0) { for (auto& p : T.particles) p.weight = p.weight / (float)sum; }
  else { for (auto& p : T.particles) p.weight = 1.0f / (float)T.particles.size(); }
}

// ParticleFilterTracker::update [impl/particle_filter.hpp], SURVEY A.6
void update(Tracker& T) {
  Particle orig = T.rep;
  Particle r = zero_particle();
  for (auto& p : T.particles) {
    double w = (double)p.weight;
    r.x = r.x + (float)((double)p.x * w); r.y = r.y + (float)((double)p.y * w); r.z = r.z + (float)((double)p.z * w);
    r.roll = r.roll + (float)((double)p.roll * w); r.pitch = r.pitch + (float)((double)p.pitch * w); r.yaw = r.yaw + (float)((double)p.yaw * w);
  }
  r.weight = 1.0f / (float)T.particles.size();
  T.rep = r;
  T.motion = zero_particle();
  T.motion.x = r.x - orig.x; T.motion.y = r.y - orig.y; T.motion.z = r.z - orig.z;
  T.motion.roll = r.roll - orig.roll; T.motion.pitch = r.pitch - orig.pitch; T.motion.yaw = r.yaw - orig.yaw;
}

// (KLDAdaptive)ParticleFilterOMPTracker::weight, no-normal branch, change detector off
// [impl/particle_filter_omp.hpp, impl/particle_filter.hpp], SURVEY A.3-A.4
void weight(Tracker& T, std::vector<int>* nn_out /*optional: [N*M] NN index into cropped*/, std::vector<float>* d2_out) {
  const int N = T.particle_num, M = (int)T.ref.size();
  const int slots = T.kld ? std::max(T.max_particle_num, N) : N;
  if ((int)T.slot_aabb.size() != slots) {
    T.slot_aabb.assign(slots, std::array<float, 6>{FLT_MAX, FLT_MAX, FLT_MAX, -FLT_MAX, -FLT_MAX, -FLT_MAX});
    T.transed.assign(slots, {});
  }
  double t0 = now_s();
  // (1) transformPointCloud per particle into its slot (materialised, as upstream does)
#pragma omp parallel for schedule(static)
  for (int i = 0; i < N; ++i) {
    Mat34 t = particle_to_matrix(T.particles[i]);
    auto& out = T.transed[i];
    out.resize(M);
    float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    for (int j = 0; j < M; ++j) {
      Pt q = T.ref[j];
      xform(t, T.ref[j].x, T.ref[j].y, T.ref[j].z, q.x, q.y, q.z);
      out[j] = q;
      mn[0] = std::min(mn[0], q.x); mn[1] = std::min(mn[1], q.y); mn[2] = std::min(mn[2], q.z);
      mx[0] = std::max(mx[0], q.x); mx[1] = std::max(mx[1], q.y); mx[2] = std::max(mx[2], q.z);
    }
    T.slot_aabb[i] = {mn[0], mn[1], mn[2], mx[0], mx[1], mx[2]};
  }
  double t1 = now_s();
  // (2) calcBoundingBox over every slot (stale slots included) + cropInputPointCloud
  double bb[6] = {DBL_MAX, DBL_MAX, DBL_MAX, -DBL_MAX, -DBL_MAX, -DBL_MAX};
  for (int s = 0; s < slots; ++s) {
    const auto& a = T.slot_aabb[s];
    for (int d = 0; d < 3; ++d) { if (bb[d] > a[d]) bb[d] = a[d]; if (bb[3 + d] < a[3 + d]) bb[3 + d] = a[3 + d]; }
  }
  for (int d = 0; d < 6; ++d) T.aabb[d] = (float)bb[d];
  for (int d = 0; d < 6; ++d) T.local_aabb[d] = T.aabb[d];
  if (T.crop_override) for (int d = 0; d < 6; ++d) T.aabb[d] = T.crop_override_box[d];
  {
    // three PassThrough passes x -> y -> z, inclusive limits, order preserving
    std::vector<Pt> a(T.input.size()), b(T.input.size());
    std::vector<int> ia(T.input.size()), ib(T.input.size());
    int n0 = passthrough(T.input.data(), (int)T.input.size(), 0, T.aabb[0], T.aabb[3], a.data(), ia.data());
    int n1 = passthrough(a.data(), n0, 1, T.aabb[1], T.aabb[4], b.data(), ib.data());
    for (int i = 0; i < n1; ++i) ib[i] = ia[ib[i]];
    int n2 = passthrough(b.data(), n1, 2, T.aabb[2], T.aabb[5], a.data(), ia.data());
    T.cropped.assign(a.begin(), a.begin() + n2);
    T.cropped_idx.resize(n2);
    for (int i = 0; i < n2; ++i) T.cropped_idx[i] = ib[ia[i]];
  }
  double t2 = now_s();
  // change_counter_ / testChangeDetection [impl/particle_filter.hpp weight()], SURVEY A.3 (3): with the detector off
  // every call computes the weights and changed_ is true for ever
  bool compute_weights = true;
  if (T.change_counter == 0) {
    bool change = true;
    if (T.use_change_detector) {
      if (!T.detector) T.detector = std::make_shared<ChangeDetector>(T.cd_resolution);  // initCompute: created once
      T.cd_last_found = T.detector->test(T.cropped.data(), (int)T.cropped.size(), T.cd_filter);
      T.cd_tests++;
      change = T.cd_last_found > 0;
    }
    if (change) { T.changed = true; T.change_counter = T.cd_interval; }
    else { T.changed = false; compute_weights = false; }
  } else {
    --T.change_counter;
    T.changed = true;  // (upstream leaves changed_ as it is, which is true here; the parity tests' set_changed hook relies on it)
  }
  if (!compute_weights) {
    // the particles keep their weights and normalizeWeight() runs on them all the same
    T.raw_weights.resize(N);
    for (int i = 0; i < N; ++i) T.raw_weights[i] = T.particles[i].weight;
    if (nn_out) nn_out->assign((size_t)N * M, -1);
    if (d2_out) d2_out->assign((size_t)N * M, FLT_MAX);
    double t3s = now_s();
    normalize_weight(T);
    T.t_stage[0] += t1 - t0; T.t_stage[1] += t2 - t1; T.t_stage[4] += now_s() - t3s;
    return;
  }
  // (3) coherence_->setTargetCloud(cropped); initCompute() => search index rebuild
  const int S = (int)T.cropped.size();
  PclOctree oct(T.octree_res);
  ExactGrid grid;
  if (T.nn_mode == NN_PCL_APPROX) oct.setInputCloud(T.cropped.data(), S);
  else if (T.nn_mode == NN_EXACT_GRID) grid.build(T.cropped.data(), S, T.grid_cell);
  double t3 = now_s();
  // (4) per particle: Nearest/ApproxNearestPairPointCloudCoherence::computeCoherence
  const double maxd2 = T.max_dist * T.max_dist;
  const float max_r = (float)std::min(T.max_dist, 1.0e3);
  T.raw_weights.assign(N, 0.f);
  if (nn_out) nn_out->assign((size_t)N * M, -1);
  if (d2_out) d2_out->assign((size_t)N * M, FLT_MAX);
#pragma omp parallel for schedule(dynamic, 4)
  for (int i = 0; i < N; ++i) {
    double val = 0.0;
    const auto& tc = T.transed[i];
    for (int j = 0; j < M; ++j) {
      const Pt& q = tc[j];
      int idx = -1; float d2 = FLT_MAX;
      if (S > 0) {
        if (T.nn_mode == NN_EXACT_BRUTE) {
          for (int k = 0; k < S; ++k) {
            float d = sqdist(q.x, q.y, q.z, T.cropped[k].x, T.cropped[k].y, T.cropped[k].z);
            if (d < d2) { d2 = d; idx = k; }
          }
        } else if (T.nn_mode == NN_EXACT_GRID) {
          idx = grid.nearest(q.x, q.y, q.z, max_r, d2);
          // the grid search stops expanding beyond max_r: anything it reports farther is not a match anyway
        } else {
          if (!oct.approxNearest(q.x, q.y, q.z, idx, d2)) idx = -1;
        }
      }
      if (nn_out) (*nn_out)[(size_t)i * M + j] = idx;
      if (d2_out) (*d2_out)[(size_t)i * M + j] = d2;
      if (idx >= 0 && (double)d2 < maxd2) {
        double c = 1.0;
        if (T.use_distance) c *= distance_coherence_d2(sqdist(q.x, q.y, q.z, T.cropped[idx].x, T.cropped[idx].y, T.cropped[idx].z), T.dist_weight);
        if (T.use_hsv) c *= hsv_coherence(q.rgba, T.cropped[idx].rgba, T.hsv_weight, T.h_weight, T.s_weight, T.v_weight);
        val += c;
      }
    }
    T.raw_weights[i] = -(float)val;
    T.particles[i].weight = -(float)val;
  }
  double t4 = now_s();
  normalize_weight(T);
  double t5 = now_s();
  T.t_stage[0] += t1 - t0; T.t_stage[1] += t2 - t1; T.t_stage[2] += t3 - t2; T.t_stage[3] += t4 - t3; T.t_stage[4] += t5 - t4;
}

void resample(Tracker& T, int slot) {
  double t0 = now_s();
  if (T.kld) resample_kld(T, slot); else resample_fixed(T, slot);
  T.t_stage[5] += now_s() - t0;
}

// Tracker::compute -> initCompute + computeTracking [impl/tracker.hpp, impl/particle_filter.hpp]
void compute(Tracker& T) {
  if (T.input.empty() || T.ref.empty()) return;  // Tracker::initCompute fails silently on empty input
  double t0 = now_s();
  if (T.particles.empty()) init_particles(T);
  for (int it = 0; it < T.iteration_num; ++it) {
    if (T.changed) resample(T, it);
    weight(T, nullptr, nullptr);
    if (T.changed) { double a = now_s(); update(T); T.t_stage[6] += now_s() - a; }
  }
  T.t_stage[7] += now_s() - t0;
}

}  // namespace

// =====================================================================================
// C API (ctypes-friendly)
// =====================================================================================
extern "C" {

struct orc_tracker { Tracker T; std::vector<int> nn; std::vector<float> d2; };

int orc_passthrough(const orc_point* in, int n, int field, float lo, float hi, orc_point* out) { return passthrough(in, n, field, lo, hi, out, nullptr); }
int orc_approx_voxel_grid_pcl(const orc_point* in, int n, float leaf, orc_point* out) { return approx_voxel_grid_pcl(in, n, leaf, out); }
int orc_voxel_grid_pcl(const orc_point* in, int n, float leaf, orc_point* out) { return voxel_grid_pcl(in, n, leaf, out); }
int orc_voxel_grid_exact(const orc_point* in, int n, float leaf, int field, float lo, float hi, orc_point* out) { return voxel_grid_exact(in, n, leaf, field, lo, hi, out); }
// removeZeroPoints, ref: src/auto_tracking.cpp:577-595
// pcl::EuclideanClusterExtraction::extract as the model builder uses it (ref: src/create_model.cpp:169-179),
// restating PCL-1.8.0 segmentation/impl/extract_clusters.hpp (extractEuclideanClusters): every unprocessed point in
// index order seeds a breadth-first growth through KdTree radius searches; FLANN's radius search keeps the points
// whose squared L2 distance -- ((dx*dx) + dy*dy) + dz*dz in fp32 -- is < (float)(tolerance * tolerance).  Clusters
// inside [min_size, max_size] are kept with their indices sorted, then ordered by size descending (upstream:
// std::sort over reverse iterators, ties unspecified; here the lower seed index first).  The radius search is
// served by a uniform grid instead of a kd-tree (same result set).  labels[i] = cluster rank or -1.
// Grid keys are floor(((double)x - min) / cell), each operation rounded once in fp64, with cell >= tolerance * 1.0001
// and at most 2^30 cells along an axis, so a key fits a long long for any finite cloud (an fp32 x / cell for points at
// 3e38 does not).  A pair that passes the fp32 test is less than (1 - 0.98e-4) cells apart and the keys err by less
// than 2^-21 cells, so the pair lands in adjacent cells (the argument in pft_cluster.cu, cl_cell_of).
int orc_euclidean_clusters(const orc_point* pts, int n, double tolerance, int min_size, int max_size, int* labels, int* sizes, int sizes_cap) {
  const float tol2 = (float)(tolerance * tolerance);
  double lo[3] = {HUGE_VAL, HUGE_VAL, HUGE_VAL}, hi[3] = {-HUGE_VAL, -HUGE_VAL, -HUGE_VAL};
  for (int i = 0; i < n; ++i) {
    if (!finite3(pts[i])) continue;
    const double c[3] = {pts[i].x, pts[i].y, pts[i].z};
    for (int d = 0; d < 3; ++d) { lo[d] = std::min(lo[d], c[d]); hi[d] = std::max(hi[d], c[d]); }
  }
  double cell = tolerance * 1.0001;
  for (int d = 0; d < 3; ++d) if (lo[d] <= hi[d]) cell = std::max(cell, (hi[d] - lo[d]) / 1073741824.0);
  struct Key { long long x, y, z; bool operator==(const Key& o) const { return x == o.x && y == o.y && z == o.z; } };
  struct KeyHash { size_t operator()(const Key& k) const { return (size_t)(k.x * 73856093ll ^ k.y * 19349663ll ^ k.z * 83492791ll); } };
  std::unordered_map<Key, std::vector<int>, KeyHash> grid;
  auto key_of = [&](const Pt& p) {
    return Key{(long long)std::floor(((double)p.x - lo[0]) / cell), (long long)std::floor(((double)p.y - lo[1]) / cell), (long long)std::floor(((double)p.z - lo[2]) / cell)};
  };
  for (int i = 0; i < n; ++i) { labels[i] = -1; if (finite3(pts[i])) grid[key_of(pts[i])].push_back(i); }
  std::vector<char> processed(n, 0);
  std::vector<std::vector<int>> clusters;
  std::vector<int> queue;
  for (int i = 0; i < n; ++i) {
    if (processed[i] || !finite3(pts[i])) continue;
    queue.clear();
    queue.push_back(i);
    processed[i] = 1;
    for (size_t q = 0; q < queue.size(); ++q) {
      const Pt& p = pts[queue[q]];
      const Key k = key_of(p);
      for (long long dz = -1; dz <= 1; ++dz) for (long long dy = -1; dy <= 1; ++dy) for (long long dx = -1; dx <= 1; ++dx) {
        auto it = grid.find(Key{k.x + dx, k.y + dy, k.z + dz});
        if (it == grid.end()) continue;
        for (int j : it->second) {
          if (processed[j]) continue;
          const float ex = p.x - pts[j].x, ey = p.y - pts[j].y, ez = p.z - pts[j].z;
          const float d2 = (ex * ex + ey * ey) + ez * ez;
          if (d2 < tol2) { processed[j] = 1; queue.push_back(j); }
        }
      }
    }
    if ((int)queue.size() >= min_size && (int)queue.size() <= max_size) {
      std::sort(queue.begin(), queue.end());
      clusters.push_back(queue);
    }
  }
  std::stable_sort(clusters.begin(), clusters.end(), [](const std::vector<int>& a, const std::vector<int>& b) {
    if (a.size() != b.size()) return a.size() > b.size();
    return a[0] < b[0];
  });
  for (size_t c = 0; c < clusters.size(); ++c) {
    if ((int)c < sizes_cap) sizes[c] = (int)clusters[c].size();
    for (int j : clusters[c]) labels[j] = (int)c;
  }
  return (int)clusters.size();
}

int orc_remove_zero_points(const orc_point* in, int n, orc_point* out) {
  int m = 0;
  for (int i = 0; i < n; ++i) {
    const orc_point& p = in[i];
    if (!(std::fabs(p.x) < 0.01 && std::fabs(p.y) < 0.01 && std::fabs(p.z) < 0.01) && !std::isnan(p.x) && !std::isnan(p.y) && !std::isnan(p.z)) out[m++] = p;
  }
  return m;
}
// pcl::compute3DCentroid (dense) [common/impl/centroid.hpp]: float accumulation, then /n; ref: src/auto_tracking.cpp:663
void orc_centroid(const orc_point* in, int n, float* c3) {
  float s[3] = {0, 0, 0};
  int cnt = 0;
  for (int i = 0; i < n; ++i) { if (!finite3(in[i])) continue; s[0] += in[i].x; s[1] += in[i].y; s[2] += in[i].z; ++cnt; }
  for (int d = 0; d < 3; ++d) c3[d] = cnt ? s[d] / (float)cnt : 0.f;
}
void orc_rgb2hsv(int r, int g, int b, int* h, int* s, int* v) { rgb2hsv_int(r, g, b, *h, *s, *v); }
int orc_div_table(int i) { return g_div.v[i & 255]; }
double orc_normal_quantile(double u) { return normal_quantile(u); }
double orc_kl_bound(int k, double delta, double eps) { return kl_bound(k, delta, eps); }
void orc_particle_to_matrix(const orc_particle* p, float* m12) { Mat34 t = particle_to_matrix(*p); std::memcpy(m12, t.m, sizeof(t.m)); }
void orc_matrix_to_particle(const float* m12, orc_particle* p) {
  *p = zero_particle(); p->x = m12[3]; p->y = m12[7]; p->z = m12[11]; matrix_to_rpy(m12, p->roll, p->pitch, p->yaw);
}
double orc_distance_coherence(const orc_point* a, const orc_point* b, double w) { return distance_coherence_d2(sqdist(a->x, a->y, a->z, b->x, b->y, b->z), w); }
double orc_hsv_coherence(uint32_t a, uint32_t b, double w, double hw, double sw, double vw) { return hsv_coherence(a, b, w, hw, sw, vw); }
void orc_particle_sample(orc_particle* p, const double* mean, const double* cov, const float* z6, int quat_mode) { particle_sample(*p, mean, cov, z6, quat_mode); }
int orc_octree_approx_nearest(const orc_point* pts, int n, double res, const float* q3, int nq, int* idx, float* d2) {
  PclOctree o(res); o.setInputCloud(pts, n);
  for (int i = 0; i < nq; ++i) { int id = -1; float d = FLT_MAX; if (!o.approxNearest(q3[3 * i], q3[3 * i + 1], q3[3 * i + 2], id, d)) id = -1; idx[i] = id; d2[i] = d; }
  return 0;
}

orc_tracker* orc_tracker_create(int kld) { auto* t = new orc_tracker(); t->T.kld = kld != 0; return t; }
void orc_tracker_destroy(orc_tracker* t) { delete t; }

enum {
  ORC_THREADS = 0, ORC_PARTICLE_NUM = 1, ORC_MAX_PARTICLE_NUM = 2, ORC_ITERATION_NUM = 3, ORC_NN_MODE = 4, ORC_USE_HSV = 5,
  ORC_USE_DISTANCE = 6, ORC_SAMPLER = 7, ORC_QUAT_SAMPLE = 8, ORC_SEED = 9,
  ORC_USE_CHANGE_DETECTOR = 10, ORC_CD_INTERVAL = 11, ORC_CD_MIN_POINTS = 12,
  ORC_DELTA = 20, ORC_EPSILON = 21, ORC_ALPHA = 22, ORC_MOTION_RATIO = 23, ORC_MAX_DIST = 24, ORC_DIST_WEIGHT = 25, ORC_HSV_WEIGHT = 26,
  ORC_H_WEIGHT = 27, ORC_S_WEIGHT = 28, ORC_V_WEIGHT = 29, ORC_OCTREE_RES = 30, ORC_GRID_CELL = 31,
  ORC_CD_RESOLUTION = 32,
  ORC_STEP_COV = 40, ORC_INIT_COV = 41, ORC_INIT_MEAN = 42, ORC_BIN_SIZE = 43
};
int orc_set_i(orc_tracker* t, int key, int v) {
  Tracker& T = t->T;
  switch (key) {
    case ORC_THREADS: T.threads = v; break;
    case ORC_PARTICLE_NUM: T.particle_num = v; break;
    case ORC_MAX_PARTICLE_NUM: T.max_particle_num = v; break;
    case ORC_ITERATION_NUM: T.iteration_num = v; break;
    case ORC_NN_MODE: T.nn_mode = v; break;
    case ORC_USE_HSV: T.use_hsv = v != 0; break;
    case ORC_USE_DISTANCE: T.use_distance = v != 0; break;
    case ORC_SAMPLER: T.sampler = v; break;
    case ORC_QUAT_SAMPLE: T.quat_sample = v; break;
    case ORC_SEED: T.rng.seed((unsigned)v); break;
    case ORC_USE_CHANGE_DETECTOR: T.use_change_detector = v != 0; break;
    case ORC_CD_INTERVAL: T.cd_interval = v; break;
    case ORC_CD_MIN_POINTS: T.cd_filter = v; break;
    default: return -1;
  }
  return 0;
}
int orc_set_d(orc_tracker* t, int key, double v) {
  Tracker& T = t->T;
  switch (key) {
    case ORC_DELTA: T.delta = v; break;
    case ORC_EPSILON: T.epsilon = v; break;
    case ORC_ALPHA: T.alpha = v; break;
    case ORC_MOTION_RATIO: T.motion_ratio = v; break;
    case ORC_MAX_DIST: T.max_dist = v; break;
    case ORC_DIST_WEIGHT: T.dist_weight = v; break;
    case ORC_HSV_WEIGHT: T.hsv_weight = v; break;
    case ORC_H_WEIGHT: T.h_weight = v; break;
    case ORC_S_WEIGHT: T.s_weight = v; break;
    case ORC_V_WEIGHT: T.v_weight = v; break;
    case ORC_OCTREE_RES: T.octree_res = v; break;
    case ORC_GRID_CELL: T.grid_cell = (float)v; break;
    case ORC_CD_RESOLUTION: T.cd_resolution = v; T.detector.reset(); break;
    default: return -1;
  }
  return 0;
}
int orc_set_vec6(orc_tracker* t, int key, const double* v) {
  Tracker& T = t->T;
  switch (key) {
    case ORC_STEP_COV: std::copy(v, v + 6, T.step_cov); break;
    case ORC_INIT_COV: std::copy(v, v + 6, T.init_cov); break;
    case ORC_INIT_MEAN: std::copy(v, v + 6, T.init_mean); break;
    case ORC_BIN_SIZE: for (int d = 0; d < 6; ++d) T.bin_size[d] = (float)v[d]; break;
    default: return -1;
  }
  return 0;
}
void orc_set_trans(orc_tracker* t, const float* m12) { std::memcpy(t->T.trans, m12, 12 * sizeof(float)); }
void orc_set_reference(orc_tracker* t, const orc_point* p, int n) { t->T.ref.assign(p, p + n); }
void orc_set_input(orc_tracker* t, const orc_point* p, int n) { t->T.input.assign(p, p + n); }
void orc_set_particles(orc_tracker* t, const orc_particle* p, int n) { t->T.particles.assign(p, p + n); t->T.particle_num = n; }
int orc_get_particles(orc_tracker* t, orc_particle* out, int cap) {
  int n = std::min<int>(cap, (int)t->T.particles.size());
  if (out) std::copy(t->T.particles.begin(), t->T.particles.begin() + n, out);
  return (int)t->T.particles.size();
}
void orc_get_result(orc_tracker* t, orc_particle* out) { *out = t->T.rep; }
void orc_set_result(orc_tracker* t, const orc_particle* in) { t->T.rep = *in; }
void orc_get_motion(orc_tracker* t, orc_particle* out) { *out = t->T.motion; }
void orc_set_motion(orc_tracker* t, const orc_particle* in) { t->T.motion = *in; }
// ParticleFilterTracker::resetTracking [tracking/particle_filter.h]: `if (particles_) particles_->points.clear ();` -- nothing else:
// particle_num_ keeps the count of the last (KLD) resample and changed_ stays as it is, so the compute() that follows re-draws
// that many particles (initParticles) and, when an earlier weight() had set changed_, resamples them in its first iteration
void orc_reset_tracking(orc_tracker* t) { t->T.particles.clear(); }
// genAliasTable of the current particle set (out arrays hold one entry per particle)
void orc_alias_table(orc_tracker* t, int* a_out, double* q_out) {
  std::vector<int> a; std::vector<double> q;
  gen_alias_table(t->T.particles, a, q);
  std::copy(a.begin(), a.end(), a_out);
  std::copy(q.begin(), q.end(), q_out);
}
void orc_set_changed(orc_tracker* t, int c) { t->T.changed = c != 0; }
int orc_get_changed(orc_tracker* t) { return t->T.changed ? 1 : 0; }
// out[4] = {change_counter_, tests run so far, point indices reported by the last test (-1: none yet), changed_}
void orc_change_detector_info(orc_tracker* t, int* out) {
  out[0] = t->T.change_counter; out[1] = t->T.cd_tests; out[2] = t->T.cd_last_found; out[3] = t->T.changed ? 1 : 0;
}
// stand-alone detector for known-answer tests: clouds[k] of sizes[k] points tested one after the other
int orc_change_detector_sequence(const orc_point* pts, const int* sizes, int n_clouds, double res, int min_points, int* found) {
  ChangeDetector d(res);
  size_t off = 0;
  for (int k = 0; k < n_clouds; ++k) { found[k] = d.test(pts + off, sizes[k], min_points); off += (size_t)sizes[k]; }
  return 0;
}
// draws: [slots][stride] uniforms for selection, [slots][stride][6] standard normals, [slots][stride] motion uniforms
void orc_inject_draws(orc_tracker* t, const float* usel, const float* normals6, const float* umotion, int slots, int stride) {
  Tracker& T = t->T;
  size_t n = (size_t)slots * stride;
  T.d_usel.assign(usel, usel + n); T.d_normals.assign(normals6, normals6 + 6 * n); T.d_umotion.assign(umotion, umotion + n);
  T.draw_stride = stride;
}
void orc_init_particles(orc_tracker* t) { init_particles(t->T); }
void orc_resample(orc_tracker* t, int slot) { resample(t->T, slot); }
void orc_weight(orc_tracker* t, int keep_nn) {
#ifdef _OPENMP
  if (t->T.threads > 0) omp_set_num_threads(t->T.threads);
#endif
  if (keep_nn) weight(t->T, &t->nn, &t->d2); else weight(t->T, nullptr, nullptr);
}
void orc_normalize(orc_tracker* t) { normalize_weight(t->T); }
void orc_update(orc_tracker* t) { update(t->T); }
void orc_compute(orc_tracker* t) {
#ifdef _OPENMP
  if (t->T.threads > 0) omp_set_num_threads(t->T.threads);
#endif
  compute(t->T);
}
void orc_get_aabb(orc_tracker* t, float* a6) { std::memcpy(a6, t->T.aabb, sizeof(float) * 6); }
void orc_get_local_aabb(orc_tracker* t, float* a6) { std::memcpy(a6, t->T.local_aabb, sizeof(float) * 6); }
// multi-rank emulation (tests): weight() crops with this box instead of the union of its own slots; NULL switches it off
void orc_set_crop_box(orc_tracker* t, const float* a6) {
  t->T.crop_override = a6 != nullptr;
  if (a6) std::memcpy(t->T.crop_override_box, a6, sizeof(float) * 6);
}
int orc_get_cropped(orc_tracker* t, int* idx, orc_point* pts, int cap) {
  int n = std::min<int>(cap, (int)t->T.cropped.size());
  for (int i = 0; i < n; ++i) { if (idx) idx[i] = t->T.cropped_idx[i]; if (pts) pts[i] = t->T.cropped[i]; }
  return (int)t->T.cropped.size();
}
// NN results of the last orc_weight(keep_nn=1): indices refer to the cropped cloud
int orc_get_nn(orc_tracker* t, int particle, int* idx, float* d2, int cap) {
  int M = (int)t->T.ref.size();
  if ((size_t)(particle + 1) * M > t->nn.size()) return -1;
  int n = std::min(cap, M);
  for (int j = 0; j < n; ++j) { idx[j] = t->nn[(size_t)particle * M + j]; d2[j] = t->d2[(size_t)particle * M + j]; }
  return M;
}
int orc_get_raw_weights(orc_tracker* t, float* w, int cap) {
  int n = std::min<int>(cap, (int)t->T.raw_weights.size());
  std::copy(t->T.raw_weights.begin(), t->T.raw_weights.begin() + n, w);
  return (int)t->T.raw_weights.size();
}
int orc_get_ancestors(orc_tracker* t, int* a, int cap) {
  int n = std::min<int>(cap, (int)t->T.last_ancestors.size());
  std::copy(t->T.last_ancestors.begin(), t->T.last_ancestors.begin() + n, a);
  return (int)t->T.last_ancestors.size();
}
double orc_get_fit_ratio(orc_tracker* t) { return t->T.fit_ratio; }
void orc_get_stage_seconds(orc_tracker* t, double* s8, int reset) {
  std::memcpy(s8, t->T.t_stage, sizeof(double) * 8);
  if (reset) std::fill(t->T.t_stage, t->T.t_stage + 8, 0.0);
}
int orc_max_threads(void) {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}
const char* orc_describe(void) { return "PCL-1.8.0 tracking algorithms restated (C++17/OpenMP), not PCL binaries; parity unpinned"; }

}  // extern "C"
