// segment.cu — the stage in front of the path (SURVEY 8f-2): what turns a Kinect frame into the cluster estimateFinalPose is
// handed (D&L/src/rosinterface.cpp:212-250 -> ProcessingPcd::getPassThrough, ObjectSegmentationPlane::getSegmentedObjectsOnPlane).
//   ope_pass_through        pcl::PassThrough on z, y, x in sequence (D&L/src/processingpcd.cpp:8-41): one ordered compaction
//   ope_euclidean_clusters  pcl::EuclideanClusterExtraction (D&L/src/objectsegmentationplane.cpp:74-90: tolerance 0.05,
//                           300 <= size <= 1e5): connected components of the "closer than the tolerance" graph by a lock-free
//                           union-find over the cloud's Morton grid; the host only renumbers the components by size
//   ope_plane_ransac        pcl::SACSegmentation, SACMODEL_PLANE / SAC_RANSAC, threshold 0.01, refined coefficients
//                           (D&L/src/objectsegmentationplane.cpp:36-55): all candidate planes of the replayed sample table scored
//                           in one launch (a block per hypothesis), the adaptive stopping rule replayed on the host
//   ope_prism_select        the polygonal-prism crop over the plane's padded bounding rectangle (:174-218)
#include <algorithm>
#include <cmath>
#include <cstring>
#include <climits>
#include <numeric>
#include <random>
#include <vector>

#include "ope_host.cuh"
#include "ope_device.cuh"

namespace ope {

static constexpr int kSegThreads = 256;

// The kernels below work on a concatenated point array whose frame f is [off[f], off[f + 1]) (device offsets); they take the frame
// from blockIdx.y (plane_refit_kernel: blockIdx.x). ope_scene_batch_create runs them on a chunk of frames; ope_pass_through,
// ope_plane_ransac and ope_segment_objects_on_plane are one-frame runs (off = {0, n}) of the same stages, so a batch's frame equals
// those calls by construction.

// ---- pass-through: keep[i] = finite && lo <= field <= hi for all three fields; order-preserving compaction ----
__global__ void pass_flag_kernel(const float4* __restrict__ pts, int n, float x0, float x1, float y0, float y1, float z0, float z1,
                                 int* __restrict__ flags) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 p = __ldg(pts + i);
  // three PassThrough filters in sequence (z, y, x): a point survives iff it is finite and inside every closed interval
  const bool keep = finite3(p.x, p.y, p.z) && !(p.z < z0 || p.z > z1) && !(p.y < y0 || p.y > y1) && !(p.x < x0 || p.x > x1);
  flags[i] = keep ? 1 : 0;
}

// ---- Euclidean clustering: union-find, the smaller index is the root ----
__device__ __forceinline__ int uf_find(int* parent, int i) {
  int p = parent[i];
  while (p != i) {
    const int gp = parent[p];
    if (gp != p) parent[i] = gp;   // path halving (benign race: any ancestor is a valid parent)
    i = p; p = gp;
  }
  return i;
}
__device__ __forceinline__ void uf_union(int* parent, int a, int b) {
  for (;;) {
    a = uf_find(parent, a); b = uf_find(parent, b);
    if (a == b) return;
    if (a < b) { const int t = a; a = b; b = t; }   // hook the larger root under the smaller
    const int old = atomicCAS(parent + a, a, b);
    if (old == a) return;
  }
}
// one warp per point: every indexed point closer than the tolerance (squared distance < tol^2, the radiusSearch of the
// reference) and with a smaller index is united with it
__global__ void __launch_bounds__(kSegThreads) cluster_union_kernel(GridView g, const float4* __restrict__ pts, int n, float r2,
                                                                    int* __restrict__ parent) {
  const int lane = threadIdx.x & 31;
  const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
  for (int i = wid; i < n; i += n_warps) {
    const float4 q = __ldg(pts + i);
    if (!finite3(q.x, q.y, q.z)) continue;
    grid_radius_ranges(g, q.x, q.y, q.z, r2, 64, [&](int b, int e) {
      for (int s = b + lane; s < e; s += 32) {
        const float4 c = __ldg(g.pts + s);
        const int j = __float_as_int(c.w);
        if (j < i && dist2(q.x, q.y, q.z, c.x, c.y, c.z) < r2) uf_union(parent, i, j);
      }
    });
  }
}
__global__ void cluster_init_kernel(const float4* __restrict__ pts, int n, int* __restrict__ parent) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) parent[i] = i;
}
__global__ void cluster_flatten_kernel(const float4* __restrict__ pts, int n, int* __restrict__ parent, int* __restrict__ root) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 q = __ldg(pts + i);
  root[i] = finite3(q.x, q.y, q.z) ? uf_find(parent, i) : -1;
}


// ---- plane RANSAC (pcl::SACSegmentation, SACMODEL_PLANE) -------------------------------------------------------------------
// Eigen's 4-float reduction order of the whole path (DESIGN.md section 2): (p0 + p1) + (p2 + p3)
OPE_HD float redux4(float p0, float p1, float p2, float p3) { return (p0 + p1) + (p2 + p3); }
OPE_HD float plane_distance(const float c[4], float x, float y, float z) { return redux4(c[0] * x, c[1] * y, c[2] * z, c[3] * 1.0f); }

// countWithinDistance for every candidate plane at once: block (h, f) counts the points of frame f with |c_h . p| < threshold
__global__ void __launch_bounds__(kSegThreads) plane_count_kernel(const float4* __restrict__ pts, const int* __restrict__ off,
                                                                  const float* __restrict__ coeffs, double threshold, int* __restrict__ counts) {
  __shared__ int total;
  const int f = blockIdx.y;
  const size_t h = (size_t)f * gridDim.x + blockIdx.x;
  const float c[4] = {coeffs[4 * h], coeffs[4 * h + 1], coeffs[4 * h + 2], coeffs[4 * h + 3]};
  if (threadIdx.x == 0) total = 0;
  __syncthreads();
  int cnt = 0;
  for (int i = off[f] + threadIdx.x, e = off[f + 1]; i < e; i += kSegThreads) {
    const float4 p = __ldg(pts + i);
    cnt += (double)fabsf(plane_distance(c, p.x, p.y, p.z)) < threshold ? 1 : 0;
  }
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if ((threadIdx.x & 31) == 0) atomicAdd(&total, cnt);
  __syncthreads();
  if (threadIdx.x == 0) counts[h] = total;
}
// selectWithinDistance: flags for the ordered compaction. Frame f uses coeff[4 f ..]; live[f] == 0: no flags.
__global__ void plane_flag_kernel(const float4* __restrict__ pts, const int* __restrict__ off, const float* __restrict__ coeff, double threshold,
                                  int invert, const int* __restrict__ live, int* __restrict__ flags) {
  const int f = blockIdx.y;
  const bool on = live[f] != 0;
  const float c[4] = {coeff[4 * f], coeff[4 * f + 1], coeff[4 * f + 2], coeff[4 * f + 3]};
  for (int i = off[f] + blockIdx.x * blockDim.x + threadIdx.x, e = off[f + 1]; i < e; i += gridDim.x * blockDim.x) {
    const float4 p = __ldg(pts + i);
    const bool in = (double)fabsf(plane_distance(c, p.x, p.y, p.z)) < threshold;
    flags[i] = (on && in != (invert != 0)) ? 1 : 0;
  }
}
__global__ void index_compact_kernel(int n, const int* __restrict__ pos, int* __restrict__ out_idx) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && pos[i + 1] > pos[i]) out_idx[pos[i]] = i;
}
__global__ void gather_points_kernel(const float4* __restrict__ pts, const int* __restrict__ idx, int m, float4* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < m) out[i] = __ldg(pts + idx[i]);
}
// optimizeModelCoefficients: computeMeanAndCovarianceMatrix accumulates nine FLOAT sums over the inliers IN INDEX ORDER, so the
// sums are order-dependent and each is one serial chain of additions. The chain is all that stays serial: warps 1.. gather the
// next chunk of inliers and write its nine term arrays (x*x, x*y, ... z) to shared memory while lanes 0..8 of warp 0 — one per
// accumulator, the same instruction stream for all nine — add up the current chunk. Thread 0 finishes with eigen33 and
// d = -n . centroid. One block per frame: block f refits in[4 f ..] over its inliers inliers[off[f] .. off[f + 1]) into out[4 f ..].
static constexpr int kRefitChunk = 512;
__global__ void __launch_bounds__(kSegThreads) plane_refit_kernel(const float4* __restrict__ pts, const int* __restrict__ inliers_all,
                                                                  const int* __restrict__ off, const float* __restrict__ in_all,
                                                                  float* __restrict__ out_all) {
  const int f = blockIdx.x;
  const int* inliers = inliers_all + off[f];
  const int m = off[f + 1] - off[f];
  const float* in = in_all + 4 * f;
  float* out = out_all + 4 * f;
  __shared__ float terms[2][9][kRefitChunk + 1];   // + 1: the nine lanes of a step read nine different banks
  __shared__ float accu[9];
  const int tid = threadIdx.x;
  auto fill = [&](int chunk) {   // by the threads of warps 1..: terms of chunk `chunk` into its buffer
    const int base = chunk * kRefitChunk;
    const int cnt = min(kRefitChunk, m - base);
    float (*t)[kRefitChunk + 1] = terms[chunk & 1];
    for (int j = tid - 32; j < cnt; j += kSegThreads - 32) {
      const float4 p = __ldg(pts + inliers[base + j]);
      t[0][j] = p.x * p.x; t[1][j] = p.x * p.y; t[2][j] = p.x * p.z;
      t[3][j] = p.y * p.y; t[4][j] = p.y * p.z; t[5][j] = p.z * p.z;
      t[6][j] = p.x; t[7][j] = p.y; t[8][j] = p.z;
    }
  };
  const int n_chunks = (m + kRefitChunk - 1) / kRefitChunk;
  float acc = 0.0f;
  if (tid >= 32 && n_chunks > 0) fill(0);
  __syncthreads();
  for (int c = 0; c < n_chunks; ++c) {
    if (tid >= 32) {
      if (c + 1 < n_chunks) fill(c + 1);
    } else if (tid < 9) {
      const int cnt = min(kRefitChunk, m - c * kRefitChunk);
      const float* t = terms[c & 1][tid];
#pragma unroll 8
      for (int j = 0; j < cnt; ++j) acc += t[j];
    }
    __syncthreads();
  }
  if (tid < 9) accu[tid] = acc / (float)m;
  __syncthreads();
  if (tid == 0) {
    if (m < 4) { for (int i = 0; i < 4; ++i) out[i] = in[i]; return; }
    float cov[9];
    cov[0] = accu[0] - accu[6] * accu[6]; cov[1] = accu[1] - accu[6] * accu[7]; cov[2] = accu[2] - accu[6] * accu[8];
    cov[4] = accu[3] - accu[7] * accu[7]; cov[5] = accu[4] - accu[7] * accu[8]; cov[8] = accu[5] - accu[8] * accu[8];
    cov[3] = cov[1]; cov[6] = cov[2]; cov[7] = cov[5];
    float ev, nv[3];
    eigen33(cov, ev, nv);
    out[0] = nv[0]; out[1] = nv[1]; out[2] = nv[2];
    out[3] = -1.0f * redux4(nv[0] * accu[6], nv[1] * accu[7], nv[2] * accu[8], 0.0f * 1.0f);
  }
}
// SampleConsensusModelPlane::projectPoints
OPE_HD void plane_project(const float c[4], float x, float y, float z, float q[3]) {
  float mc[4] = {c[0], c[1], c[2], 0.0f};
  const float nrm = sqrtf(redux4(mc[0] * mc[0], mc[1] * mc[1], mc[2] * mc[2], mc[3] * mc[3]));
  for (int i = 0; i < 4; ++i) mc[i] /= nrm;
  const float dist = redux4(mc[0] * x, mc[1] * y, mc[2] * z, c[3] * 1.0f);
  q[0] = x - mc[0] * dist; q[1] = y - mc[1] * dist; q[2] = z - mc[2] * dist;
}
// bounding box (x, y) of the projected inliers: out = {min x, min y, max x, max y}, float bits compared through atomics on ints
__device__ __forceinline__ void atomic_min_f(float* a, float v) { v += 0.0f; if (v >= 0) atomicMin((int*)a, __float_as_int(v)); else atomicMax((unsigned*)a, __float_as_uint(v)); }
__device__ __forceinline__ void atomic_max_f(float* a, float v) { v += 0.0f; if (v >= 0) atomicMax((int*)a, __float_as_int(v)); else atomicMin((unsigned*)a, __float_as_uint(v)); }
// frame f (blockIdx.y): inliers[off[f] .. off[f + 1]), plane coeff[4 f ..], box out[4 f ..]
__global__ void projected_bbox_kernel(const float4* __restrict__ pts, const int* __restrict__ inliers, const int* __restrict__ off,
                                      const float* __restrict__ coeff_all, float* __restrict__ out_all) {
  const int f = blockIdx.y;
  const float* coeff = coeff_all + 4 * f;
  float* out = out_all + 4 * f;
  const float c[4] = {coeff[0], coeff[1], coeff[2], coeff[3]};
  float mnx = INFINITY, mny = INFINITY, mxx = -INFINITY, mxy = -INFINITY;
  for (int i = off[f] + blockIdx.x * blockDim.x + threadIdx.x, e = off[f + 1]; i < e; i += gridDim.x * blockDim.x) {
    const float4 p = __ldg(pts + inliers[i]);
    float q[3];
    plane_project(c, p.x, p.y, p.z, q);
    mnx = fminf(mnx, q[0]); mny = fminf(mny, q[1]); mxx = fmaxf(mxx, q[0]); mxy = fmaxf(mxy, q[1]);
  }
  for (int o = 16; o > 0; o >>= 1) {
    mnx = fminf(mnx, __shfl_xor_sync(0xffffffffu, mnx, o)); mny = fminf(mny, __shfl_xor_sync(0xffffffffu, mny, o));
    mxx = fmaxf(mxx, __shfl_xor_sync(0xffffffffu, mxx, o)); mxy = fmaxf(mxy, __shfl_xor_sync(0xffffffffu, mxy, o));
  }
  if ((threadIdx.x & 31) == 0 && mnx <= mxx) { atomic_min_f(out, mnx); atomic_min_f(out + 1, mny); atomic_max_f(out + 2, mxx); atomic_max_f(out + 3, mxy); }
}
// pcl::ExtractPolygonalPrismData over the 4-corner rectangle: signed height in [0, FLT_MAX] and the projected point inside the polygon.
// k1 < 0: the frame has no table plane, nothing is inside.
struct PrismArgs { float mc[4]; float poly[4][2]; int k1, k2; };
__device__ __forceinline__ bool prism_keep(const PrismArgs& a, float4 p) {
  if (a.k1 < 0) return false;
  const double distance = (double)(a.mc[0] * p.x + a.mc[1] * p.y + a.mc[2] * p.z + a.mc[3]);
  bool keep = !(distance < 0.0 || distance > (double)FLT_MAX);
  if (keep) {
    float q[3];
    plane_project(a.mc, p.x, p.y, p.z, q);
    const double px = q[a.k1], py = q[a.k2];
    bool in = false;
    double xold = a.poly[3][0], yold = a.poly[3][1];
    for (int e = 0; e < 4; ++e) {
      const double xnew = a.poly[e][0], ynew = a.poly[e][1];
      double x1, x2, y1, y2;
      if (xnew > xold) { x1 = xold; x2 = xnew; y1 = yold; y2 = ynew; } else { x1 = xnew; x2 = xold; y1 = ynew; y2 = yold; }
      if ((xnew < px) == (px <= xold) && (py - y1) * (x2 - x1) < (y2 - y1) * (px - x1)) in = !in;
      xold = xnew; yold = ynew;
    }
    keep = in;
  }
  return keep;
}
// frame f (blockIdx.y) is cropped by pa[f]
__global__ void prism_flag_kernel(const float4* __restrict__ pts, const int* __restrict__ off, const PrismArgs* __restrict__ pa,
                                  int* __restrict__ flags) {
  const int f = blockIdx.y;
  const PrismArgs a = pa[f];
  for (int i = off[f] + blockIdx.x * blockDim.x + threadIdx.x, e = off[f + 1]; i < e; i += gridDim.x * blockDim.x)
    flags[i] = prism_keep(a, __ldg(pts + i)) ? 1 : 0;
}

}  // namespace ope

using namespace ope;

namespace {

// SampleConsensusModel::drawIndexSample: boost::mt19937(12345) through uniform_int<>(0, INT_MAX) = mt() >> 1, Fisher-Yates swaps on
// shuffled_indices_ (initially 0 .. n-1). Only the entries a swap has touched are stored (at most 6 per draw), so drawing costs the
// same for every n: a batch draws for every frame.
struct PlaneSampler {
  std::mt19937 rng{12345u};
  size_t index_size;
  int head[3] = {0, 1, 2};                      // positions 0..2
  std::vector<std::pair<size_t, int>> moved;    // (position, value) of the other entries that differ from the identity
  explicit PlaneSampler(size_t n) : index_size(n) {}
  int* at(size_t pos) {
    if (pos < 3) return &head[pos];
    for (auto& e : moved) if (e.first == pos) return &e.second;
    moved.emplace_back(pos, (int)pos);
    return &moved.back().second;
  }
  void draw(int out[3]) {
    for (unsigned i = 0; i < 3; ++i) {
      const size_t j = i + ((unsigned)(rng() >> 1) % (index_size - i));
      int* b = at(j);   // may grow `moved`; head[i] does not move
      std::swap(head[i], *b);
    }
    out[0] = head[0]; out[1] = head[1]; out[2] = head[2];
  }
};
bool sample_good(const float4& p0, const float4& p1, const float4& p2) {
  const float d0 = (p1.x - p0.x) / (p2.x - p0.x), d1 = (p1.y - p0.y) / (p2.y - p0.y), d2 = (p1.z - p0.z) / (p2.z - p0.z);
  return (d0 != d1) || (d2 != d1);
}
bool plane_from_sample(const float4& p0, const float4& p1, const float4& p2, float c[4]) {
  const float a[3] = {p1.x - p0.x, p1.y - p0.y, p1.z - p0.z}, b[3] = {p2.x - p0.x, p2.y - p0.y, p2.z - p0.z};
  const float d0 = a[0] / b[0], d1 = a[1] / b[1], d2 = a[2] / b[2];
  if ((d0 == d1) && (d2 == d1)) return false;
  c[0] = a[1] * b[2] - a[2] * b[1];
  c[1] = a[2] * b[0] - a[0] * b[2];
  c[2] = a[0] * b[1] - a[1] * b[0];
  c[3] = 0.0f;
  const float nrm = std::sqrt(redux4(c[0] * c[0], c[1] * c[1], c[2] * c[2], c[3] * c[3]));
  for (int i = 0; i < 4; ++i) c[i] /= nrm;
  c[3] = -1.0f * redux4(c[0] * p0.x, c[1] * p0.y, c[2] * p0.z, c[3] * 1.0f);
  return true;
}

// The padded bounding rectangle of the projected table inliers (box = min x, min y, max x, max y), z from the plane equation
// (objectsegmentationplane.cpp:174-196), and ExtractPolygonalPrismData's plane of its four corners (mean + covariance + eigen33),
// flipped towards the viewpoint (0, 0, 0)
PrismArgs prism_args(const float c1[4], const float box[4], double hull_margin) {
  const float vx[4] = {(float)(box[0] - hull_margin), (float)(box[0] - hull_margin), (float)(box[2] + hull_margin), (float)(box[2] + hull_margin)};
  const float vy[4] = {(float)(box[1] - hull_margin), (float)(box[3] + hull_margin), (float)(box[3] + hull_margin), (float)(box[1] - hull_margin)};
  float rect[4][3];
  for (int i = 0; i < 4; ++i) { rect[i][0] = vx[i]; rect[i][1] = vy[i]; rect[i][2] = -((c1[0] * vx[i]) + (c1[1] * vy[i]) + c1[3]) / c1[2]; }
  PrismArgs pa;
  {
    float accu[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = 0; i < 4; ++i) {
      const float* p = rect[i];
      accu[0] += p[0] * p[0]; accu[1] += p[0] * p[1]; accu[2] += p[0] * p[2];
      accu[3] += p[1] * p[1]; accu[4] += p[1] * p[2]; accu[5] += p[2] * p[2];
      accu[6] += p[0]; accu[7] += p[1]; accu[8] += p[2];
    }
    for (int i = 0; i < 9; ++i) accu[i] /= 4.0f;
    float cov[9];
    cov[0] = accu[0] - accu[6] * accu[6]; cov[1] = accu[1] - accu[6] * accu[7]; cov[2] = accu[2] - accu[6] * accu[8];
    cov[4] = accu[3] - accu[7] * accu[7]; cov[5] = accu[4] - accu[7] * accu[8]; cov[8] = accu[5] - accu[8] * accu[8];
    cov[3] = cov[1]; cov[6] = cov[2]; cov[7] = cov[5];
    float ev, nv[3];
    eigen33(cov, ev, nv);
    float* mc = pa.mc;
    mc[0] = nv[0]; mc[1] = nv[1]; mc[2] = nv[2]; mc[3] = 0.0f;
    mc[3] = -1.0f * redux4(mc[0] * accu[6], mc[1] * accu[7], mc[2] * accu[8], mc[3] * 1.0f);
    const float vp[3] = {0.0f - rect[0][0], 0.0f - rect[0][1], 0.0f - rect[0][2]};
    const float cos_theta = redux4(vp[0] * mc[0], vp[1] * mc[1], vp[2] * mc[2], 0.0f * mc[3]);
    if (cos_theta < 0) {
      for (int i = 0; i < 4; ++i) mc[i] *= -1.0f;
      mc[3] = 0.0f;
      mc[3] = -1.0f * redux4(mc[0] * rect[0][0], mc[1] * rect[0][1], mc[2] * rect[0][2], mc[3] * 1.0f);
    }
    int k0 = (std::fabs(mc[0]) > std::fabs(mc[1])) ? 0 : 1;
    k0 = (std::fabs(mc[k0]) > std::fabs(mc[2])) ? k0 : 2;
    pa.k1 = (k0 + 1) % 3; pa.k2 = (k0 + 2) % 3;
    for (int i = 0; i < 4; ++i) { pa.poly[i][0] = rect[i][pa.k1]; pa.poly[i][1] = rect[i][pa.k2]; }
  }
  return pa;
}

// RandomSampleConsensus::computeModel [UPSTREAM ransac.hpp] replayed over the inlier counts of the max_iterations + 1 drawn
// hypotheses of a cloud of n points: returns the iteration count, *best = the winning hypothesis (-1: none)
int ransac_replay(const int* counts, size_t n, const ope_segment_params& P, int* best_out) {
  const int M = P.max_iterations + 1;
  int it = 0, n_best = -INT_MAX, best = -1;
  double k = 1.0;
  const double log_probability = std::log(1.0 - P.probability), one_over_indices = 1.0 / (double)n;
  while (it < k && it < M) {
    if (counts[(size_t)it] > n_best) {
      n_best = counts[(size_t)it]; best = it;
      const double w = (double)n_best * one_over_indices;
      double p_no_outliers = 1.0 - std::pow(w, 3.0);
      p_no_outliers = std::max(std::numeric_limits<double>::epsilon(), p_no_outliers);
      p_no_outliers = std::min(1.0 - std::numeric_limits<double>::epsilon(), p_no_outliers);
      k = log_probability / std::log(p_no_outliers);
    }
    ++it;
    if (it > P.max_iterations) break;
  }
  *best_out = best;
  return it;
}

}  // namespace

extern "C" {

void ope_segment_params_default(ope_segment_params* p) {
  std::memset(p, 0, sizeof(*p));
  p->distance_threshold = 0.01; p->max_iterations = 50; p->probability = 0.99; p->hull_margin = 0.1;
  p->cluster_tolerance = 0.05f; p->min_cluster_size = 300; p->max_cluster_size = 100000;
}

// labels: n entries — cluster number (0 = largest; equal sizes by the smaller first index) or -1 (not finite / component outside
// [min_size, max_size]). Returns the number of clusters kept in *n_clusters.
int ope_euclidean_clusters(ope_ctx* ctx, const ope_cloud* cloud, float tolerance, int min_size, int max_size, int32_t* labels, int* n_clusters) {
  OPE_ENTER(ctx);
  if (!ctx || !cloud || !labels || !n_clusters || !(tolerance > 0)) return OPE_ERR_INVALID;
  *n_clusters = 0;
  const size_t n = cloud->n;
  if (n == 0) return OPE_OK;
  if (n > 0x7ffffffeull) return fail(ctx, OPE_ERR_INVALID, "cloud too large");
  OPE_TRY(cloud_bbox(ctx, const_cast<ope_cloud*>(cloud)));
  std::vector<int> root(n, -1);
  if (cloud->n_finite > 0) {
    GridView g;
    OPE_TRY(cloud_grid(ctx, cloud, tolerance, &g));
    Scratch<int> parent(ctx), d_root(ctx);
    OPE_TRY(parent.alloc(n)); OPE_TRY(d_root.alloc(n));
    cluster_init_kernel<<<div_up(n, kSegThreads), kSegThreads, 0, ctx->stream>>>(cloud->pts, (int)n, parent.p);
    OPE_TRY(check_launch(ctx, "cluster_init_kernel"));
    const unsigned blocks = (unsigned)std::min<size_t>(div_up(n * 32, kSegThreads), (size_t)ctx->sm_count * 16);
    cluster_union_kernel<<<blocks, kSegThreads, 0, ctx->stream>>>(g, cloud->pts, (int)n, tolerance * tolerance, parent.p);
    OPE_TRY(check_launch(ctx, "cluster_union_kernel"));
    cluster_flatten_kernel<<<div_up(n, kSegThreads), kSegThreads, 0, ctx->stream>>>(cloud->pts, (int)n, parent.p, d_root.p);
    OPE_TRY(check_launch(ctx, "cluster_flatten_kernel"));
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(root.data(), d_root.p, n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    OPE_CUDA_TRY(ctx, stream_sync(ctx));
  }
  // bookkeeping on the host: component sizes, the size window, the reference's ordering (largest first)
  std::vector<int> size(n, 0);
  for (size_t i = 0; i < n; ++i) if (root[i] >= 0) size[(size_t)root[i]]++;
  std::vector<int> roots;
  for (size_t i = 0; i < n; ++i) if (size[i] >= min_size && size[i] <= max_size && size[i] > 0) roots.push_back((int)i);   // a root is its component's smallest index
  std::sort(roots.begin(), roots.end(), [&](int a, int b) { return size[(size_t)a] != size[(size_t)b] ? size[(size_t)a] > size[(size_t)b] : a < b; });
  std::vector<int> number(n, -1);
  for (size_t c = 0; c < roots.size(); ++c) number[(size_t)roots[c]] = (int)c;
  for (size_t i = 0; i < n; ++i) labels[i] = root[i] >= 0 ? number[(size_t)root[i]] : -1;
  *n_clusters = (int)roots.size();
  return OPE_OK;
}

}  // extern "C"

// ---- many frames per call: ope_scene_batch_create / ope_scene_pose_batch ---------------------------------------------------------
// A chunk of frames runs through the kernels above as ONE concatenated point array whose frames are contiguous and in order (every
// compaction is order-preserving, so frame boundaries after a compaction are the scan at the old boundaries). Each segmented launch
// takes its frame from blockIdx.y and the frame's bounds from device memory; the host only draws the RANSAC samples, replays the
// stopping rule, builds the prism planes and numbers the clusters, from small per-frame read-backs.
namespace ope {

// out[f] = pos[off ? off[f] : f * stride], f = 0 .. frames: frame boundaries after a compaction (pos = the exclusive scan of the
// flags, off = the boundaries before it) or of a batched depth cloud (pos = col_start, stride = columns)
__global__ void span_bounds_kernel(const int* __restrict__ pos, const int* __restrict__ off, int stride, int frames, int* __restrict__ out) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f <= frames) out[f] = pos[off ? off[f] : f * stride];
}
__global__ void fill_kernel(float* __restrict__ p, int n, float v0, float v1, int period) {   // p[i] = i % period < period / 2 ? v0 : v1
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = (i % period) < period / 2 ? v0 : v1;
}
__global__ void fill_i32_kernel(int* __restrict__ p, int n, int v) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}
// per-frame bounding box (min xyz, max xyz) of pts[idx[k]], k in frame f's span
__global__ void span_bbox_kernel(const float4* __restrict__ pts, const int* __restrict__ idx, const int* __restrict__ off, float* __restrict__ out6) {
  const int f = blockIdx.y;
  float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int k = off[f] + blockIdx.x * blockDim.x + threadIdx.x, e = off[f + 1]; k < e; k += gridDim.x * blockDim.x) {
    const float4 p = __ldg(pts + idx[k]);
    mn[0] = fminf(mn[0], p.x); mn[1] = fminf(mn[1], p.y); mn[2] = fminf(mn[2], p.z);
    mx[0] = fmaxf(mx[0], p.x); mx[1] = fmaxf(mx[1], p.y); mx[2] = fmaxf(mx[2], p.z);
  }
  for (int o = 16; o > 0; o >>= 1)
    for (int a = 0; a < 3; ++a) { mn[a] = fminf(mn[a], __shfl_xor_sync(0xffffffffu, mn[a], o)); mx[a] = fmaxf(mx[a], __shfl_xor_sync(0xffffffffu, mx[a], o)); }
  if ((threadIdx.x & 31) == 0 && mn[0] <= mx[0])
    for (int a = 0; a < 3; ++a) { atomic_min_f(out6 + 6 * f + a, mn[a]); atomic_max_f(out6 + 6 * f + 3 + a, mx[a]); }
}

// The clustering grid of a chunk: frame f owns cells [base, base + dim x * dim y * dim z), so that no radius traversal crosses frames.
// Cell edge >= the tolerance: every neighbour closer than the tolerance lies in the 27 cells around a point's own cell.
struct CellFrame { float o[3]; float inv; int dim[3]; int base; };
__device__ __forceinline__ void cell_coords(const CellFrame& g, float4 p, int c[3]) {
  const float v[3] = {p.x, p.y, p.z};
  for (int a = 0; a < 3; ++a) c[a] = min(max((int)floorf((v[a] - g.o[a]) * g.inv), 0), g.dim[a] - 1);
}
__global__ void scene_cell_count_kernel(const float4* __restrict__ pts, const int* __restrict__ off, const CellFrame* __restrict__ grid, int* __restrict__ cell_of,
                                        int* __restrict__ cell_count) {
  const int f = blockIdx.y;
  const CellFrame g = grid[f];
  for (int i = off[f] + blockIdx.x * blockDim.x + threadIdx.x, e = off[f + 1]; i < e; i += gridDim.x * blockDim.x) {
    int c[3];
    cell_coords(g, __ldg(pts + i), c);
    const int cell = g.base + c[0] + g.dim[0] * (c[1] + g.dim[1] * c[2]);
    cell_of[i] = cell;
    atomicAdd(cell_count + cell, 1);
  }
}
__global__ void scene_cell_fill_kernel(int n, const int* __restrict__ cell_of, const int* __restrict__ cell_start, int* __restrict__ fill,
                                       int* __restrict__ sorted) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) sorted[cell_start[cell_of[i]] + atomicAdd(fill + cell_of[i], 1)] = i;   // order inside a cell does not matter
}
// one warp per point: every point of the 27 surrounding cells closer than the tolerance and with a smaller index is united with it —
// the same graph as cluster_union_kernel, so the components (and their smallest indices, the roots) are the same
__global__ void __launch_bounds__(kSegThreads) scene_cluster_union_kernel(const float4* __restrict__ pts, const int* __restrict__ off, const CellFrame* __restrict__ grid,
                                                                          const int* __restrict__ cell_start, const int* __restrict__ sorted, float r2,
                                                                          int* __restrict__ parent) {
  const int f = blockIdx.y;
  const CellFrame g = grid[f];
  const int lane = threadIdx.x & 31;
  const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
  for (int i = off[f] + wid, e = off[f + 1]; i < e; i += n_warps) {
    const float4 q = __ldg(pts + i);
    int c[3];
    cell_coords(g, q, c);
    for (int dz = -1; dz <= 1; ++dz) for (int dy = -1; dy <= 1; ++dy) for (int dx = -1; dx <= 1; ++dx) {
      const int x = c[0] + dx, y = c[1] + dy, z = c[2] + dz;
      if (x < 0 || y < 0 || z < 0 || x >= g.dim[0] || y >= g.dim[1] || z >= g.dim[2]) continue;
      const int cell = g.base + x + g.dim[0] * (y + g.dim[1] * z);
      for (int t = cell_start[cell] + lane, te = cell_start[cell + 1]; t < te; t += 32) {
        const int j = sorted[t];
        if (j < i) {
          const float4 p = __ldg(pts + j);
          if (dist2(q.x, q.y, q.z, p.x, p.y, p.z) < r2) uf_union(parent, i, j);
        }
      }
    }
  }
}
__global__ void component_size_kernel(int n, const int* __restrict__ root, int* __restrict__ size) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) atomicAdd(size + root[i], 1);
}
// roots (a component's smallest index) whose component size is inside [min_size, max_size]
__global__ void root_flag_kernel(int n, const int* __restrict__ root, const int* __restrict__ size, int min_size, int max_size, int* __restrict__ flags) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) flags[i] = (root[i] == i && size[i] >= min_size && size[i] <= max_size && size[i] > 0) ? 1 : 0;
}
__global__ void root_compact_kernel(int n, const int* __restrict__ pos, const int* __restrict__ size, int* __restrict__ out_idx, int* __restrict__ out_size) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && pos[i + 1] > pos[i]) { out_idx[pos[i]] = i; out_size[pos[i]] = size[i]; }
}
__global__ void scatter_number_kernel(int m, const int2* __restrict__ root_number, int* __restrict__ number) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k < m) number[root_number[k].x] = root_number[k].y;
}
// the labels of ope_segment_objects_on_plane: prism points NO_CLUSTER, second-plane inliers PLANE, the rest their cluster number
__global__ void label_prism_kernel(const int* __restrict__ off, const int* __restrict__ live, const int* __restrict__ prism, int* __restrict__ labels) {
  const int f = blockIdx.y;
  if (!live[f]) return;
  for (int j = off[f] + blockIdx.x * blockDim.x + threadIdx.x, e = off[f + 1]; j < e; j += gridDim.x * blockDim.x) labels[prism[j]] = OPE_SEG_NO_CLUSTER;
}
__global__ void label_plane_kernel(const int* __restrict__ off, const int* __restrict__ inliers, const int* __restrict__ prism, int* __restrict__ labels) {
  const int f = blockIdx.y;
  for (int k = off[f] + blockIdx.x * blockDim.x + threadIdx.x, e = off[f + 1]; k < e; k += gridDim.x * blockDim.x) labels[prism[inliers[k]]] = OPE_SEG_PLANE;
}
__global__ void label_rest_kernel(const int* __restrict__ off, const int* __restrict__ rest, const int* __restrict__ prism, const int* __restrict__ root,
                                  const int* __restrict__ number, int* __restrict__ labels) {
  const int f = blockIdx.y;
  for (int k = off[f] + blockIdx.x * blockDim.x + threadIdx.x, e = off[f + 1]; k < e; k += gridDim.x * blockDim.x) {
    const int c = number[root[k]];
    labels[prism[rest[k]]] = c >= 0 ? c : OPE_SEG_NO_CLUSTER;
  }
}

// ope_scene_pose_batch, ope_scene_track_step: block b copies the points of cut b whose label is `want` (INT_MIN: every point) in
// index order to out + out_off
__global__ void __launch_bounds__(1024) scene_cut_kernel(const SceneCut* __restrict__ cuts, float4* __restrict__ out) {
  __shared__ int warp_count[32];
  const SceneCut c = cuts[blockIdx.x];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int base = 0;
  for (int t0 = 0; t0 < c.n; t0 += 1024) {
    const int i = t0 + threadIdx.x;
    const bool keep = i < c.n && (c.want == INT_MIN || c.labels[i] == c.want);
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) warp_count[w] = __popc(m);
    __syncthreads();
    int before = 0, total = 0;
    for (int k = 0; k < 32; ++k) { const int v = warp_count[k]; before += k < w ? v : 0; total += v; }
    if (keep) out[c.out_off + base + before + __popc(m & ((1u << lane) - 1u))] = c.pts[i];
    base += total;
    __syncthreads();
  }
}

int scene_cut_device(ope_ctx* ctx, const SceneCut* d_cuts, int n_cuts, float4* out) {
  if (n_cuts == 0) return OPE_OK;
  scene_cut_kernel<<<(unsigned)n_cuts, 1024, 0, ctx->stream>>>(d_cuts, out);
  return check_launch(ctx, "scene_cut_kernel");
}

}  // namespace ope

namespace {

unsigned span_blocks(size_t max_per_frame) { return (unsigned)std::max<size_t>(1, std::min<size_t>(div_up(max_per_frame, kSegThreads), 1024)); }

size_t max_span(const std::vector<int>& off) {
  size_t m = 0;
  for (size_t f = 0; f + 1 < off.size(); ++f) m = std::max<size_t>(m, (size_t)(off[f + 1] - off[f]));
  return m;
}

template <typename T>
int download(ope_ctx* ctx, std::vector<T>& dst, const T* src, size_t count) {
  dst.resize(count);
  if (count) OPE_CUDA_TRY(ctx, cudaMemcpyAsync(dst.data(), src, count * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
  return OPE_OK;
}
template <typename T>
int upload(ope_ctx* ctx, T* dst, const std::vector<T>& src) {
  if (!src.empty()) OPE_CUDA_TRY(ctx, cudaMemcpyAsync(dst, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
  return OPE_OK;
}

// ordered compaction of a chunk: d_idx[0 .. total) = the flagged indices ascending, d_off_out = the frame boundaries in d_idx.
// flags: n + 1 entries, the first n written by a flag kernel.
int compact_frames(ope_ctx* ctx, int* flags, size_t n, int frames, const int* d_off_in, int* d_idx, int* d_off_out) {
  OPE_CUDA_TRY(ctx, cudaMemsetAsync(flags + n, 0, sizeof(int), ctx->stream));
  OPE_TRY(exclusive_scan_i32(ctx, flags, n + 1));
  if (n) {
    index_compact_kernel<<<div_up(n, kSegThreads), kSegThreads, 0, ctx->stream>>>((int)n, flags, d_idx);
    OPE_TRY(check_launch(ctx, "index_compact_kernel"));
  }
  span_bounds_kernel<<<div_up((size_t)frames + 1, kSegThreads), kSegThreads, 0, ctx->stream>>>(flags, d_off_in, 0, frames, d_off_out);
  return check_launch(ctx, "span_bounds_kernel");
}

// pcl::SACSegmentation::segment (SACMODEL_PLANE, SAC_RANSAC, optimized coefficients) for every frame of a concatenated point array
// without NaN points. pts: the frames' points, frame f at [off[f], off[f + 1]) (host h_off and device d_off). The samples are drawn
// on the host exactly as PCL draws them, their points fetched in one gather, every candidate plane of every frame scored in one
// launch, the adaptive stopping rule replayed over the counts. live[f] (in): fit frame f; (out): frame f has a plane (not below 3
// points). Outputs per frame: iterations, status (a degenerate sample fails the frame), the refined plane in d_plane[4 f ..]; the
// refined plane's inliers (ascending indices into pts) in d_inl, frame f at [d_inl_off[f], d_inl_off[f + 1]); d_live (device copy
// of live). d_inl and flags have room for n and n + 1 entries. Two host waits.
int plane_segment_frames(ope_ctx* ctx, const float4* pts, const std::vector<int>& h_off, const int* d_off, const ope_segment_params& P,
                         std::vector<int>& live, std::vector<int>& iterations, std::vector<int>& status, float* d_plane, int* d_live,
                         int* d_inl, int* d_inl_off, int* flags) {
  const int B = (int)live.size();
  const size_t n = (size_t)h_off[(size_t)B];
  const int M = P.max_iterations + 1;
  iterations.assign((size_t)B, 0);
  bool any = false;
  for (int f = 0; f < B; ++f) {
    if (h_off[(size_t)f + 1] - h_off[(size_t)f] < 3) live[(size_t)f] = 0;   // no plane below 3 points
    any |= live[(size_t)f] != 0;
  }
  std::vector<float> h_best((size_t)4 * B, 0.0f);
  if (any) {
    std::vector<int> h_idx((size_t)3 * M * B, 0);
    for (int f = 0; f < B; ++f) {
      if (!live[(size_t)f]) continue;
      PlaneSampler sampler((size_t)(h_off[(size_t)f + 1] - h_off[(size_t)f]));
      int* o = &h_idx[(size_t)3 * M * f];
      for (int h = 0; h < M; ++h) {
        sampler.draw(o + 3 * h);
        for (int k = 0; k < 3; ++k) o[3 * h + k] += h_off[(size_t)f];
      }
    }
    Scratch<int> d_idx(ctx), d_counts(ctx);
    Scratch<float4> d_spts(ctx);
    Scratch<float> d_coeffs(ctx);
    OPE_TRY(d_idx.alloc(h_idx.size())); OPE_TRY(d_spts.alloc(h_idx.size())); OPE_TRY(d_coeffs.alloc((size_t)4 * M * B));
    OPE_TRY(d_counts.alloc((size_t)M * B));
    OPE_TRY(upload(ctx, d_idx.p, h_idx));
    gather_points_kernel<<<div_up(h_idx.size(), kSegThreads), kSegThreads, 0, ctx->stream>>>(pts, d_idx.p, (int)h_idx.size(), d_spts.p);
    OPE_TRY(check_launch(ctx, "gather_points_kernel"));
    std::vector<float4> sp;
    OPE_TRY(download(ctx, sp, (const float4*)d_spts.p, h_idx.size()));
    OPE_CUDA_TRY(ctx, stream_sync(ctx));
    std::vector<float> h_coeffs((size_t)4 * M * B, 0.0f);
    for (int f = 0; f < B; ++f) {
      if (!live[(size_t)f]) continue;
      for (int h = 0; h < M; ++h) {
        const size_t q = (size_t)M * f + h;
        const float4 &p0 = sp[3 * q], &p1 = sp[3 * q + 1], &p2 = sp[3 * q + 2];
        // a degenerate draw makes PCL draw again / skip the iteration, which shifts the whole random sequence: practically never
        // (three exactly collinear float points), and then this one-gather scheme does not apply: the frame fails
        if (!sample_good(p0, p1, p2) || !plane_from_sample(p0, p1, p2, &h_coeffs[4 * q])) {
          status[(size_t)f] = fail(ctx, OPE_ERR_UNSUPPORTED, "plane RANSAC drew a degenerate sample (hypothesis %d)", h);
          live[(size_t)f] = 0;
          break;
        }
      }
    }
    OPE_TRY(upload(ctx, d_coeffs.p, h_coeffs));
    plane_count_kernel<<<dim3(M, B), kSegThreads, 0, ctx->stream>>>(pts, d_off, d_coeffs.p, P.distance_threshold, d_counts.p);
    OPE_TRY(check_launch(ctx, "plane_count_kernel"));
    std::vector<int> counts;
    OPE_TRY(download(ctx, counts, (const int*)d_counts.p, (size_t)M * B));
    OPE_CUDA_TRY(ctx, stream_sync(ctx));
    for (int f = 0; f < B; ++f) {
      if (!live[(size_t)f]) continue;
      int best = -1;
      iterations[(size_t)f] = ransac_replay(&counts[(size_t)M * f], (size_t)(h_off[(size_t)f + 1] - h_off[(size_t)f]), P, &best);
      std::memcpy(&h_best[(size_t)4 * f], &h_coeffs[(size_t)4 * ((size_t)M * f + best)], 4 * sizeof(float));
    }
  }
  // inliers of the best model, the refit over them (one block per frame), inliers of the refined model
  Scratch<float> d_best(ctx);
  OPE_TRY(d_best.alloc((size_t)4 * B));
  OPE_TRY(upload(ctx, d_best.p, h_best));
  OPE_TRY(upload(ctx, d_live, live));
  const dim3 grid(span_blocks(max_span(h_off)), B);
  plane_flag_kernel<<<grid, kSegThreads, 0, ctx->stream>>>(pts, d_off, d_best.p, P.distance_threshold, 0, d_live, flags);
  OPE_TRY(check_launch(ctx, "plane_flag_kernel"));
  OPE_TRY(compact_frames(ctx, flags, n, B, d_off, d_inl, d_inl_off));
  plane_refit_kernel<<<B, kSegThreads, 0, ctx->stream>>>(pts, d_inl, d_inl_off, d_best.p, d_plane);
  OPE_TRY(check_launch(ctx, "plane_refit_kernel"));
  plane_flag_kernel<<<grid, kSegThreads, 0, ctx->stream>>>(pts, d_off, d_plane, P.distance_threshold, 0, d_live, flags);
  OPE_TRY(check_launch(ctx, "plane_flag_kernel"));
  return compact_frames(ctx, flags, n, B, d_off, d_inl, d_inl_off);
}

// {0, n}: the offsets of a one-frame run of the stages below, on the host and on the device
int one_span(ope_ctx* ctx, size_t n, std::vector<int>& h_off, Scratch<int>& d_off) {
  h_off = {0, (int)n};
  OPE_TRY(d_off.alloc(2));
  return upload(ctx, d_off.p, h_off);
}

// The crop (ProcessingPcd::getPassThrough) of every frame of a concatenated cloud, frame f at [off[f], off[f + 1]) (host h_off and
// device d_off). The crop does not depend on the frame: one flag pass and one ordered compaction over the whole array. idx (room for
// n entries): the kept indices, ascending; d_crop_off / h_crop: the frames' bounds among them. The kept points are gathered into *out,
// which new_points(m, out) allocates once their number m is known. One host wait.
template <typename NewPoints>
int crop_frames(ope_ctx* ctx, const float4* cloud, const std::vector<int>& h_off, const int* d_off, const float lim[6], int* idx,
                int* d_crop_off, std::vector<int>& h_crop, NewPoints new_points, float4** out) {
  const int B = (int)h_off.size() - 1;
  const size_t n = (size_t)h_off[(size_t)B];
  Scratch<int> flags(ctx);
  OPE_TRY(flags.alloc(n + 1));
  if (n) {
    pass_flag_kernel<<<div_up(n, kSegThreads), kSegThreads, 0, ctx->stream>>>(cloud, (int)n, lim[0], lim[1], lim[2], lim[3], lim[4], lim[5], flags.p);
    OPE_TRY(check_launch(ctx, "pass_flag_kernel"));
  }
  OPE_TRY(compact_frames(ctx, flags.p, n, B, d_off, idx, d_crop_off));
  OPE_TRY(download(ctx, h_crop, (const int*)d_crop_off, (size_t)B + 1));
  OPE_CUDA_TRY(ctx, stream_sync(ctx));
  const size_t m = (size_t)h_crop[(size_t)B];
  OPE_TRY(new_points(m, out));
  if (m) {
    gather_points_kernel<<<div_up(m, kSegThreads), kSegThreads, 0, ctx->stream>>>(cloud, idx, (int)m, *out);
    OPE_TRY(check_launch(ctx, "gather_points_kernel"));
  }
  return OPE_OK;
}

// The segmentation (ObjectSegmentationPlane::getSegmentedObjectsOnPlane, D&L/src/objectsegmentationplane.cpp:122-282) of every frame
// of a concatenated, cropped point array, frame f at [off[f], off[f + 1]) (host h_off and device d_off): table plane, prism over the
// padded bounding rectangle of its projected inliers, second plane on the prism's points, Euclidean clusters of the rest. Writes each
// frame's status, iterations, and, when both planes were found, planes, n_clusters and cluster sizes to out[f] (else n_clusters = -1),
// and every point's label to labels (device). Eight host waits; the last label kernels may still be running on return.
int segment_frames(ope_ctx* ctx, const ope_segment_params& S, const float4* pts, const std::vector<int>& h_off, const int* d_off, int* labels,
                   ope_scene_batch::Frame* out) {
  const int B = (int)h_off.size() - 1;
  const size_t m = (size_t)h_off[(size_t)B];
  if (m) {
    fill_i32_kernel<<<div_up(m, kSegThreads), kSegThreads, 0, ctx->stream>>>(labels, (int)m, OPE_SEG_OUTSIDE_PRISM);
    OPE_TRY(check_launch(ctx, "fill_i32_kernel"));
  }
  std::vector<int> status((size_t)B, OPE_OK);
  // the table plane
  std::vector<int> live1((size_t)B, 1), it1, live2, it2;
  Scratch<float> c1(ctx), c2(ctx), box(ctx);
  Scratch<int> d_live1(ctx), d_live2(ctx), in1(ctx), in1_off(ctx), flags(ctx);
  OPE_TRY(c1.alloc((size_t)4 * B)); OPE_TRY(c2.alloc((size_t)4 * B)); OPE_TRY(box.alloc((size_t)6 * B));
  OPE_TRY(d_live1.alloc(B)); OPE_TRY(d_live2.alloc(B)); OPE_TRY(in1.alloc(m)); OPE_TRY(in1_off.alloc((size_t)B + 1)); OPE_TRY(flags.alloc(m + 1));
  OPE_TRY(plane_segment_frames(ctx, pts, h_off, d_off, S, live1, it1, status, c1.p, d_live1.p, in1.p, in1_off.p, flags.p));
  // bounding rectangle of the projected inliers -> prism plane per frame
  fill_kernel<<<div_up((size_t)4 * B, kSegThreads), kSegThreads, 0, ctx->stream>>>(box.p, 4 * B, INFINITY, -INFINITY, 4);
  OPE_TRY(check_launch(ctx, "fill_kernel"));
  const unsigned gx_crop = span_blocks(max_span(h_off));
  projected_bbox_kernel<<<dim3(std::min(gx_crop, 64u), B), kSegThreads, 0, ctx->stream>>>(pts, in1.p, in1_off.p, c1.p, box.p);
  OPE_TRY(check_launch(ctx, "projected_bbox_kernel"));
  std::vector<float> h_box, h_c1;
  OPE_TRY(download(ctx, h_box, (const float*)box.p, (size_t)4 * B));
  OPE_TRY(download(ctx, h_c1, (const float*)c1.p, (size_t)4 * B));
  OPE_CUDA_TRY(ctx, stream_sync(ctx));
  std::vector<PrismArgs> pa((size_t)B);
  for (int f = 0; f < B; ++f) {
    if (live1[(size_t)f]) pa[(size_t)f] = prism_args(&h_c1[(size_t)4 * f], &h_box[(size_t)4 * f], S.hull_margin);
    else { std::memset(&pa[(size_t)f], 0, sizeof(PrismArgs)); pa[(size_t)f].k1 = -1; }
  }
  Scratch<PrismArgs> d_pa(ctx);
  Scratch<int> prism(ctx), prism_off(ctx);
  OPE_TRY(d_pa.alloc(B)); OPE_TRY(prism.alloc(m)); OPE_TRY(prism_off.alloc((size_t)B + 1));
  OPE_TRY(upload(ctx, d_pa.p, pa));
  prism_flag_kernel<<<dim3(gx_crop, B), kSegThreads, 0, ctx->stream>>>(pts, d_off, d_pa.p, flags.p);
  OPE_TRY(check_launch(ctx, "prism_flag_kernel"));
  OPE_TRY(compact_frames(ctx, flags.p, m, B, d_off, prism.p, prism_off.p));
  std::vector<int> h_prism;
  OPE_TRY(download(ctx, h_prism, (const int*)prism_off.p, (size_t)B + 1));
  OPE_CUDA_TRY(ctx, stream_sync(ctx));
  const size_t mp = (size_t)h_prism[(size_t)B];
  // cloudObjWithPlane and the second plane
  Scratch<float4> sub(ctx);
  Scratch<int> in2(ctx), in2_off(ctx), rest(ctx), rest_off(ctx);
  OPE_TRY(sub.alloc(mp)); OPE_TRY(in2.alloc(mp)); OPE_TRY(in2_off.alloc((size_t)B + 1)); OPE_TRY(rest.alloc(mp)); OPE_TRY(rest_off.alloc((size_t)B + 1));
  if (mp) {
    gather_points_kernel<<<div_up(mp, kSegThreads), kSegThreads, 0, ctx->stream>>>(pts, prism.p, (int)mp, sub.p);
    OPE_TRY(check_launch(ctx, "gather_points_kernel"));
  }
  live2 = live1;
  OPE_TRY(plane_segment_frames(ctx, sub.p, h_prism, prism_off.p, S, live2, it2, status, c2.p, d_live2.p, in2.p, in2_off.p, flags.p));
  // the rest: prism points off the second plane, and the bounding box of every frame's rest for the clustering grid
  const unsigned gx_prism = span_blocks(max_span(h_prism));
  plane_flag_kernel<<<dim3(gx_prism, B), kSegThreads, 0, ctx->stream>>>(sub.p, prism_off.p, c2.p, S.distance_threshold, 1, d_live2.p, flags.p);
  OPE_TRY(check_launch(ctx, "plane_flag_kernel"));
  OPE_TRY(compact_frames(ctx, flags.p, mp, B, prism_off.p, rest.p, rest_off.p));
  fill_kernel<<<div_up((size_t)6 * B, kSegThreads), kSegThreads, 0, ctx->stream>>>(box.p, 6 * B, INFINITY, -INFINITY, 6);
  OPE_TRY(check_launch(ctx, "fill_kernel"));
  span_bbox_kernel<<<dim3(std::min(gx_prism, 64u), B), kSegThreads, 0, ctx->stream>>>(sub.p, rest.p, rest_off.p, box.p);
  OPE_TRY(check_launch(ctx, "span_bbox_kernel"));
  std::vector<int> h_rest;
  std::vector<float> h_box6, h_c2;
  OPE_TRY(download(ctx, h_rest, (const int*)rest_off.p, (size_t)B + 1));
  OPE_TRY(download(ctx, h_box6, (const float*)box.p, (size_t)6 * B));
  OPE_TRY(download(ctx, h_c2, (const float*)c2.p, (size_t)4 * B));
  OPE_CUDA_TRY(ctx, stream_sync(ctx));
  const size_t mr = (size_t)h_rest[(size_t)B];
  // Euclidean clusters of every frame's rest at once: union-find over the frame-aware grid
  std::vector<std::vector<int>> sizes((size_t)B);
  Scratch<float4> rpts(ctx);
  Scratch<int> root(ctx), number(ctx);
  OPE_TRY(rpts.alloc(mr)); OPE_TRY(root.alloc(mr)); OPE_TRY(number.alloc(mr));
  if (mr) {
    gather_points_kernel<<<div_up(mr, kSegThreads), kSegThreads, 0, ctx->stream>>>(sub.p, rest.p, (int)mr, rpts.p);
    OPE_TRY(check_launch(ctx, "gather_points_kernel"));
    std::vector<CellFrame> cf((size_t)B);
    size_t cells = 0;
    for (int f = 0; f < B; ++f) {
      CellFrame& g = cf[(size_t)f];
      const size_t nf = (size_t)(h_rest[(size_t)f + 1] - h_rest[(size_t)f]);
      const float* bx = &h_box6[(size_t)6 * f];
      double h = (double)S.cluster_tolerance * 1.001;   // a hair above the tolerance: float binning never splits a closer pair by two cells
      int64_t dim[3] = {1, 1, 1};
      for (;;) {
        for (int a = 0; a < 3; ++a) dim[a] = nf ? (int64_t)std::floor(((double)bx[3 + a] - (double)bx[a]) / h) + 1 : 1;
        if (dim[0] * dim[1] * dim[2] <= (int64_t)std::max<size_t>(8 * nf, 4096)) break;
        h *= 1.25;
      }
      for (int a = 0; a < 3; ++a) { g.o[a] = nf ? bx[a] : 0.0f; g.dim[a] = (int)dim[a]; }
      g.inv = (float)(1.0 / h);
      g.base = (int)cells;
      cells += (size_t)(dim[0] * dim[1] * dim[2]);
    }
    if (cells + mr > 0x7ffffffeull) return fail(ctx, OPE_ERR_INVALID, "clustering grid too large");
    Scratch<CellFrame> d_cf(ctx);
    Scratch<int> cell_of(ctx), cell_start(ctx), fill(ctx), sorted(ctx), parent(ctx), size(ctx);
    OPE_TRY(d_cf.alloc(B)); OPE_TRY(cell_of.alloc(mr)); OPE_TRY(cell_start.alloc(cells + 1)); OPE_TRY(fill.alloc(cells));
    OPE_TRY(sorted.alloc(mr)); OPE_TRY(parent.alloc(mr)); OPE_TRY(size.alloc(mr));
    OPE_TRY(upload(ctx, d_cf.p, cf));
    OPE_CUDA_TRY(ctx, cudaMemsetAsync(cell_start.p, 0, (cells + 1) * sizeof(int), ctx->stream));
    OPE_CUDA_TRY(ctx, cudaMemsetAsync(fill.p, 0, cells * sizeof(int), ctx->stream));
    OPE_CUDA_TRY(ctx, cudaMemsetAsync(size.p, 0, mr * sizeof(int), ctx->stream));
    OPE_CUDA_TRY(ctx, cudaMemsetAsync(number.p, 0xff, mr * sizeof(int), ctx->stream));
    const unsigned gx_rest = span_blocks(max_span(h_rest));
    scene_cell_count_kernel<<<dim3(gx_rest, B), kSegThreads, 0, ctx->stream>>>(rpts.p, rest_off.p, d_cf.p, cell_of.p, cell_start.p);
    OPE_TRY(check_launch(ctx, "scene_cell_count_kernel"));
    OPE_TRY(exclusive_scan_i32(ctx, cell_start.p, cells + 1));
    scene_cell_fill_kernel<<<div_up(mr, kSegThreads), kSegThreads, 0, ctx->stream>>>((int)mr, cell_of.p, cell_start.p, fill.p, sorted.p);
    OPE_TRY(check_launch(ctx, "scene_cell_fill_kernel"));
    cluster_init_kernel<<<div_up(mr, kSegThreads), kSegThreads, 0, ctx->stream>>>(rpts.p, (int)mr, parent.p);
    OPE_TRY(check_launch(ctx, "cluster_init_kernel"));
    // a warp per point; up to 256 blocks per frame, more when a few frames would leave the device idle (with 256 blocks,
    // ope_pass_through + ope_segment_objects_on_plane on one 640x480 frame took 4.5 ms instead of 2.2 ms on a B200). The launch shape
    // cannot change the result: a root is its component's smallest index however the unions are scheduled.
    const size_t max_union = std::max<size_t>(256, (size_t)ctx->sm_count * 16 / (size_t)B);
    const unsigned gx_union = (unsigned)std::max<size_t>(1, std::min<size_t>(div_up(max_span(h_rest) * 32, kSegThreads), max_union));
    scene_cluster_union_kernel<<<dim3(gx_union, B), kSegThreads, 0, ctx->stream>>>(rpts.p, rest_off.p, d_cf.p, cell_start.p, sorted.p,
                                                                                    S.cluster_tolerance * S.cluster_tolerance, parent.p);
    OPE_TRY(check_launch(ctx, "scene_cluster_union_kernel"));
    cluster_flatten_kernel<<<div_up(mr, kSegThreads), kSegThreads, 0, ctx->stream>>>(rpts.p, (int)mr, parent.p, root.p);
    OPE_TRY(check_launch(ctx, "cluster_flatten_kernel"));
    component_size_kernel<<<div_up(mr, kSegThreads), kSegThreads, 0, ctx->stream>>>((int)mr, root.p, size.p);
    OPE_TRY(check_launch(ctx, "component_size_kernel"));
    // the roots inside [min, max] size with their sizes; at most mr / min_size of them
    const size_t cap = std::min<size_t>(mr, mr / (size_t)std::max(S.min_cluster_size, 1)) + 1;
    Scratch<int> rflags(ctx), roots(ctx), rsize(ctx), root_off(ctx);
    OPE_TRY(rflags.alloc(mr + 1)); OPE_TRY(roots.alloc(cap)); OPE_TRY(rsize.alloc(cap)); OPE_TRY(root_off.alloc((size_t)B + 1));
    root_flag_kernel<<<div_up(mr, kSegThreads), kSegThreads, 0, ctx->stream>>>((int)mr, root.p, size.p, S.min_cluster_size, S.max_cluster_size, rflags.p);
    OPE_TRY(check_launch(ctx, "root_flag_kernel"));
    OPE_CUDA_TRY(ctx, cudaMemsetAsync(rflags.p + mr, 0, sizeof(int), ctx->stream));
    OPE_TRY(exclusive_scan_i32(ctx, rflags.p, mr + 1));
    root_compact_kernel<<<div_up(mr, kSegThreads), kSegThreads, 0, ctx->stream>>>((int)mr, rflags.p, size.p, roots.p, rsize.p);
    OPE_TRY(check_launch(ctx, "root_compact_kernel"));
    span_bounds_kernel<<<div_up((size_t)B + 1, kSegThreads), kSegThreads, 0, ctx->stream>>>(rflags.p, rest_off.p, 0, B, root_off.p);
    OPE_TRY(check_launch(ctx, "span_bounds_kernel"));
    std::vector<int> h_root_off, h_roots, h_rsize;
    OPE_TRY(download(ctx, h_root_off, (const int*)root_off.p, (size_t)B + 1));
    OPE_TRY(download(ctx, h_roots, (const int*)roots.p, cap));
    OPE_TRY(download(ctx, h_rsize, (const int*)rsize.p, cap));
    OPE_CUDA_TRY(ctx, stream_sync(ctx));
    // the reference's order per frame: largest first, equal sizes by the smaller first index (= the root)
    std::vector<int2> numbering;
    for (int f = 0; f < B; ++f) {
      if (!live2[(size_t)f]) continue;
      std::vector<int> k((size_t)(h_root_off[(size_t)f + 1] - h_root_off[(size_t)f]));
      std::iota(k.begin(), k.end(), h_root_off[(size_t)f]);
      std::sort(k.begin(), k.end(), [&](int a, int b) { return h_rsize[(size_t)a] != h_rsize[(size_t)b] ? h_rsize[(size_t)a] > h_rsize[(size_t)b] : h_roots[(size_t)a] < h_roots[(size_t)b]; });
      for (size_t c = 0; c < k.size(); ++c) { numbering.push_back(make_int2(h_roots[(size_t)k[c]], (int)c)); sizes[(size_t)f].push_back(h_rsize[(size_t)k[c]]); }
    }
    Scratch<int2> d_numbering(ctx);
    OPE_TRY(d_numbering.alloc(numbering.size()));
    OPE_TRY(upload(ctx, d_numbering.p, numbering));
    if (!numbering.empty()) {
      scatter_number_kernel<<<div_up(numbering.size(), kSegThreads), kSegThreads, 0, ctx->stream>>>((int)numbering.size(), d_numbering.p, number.p);
      OPE_TRY(check_launch(ctx, "scatter_number_kernel"));
    }
    // labels (in ope_segment_objects_on_plane's order of writes)
    label_prism_kernel<<<dim3(gx_prism, B), kSegThreads, 0, ctx->stream>>>(prism_off.p, d_live2.p, prism.p, labels);
    OPE_TRY(check_launch(ctx, "label_prism_kernel"));
    label_plane_kernel<<<dim3(gx_prism, B), kSegThreads, 0, ctx->stream>>>(in2_off.p, in2.p, prism.p, labels);
    OPE_TRY(check_launch(ctx, "label_plane_kernel"));
    label_rest_kernel<<<dim3(gx_rest, B), kSegThreads, 0, ctx->stream>>>(rest_off.p, rest.p, prism.p, root.p, number.p, labels);
    OPE_TRY(check_launch(ctx, "label_rest_kernel"));
  } else if (mp) {
    label_prism_kernel<<<dim3(gx_prism, B), kSegThreads, 0, ctx->stream>>>(prism_off.p, d_live2.p, prism.p, labels);
    OPE_TRY(check_launch(ctx, "label_prism_kernel"));
    label_plane_kernel<<<dim3(gx_prism, B), kSegThreads, 0, ctx->stream>>>(in2_off.p, in2.p, prism.p, labels);
    OPE_TRY(check_launch(ctx, "label_plane_kernel"));
  }
  for (int f = 0; f < B; ++f) {
    ope_scene_batch::Frame& F = out[f];
    F.status = status[(size_t)f];
    F.info.iterations[0] = it1[(size_t)f];
    F.info.iterations[1] = live1[(size_t)f] ? it2[(size_t)f] : 0;
    F.info.n_clusters = -1;
    if (live2[(size_t)f] && F.status == OPE_OK) {
      std::memcpy(F.info.plane1, &h_c1[(size_t)4 * f], 16);
      std::memcpy(F.info.plane2, &h_c2[(size_t)4 * f], 16);
      F.info.n_clusters = (int)sizes[(size_t)f].size();
      F.sizes = sizes[(size_t)f];
    }
  }
  return OPE_OK;
}

// One chunk of frames (device depth): depth -> cloud, crop, segmentation. Appends the frames to s (their points and labels in two new
// device blocks). Eleven host waits, whatever the number of frames.
int scene_chunk(ope_ctx* ctx, const ope_scene_params& P, const uint16_t* d_depth, int B, int rows, int cols, ope_scene_batch* s) {
  const size_t npx = (size_t)B * rows * cols;
  // depth -> cloud (ope_depth_to_cloud_batch: column-outer order, frame after frame)
  Scratch<float4> cloud(ctx);
  Scratch<int> col(ctx), dep_off(ctx);
  OPE_TRY(cloud.alloc(npx)); OPE_TRY(col.alloc((size_t)B * cols + 1)); OPE_TRY(dep_off.alloc((size_t)B + 1));
  OPE_TRY(ope_depth_to_cloud_batch(ctx, d_depth, B, rows, cols, P.fx, P.fy, P.cx, P.cy, P.scale, P.z_max, cloud.p, col.p));
  span_bounds_kernel<<<div_up((size_t)B + 1, kSegThreads), kSegThreads, 0, ctx->stream>>>(col.p, nullptr, cols, B, dep_off.p);
  OPE_TRY(check_launch(ctx, "span_bounds_kernel"));
  std::vector<int> h_dep;
  OPE_TRY(download(ctx, h_dep, (const int*)dep_off.p, (size_t)B + 1));
  OPE_CUDA_TRY(ctx, stream_sync(ctx));
  Scratch<int> idx(ctx), crop_off(ctx);
  OPE_TRY(idx.alloc((size_t)h_dep[(size_t)B])); OPE_TRY(crop_off.alloc((size_t)B + 1));
  std::vector<int> h_crop;
  float4* pts = nullptr;
  int* labels = nullptr;
  OPE_TRY(crop_frames(ctx, cloud.p, h_dep, dep_off.p, P.limits, idx.p, crop_off.p, h_crop, [&](size_t m, float4** p) -> int {
    OPE_TRY(dalloc(ctx, p, m));
    s->blocks.push_back(*p);
    return OPE_OK;
  }, &pts));
  OPE_TRY(dalloc(ctx, &labels, (size_t)h_crop[(size_t)B]));
  s->blocks.push_back(labels);
  const size_t first = s->frames.size();
  s->frames.resize(first + (size_t)B);
  OPE_TRY(segment_frames(ctx, P.seg, pts, h_crop, crop_off.p, labels, &s->frames[first]));
  OPE_CUDA_TRY(ctx, stream_sync(ctx));
  for (int f = 0; f < B; ++f) {
    ope_scene_batch::Frame& F = s->frames[first + (size_t)f];
    F.info.n_points = h_dep[(size_t)f + 1] - h_dep[(size_t)f];
    F.info.n_cropped = h_crop[(size_t)f + 1] - h_crop[(size_t)f];
    F.pts = pts + h_crop[(size_t)f];
    F.labels = labels + h_crop[(size_t)f];
  }
  return OPE_OK;
}

}  // namespace

extern "C" {

// limits: x_min, x_max, y_min, y_max, z_min, z_max (ProcessingPcd::getPassThrough's argument order). out_idx (n entries) may be NULL.
int ope_pass_through(ope_ctx* ctx, const ope_cloud* cloud, const float limits[6], ope_cloud** out, int32_t* out_idx, size_t* out_n) {
  OPE_ENTER(ctx);
  if (!ctx || !cloud || !limits || !out) return OPE_ERR_INVALID;
  *out = nullptr;
  if (out_n) *out_n = 0;
  const size_t n = cloud->n;
  if (n > 0x7ffffffeull) return fail(ctx, OPE_ERR_INVALID, "cloud too large");
  std::vector<int> h_off, h_crop;
  Scratch<int> off(ctx), idx(ctx), crop_off(ctx);   // idx: the compaction's index list, which the gather reads, out_idx or not
  OPE_TRY(one_span(ctx, n, h_off, off)); OPE_TRY(idx.alloc(n)); OPE_TRY(crop_off.alloc(2));
  ope_cloud* o = nullptr;
  float4* pts = nullptr;
  int rc = crop_frames(ctx, cloud->pts, h_off, off.p, limits, idx.p, crop_off.p, h_crop, [&](size_t m, float4** p) -> int {
    OPE_TRY(cloud_alloc(ctx, m, false, &o));
    *p = o->pts;
    return OPE_OK;
  }, &pts);
  const size_t m = rc == OPE_OK ? (size_t)h_crop[1] : 0;
  if (rc == OPE_OK && out_idx && m > 0) {
    cudaError_t e = cudaMemcpyAsync(out_idx, idx.p, m * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = stream_sync(ctx);
    if (e != cudaSuccess) rc = fail(ctx, OPE_ERR_CUDA, "index download failed: %s", cudaGetErrorString(e));
  }
  if (rc != OPE_OK) { if (o) ope_cloud_free(ctx, o); return rc; }
  if (out_n) *out_n = m;
  *out = o;
  return OPE_OK;
}

// pcl::SACSegmentation on a device cloud without NaN points: refined plane coefficients, the inlier indices (ascending; out_idx has
// room for ope_cloud_size entries, may be NULL), the RANSAC iteration count. *found = 0 when no plane exists (fewer than 3 points).
int ope_plane_ransac(ope_ctx* ctx, const ope_cloud* cloud, const ope_segment_params* prm, float coeff[4], int32_t* out_idx, size_t* out_n,
                     int32_t* iterations, int32_t* found) {
  OPE_ENTER(ctx);
  if (!ctx || !cloud || !coeff || !found) return OPE_ERR_INVALID;
  ope_segment_params P;
  if (prm) P = *prm; else ope_segment_params_default(&P);
  const size_t n = cloud->n;
  if (n > 0x7ffffffeull) return fail(ctx, OPE_ERR_INVALID, "cloud too large");
  std::vector<int> h_off, live{1}, it, status{OPE_OK};
  Scratch<int> off(ctx), d_live(ctx), inl(ctx), inl_off(ctx), flags(ctx);
  Scratch<float> plane(ctx);
  OPE_TRY(one_span(ctx, n, h_off, off)); OPE_TRY(d_live.alloc(1)); OPE_TRY(inl.alloc(n)); OPE_TRY(inl_off.alloc(2));
  OPE_TRY(flags.alloc(n + 1)); OPE_TRY(plane.alloc(4));
  OPE_TRY(plane_segment_frames(ctx, cloud->pts, h_off, off.p, P, live, it, status, plane.p, d_live.p, inl.p, inl_off.p, flags.p));
  OPE_TRY(status[0]);
  size_t m = 0;
  if (live[0]) {
    std::vector<float> c;
    std::vector<int> end;
    OPE_TRY(download(ctx, c, (const float*)plane.p, 4));
    OPE_TRY(download(ctx, end, (const int*)inl_off.p + 1, 1));
    OPE_CUDA_TRY(ctx, stream_sync(ctx));
    std::memcpy(coeff, c.data(), 16);
    m = (size_t)end[0];
    if (out_idx && m > 0) {
      OPE_CUDA_TRY(ctx, cudaMemcpyAsync(out_idx, inl.p, m * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
      OPE_CUDA_TRY(ctx, stream_sync(ctx));
    }
  }
  if (out_n) *out_n = m;
  if (iterations) *iterations = it[0];
  *found = live[0];
  return OPE_OK;
}

// ObjectSegmentationPlane::getSegmentedObjectsOnPlane (D&L/src/objectsegmentationplane.cpp:122-282) on a pass-through-filtered
// device cloud: plane, prism over the padded hull rectangle, second plane on the prism's points, Euclidean clusters of the rest.
// labels (n entries): OPE_SEG_OUTSIDE_PRISM / OPE_SEG_PLANE / OPE_SEG_NO_CLUSTER / cluster number (0 = largest).
// *n_clusters = -1 when no plane was found (the reference then passes the whole cloud on). The clusters come from the frame-aware dense
// grid of the batch: a cloud that was not cropped, with prism points far above the table, coarsens that grid until the union search is
// close to quadratic in the rest's size (correct, but slow); ope_euclidean_clusters' Morton grid does not have this limit.
int ope_segment_objects_on_plane(ope_ctx* ctx, const ope_cloud* cloud, const ope_segment_params* prm, int32_t* labels, float plane1[4],
                                 float plane2[4], int32_t iters[2], int32_t* n_clusters) {
  OPE_ENTER(ctx);
  if (!ctx || !cloud || !labels || !n_clusters) return OPE_ERR_INVALID;
  ope_segment_params P;
  if (prm) P = *prm; else ope_segment_params_default(&P);
  const size_t n = cloud->n;
  *n_clusters = -1;
  for (size_t i = 0; i < n; ++i) labels[i] = OPE_SEG_OUTSIDE_PRISM;
  if (n > 0x7ffffffeull) return fail(ctx, OPE_ERR_INVALID, "cloud too large");
  std::vector<int> h_off;
  Scratch<int> off(ctx), d_labels(ctx);
  OPE_TRY(one_span(ctx, n, h_off, off)); OPE_TRY(d_labels.alloc(n));
  ope_scene_batch::Frame F;
  OPE_TRY(segment_frames(ctx, P, cloud->pts, h_off, off.p, d_labels.p, &F));
  const ope_scene_frame& I = F.info;
  // a degenerate sample of the table plane leaves iters untouched; one of the second plane leaves {table plane's iterations, 0}. The
  // two are told apart by iterations[0]: 0 when the table plane's sample failed (no count was replayed), else >= 1, because
  // ransac_replay runs at least one iteration for every frame it fits.
  if (iters && (F.status == OPE_OK || I.iterations[0] > 0)) { iters[0] = I.iterations[0]; iters[1] = I.iterations[1]; }
  OPE_TRY(F.status);
  if (n) {
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(labels, d_labels.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    OPE_CUDA_TRY(ctx, stream_sync(ctx));
  }
  if (I.n_clusters >= 0) {
    if (plane1) std::memcpy(plane1, I.plane1, 16);
    if (plane2) std::memcpy(plane2, I.plane2, 16);
  }
  *n_clusters = I.n_clusters;
  return OPE_OK;
}

void ope_scene_params_default(ope_scene_params* p) {
  std::memset(p, 0, sizeof(*p));
  p->fx = 525.0f; p->fy = 525.0f; p->cx = 319.5f; p->cy = 239.5f; p->scale = 1000.0f; p->z_max = 2.0f;
  const float lim[6] = {-0.5f, 0.5f, -0.5f, 0.3f, 0.5f, 1.6f};
  std::memcpy(p->limits, lim, sizeof(lim));
  ope_segment_params_default(&p->seg);
}

// Every frame equals ope_depth_to_cloud -> ope_pass_through -> ope_segment_objects_on_plane by construction: those calls are one-frame
// runs of scene_chunk's crop and segmentation stages.
int ope_scene_batch_create(ope_ctx* ctx, const ope_scene_params* prm, const uint16_t* depth, int frames, int rows, int cols,
                           ope_scene_batch** out, ope_scene_frame* info, int32_t* status) {
  OPE_ENTER(ctx);
  if (!ctx || !depth || !out || !info || frames <= 0 || rows <= 0 || cols <= 0) return OPE_ERR_INVALID;
  *out = nullptr;
  ope_scene_params P;
  if (prm) P = *prm; else ope_scene_params_default(&P);
  if (!(P.scale > 0) || !(P.seg.cluster_tolerance > 0)) return OPE_ERR_INVALID;
  const size_t px = (size_t)rows * cols;
  if (px > 0x3fffffffull) return fail(ctx, OPE_ERR_INVALID, "image too large");
  cudaPointerAttributes attr;
  const cudaError_t pe = cudaPointerGetAttributes(&attr, depth);
  if (pe != cudaSuccess) cudaGetLastError();
  const bool on_device = pe == cudaSuccess && (attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged);
  // frames per chunk: the chunk's scratch (depth, cloud, flags and indices, about 64 bytes per pixel at most) within 4 GiB and the
  // 32-bit point offsets of the scans; OPE_SCENE_CHUNK overrides
  size_t chunk = std::max<size_t>(1, ((size_t)4 << 30) / (px * 64));
  chunk = std::min(chunk, (size_t)0x7ffffffe / px);
  if (const char* e = std::getenv("OPE_SCENE_CHUNK")) chunk = (size_t)std::max(1, std::atoi(e));
  chunk = std::min(chunk, (size_t)frames);
  ope_scene_batch* s = new (std::nothrow) ope_scene_batch;
  if (!s) return fail(ctx, OPE_ERR_INVALID, "out of host memory");
  s->ctx = ctx;
  s->frames.reserve((size_t)frames);
  int rc = OPE_OK;
  {
    Scratch<uint16_t> staged(ctx);
    if (!on_device) rc = staged.alloc(chunk * px);
    for (size_t f0 = 0; rc == OPE_OK && f0 < (size_t)frames; f0 += chunk) {
      const int nb = (int)std::min(chunk, (size_t)frames - f0);
      const uint16_t* d = depth + f0 * px;
      if (!on_device) {
        const cudaError_t e = cudaMemcpyAsync(staged.p, d, (size_t)nb * px * sizeof(uint16_t), cudaMemcpyHostToDevice, ctx->stream);
        if (e != cudaSuccess) { rc = fail(ctx, OPE_ERR_CUDA, "depth upload failed: %s", cudaGetErrorString(e)); break; }
        d = staged.p;
      }
      rc = scene_chunk(ctx, P, d, nb, rows, cols, s);
    }
  }
  if (rc != OPE_OK) { ope_scene_batch_destroy(s); return rc; }
  int first = OPE_OK;
  for (int f = 0; f < frames; ++f) {
    info[f] = s->frames[(size_t)f].info;
    if (status) status[f] = s->frames[(size_t)f].status;
    if (first == OPE_OK) first = s->frames[(size_t)f].status;
  }
  *out = s;
  return first;
}

int ope_scene_batch_frame(const ope_scene_batch* s, size_t frame, float* xyz, int32_t* labels, ope_scene_frame* info) {
  if (!s || frame >= s->frames.size()) return OPE_ERR_INVALID;
  ope_ctx* ctx = s->ctx;
  OPE_ENTER(ctx);
  const ope_scene_batch::Frame& F = s->frames[frame];
  const size_t n = (size_t)F.info.n_cropped;
  if (info) *info = F.info;
  if (n && xyz) {
    std::vector<float4> h;
    OPE_TRY(download(ctx, h, F.pts, n));
    OPE_CUDA_TRY(ctx, stream_sync(ctx));
    for (size_t i = 0; i < n; ++i) { xyz[3 * i] = h[i].x; xyz[3 * i + 1] = h[i].y; xyz[3 * i + 2] = h[i].z; }
  }
  if (n && labels) {
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(labels, F.labels, n * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    OPE_CUDA_TRY(ctx, stream_sync(ctx));
  }
  return OPE_OK;
}

void ope_scene_batch_destroy(ope_scene_batch* s) {
  if (!s) return;
  OPE_ENTER(s->ctx);
  for (void* p : s->blocks) dfree(s->ctx, p);
  delete s;
}

int ope_scene_pose_batch(const ope_scene_batch* s, const ope_pose_params* prm, const float* model_xyz, size_t n_model, const int32_t* cluster,
                         const ope_rng_table* tables, int workers, ope_pose_result* results, int32_t* status) {
  if (!s || !model_xyz || n_model == 0 || !results) return OPE_ERR_INVALID;
  ope_ctx* ctx = s->ctx;
  OPE_ENTER(ctx);
  const size_t B = s->frames.size();
  std::vector<SceneCut> cuts;
  std::vector<size_t> n_out(B, 0), off(B, 0);
  size_t total = 0;
  for (size_t f = 0; f < B; ++f) {
    const ope_scene_batch::Frame& F = s->frames[f];
    const int r = cluster ? cluster[f] : 0;
    if (r < 0) return fail(ctx, OPE_ERR_INVALID, "negative cluster rank for frame %zu", f);
    SceneCut c{F.pts, F.labels, F.info.n_cropped, INT_MIN, (long long)total};
    if (F.status != OPE_OK) continue;                                         // an empty target
    if (F.info.n_clusters >= 0) {
      if (r >= F.info.n_clusters) continue;                                   // an empty target
      c.want = r;
      n_out[f] = (size_t)F.sizes[(size_t)r];
    } else {
      n_out[f] = (size_t)F.info.n_cropped;                                    // no plane: the whole cropped cloud (:149-152)
    }
    if (!n_out[f]) continue;
    off[f] = total;
    total += n_out[f];
    cuts.push_back(c);
  }
  Scratch<float4> buf(ctx);
  Scratch<SceneCut> d_cuts(ctx);
  OPE_TRY(buf.alloc(total)); OPE_TRY(d_cuts.alloc(cuts.size()));
  if (!cuts.empty()) {
    OPE_TRY(upload(ctx, d_cuts.p, cuts));
    OPE_TRY(scene_cut_device(ctx, d_cuts.p, (int)cuts.size(), buf.p));
  }
  OPE_CUDA_TRY(ctx, stream_sync(ctx));   // the pose batch reads the clusters from other streams
  std::vector<ope_cloud> views(B);
  std::vector<ope_frame_input> inputs(B);
  for (size_t f = 0; f < B; ++f) {
    inputs[f] = ope_frame_input{nullptr, 0, 0, 0, nullptr};
    if (!n_out[f]) continue;
    views[f].ctx = ctx; views[f].n = n_out[f]; views[f].pts = buf.p + off[f];
    inputs[f].cloud = &views[f];
  }
  return ope_pose_batch(ctx, prm, model_xyz, n_model, inputs.data(), B, tables, workers, results, status);
}

}  // extern "C"
