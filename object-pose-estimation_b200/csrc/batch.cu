// batch.cu — frame-spanning launches (BASELINE.json configs[4], SURVEY 8e row 1): pose_chunk runs every stage of
// PoseEstimator::estimateFinalPose (D&L/src/poseestimator.cpp:383-448) as ONE launch for a whole chunk of frames — blockIdx.y (or a
// ticket) selects the frame, sizes are read from device memory — instead of ~40 launches and ~25 host round trips per frame. Per
// chunk the host waits a handful of times (to size the next stage's grid). Its callers: ope_pose_batch and ope_pose_tracker_step_batch.
//
//   stage                                  launch(es)                                        per-frame data
//   target UniformSampling 1 cm + 8 mm     bsample_kernel<false>      grid (frames, 2)        cluster -> tp1, tp2 (voxel-key order)
//   normals k = 30 of tp1, tp2             normals_smem_batch_kernel  grid (<=8, 2 frames)    (+ a tracker's own 1 cm source sample)
//   SPFH + FPFH of tp1                     spfh_/fpfh_batch_kernel    grid (n/8, frames)
//   5 nearest target features per source   feature_knn_kernel (+ merge) grid (nq/128, <=4, frames)   the model's descriptors are shared
//   SAC-IA 400 x 5                         sacia_transform_/seed_/score_batch_kernel         + select: coarse pose per frame
//                                                                     score grid (frames, 400/16)
//   source under the coarse pose, 8 mm     bsample_kernel<true>       grid (frames)           157 825 points, never materialised
//   normals k = 30 of sp2                  normals_smem_batch_kernel
//   removeNaNNormalsFromPointCloud x 2     compact_normals_batch_kernel
//   ICP-with-normals <= 100 iterations     icp_small_batch_kernel     ticketed blocks of all frames
//   getFitnessScore                        fitness_smem_batch_kernel  grid (frames)
//
// The kernels are the single-frame kernels, or their bodies (features.cu, registration.cu), behind a frame index, so a frame's
// result is what ope_pose_estimate_final returns for it — bit for bit, tests/test_gpu_parity.py. Frames outside the fast path's envelope
// (empty or tiny clusters, clouds beyond the shared-memory capacities, voxel tables that overflow) are finished by the caller's
// per-frame path. ope_pose_batch computes the frame-invariant model side (1 cm sample, normals, FPFH; dense Umeyama of the model
// onto itself) once per call (SURVEY 8f-3); a tracker brings its own source, which the chunk samples and describes.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

#include <chrono>
#include <cstdio>
#include "ope_host.cuh"
#include "ope_device.cuh"

namespace ope {

static constexpr int kBTable = 8192;      // voxel hash slots per block (load factor <= 0.5 at kBCap voxels)
static constexpr int kBThreads = 1024;
static constexpr unsigned long long kEmpty = ~0ull;


struct SampleSmem {
  unsigned long long keys[kBTable];
  unsigned long long vals[kBTable];
  unsigned long long list_key[kBCap];
  unsigned long long list_val[kBCap];
  float red[6][kBThreads / 32];
  int scan[kBThreads / 32];
  int n_finite, occupied, overflow, total;
  float bbox[6];
};

__device__ __forceinline__ unsigned hash_cell(long long c) {
  unsigned long long x = (unsigned long long)c * 0x9E3779B97F4A7C15ull;
  return (unsigned)(x >> 40);
}

// pcl::UniformSampling (SURVEY A.1) of one cloud per block: bounding box -> voxel frame -> per voxel the point with the smallest
// (||p4 - ijk4||^2, index) -> selected points in ascending voxel index. The voxel table is a shared-memory hash (linear probing,
// 64-bit keys); the result equals uniform_sample_device + gather_cloud (grid.cu) point for point.
__global__ void __launch_bounds__(kBThreads) bsample_kernel(BSampleArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SampleSmem* sm = reinterpret_cast<SampleSmem*>(smem_raw);
  const int f = blockIdx.x, leaf = blockIdx.y;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (a.active && !a.active[f]) return;
  const float4* pts = a.src[f];
  const int n = a.counts[f];
  const bool xf = a.xforms && (!a.xform_on || a.xform_on[f]);
  Mat4 T;
  if (xf) for (int i = 0; i < 16; ++i) T.m[i] = a.xforms[f].T[i];
  auto load = [&](int i) {
    float4 p = __ldg(pts + i);
    if (xf) { float x, y, z; xform_point(T, p.x, p.y, p.z, x, y, z); p.x = x; p.y = y; p.z = z; }
    return p;
  };
  // ---- bounding box of the finite points ----
  float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  int fin = 0;
  for (int i = tid; i < n; i += kBThreads) {
    const float4 p = load(i);
    if (!finite3(p.x, p.y, p.z)) continue;
    ++fin;
    lo[0] = fminf(lo[0], p.x); lo[1] = fminf(lo[1], p.y); lo[2] = fminf(lo[2], p.z);
    hi[0] = fmaxf(hi[0], p.x); hi[1] = fmaxf(hi[1], p.y); hi[2] = fmaxf(hi[2], p.z);
  }
  for (int o = 16; o > 0; o >>= 1) {
    for (int d = 0; d < 3; ++d) { lo[d] = fminf(lo[d], __shfl_xor_sync(0xffffffffu, lo[d], o)); hi[d] = fmaxf(hi[d], __shfl_xor_sync(0xffffffffu, hi[d], o)); }
    fin += __shfl_xor_sync(0xffffffffu, fin, o);
  }
  if (tid == 0) { sm->n_finite = 0; sm->occupied = 0; sm->overflow = 0; }
  if (lane == 0) for (int d = 0; d < 3; ++d) { sm->red[d][warp] = lo[d]; sm->red[3 + d][warp] = hi[d]; }
  for (int s = tid; s < kBTable; s += kBThreads) { sm->keys[s] = kEmpty; sm->vals[s] = kEmpty; }
  __syncthreads();
  if (lane == 0) atomicAdd(&sm->n_finite, fin);
  if (tid < 6) {
    float v = sm->red[tid][0];
    for (int w = 1; w < kBThreads / 32; ++w) v = tid < 3 ? fminf(v, sm->red[tid][w]) : fmaxf(v, sm->red[tid][w]);
    sm->bbox[tid] = v;
  }
  __syncthreads();
  int* out_count = a.out_counts[leaf] + f;
  if (sm->n_finite == 0) { if (tid == 0) *out_count = 0; return; }
  // ---- the voxel frame of PCL (pcl_voxel_frame, grid.cu): min_b = floor(min * inv), dim = max_b - min_b + 1 ----
  const float inv = a.inv_leaf[leaf];
  int min_b[3];
  long long dim[3];
  bool too_large = false;
  for (int d = 0; d < 3; ++d) {
    const float l = sm->bbox[d] * inv, h = sm->bbox[3 + d] * inv;
    min_b[d] = (int)floorf(l);
    dim[d] = (long long)(int)floorf(h) - min_b[d] + 1;
    if (dim[d] > 0x7fffffffll) too_large = true;
  }
  if (!too_large && (double)dim[0] * (double)dim[1] * (double)dim[2] > (double)(1ll << 28)) too_large = true;
  if (too_large) { if (tid == 0) { *out_count = 0; atomicOr(a.flags + f, 1); } return; }
  // ---- per voxel: argmin over (||p4 - ijk4||^2, index) ----
  for (int i = tid; i < n; i += kBThreads) {
    const float4 p = load(i);
    if (!finite3(p.x, p.y, p.z)) continue;
    const int ix = (int)floorf(p.x * inv), iy = (int)floorf(p.y * inv), iz = (int)floorf(p.z * inv);
    const long long cell = ((long long)(iz - min_b[2]) * dim[1] + (iy - min_b[1])) * dim[0] + (ix - min_b[0]);
    const float da = p.x - (float)ix, db = p.y - (float)iy, dc = p.z - (float)iz;
    float d = da * da;
    d = d + db * db;
    d = d + dc * dc;
    d = d + 1.0f;  // 4th component of (p4 - ijk4): (1 - 0)^2
    const unsigned long long packed = ((unsigned long long)__float_as_uint(d) << 32) | (unsigned)i;
    unsigned slot = hash_cell(cell) & (kBTable - 1);
    bool placed = false;
    for (int probe = 0; probe < kBTable; ++probe) {
      unsigned long long k = sm->keys[slot];
      if (k == kEmpty) {
        if (sm->occupied >= kBTable / 2) break;                 // table full: give up (the frame is flagged below)
        k = atomicCAS(&sm->keys[slot], kEmpty, (unsigned long long)cell);
        if (k == kEmpty) { atomicAdd(&sm->occupied, 1); k = (unsigned long long)cell; }
      }
      if (k == (unsigned long long)cell) { placed = true; break; }
      slot = (slot + 1) & (kBTable - 1);
    }
    if (!placed) { sm->overflow = 1; continue; }
    if (sm->vals[slot] > packed) atomicMin(&sm->vals[slot], packed);
  }
  __syncthreads();
  const int cap = a.cap[leaf];
  if (sm->overflow || sm->occupied > cap) { if (tid == 0) { *out_count = 0; atomicOr(a.flags + f, 1); } return; }
  // ---- compact the occupied slots, sort by voxel index, emit the points ----
  constexpr int kPer = kBTable / kBThreads;
  int mine = 0;
  for (int u = 0; u < kPer; ++u) mine += sm->keys[tid * kPer + u] != kEmpty ? 1 : 0;
  int incl = mine;
  for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
  if (lane == 31) sm->scan[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int v = sm->scan[lane];
    int inc2 = v;
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc2, o); if (lane >= o) inc2 += t; }
    sm->scan[lane] = inc2 - v;
    if (lane == 31) sm->total = inc2;
  }
  __syncthreads();
  int pos = sm->scan[warp] + incl - mine;
  for (int u = 0; u < kPer; ++u) {
    const int s = tid * kPer + u;
    if (sm->keys[s] != kEmpty) { sm->list_key[pos] = sm->keys[s]; sm->list_val[pos] = sm->vals[s]; ++pos; }
  }
  const int m = sm->total;
  int m2 = 1;
  while (m2 < m) m2 <<= 1;
  for (int j = m + tid; j < m2; j += kBThreads) { sm->list_key[j] = kEmpty; sm->list_val[j] = kEmpty; }
  __syncthreads();
  for (int k2 = 2; k2 <= m2; k2 <<= 1)
    for (int j2 = k2 >> 1; j2 > 0; j2 >>= 1) {
      for (int i = tid; i < m2; i += kBThreads) {
        const int l = i ^ j2;
        if (l > i) {
          const bool up = (i & k2) == 0;
          const unsigned long long ki = sm->list_key[i], kl = sm->list_key[l];
          if ((ki > kl) == up) {
            sm->list_key[i] = kl; sm->list_key[l] = ki;
            const unsigned long long vi = sm->list_val[i];
            sm->list_val[i] = sm->list_val[l]; sm->list_val[l] = vi;
          }
        }
      }
      __syncthreads();
    }
  float4* out = a.out[leaf] + (size_t)f * kBCap;
  for (int j = tid; j < m; j += kBThreads) {
    const int idx = (int)(unsigned)(sm->list_val[j] & 0xffffffffull);
    float4 p = load(idx);
    out[j] = p;
  }
  if (tid == 0) *out_count = m;
}

// UniformSampling of every frame's cloud at each leaf, one block per (frame, leaf): grid (frames, leaves)
static int bsample_batch(ope_ctx* ctx, const BSampleArgs& a, int frames, int leaves) {
  OPE_TRY(dyn_smem(ctx, (const void*)bsample_kernel, sizeof(SampleSmem)));
  bsample_kernel<<<dim3(frames, leaves), kBThreads, sizeof(SampleSmem), ctx->stream>>>(a);
  return check_launch(ctx, "bsample_kernel");
}

// pcl::removeNaNNormalsFromPointCloud (D&L/src/poseestimator.cpp:215-216) for one cloud per block: points whose normal is finite,
// in order; the compacted points carry their new index in .w (the ICP kernel's work order).
__global__ void __launch_bounds__(kBThreads) compact_normals_batch_kernel(const float4* __restrict__ pts, const float4* __restrict__ nrm,
                                                                          const int* __restrict__ counts, const int* __restrict__ active,
                                                                          int frames, float4* __restrict__ opts, float4* __restrict__ onrm,
                                                                          int* __restrict__ ocounts) {
  __shared__ int scan[kBThreads / 32];
  __shared__ int total;
  const int c = blockIdx.x;   // cloud: [which][frame]
  const int f = c % frames;
  if (active && !active[f]) return;
  const int n = counts[c];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int kPer = kBCap / kBThreads;
  const size_t base = (size_t)c * kBCap;
  bool keep[kPer];
  int mine = 0;
  for (int u = 0; u < kPer; ++u) {
    const int i = tid * kPer + u;
    keep[u] = false;
    if (i < n) { const float4 v = __ldg(nrm + base + i); keep[u] = finite3(v.x, v.y, v.z); }
    mine += keep[u] ? 1 : 0;
  }
  int incl = mine;
  for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
  if (lane == 31) scan[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int v = scan[lane];
    int inc2 = v;
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc2, o); if (lane >= o) inc2 += t; }
    scan[lane] = inc2 - v;
    if (lane == 31) total = inc2;
  }
  __syncthreads();
  int pos = scan[warp] + incl - mine;
  for (int u = 0; u < kPer; ++u) {
    const int i = tid * kPer + u;
    if (keep[u]) {
      float4 p = __ldg(pts + base + i);
      p.w = __int_as_float(pos);
      opts[base + pos] = p;
      onrm[base + pos] = __ldg(nrm + base + i);
      ++pos;
    }
  }
  if (tid == 0) ocounts[c] = total;
}

// Work order of the ICP kernel: both fine clouds re-ordered along the Morton curve of their own bounding box, so that the 32 points
// of a warp and the 8 points of a target group are spatial neighbours (the voxel-key order of the sampling is a z-major raster:
// thin rows). One block per cloud: bounding box, 30-bit Morton key | position, bitonic sort in shared memory, gather. The clouds
// stay self-consistent (points and normals move together, .w = new position), so nothing but the order of equal-distance ties
// and of the double-precision moment sums changes.
__device__ __forceinline__ unsigned spread10(unsigned v) {
  v &= 0x3ffu;
  v = (v | (v << 16)) & 0x030000ffu;
  v = (v | (v << 8)) & 0x0300f00fu;
  v = (v | (v << 4)) & 0x030c30c3u;
  v = (v | (v << 2)) & 0x09249249u;
  return v;
}
__global__ void __launch_bounds__(kBThreads) morton_sort_batch_kernel(const float4* __restrict__ pts, const float4* __restrict__ nrm,
                                                                     const int* __restrict__ counts, const int* __restrict__ active, int frames,
                                                                     float4* __restrict__ opts, float4* __restrict__ onrm) {
  __shared__ unsigned long long keys[kBCap];
  __shared__ float red[6][kBThreads / 32];
  __shared__ float box[6];
  const int c = blockIdx.x, f = c % frames;
  if (active && !active[f]) return;
  const int n = counts[c];
  if (n <= 0) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t base = (size_t)c * kBCap;
  float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int i = tid; i < n; i += kBThreads) {
    const float4 p = __ldg(pts + base + i);
    lo[0] = fminf(lo[0], p.x); lo[1] = fminf(lo[1], p.y); lo[2] = fminf(lo[2], p.z);
    hi[0] = fmaxf(hi[0], p.x); hi[1] = fmaxf(hi[1], p.y); hi[2] = fmaxf(hi[2], p.z);
  }
  for (int o = 16; o > 0; o >>= 1)
    for (int d = 0; d < 3; ++d) { lo[d] = fminf(lo[d], __shfl_xor_sync(0xffffffffu, lo[d], o)); hi[d] = fmaxf(hi[d], __shfl_xor_sync(0xffffffffu, hi[d], o)); }
  if (lane == 0) for (int d = 0; d < 3; ++d) { red[d][warp] = lo[d]; red[3 + d][warp] = hi[d]; }
  __syncthreads();
  if (tid < 6) {
    float v = red[tid][0];
    for (int w = 1; w < kBThreads / 32; ++w) v = tid < 3 ? fminf(v, red[tid][w]) : fmaxf(v, red[tid][w]);
    box[tid] = v;
  }
  __syncthreads();
  const float ext = fmaxf(fmaxf(box[3] - box[0], box[4] - box[1]), fmaxf(box[5] - box[2], 1e-9f));
  const float scale = 1023.0f / ext;
  int m2 = 1;
  while (m2 < n) m2 <<= 1;
  for (int i = tid; i < m2; i += kBThreads) {
    unsigned long long k = ~0ull;
    if (i < n) {
      const float4 p = __ldg(pts + base + i);
      const unsigned x = (unsigned)fminf(fmaxf((p.x - box[0]) * scale, 0.0f), 1023.0f), y = (unsigned)fminf(fmaxf((p.y - box[1]) * scale, 0.0f), 1023.0f),
                     z = (unsigned)fminf(fmaxf((p.z - box[2]) * scale, 0.0f), 1023.0f);
      k = ((unsigned long long)(spread10(x) | (spread10(y) << 1) | (spread10(z) << 2)) << 32) | (unsigned)i;
    }
    keys[i] = k;
  }
  __syncthreads();
  for (int k2 = 2; k2 <= m2; k2 <<= 1)
    for (int j2 = k2 >> 1; j2 > 0; j2 >>= 1) {
      for (int i = tid; i < m2; i += kBThreads) {
        const int l = i ^ j2;
        if (l > i) {
          const bool up = (i & k2) == 0;
          const unsigned long long ki = keys[i], kl = keys[l];
          if ((ki > kl) == up) { keys[i] = kl; keys[l] = ki; }
        }
      }
      __syncthreads();
    }
  for (int j = tid; j < n; j += kBThreads) {
    const int src = (int)(unsigned)(keys[j] & 0xffffffffull);
    float4 p = __ldg(pts + base + src);
    p.w = __int_as_float(j);
    opts[base + j] = p;
    onrm[base + j] = __ldg(nrm + base + src);
  }
}

// per-stage device time of the chunk (CUDA events on the context's stream), accumulated into ctx->batch_stage_ms
struct ChunkTimer {
  ope_ctx* ctx;
  cudaEvent_t ev[16];
  std::chrono::steady_clock::time_point host[16];
  int n = 0;
  bool on, trace;
  explicit ChunkTimer(ope_ctx* c) : ctx(c), on(c->batch_timing), trace(c->batch_timing && std::getenv("OPE_BATCH_TRACE") != nullptr) {
    if (on) for (auto& e : ev) cudaEventCreate(&e);
    mark();
  }
  void mark() { if (on && n < 16) { host[n] = std::chrono::steady_clock::now(); cudaEventRecord(ev[n++], ctx->stream); } }
  ~ChunkTimer() {
    if (!on) return;
    cudaEventSynchronize(ev[n - 1]);
    for (int i = 1; i < n; ++i) {
      float ms = 0;
      cudaEventElapsedTime(&ms, ev[i - 1], ev[i]);
      ctx->batch_stage_ms[i - 1] += ms;
      // OPE_BATCH_TRACE: the host's wall clock between the same marks (the device time includes what the device waited for the host)
      if (trace) fprintf(stderr, "[ope batch] stage %2d: device %8.3f ms, host %8.3f ms\n", i - 1, ms,
                         std::chrono::duration<double, std::milli>(host[i] - host[i - 1]).count());
    }
    for (auto& e : ev) cudaEventDestroy(e);
  }
};
// a chunk's sampled clouds: [0] 1 cm target, [1] 8 mm target, [2] source, each frames x kBCap points (and their normals, their
// NaN-normal compactions); counts / ccounts: 3 x frames; flags, active: per frame
struct BatchClouds { float4 *sampled, *normals, *compacted, *cnormals; int *counts, *ccounts, *flags, *active; };

// The fine stage of a chunk (estimateFinePose, :161-379): frame f's source (sa.src / sa.counts, through sa.xforms where set) sampled
// at the fine leaf into slab [2], its normals, removeNaNNormalsFromPointCloud of tp2 (slab [1], sampled with its normals by the
// caller) and sp2, the ICP's Morton work order, ICP, getFitnessScore. A frame that leaves the envelope leaves h_active; for the
// others by_frame (ICP), h_fit and h_cc (compacted counts: [0, B) tp2, [B, 2B) sp2) hold the results.
static int fine_stage(ope_ctx* ctx, const ope_pose_params& P, int B, const BatchClouds& c, BSampleArgs sa, std::vector<int>& h_active,
                      std::vector<ope_reg_result>& by_frame, std::vector<double>& h_fit, std::vector<int>& h_cc, ChunkTimer* tm) {
  const size_t slab = (size_t)B * kBCap;
  float4 *sampled = c.sampled, *normals = c.normals, *compacted = c.compacted, *cnormals = c.cnormals;
  int *d_counts = c.counts, *d_ccounts = c.ccounts, *d_flags = c.flags, *d_active = c.active;
  const float vp[3] = {0, 0, 0};
  sa.active = d_active; sa.flags = d_flags;
  sa.inv_leaf[0] = 1.0f / P.fine_leaf; sa.cap[0] = kBCap; sa.out[0] = sampled + 2 * slab; sa.out_counts[0] = d_counts + 2 * (size_t)B;
  bsample_kernel<<<dim3(B, 1), kBThreads, sizeof(SampleSmem), ctx->stream>>>(sa);
  OPE_TRY(check_launch(ctx, "bsample_kernel<source>"));
  std::vector<int> h_sp2;
  OPE_TRY(download(ctx, d_counts + 2 * (size_t)B, (size_t)B, h_sp2));
  std::vector<int> h_flags;
  OPE_TRY(download(ctx, d_flags, (size_t)B, h_flags));
  int max_sp2 = 0;
  for (int i = 0; i < B; ++i) {
    if (!h_active[(size_t)i]) continue;
    if (h_flags[(size_t)i] || h_sp2[(size_t)i] <= 0) { h_active[(size_t)i] = 0; continue; }
    max_sp2 = std::max(max_sp2, h_sp2[(size_t)i]);
  }
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_active, h_active.data(), B * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  if (tm) tm->mark();   // [6] model sampling
  OPE_TRY(normals_smem_batch(ctx, sampled + 2 * slab, d_counts + 2 * (size_t)B, kBCap, B, max_sp2, P.normal_k, vp, normals + 2 * slab));
  if (tm) tm->mark();   // [7] source normals
  // removeNaNNormalsFromPointCloud on both fine clouds (:215-216): clouds [1] (tp2) and [2] (sp2)
  compact_normals_batch_kernel<<<2 * B, kBThreads, 0, ctx->stream>>>(sampled + slab, normals + slab, d_counts + B, d_active, B,
                                                                     compacted + slab, cnormals + slab, d_ccounts + B);
  OPE_TRY(check_launch(ctx, "compact_normals_batch_kernel"));
  OPE_TRY(download(ctx, d_ccounts + B, 2 * (size_t)B, h_cc));   // [0..B) tp2, [B..2B) sp2
  // the ICP's work order: both fine clouds along their Morton curve (the raw samples' arrays are free by now)
  const char* me = std::getenv("OPE_BATCH_MORTON");
  const bool morton = !(me && std::atoi(me) == 0);
  const float4* fine_pts = compacted;
  const float4* fine_nrm = cnormals;
  if (morton) {
    morton_sort_batch_kernel<<<2 * B, kBThreads, 0, ctx->stream>>>(compacted + slab, cnormals + slab, d_ccounts + B, d_active, B,
                                                                   sampled + slab, normals + slab);
    OPE_TRY(check_launch(ctx, "morton_sort_batch_kernel"));
    fine_pts = sampled; fine_nrm = normals;
  }
  std::vector<IcpBatchFrame> icp_frames;
  std::vector<int> icp_of;
  int max_tgt = 0;
  for (int i = 0; i < B; ++i) {
    if (!h_active[(size_t)i]) continue;
    const int nt = h_cc[(size_t)i], nsrc = h_cc[(size_t)B + i];
    if (nt < P.min_target_points || !icp_small_batch_applicable(P.icp, (size_t)nsrc, (size_t)nt)) { h_active[(size_t)i] = 0; continue; }
    IcpBatchFrame fr;
    fr.tgt_pts = fine_pts + slab + (size_t)i * kBCap; fr.tgt_nrm = fine_nrm + slab + (size_t)i * kBCap; fr.n_tgt = nt;
    fr.src_pts = fine_pts + 2 * slab + (size_t)i * kBCap; fr.src_nrm = fine_nrm + 2 * slab + (size_t)i * kBCap; fr.n_src = nsrc;
    icp_frames.push_back(fr);
    icp_of.push_back(i);
    max_tgt = std::max(max_tgt, nt);
  }
  if (icp_frames.empty()) return OPE_OK;
  Scratch<ope_reg_result> d_fine(ctx);
  Scratch<double> d_fit(ctx);
  OPE_TRY(d_fine.alloc(B));
  Scratch<ope_reg_result> d_icp(ctx);
  const int NI = (int)icp_frames.size();
  OPE_TRY(d_icp.alloc(NI));
  if (tm) tm->mark();   // [8] NaN-normal compaction
  OPE_TRY(icp_small_batch_device(ctx, P.icp, icp_frames.data(), NI, d_icp.p));
  if (tm) tm->mark();   // [9] ICP
  // ---- getFitnessScore (:354) of every aligned pair; the ICP results are indexed by their position in icp_frames ----
  OPE_TRY(d_fit.alloc(B));
  {
    // scatter the compact ICP results back to frame order so that the fitness kernel can index by frame
    std::vector<ope_reg_result> h_icp;
    OPE_TRY(download(ctx, d_icp.p, (size_t)NI, h_icp));
    by_frame.assign((size_t)B, ope_reg_result());
    std::memset(by_frame.data(), 0, by_frame.size() * sizeof(ope_reg_result));
    for (int j = 0; j < NI; ++j) by_frame[(size_t)icp_of[(size_t)j]] = h_icp[(size_t)j];
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_fine.p, by_frame.data(), (size_t)B * sizeof(ope_reg_result), cudaMemcpyHostToDevice, ctx->stream));
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_active, h_active.data(), B * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    OPE_TRY(fitness_batch_device(ctx, fine_pts + slab, d_ccounts + B, fine_pts + 2 * slab, d_ccounts + 2 * (size_t)B, kBCap, B, max_tgt,
                                 d_fine.p, d_active, d_fit.p));
    if (tm) tm->mark();   // [10] fitness
    OPE_TRY(download(ctx, d_fit.p, (size_t)B, h_fit));   // also orders the host vectors above after their copies
  }
  return OPE_OK;
}

// Stages a chunk's targets in one device array (host points through the pinned arena, device clouds device-to-device) and
// fills `d_src` with each frame's first point. h_active[i] == 0 on entry excludes frame i; empty frames are excluded here.
// h_cnt[i]: the points of frame i (0 when excluded); *total == 0: nothing was staged.
static int stage_frames(ope_ctx* ctx, const ope_frame_input* frames, int B, std::vector<int>& h_active, std::vector<int>& h_off,
                        std::vector<int>& h_cnt, Scratch<float4>& clusters, Scratch<const float4*>& d_src, size_t* total_out) {
  h_off.assign((size_t)B, 0); h_cnt.assign((size_t)B, 0);
  size_t total = 0;
  *total_out = 0;
  for (int i = 0; i < B; ++i) {
    const ope_frame_input& in = frames[i];
    const size_t n = in.points ? in.n : (in.cloud ? ((const ope_cloud*)in.cloud)->n : 0);
    if (n == 0 || n > 0x3fffffff) h_active[(size_t)i] = 0;
    h_off[(size_t)i] = (int)total; h_cnt[(size_t)i] = h_active[(size_t)i] ? (int)n : 0;
    total += (size_t)h_cnt[(size_t)i];
  }
  if (total == 0 || total > 0x7fffffffull) return OPE_OK;
  OPE_TRY(clusters.alloc(total));
  OPE_TRY(d_src.alloc((size_t)B));
  void* stage = nullptr;
  OPE_TRY(stage_reserve(ctx, total * sizeof(float4) + (size_t)B * sizeof(const float4*), &stage));
  float4* h = (float4*)stage;
  for (int i = 0; i < B; ++i) {
    if (!h_active[(size_t)i]) continue;
    const ope_frame_input& in = frames[i];
    float4* dst = h + h_off[(size_t)i];
    if (in.points) {
      const unsigned char* base = (const unsigned char*)in.points + in.offset;
      for (size_t j = 0; j < in.n; ++j) { float v[3]; std::memcpy(v, base + j * in.stride, 12); dst[j] = make_float4(v[0], v[1], v[2], 1.0f); }
    }
  }
  const float4** hp = (const float4**)(h + total);
  for (int i = 0; i < B; ++i) hp[i] = clusters.p + h_off[(size_t)i];
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(clusters.p, stage, total * sizeof(float4), cudaMemcpyHostToDevice, ctx->stream));
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_src.p, hp, (size_t)B * sizeof(const float4*), cudaMemcpyHostToDevice, ctx->stream));
  for (int i = 0; i < B; ++i) {   // device-resident clusters: device-to-device into their slot
    const ope_frame_input& in = frames[i];
    if (h_active[(size_t)i] && !in.points)
      OPE_CUDA_TRY(ctx, cudaMemcpyAsync(clusters.p + h_off[(size_t)i], ((const ope_cloud*)in.cloud)->pts, (size_t)h_cnt[(size_t)i] * sizeof(float4),
                                        cudaMemcpyDeviceToDevice, ctx->stream));
  }
  *total_out = total;
  return OPE_OK;
}

// One chunk of frames through the frame-spanning launches: estimateCoarsePose (:16-73) for the frames that run SAC-IA, then
// estimateFinePose (:161-379). A frame outside the fast path's envelope leaves c.active (the caller finishes it on its per-frame
// path); the others have their results in c. The table hook runs exactly once, whatever happens before it (see PoseChunk).
int pose_chunk(ope_ctx* ctx, const ope_pose_params& P, int B, PoseChunk& c, const std::function<int(PoseChunk&)>& tables_hook) {
  const int H = P.sacia.max_iterations, S = P.sacia.nr_samples, K = P.sacia.k_correspondences;
  const bool own_src = !c.src_clouds.empty();
  const int clouds = (own_src ? 3 : 2) * B;   // sampled clouds the coarse stage describes: tp1, tp2 (, the sources' 1 cm samples)
  std::vector<int>& act = c.active;
  auto any_active = [&]() { return std::any_of(act.begin(), act.end(), [](int a) { return a != 0; }); };
  c.tables.assign((size_t)B, nullptr); c.n_src_coarse.assign((size_t)B, 0); c.n_tgt_coarse.assign((size_t)B, 0);
  std::vector<int> h_off, h_cnt, h_re((size_t)B, 0), h_counts, h_flags((size_t)B, 0);   // counts: tp1, tp2, source samples (B each)
  Scratch<float4> clusters(ctx), sampled(ctx), normals(ctx), compacted(ctx), cnormals(ctx);
  Scratch<const float4*> d_src(ctx);
  Scratch<int> d_cnt(ctx), d_active(ctx), d_re(ctx), d_counts(ctx), d_ccounts(ctx), d_flags(ctx), d_samples(ctx), d_picks(ctx), d_knn(ctx);
  Scratch<float> spfh(ctx), fpfh(ctx), sspfh(ctx), sfpfh(ctx), errors(ctx), transforms(ctx);
  Scratch<ope_reg_result> d_coarse(ctx);
  // sampled clouds: [0] tp1 (1 cm target), [1] tp2 (8 mm target), [2] the frame's source at 1 cm, then at 8 mm; each B x kBCap
  const size_t slab = (size_t)B * kBCap;
  BSampleArgs sa;
  std::memset(&sa, 0, sizeof(sa));
  ChunkTimer tm(ctx);
  size_t total = 0;
  OPE_TRY(stage_frames(ctx, c.targets, B, act, h_off, h_cnt, clusters, d_src, &total));
  if (total == 0) std::fill(act.begin(), act.end(), 0);
  else {
    OPE_TRY(sampled.alloc(3 * slab)); OPE_TRY(normals.alloc(3 * slab)); OPE_TRY(compacted.alloc(3 * slab)); OPE_TRY(cnormals.alloc(3 * slab));
    OPE_TRY(d_cnt.alloc(B)); OPE_TRY(d_active.alloc(B)); OPE_TRY(d_re.alloc(B)); OPE_TRY(d_counts.alloc(3 * (size_t)B)); OPE_TRY(d_ccounts.alloc(3 * (size_t)B));
    OPE_TRY(d_flags.alloc(B)); OPE_TRY(d_coarse.alloc(B));
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_cnt.p, h_cnt.data(), B * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_active.p, act.data(), B * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    OPE_CUDA_TRY(ctx, cudaMemsetAsync(d_flags.p, 0, B * sizeof(int), ctx->stream));
    OPE_CUDA_TRY(ctx, cudaMemsetAsync(d_counts.p, 0, 3 * (size_t)B * sizeof(int), ctx->stream));
    OPE_CUDA_TRY(ctx, cudaMemsetAsync(d_ccounts.p, 0, 3 * (size_t)B * sizeof(int), ctx->stream));
    tm.mark();   // [0] staging + H2D of the targets
    // ---- target UniformSampling at the coarse and the fine leaf (subSampleAndCalculateNormals, :131-158) ----
    sa.src = d_src.p; sa.counts = d_cnt.p; sa.active = d_active.p; sa.flags = d_flags.p;
    sa.inv_leaf[0] = 1.0f / P.coarse_leaf; sa.inv_leaf[1] = 1.0f / P.fine_leaf;
    sa.cap[0] = kBFeatCap; sa.cap[1] = kBCap;
    sa.out[0] = sampled.p; sa.out[1] = sampled.p + slab;
    sa.out_counts[0] = d_counts.p; sa.out_counts[1] = d_counts.p + B;
    OPE_TRY(bsample_batch(ctx, sa, B, 2));
    if (own_src) {   // ---- the per-frame sources of the frames that run SAC-IA at the coarse leaf, into slab [2] ----
      for (int i = 0; i < B; ++i) h_re[(size_t)i] = act[(size_t)i] && c.ran_coarse(i);
      OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_src.p, c.src_clouds.data(), B * sizeof(const float4*), cudaMemcpyHostToDevice, ctx->stream));
      OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_cnt.p, c.src_cloud_n.data(), B * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
      OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_re.p, h_re.data(), B * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
      std::memset(&sa, 0, sizeof(sa));
      sa.src = d_src.p; sa.counts = d_cnt.p; sa.active = d_re.p; sa.flags = d_flags.p;
      sa.inv_leaf[0] = 1.0f / P.coarse_leaf; sa.cap[0] = kBFeatCap; sa.out[0] = sampled.p + 2 * slab; sa.out_counts[0] = d_counts.p + 2 * (size_t)B;
      OPE_TRY(bsample_batch(ctx, sa, B, 1));
    }
    OPE_TRY(download(ctx, d_counts.p, (size_t)clouds, h_counts));
    OPE_TRY(download(ctx, d_flags.p, (size_t)B, h_flags));
  }
  h_counts.resize(3 * (size_t)B, 0);
  int max_tp = 0, max_tp1 = 0, max_ns = 0, n_re = 0;
  for (int i = 0; i < B; ++i) {
    const int n1 = h_counts[(size_t)i], n2 = h_counts[(size_t)B + i], ns = own_src ? h_counts[2 * (size_t)B + i] : c.src_n;
    // the envelope of the fast path: the fine stage runs ICP, every cloud fits its shared-memory kernel; a frame that runs SAC-IA
    // needs its coarse target and S source points (a per-frame source sample lives in a slab)
    bool ok = act[(size_t)i] && !h_flags[(size_t)i] && n2 >= std::max(P.min_target_points, 1) && n2 <= kBCap;
    if (c.ran_coarse(i))
      ok = ok && n1 >= std::max(P.min_target_features, 1) && n1 <= kBFeatCap && ns >= std::max(S, 1) && (!own_src || ns <= kBFeatCap);
    act[(size_t)i] = ok;
    h_re[(size_t)i] = ok && c.ran_coarse(i);
    if (!h_re[(size_t)i]) { h_counts[(size_t)i] = 0; h_counts[2 * (size_t)B + i] = 0; }   // no coarse stage: no 1 cm samples
    if (!ok) { h_counts[(size_t)B + i] = 0; continue; }
    c.n_tgt_coarse[(size_t)i] = h_counts[(size_t)i];
    if (h_re[(size_t)i]) c.n_src_coarse[(size_t)i] = own_src ? h_counts[2 * (size_t)B + i] : c.src_n;
    max_tp = std::max(max_tp, std::max(h_counts[(size_t)i], h_counts[(size_t)B + i]));
    max_tp1 = std::max(max_tp1, h_counts[(size_t)i]);
    max_ns = std::max(max_ns, h_counts[2 * (size_t)B + i]);
    n_re += h_re[(size_t)i];
  }
  int* d_sacia = c.coarse.empty() ? d_active.p : d_re.p;   // the frames that run SAC-IA
  const int ns = own_src ? max_ns : c.src_n;                // SAC-IA's source points per frame (at most)
  const float* fsrc = c.src_fpfh;
  if (any_active()) {
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_active.p, act.data(), B * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    if (d_sacia != d_active.p) OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_sacia, h_re.data(), B * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_counts.p, h_counts.data(), (size_t)clouds * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    tm.mark();   // [1] sampling
    // ---- normals of all the 1 cm and 8 mm samples in one launch, FPFH of tp1 and of the sources' samples (:16-48) ----
    const float vp[3] = {0, 0, 0};
    OPE_TRY(normals_smem_batch(ctx, sampled.p, d_counts.p, kBCap, clouds, std::max(max_tp, max_ns), P.normal_k, vp, normals.p));
    tm.mark();   // [2] normals
    if (n_re) {
      OPE_TRY(spfh.alloc(slab * 33)); OPE_TRY(fpfh.alloc(slab * 33));
      OPE_TRY(fpfh_smem_batch(ctx, sampled.p, normals.p, d_counts.p, kBCap, B, max_tp1, P.fpfh_radius, spfh.p, fpfh.p));
      if (own_src) {
        OPE_TRY(sspfh.alloc(slab * 33)); OPE_TRY(sfpfh.alloc(slab * 33));
        OPE_TRY(fpfh_smem_batch(ctx, sampled.p + 2 * slab, normals.p + 2 * slab, d_counts.p + 2 * (size_t)B, kBCap, B, max_ns, P.fpfh_radius,
                                sspfh.p, sfpfh.p));
        fsrc = sfpfh.p;
      }
      tm.mark();   // [3] FPFH
      // ---- findSimilarFeatures for every source point of every frame at once (:50-64) ----
      OPE_TRY(d_knn.alloc((size_t)B * ns * K));
      OPE_TRY(feature_knn_batch(ctx, fpfh.p, d_counts.p, kBCap, B, max_tp1, fsrc, ns, own_src ? kBCap : 0, own_src ? d_counts.p + 2 * (size_t)B : nullptr,
                                33, K, d_knn.p));
      tm.mark();   // [4] feature k-NN
    }
  }
  c.src_samples = own_src && sampled.p ? sampled.p + 2 * slab : nullptr;
  OPE_TRY(tables_hook(c));
  if (!any_active()) return OPE_OK;
  if (n_re) {   // ---- SAC-IA pool with the frames' decision tables, first strictly-lower error wins (:50-64) ----
    const size_t tb = (size_t)B * H * S;
    OPE_TRY(d_samples.alloc(tb)); OPE_TRY(d_picks.alloc(tb));
    void* stage = nullptr;
    OPE_CUDA_TRY(ctx, stream_sync(ctx));   // the target staging buffer is reused
    OPE_TRY(stage_reserve(ctx, 2 * tb * sizeof(int), &stage));
    int* hs = (int*)stage;
    int* hp = hs + tb;
    for (int i = 0; i < B; ++i) {
      int* s = hs + (size_t)i * H * S;
      int* p = hp + (size_t)i * H * S;
      if (!h_re[(size_t)i]) { std::memset(s, 0, (size_t)H * S * sizeof(int)); std::memset(p, 0, (size_t)H * S * sizeof(int)); continue; }
      // the single call's rule: at least H hypotheses of S samples (the first H are used), entries within the source and K
      const ope_rng_table* t = c.tables[(size_t)i];
      if (!t || t->n_hypotheses < H || t->nr_samples != S || !t->samples || !t->picks)
        return fail(ctx, OPE_ERR_INVALID, "decision table of frame %zu does not match the SAC-IA parameters", c.first + (size_t)i);
      std::memcpy(s, t->samples, (size_t)H * S * sizeof(int));
      std::memcpy(p, t->picks, (size_t)H * S * sizeof(int));
      for (size_t e = 0; e < (size_t)H * S; ++e)
        if (s[e] < 0 || s[e] >= c.n_src_coarse[(size_t)i] || p[e] < 0 || p[e] >= K) return fail(ctx, OPE_ERR_INVALID, "rng table entry out of range");
    }
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_samples.p, hs, tb * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_picks.p, hp, tb * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    OPE_TRY(errors.alloc((size_t)B * H)); OPE_TRY(transforms.alloc((size_t)B * H * 16));
    SaciaBatch sb;
    std::memset(&sb, 0, sizeof(sb));
    sb.src = own_src ? sampled.p + 2 * slab : c.src_pts; sb.ns = ns;
    if (own_src) { sb.src_stride = kBCap; sb.src_counts = d_counts.p + 2 * (size_t)B; }
    sb.tgt = sampled.p; sb.counts = d_counts.p; sb.stride = kBCap;
    sb.nr_samples = S; sb.k_corr = K; sb.H = H; sb.samples = d_samples.p; sb.picks = d_picks.p; sb.knn_idx = d_knn.p; sb.active = d_sacia;
    sb.h_begin = 0; sb.h_end = H; sb.early_exit = 1;
    sb.threshold = (float)P.sacia.max_correspondence_distance; sb.errors = errors.p; sb.transforms = transforms.p;
    const char* me = std::getenv("OPE_BATCH_MORTON");
    if (!(me && std::atoi(me) == 0)) {   // the distance scan reads a Morton-ordered copy of the target (slot [0] of the compaction arrays is free)
      morton_sort_batch_kernel<<<B, kBThreads, 0, ctx->stream>>>(sampled.p, normals.p, d_counts.p, d_sacia, B, compacted.p, cnormals.p);
      OPE_TRY(check_launch(ctx, "morton_sort_batch_kernel"));
      sb.tgt_scan = compacted.p;
    }
    OPE_TRY(sacia_batch_device(ctx, sb, B, max_tp1, nullptr, d_coarse.p));
    tm.mark();   // [5] SAC-IA
  }
  // ---- estimateFinePose (:161-379): each frame's fine source, through its coarse pose where it ran SAC-IA (never materialised) ----
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_src.p, c.fine_src.data(), B * sizeof(const float4*), cudaMemcpyHostToDevice, ctx->stream));
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_cnt.p, c.fine_n.data(), B * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  std::memset(&sa, 0, sizeof(sa));
  sa.src = d_src.p; sa.counts = d_cnt.p; sa.xforms = d_coarse.p; sa.xform_on = c.coarse.empty() ? nullptr : d_re.p;
  BatchClouds bc{sampled.p, normals.p, compacted.p, cnormals.p, d_counts.p, d_ccounts.p, d_flags.p, d_active.p};
  std::vector<int> h_cc;
  OPE_TRY(fine_stage(ctx, P, B, bc, sa, act, c.fine, c.fitness, h_cc, &tm));
  if (!any_active()) return OPE_OK;
  c.n_tgt_fine.assign(h_cc.begin(), h_cc.begin() + B); c.n_src_fine.assign(h_cc.begin() + B, h_cc.end());
  return download(ctx, d_coarse.p, (size_t)B, c.coarse_res);
}

ope_pose_result chunk_pose_result(const PoseChunk& c, int i, const Mat4& rigid) {
  ope_pose_result r;
  std::memset(&r, 0, sizeof(r));
  const ope_reg_result& f = c.fine[(size_t)i];
  Mat4 coarse = mat4_identity(), fine;
  if (c.ran_coarse(i)) std::memcpy(coarse.m, c.coarse_res[(size_t)i].T, 64);
  std::memcpy(fine.m, f.T, 64);
  const Mat4 final_pose = mat4_mul(rigid, mat4_mul(coarse, fine));
  std::memcpy(r.final_pose, final_pose.m, 64); std::memcpy(r.coarse_pose, coarse.m, 64);
  std::memcpy(r.fine_pose, fine.m, 64); std::memcpy(r.rigid_model_pose, rigid.m, 64);
  const int nsrc = c.n_src_fine[(size_t)i], nt = c.n_tgt_fine[(size_t)i];
  r.fitness = c.fitness[(size_t)i];
  r.align_strength = (double)f.n_correspondences / (double)((long)nsrc + (long)nt);   // VP/icp_mod.h:249-260
  r.icp_iterations = f.iterations; r.icp_converged = f.converged; r.icp_state = f.state;
  r.n_src_fine = nsrc; r.n_tgt_fine = nt;
  if (c.ran_coarse(i)) {
    r.ran_coarse = 1;
    r.n_src_coarse = c.n_src_coarse[(size_t)i]; r.n_tgt_coarse = c.n_tgt_coarse[(size_t)i];
    r.sacia_best_iteration = c.coarse_res[(size_t)i].best_iteration; r.sacia_best_error = c.coarse_res[(size_t)i].best_error;
  }
  return r;
}

}  // namespace ope
