// registration.cu — rigid transform estimation (K10/K11), fitness (K9), the fused ICP loop (K8) and the SAC-IA
// hypothesis pool (K7).
//
// ICP is ONE persistent cooperative kernel per align(): every iteration fuses correspondence search on the
// target grid, the rejector chain, the centroid / 3x3 cross-covariance reduction (double, fixed-shape tree:
// thread -> warp shuffle -> block -> per-block partials in HBM), ONE grid barrier, then in every block
// redundantly the reduction of the per-block partials in a fixed order, the 3x3 Jacobi SVD (Umeyama), the
// convergence test and the in-place rigid transform of the block's own source points. Nothing but the 4x4,
// the flags and the iteration count returns to the host (SURVEY 3.2, K8).
#include <cooperative_groups.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>

#include <map>
#include <mutex>

#include <chrono>
#include "ope_host.cuh"
#include "ope_octet.cuh"

namespace cg = cooperative_groups;

namespace ope {

// ===================================================================================== small kernels ===
__global__ void transform_kernel(const float4* __restrict__ in, const float4* __restrict__ in_n, int n, Mat4 T,
                                 float4* __restrict__ out, float4* __restrict__ out_n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float4 p = __ldg(in + i);
  float4 o = p;
  xform_point(T, p.x, p.y, p.z, o.x, o.y, o.z);
  out[i] = o;
  if (in_n && out_n) {
    float4 v = __ldg(in_n + i);
    float4 w = v;
    xform_normal(T, v.x, v.y, v.z, w.x, w.y, w.z);
    out_n[i] = w;
  }
}

static constexpr int kRedThreads = 256;
static constexpr int kMomentAcc = 16;  // n, Ss[3], St[3], Sts[9]

__device__ __forceinline__ double warp_sum_d(double v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// block-level sum of NACC doubles per thread -> out[NACC] valid in ALL threads of warp 0 / written to dst by thread 0.
template <int NACC>
__device__ __forceinline__ void block_reduce_store(double* acc, double* smem /* (blockDim/32)*NACC */, double* dst) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
  for (int a = 0; a < NACC; ++a) acc[a] = warp_sum_d(acc[a]);
  if (lane == 0)
    for (int a = 0; a < NACC; ++a) smem[warp * NACC + a] = acc[a];
  __syncthreads();
  if (threadIdx.x < NACC) {
    double s = 0.0;
    for (int w = 0; w < nw; ++w) s += smem[w * NACC + threadIdx.x];
    dst[threadIdx.x] = s;
  }
  __syncthreads();
}

// raw moments of n pairs (src[is[i]], tgt[it[i]]) -> partials[block][16]
__global__ void moments_kernel(const float4* __restrict__ src, const float4* __restrict__ tgt, const int* __restrict__ is,
                               const int* __restrict__ it, int n, double* __restrict__ partials) {
  __shared__ double smem[(kRedThreads / 32) * kMomentAcc];
  double acc[kMomentAcc];
  for (int a = 0; a < kMomentAcc; ++a) acc[a] = 0.0;
  double o[3];
  { const float4 t0 = __ldg(tgt); moment_origin(t0.x, t0.y, t0.z, o[0], o[1], o[2]); }   // relative to the target's first point
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 s = __ldg(src + (is ? is[i] : i));
    const float4 t = __ldg(tgt + (it ? it[i] : i));
    const double sv[3] = {(double)s.x - o[0], (double)s.y - o[1], (double)s.z - o[2]};
    const double tv[3] = {(double)t.x - o[0], (double)t.y - o[1], (double)t.z - o[2]};
    acc[0] += 1.0;
    acc[1] += sv[0]; acc[2] += sv[1]; acc[3] += sv[2];
    acc[4] += tv[0]; acc[5] += tv[1]; acc[6] += tv[2];
    for (int c = 0; c < 3; ++c)
      for (int r = 0; r < 3; ++r) acc[7 + c * 3 + r] += tv[r] * sv[c];
  }
  block_reduce_store<kMomentAcc>(acc, smem, partials + (size_t)blockIdx.x * kMomentAcc);
}
// one warp per accumulator (lanes stride over the blocks, fixed shuffle tree), then one thread runs the 3x3 Umeyama
__device__ __forceinline__ void umeyama_final(const double* __restrict__ partials, int nblocks, float* __restrict__ out16, const float4* __restrict__ tgt) {
  __shared__ double acc[kMomentAcc];
  const int a = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (a < kMomentAcc) {
    double s = 0.0;
    for (int b = lane; b < nblocks; b += 32) s += partials[(size_t)b * kMomentAcc + a];
    s = warp_sum_d(s);
    if (lane == 0) acc[a] = s;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    Mat4 T;
    double o[3];
    const float4 t0 = __ldg(tgt);
    moment_origin(t0.x, t0.y, t0.z, o[0], o[1], o[2]);
    umeyama_from_moments(acc, T, o[0], o[1], o[2]);
    for (int i = 0; i < 16; ++i) out16[i] = T.m[i];
  }
}
__global__ void umeyama_final_kernel(const double* __restrict__ partials, int nblocks, float* __restrict__ out16,
                                     const float4* __restrict__ tgt) {
  umeyama_final(partials, nblocks, out16, tgt);
}

// The state commit of a tracker step (ope_pose_tracker_step_batch), blockIdx.y = tracker, one read of its big clouds:
//   out_aligned = out_source = fine(coarse(in)) (re-coarse; rounded to float after each transform, as two transform_kernel
//                              passes) or fine(in) (tracking)
//   the moments of the dense Umeyama model -> source with umeyama_device's shape: c.nb blocks, the same grid-stride loop, the
//   same block reduction, so that track_umeyama_final_kernel returns its bits
__global__ void __launch_bounds__(kRedThreads) track_commit_kernel(const TrackCommit* __restrict__ commits, double* __restrict__ partials) {
  __shared__ double smem[(kRedThreads / 32) * kMomentAcc];
  const TrackCommit& c = commits[blockIdx.y];
  if ((int)blockIdx.x >= c.nb) return;
  const int stride = c.nb * kRedThreads;
  Mat4 C, F;
  for (int i = 0; i < 16; ++i) { C.m[i] = c.coarse[i]; F.m[i] = c.fine[i]; }
  for (int i = blockIdx.x * kRedThreads + threadIdx.x; i < c.n_in; i += stride) {
    float4 p = __ldg(c.in + i);
    if (c.pre) { float4 q = p; xform_point(C, p.x, p.y, p.z, q.x, q.y, q.z); p = q; }
    float4 o = p;
    xform_point(F, p.x, p.y, p.z, o.x, o.y, o.z);
    c.out_aligned[i] = o;
    c.out_source[i] = o;
  }
  if (c.n_model == 0) return;
  double acc[kMomentAcc];
  for (int a = 0; a < kMomentAcc; ++a) acc[a] = 0.0;
  double o[3];
  { const float4 t0 = __ldg(c.src); moment_origin(t0.x, t0.y, t0.z, o[0], o[1], o[2]); }
  for (int i = blockIdx.x * kRedThreads + threadIdx.x; i < c.n_model; i += stride) {
    const float4 s = __ldg(c.model + i);
    const float4 t = __ldg(c.src + i);
    const double sv[3] = {(double)s.x - o[0], (double)s.y - o[1], (double)s.z - o[2]};
    const double tv[3] = {(double)t.x - o[0], (double)t.y - o[1], (double)t.z - o[2]};
    acc[0] += 1.0;
    acc[1] += sv[0]; acc[2] += sv[1]; acc[3] += sv[2];
    acc[4] += tv[0]; acc[5] += tv[1]; acc[6] += tv[2];
    for (int cc = 0; cc < 3; ++cc)
      for (int r = 0; r < 3; ++r) acc[7 + cc * 3 + r] += tv[r] * sv[cc];
  }
  block_reduce_store<kMomentAcc>(acc, smem, partials + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * kMomentAcc);
}
__global__ void track_umeyama_final_kernel(const TrackCommit* __restrict__ commits, const double* __restrict__ partials, int max_nb,
                                           float* __restrict__ out16) {
  const TrackCommit& c = commits[blockIdx.x];
  if (c.n_model == 0) return;
  umeyama_final(partials + (size_t)blockIdx.x * max_nb * kMomentAcc, c.nb, out16 + (size_t)blockIdx.x * 16, c.src);
}

// fitness: sum of NN-1 squared distances <= max_range of the transformed source (double), plus the count.
// One query per thread through block_nn1 (fast path per thread, far queries finished by octets).
static constexpr int kNnThreads = 256;
__global__ void __launch_bounds__(kNnThreads) fitness_kernel(GridView g, const float4* __restrict__ src, int n, Mat4 T,
                                                             float max_range_f, double* __restrict__ partials) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Nn1Smem<kNnThreads>* nn = reinterpret_cast<Nn1Smem<kNnThreads>*>(smem_raw);
  __shared__ double smem[(kNnThreads / 32) * 2];
  double acc[2] = {0.0, 0.0};
  for (int base = blockIdx.x * kNnThreads; base < n; base += gridDim.x * kNnThreads) {
    const int i = base + (int)threadIdx.x;
    float x = 0, y = 0, z = 0;
    bool ok = false;
    if (i < n) {
      const float4 p = __ldg(src + i);
      xform_point(T, p.x, p.y, p.z, x, y, z);
      ok = finite3(x, y, z);
    }
    float d2;
    const int idx = block_nn1<kNnThreads>(g, nn, ok, x, y, z, FLT_MAX, -1, nullptr, d2);
    if (ok && idx >= 0 && d2 <= max_range_f) { acc[0] += (double)d2; acc[1] += 1.0; }
  }
  block_reduce_store<2>(acc, smem, partials + (size_t)blockIdx.x * 2);
}
// The same against a small target (a down-sampled cluster) held in shared memory: exact brute force, one query per thread, eight
// independent distances per step (broadcast loads). No spatial index to build, so the call is two launches instead of eight.
static constexpr int kFitSmemMax = 4096;
__global__ void __launch_bounds__(kNnThreads) fitness_smem_kernel(const float4* __restrict__ tgt, int nt, const float4* __restrict__ src, int n,
                                                                  Mat4 T, float max_range_f, double* __restrict__ partials) {
  extern __shared__ __align__(16) float4 tg_fit[];
  __shared__ double smem[(kNnThreads / 32) * 2];
  const int nt8 = (nt + 7) & ~7;
  for (int j = threadIdx.x; j < nt8; j += kNnThreads) tg_fit[j] = j < nt ? __ldg(tgt + j) : make_float4(INFINITY, INFINITY, INFINITY, 0.0f);
  __syncthreads();
  double acc[2] = {0.0, 0.0};
  for (int base = blockIdx.x * kNnThreads; base < n; base += gridDim.x * kNnThreads) {
    const int i = base + (int)threadIdx.x;
    float x = 0, y = 0, z = 0;
    bool ok = false;
    if (i < n) {
      const float4 p = __ldg(src + i);
      xform_point(T, p.x, p.y, p.z, x, y, z);
      ok = finite3(x, y, z);
    }
    float best = INFINITY;
    if (ok) {
      for (int j0 = 0; j0 < nt8; j0 += 8) {
        float d2[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) { const float4 t = tg_fit[j0 + u]; d2[u] = dist2(x, y, z, t.x, t.y, t.z); }
#pragma unroll
        for (int u = 0; u < 8; ++u) if (d2[u] < best) best = d2[u];   // NaN (non-finite target point) never wins
      }
    }
    if (ok && best <= max_range_f) { acc[0] += (double)best; acc[1] += 1.0; }   // best = inf: no finite target point
  }
  block_reduce_store<2>(acc, smem, partials + (size_t)blockIdx.x * 2);
}
__global__ void sum_partials_kernel(const double* __restrict__ partials, int nblocks, int nacc, double* __restrict__ out) {
  // one warp per accumulator, lanes stride over the blocks, fixed shuffle tree
  const int a = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (blockIdx.x != 0 || a >= nacc) return;
  double s = 0.0;
  for (int b = lane; b < nblocks; b += 32) s += partials[(size_t)b * nacc + a];
  s = warp_sum_d(s);
  if (lane == 0) out[a] = s;
}

// =============================================================================================== ICP ====
// Work layout. The source is processed in the Morton order of its own cached grid (spatially coherent neighbours
// sit in the same warp: their searches touch the same cells, so the divergent 4- and 16-byte loads coalesce and hit
// L1); `cur_pts[s].w` carries the ORIGINAL index, which is what every caller-visible array is indexed by.
//
//  nearest estimator — two grid barriers per iteration:
//    A  one source point per THREAD: seed the bound with the previous iteration's exact neighbour, ope::nn1_fast; the
//       queries whose candidate set is too large (far from the target surface) are compacted — deterministically —
//       into the block's segment of a grid-wide queue;                                                  [barrier 1]
//    B  ALL warps of the grid drain the queue round-robin, one far query per WARP (coop_nn1, large leaves), so the
//       blocks that happened to own many far points do not hold the others at the barrier;              [barrier 2]
//    C  every block reduces the per-block double moments in the same order, warp 0 forms the means and the float
//       cross-covariance with one division per lane, lane 0 runs the 3x3 Jacobi SVD (Umeyama) and the convergence
//       test, then the block transforms its own slice of the source in place.
//  normal shooting — one barrier per iteration: one source point per WARP (warp_knn bounded by the previous iteration's
//       k-th distance), each warp owns a contiguous run of points and transforms it with all its lanes.
struct IcpDev {
  GridView grid;
  const float4* tgt_pts;      // original order (match index -> point)
  const float4* tgt_nrm;      // original order or null
  const float4* src0_pts;     // untouched input, original order (variant MODCORR reads stale normals/points from here)
  const float4* src0_nrm;
  const float4* src_sorted;   // finite source points in Morton order of the source's own grid, .w = original index
  int n_src;                  // points in the source cloud
  int n_work;                 // finite points = entries of src_sorted / cur_*
  float4* cur_pts;            // working copy (sorted order), transformed in place every iteration, .w = original index
  float4* cur_nrm;
  // parameters
  int max_iterations, min_corr, estimator, k_search, n_rej, transformation, variant, force_all;
  int rej_kind[OPE_MAX_REJECTORS];
  double rej_thr[OPE_MAX_REJECTORS];
  double max_corr_dist;       // as given (unsquared)
  float max_d2_f;             // squared, clamped to FLT_MAX (nearest estimator search bound)
  double rot_thr, trans_thr, rel_mse_thr, abs_mse_thr;
  int max_similar, fail_after_max;
  // outputs / state
  int* corr_match;            // n_src by ORIGINAL index, -1 = no correspondence this iteration (pre-filled by the host)
  float* corr_d2;             // n_src
  int* seed;                  // nearest: n_work (sorted position) last exact neighbour, -1 = none
                              // normal shooting: n_work * k_search, last k-NN list, -1 = none
  float4* ref;                // nearest: n_work certificates {query position when issued, R}: every target point other than
                              // seed[s] is at least R away from that position (R <= 0: none)
  float cert_gap;             // how far beyond the neighbour a search looks so that R exceeds the neighbour's distance
  int dfs_max;                // candidate-set size up to which a thread finishes its own query (above: the warp queue)
  int tgt_in_smem;            // normal shooting against a small target: the target lives in shared memory (warp_knn_smem)
  int n_tgt;                  // points in the target cloud
  int split_min;              // far queries with more candidate points than this are split by start node
  float4* def_q;              // far-query queue: x, y, z, seed d2          (block b's segment starts at its slice)
  int4* def_m;                //                  sorted position, seed index, original index, start node (-1: all)
  float4* def_res;            // result of a queue entry: d1, i1 (bits), s2, r2
  int* def_count;             // [2][gridDim]: per block, small then large
  int* def_head;              // [2 parities][2 kinds] claim counters of the far queues (zeroed by the host / by block 0)
  double* partials;           // 2 * gridDim * kIcpAcc (double buffered)
  unsigned* barrier;          // monotonic arrival counter of the grid barrier (zeroed by the host)
  ope_reg_result* result;     // device copy
  long long* phase_cycles;    // optional (OPE_PROFILE=1): block 0's cycles per phase
  Mat4 guess;
};

static constexpr int kIcpThreads = 512;
static constexpr int kIcpWarps = kIcpThreads / 32;
static constexpr int kIcpAcc = 17;  // moments[16] + sum of correspondence distances
static constexpr int kIcpMaxBlocks = 1024;
static constexpr int kIcpSmemMaxTargets = 4096;   // 64 KB of target points next to the kernel's other shared memory
static constexpr int kIcpSplitMin = 6144;   // far queries with more candidate points than this are split by start node (<= 8 entries)


struct IcpSmem {
  OctStack wstack[kIcpWarps];   // one traversal stack per warp (far queries / k-NN)
  float2 knn_buf[kIcpWarps][kKnnBufCap + 32];   // warp_knn_smem_bounded: candidates within the bound + the sorted k best
  LeafList leaves[kIcpWarps];   // collected leaf ranges of the warp's far query
  int dir[kDirEntries];         // upper levels of the target's implicit octree (coop_nn1_far)
  Nn1Smem<kIcpThreads> nn;      // only the one-pass kernel uses the block-local variant
  double red[kIcpWarps][kIcpAcc];
  double totals[kIcpAcc];
  int prefix[2][kIcpMaxBlocks]; // inclusive prefixes of the blocks' far-query counts: [0] small (octets), [1] large (warps)
  int warp_cnt[2][kIcpWarps];
  int n_def[2];
  Mat4 T_inc;
  int stop;  // 0 continue, 1 stop, 2 stop without a transform (not enough correspondences)
};

// ---- grid barrier: monotonic counter, release on arrival, acquire on the spin (cooperative launch => co-resident) ----
__device__ __forceinline__ void grid_barrier(unsigned* counter, unsigned target) {
  __syncthreads();
  if (threadIdx.x == 0) {
    asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(counter) : "memory");
    unsigned v;
    do {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
    } while (v < target);
  }
  __syncthreads();
}

// Sum v[0..15] over the 32 lanes with 16 double shuffles instead of 80: at every level a lane keeps half of its
// values and hands the other half to its partner. Afterwards lane l holds the warp total of slot
// ((l>>4)&1)*8 + ((l>>3)&1)*4 + ((l>>2)&1)*2 + ((l>>1)&1) (both lanes of a pair hold the same one). Fixed shape.
__device__ __forceinline__ double warp_reduce16(const double* v, int lane, int& slot) {
  double w8[8], w4[4], w2[2], w1;
  const bool b16 = lane & 16, b8 = lane & 8, b4 = lane & 4, b2 = lane & 2;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const double keep = b16 ? v[j + 8] : v[j], give = b16 ? v[j] : v[j + 8];
    w8[j] = keep + __shfl_xor_sync(0xffffffffu, give, 16);
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const double keep = b8 ? w8[j + 4] : w8[j], give = b8 ? w8[j] : w8[j + 4];
    w4[j] = keep + __shfl_xor_sync(0xffffffffu, give, 8);
  }
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const double keep = b4 ? w4[j + 2] : w4[j], give = b4 ? w4[j] : w4[j + 2];
    w2[j] = keep + __shfl_xor_sync(0xffffffffu, give, 4);
  }
  {
    const double keep = b2 ? w2[1] : w2[0], give = b2 ? w2[0] : w2[1];
    w1 = keep + __shfl_xor_sync(0xffffffffu, give, 2);
  }
  w1 += __shfl_xor_sync(0xffffffffu, w1, 1);
  slot = (b16 ? 8 : 0) + (b8 ? 4 : 0) + (b4 ? 2 : 0) + (b2 ? 1 : 0);
  return w1;
}

// term e (0..16) of the moments of one correspondence (p -> t, squared distance d2)
// (coordinates relative to the origin o: see ope::umeyama_from_moments)
__device__ __forceinline__ double moment_term(int e, const float4 p, const float4 t, float d2, const double o[3]) {
  if (e == 0) return 1.0;
  if (e < 4) return e == 1 ? (double)p.x - o[0] : (e == 2 ? (double)p.y - o[1] : (double)p.z - o[2]);
  if (e < 7) return e == 4 ? (double)t.x - o[0] : (e == 5 ? (double)t.y - o[1] : (double)t.z - o[2]);
  if (e < 16) {
    const int c = (e - 7) / 3, r = (e - 7) % 3;
    const double sv = c == 0 ? (double)p.x - o[0] : (c == 1 ? (double)p.y - o[1] : (double)p.z - o[2]);
    const double tv = r == 0 ? (double)t.x - o[0] : (r == 1 ? (double)t.y - o[1] : (double)t.z - o[2]);
    return tv * sv;
  }
  return (double)d2;
}

// rejector chain for one candidate correspondence (VP/impl/icp_mod.hpp:194-208); s = position in cur_*, orig = original
// index. Returns the match or -1.
__device__ __forceinline__ int icp_reject(const IcpDev& a, int s, int orig, const float4 p, int match) {
  const bool stale = a.variant == OPE_ICP_VARIANT_MODCORR;
  for (int r = 0; r < a.n_rej && match >= 0; ++r) {
    const float4 sn = stale ? __ldg(a.src0_nrm + orig) : a.cur_nrm[s];
    double score;
    if (a.rej_kind[r] == OPE_REJ_SURFACE_NORMAL) {
      const float4 tn = __ldg(a.tgt_nrm + match);
      score = (double)((sn.x * tn.x) + (sn.y * tn.y) + (sn.z * tn.z));
    } else {
      const float4 sp = stale ? __ldg(a.src0_pts + orig) : p;
      const double sl = (double)sqrtf(sp.x * sp.x + sp.y * sp.y + sp.z * sp.z);
      score = (double)((sn.x * (-sp.x / sl)) + (sn.y * (-sp.y / sl)) + (sn.z * (-sp.z / sl)));
    }
    if (!(score > a.rej_thr[r])) match = -1;
  }
  return match;
}

// exact neighbour -> correspondence: distance gate (VP/impl/correspondence_estimation_mod.hpp:171) + rejector chain
__device__ __forceinline__ int icp_gate(const IcpDev& a, int s, int orig, const float4 p, int nn, float d2) {
  int match = nn;
  if (match >= 0 && (double)d2 > a.max_corr_dist * a.max_corr_dist) match = -1;
  if (match >= 0) match = icp_reject(a, s, orig, p, match);
  return match;
}

// CorrespondenceEstimationNormalShooting: one source point per WARP. Among the k nearest, the one with the smallest
// squared distance to the line through p along the source normal (double); the first minimum in list order wins.
__device__ __forceinline__ int icp_correspond_shooting(const IcpDev& a, OctStack* st, int s, int orig, const float4 p, bool use_seed,
                                                       float& d2_out, const float4* tg_smem = nullptr, float2* knn_buf = nullptr) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const bool ok = finite3(p.x, p.y, p.z);
  const bool stale = a.variant == OPE_ICP_VARIANT_MODCORR;
  const int k = a.k_search < a.grid.n ? a.k_search : a.grid.n;
  // the previous iteration's k neighbours bound this iteration's k-th distance
  float bound = FLT_MAX;
  if (use_seed && ok) {
    int pj = -1;
    if (lane < k) pj = a.seed[(size_t)s * a.k_search + lane];
    float d = 0.0f;
    if (pj >= 0) { const float4 t = tg_smem ? tg_smem[pj] : __ldg(a.tgt_pts + pj); d = dist2(p.x, p.y, p.z, t.x, t.y, t.z); }
    const bool all_valid = __ballot_sync(full, lane >= k || pj >= 0) == full;
    for (int o = 16; o > 0; o >>= 1) d = fmaxf(d, __shfl_xor_sync(full, d, o));
    if (all_valid) bound = d;
  }
  float ld;
  int li;
  const int cnt = tg_smem ? (knn_buf ? warp_knn_smem_bounded(tg_smem, a.n_tgt, a.grid.n, ok, p.x, p.y, p.z, a.k_search, bound, knn_buf, ld, li)
                                     : warp_knn_smem(tg_smem, a.n_tgt, a.grid.n, ok, p.x, p.y, p.z, a.k_search, bound, ld, li))
                          : warp_knn(a.grid, st, ok, p.x, p.y, p.z, a.k_search, bound, ld, li);
  if (a.seed && lane < a.k_search) a.seed[(size_t)s * a.k_search + lane] = (lane < cnt) ? li : -1;
  int match = -1;
  float d2 = 0.0f;
  if (cnt > 0) {
    const float4 nr = stale ? __ldg(a.src0_nrm + orig) : a.cur_nrm[s];
    const double N[3] = {nr.x, nr.y, nr.z};
    double dist = DBL_MAX;
    int jdx = 0x7fffffff;
    if (lane < cnt) {
      const float4 t = tg_smem ? tg_smem[li] : __ldg(a.tgt_pts + li);
      const float px = t.x - p.x, py = t.y - p.y, pz = t.z - p.z;
      const double V[3] = {px, py, pz};
      const double C0 = N[1] * V[2] - N[2] * V[1], C1 = N[2] * V[0] - N[0] * V[2], C2 = N[0] * V[1] - N[1] * V[0];
      dist = C0 * C0 + C1 * C1 + C2 * C2;
      jdx = lane;
      if (!(dist < DBL_MAX)) { dist = DBL_MAX; jdx = 0x7fffffff; }  // NaN / inf never win (`dist < min_dist` in the reference)
    }
    for (int o = 16; o > 0; o >>= 1) {
      const double od = __shfl_xor_sync(full, dist, o);
      const int oj = __shfl_xor_sync(full, jdx, o);
      if (od < dist || (od == dist && oj < jdx)) { dist = od; jdx = oj; }
    }
    // the reference starts from min_index = 0: with no finite candidate it still reports neighbour 0 unless rejected below
    const int pick = jdx == 0x7fffffff ? 0 : jdx;
    const double min_dist = jdx == 0x7fffffff ? DBL_MAX : dist;
    if (!(min_dist > a.max_corr_dist)) {  // sic (SURVEY A.8): squared cross norm vs unsquared threshold
      match = __shfl_sync(full, li, pick);
      d2 = __shfl_sync(full, ld, pick);
    }
  }
  if (match >= 0) match = icp_reject(a, s, orig, p, match);
  d2_out = d2;
  return match;
}

// in-place rigid transform of cur_pts[s] / cur_nrm[s]
__device__ __forceinline__ void icp_move(const IcpDev& a, const Mat4& T, int s) {
  float4 p = a.cur_pts[s];
  if (!finite3(p.x, p.y, p.z)) return;
  float x, y, z;
  xform_point(T, p.x, p.y, p.z, x, y, z);
  p.x = x; p.y = y; p.z = z;
  a.cur_pts[s] = p;
  if (a.cur_nrm) {
    float4 v = a.cur_nrm[s];
    if (finite3(v.x, v.y, v.z)) {
      xform_normal(T, v.x, v.y, v.z, x, y, z);
      v.x = x; v.y = y; v.z = z;
      a.cur_nrm[s] = v;
    }
  }
}

__global__ void __launch_bounds__(kIcpThreads, 1) icp_kernel(IcpDev a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  IcpSmem* sm = reinterpret_cast<IcpSmem*>(smem_raw);
  double morg[3];   // origin of the moment accumulation: the target's first point (ope::umeyama_from_moments)
  { const float4 t0 = a.n_tgt > 0 ? __ldg(a.tgt_pts) : make_float4(0, 0, 0, 0); moment_origin(t0.x, t0.y, t0.z, morg[0], morg[1], morg[2]); }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int gwarp = blockIdx.x * kIcpWarps + warp, n_gwarps = gridDim.x * kIcpWarps;
  const bool shooting = a.estimator == OPE_EST_NORMAL_SHOOTING;
  OctStack* st = &sm->wstack[warp];

  // nearest: block b owns the slice [lo, hi) of the sorted source; shooting: warp gw owns [wlo, whi)
  const int chunk = (a.n_work + (int)gridDim.x - 1) / (int)gridDim.x;
  const int lo = min(a.n_work, (int)blockIdx.x * chunk), hi = min(a.n_work, lo + chunk);
  const int wchunk = (a.n_work + n_gwarps - 1) / n_gwarps;
  const int wlo = min(a.n_work, gwarp * wchunk), whi = min(a.n_work, wlo + wchunk);

  // input_transformed = guess applied to input (VP/impl/icp_mod.hpp:132-139), in sorted order
  const bool have_guess = !mat4_is_identity(a.guess);
  for (int s = blockIdx.x * kIcpThreads + threadIdx.x; s < a.n_work; s += gridDim.x * kIcpThreads) {
    float4 p = __ldg(a.src_sorted + s);
    const int orig = __float_as_int(p.w);
    float4 v = a.src0_nrm ? __ldg(a.src0_nrm + orig) : make_float4(0, 0, 0, 0);
    if (have_guess) {
      float x, y, z;
      xform_point(a.guess, p.x, p.y, p.z, x, y, z);
      p.x = x; p.y = y; p.z = z;
      if (a.src0_nrm && finite3(v.x, v.y, v.z)) {
        xform_normal(a.guess, v.x, v.y, v.z, x, y, z);
        v.x = x; v.y = y; v.z = z;
      }
    }
    a.cur_pts[s] = p;
    if (a.cur_nrm) a.cur_nrm[s] = v;
  }
  float4* tg_smem = nullptr;
  if (a.tgt_in_smem) {   // small target: resident in shared memory for the whole alignment
    tg_smem = reinterpret_cast<float4*>(smem_raw + ((sizeof(IcpSmem) + 15) & ~(size_t)15));
    for (int j = threadIdx.x; j < a.n_tgt; j += kIcpThreads) tg_smem[j] = __ldg(a.tgt_pts + j);
  } else {
    far_dir_load(a.grid, sm->dir);
  }
  FarDir fdir;
  fdir.sdir = sm->dir; fdir.dl = far_dir_level(a.grid);
  // the initialisation above is grid-strided, the iterations use their own ownership maps: one barrier in between
  unsigned bar_target = gridDim.x;
  grid_barrier(a.barrier, bar_target);

  // per-block replicated state (identical in every block: same inputs, same order of operations)
  Mat4 final_t = a.guess;
  double prev_mse = DBL_MAX, cur_mse = DBL_MAX;
  int similar = 0, iterations = 0, state = OPE_CONV_NOT_CONVERGED, converged = 0, n_corr = 0;
  int pass = 0;  // uniform across all threads: selects the partials buffer

  long long t_phase[7] = {0, 0, 0, 0, 0, 0, 0};
  long long t_prev[7] = {0, 0, 0, 0, 0, 0, 0};
  const bool prof_any = a.phase_cycles != nullptr;
  long long n_far = 0;
  const bool prof = a.phase_cycles != nullptr && blockIdx.x == 0 && threadIdx.x == 0;
  for (;; ++pass) {
    long long t0 = prof ? clock64() : 0;
    for (int e = lane; e < kIcpAcc; e += 32) sm->red[warp][e] = 0.0;
    if (threadIdx.x < 2) sm->n_def[threadIdx.x] = 0;
    __syncthreads();
    if (!shooting) {
      // ---- phase A: thread per point, fast path; far queries go to the grid-wide queue ----
      for (int base = lo; base < hi; base += kIcpThreads) {
        const int s = base + (int)threadIdx.x;
        const bool in_range = s < hi;
        float4 p = make_float4(0, 0, 0, 0);
        int sd = -1;
        if (in_range) { p = a.cur_pts[s]; if (pass > 0) sd = __ldcg(a.seed + s); }  // seed/ref may have been written by another SM
        const int orig = __float_as_int(p.w);
        const bool ok = in_range && a.grid.n > 0 && finite3(p.x, p.y, p.z);
        Nn1State nst;
        nst.d1 = FLT_MAX; nst.i1 = 0x7fffffff; nst.s2 = FLT_MAX;
        bool far = false, certified = false;
        int total = 0;  // candidate points in the start nodes of an uncertified query
        unsigned node_mask = 0u;
        if (ok) {
          const float ux = (p.x - a.grid.ox) * a.grid.inv_h, uy = (p.y - a.grid.oy) * a.grid.inv_h, uz = (p.z - a.grid.oz) * a.grid.inv_h;
          if (sd >= 0) {
            const float4 t = __ldg(a.tgt_pts + sd);
            nst.d1 = dist2(p.x, p.y, p.z, t.x, t.y, t.z);
            nst.i1 = sd;
            // certificate of an earlier iteration: every other target point was at least R from the position rf; the point
            // has moved by delta since, so they are at least R - delta away now. If the old neighbour is strictly closer
            // than that (with a margin far above float rounding) it is still THE nearest neighbour: no search.
            const float4 rf = __ldcg(a.ref + s);
            if (rf.w > 0.0f) {
              const float delta = sqrtf(dist2(p.x, p.y, p.z, rf.x, rf.y, rf.z));
              const float d1n = sqrtf(nst.d1);
              certified = (d1n + 2.0f * delta) * 1.00001f + 2e-6f < rf.w;
              // range certificate: the old neighbour and everything else are still beyond the correspondence limit, so the
              // point has no correspondence whatever its exact neighbour is (the gate below rejects d2 > max^2)
              if (!certified && a.max_d2_f < FLT_MAX) {
                const float lim = sqrtf(a.max_d2_f) * 1.00001f + 2e-6f;
                certified = d1n > lim && rf.w - delta > lim;
              }
            }
          } else {
            nn1_probe(a.grid, p.x, p.y, p.z, ux, uy, uz, [&](int b, int e) {
              for (int i = b; i < e; ++i) {
                const float4 c = __ldg(a.grid.pts + i);
                nn1_offer(nst, dist2(p.x, p.y, p.z, c.x, c.y, c.z), __float_as_int(c.w));
              }
            });
            nst.s2 = FLT_MAX;  // the probe only seeds the bound
          }
          if (!certified) {
            // three tiers by the size of the candidate set: direct scan (<= 96 points), this thread's own pruned traversal
            // (<= dfs_max points in the ball's start nodes: every thread works in parallel), the grid-wide warp queue
            float r2 = 0.0f;
            far = !nn1_fast(a.grid, p.x, p.y, p.z, ux, uy, uz, a.max_d2_f, a.cert_gap, nst, &r2, &total, &node_mask);
            if (far && total <= a.dfs_max) {
              nn1_thread_dfs(a.grid, p.x, p.y, p.z, ux, uy, uz, a.max_d2_f, a.cert_gap, nst, &r2);
              far = false;
            }
            if (!far) a.ref[s] = make_float4(p.x, p.y, p.z, sqrtf(fminf(nst.s2, r2)));
          }
        }
        const float best_d2 = nst.d1;
        const int best_i = nst.i1;
        // Deterministic compaction of the far queries into this block's queue segment (filled from the back). A query whose
        // candidate set is huge (e.g. a point near the axis of a cylinder: thousands of near-equidistant neighbours, all of
        // which an exact search must test) is split into one entry per non-empty start node, so that up to eight warps of
        // the grid share it; the entries of one query are adjacent and are merged by the owner after barrier 2.
        int nsub = far ? ((total > a.split_min) ? __popc(node_mask) : 1) : 0;
        for (int attempt = 0; attempt < 2; ++attempt) {
          int incl = nsub;
          for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
          if (lane == 31) sm->warp_cnt[1][warp] = incl;
          __syncthreads();
          int before = sm->n_def[1], block_total = sm->n_def[1];
          for (int w = 0; w < kIcpWarps; ++w) { if (w < warp) before += sm->warp_cnt[1][w]; block_total += sm->warp_cnt[1][w]; }
          __syncthreads();
          if (block_total > hi - lo) { nsub = nsub > 1 ? 1 : nsub; continue; }  // no room for the split entries: one entry per query
          before += incl - nsub;
          if (far) {
            int k = 0;
            for (int j = 0; j < 8; ++j) {
              if (nsub > 1 && !((node_mask >> j) & 1u)) continue;
              if (nsub == 1 && j > 0) break;
              const int slot = hi - 1 - (before + k);
              a.def_q[slot] = make_float4(p.x, p.y, p.z, nst.d1);
              a.def_m[slot] = make_int4(s, nst.i1, orig, nsub > 1 ? j : -1);
              ++k;
            }
          }
          if (threadIdx.x == 0) sm->n_def[1] = block_total;
          break;
        }
        __syncthreads();
        // finish the near queries: gate, rejectors, outputs, moments
        int m = -1;
        float d2 = 0.0f;
        if (ok && !far) {
          const int nn = best_i == 0x7fffffff ? -1 : best_i;
          a.seed[s] = nn;
          d2 = best_d2;
          m = icp_gate(a, s, orig, p, nn, d2);
          a.corr_match[orig] = m;
          a.corr_d2[orig] = d2;
        } else if (in_range && !far) {
          a.seed[s] = -1;
          a.corr_match[orig] = -1;
        }
        if (__ballot_sync(0xffffffffu, m >= 0) != 0u) {  // warp-uniform
          double v[16];
#pragma unroll
          for (int e = 0; e < 16; ++e) v[e] = 0.0;
          double dsum = 0.0;
          if (m >= 0) {
            const float4 t = __ldg(a.tgt_pts + m);
#pragma unroll
            for (int e = 0; e < 16; ++e) v[e] = moment_term(e, p, t, d2, morg);
            dsum = (double)d2;
          }
          int slot;
          const double w = warp_reduce16(v, lane, slot);
          dsum = warp_sum_d(dsum);
          if ((lane & 1) == 0) sm->red[warp][slot] += w;
          if (lane == 1) sm->red[warp][16] += dsum;
        }
        __syncthreads();
      }
      if (threadIdx.x < 2) a.def_count[threadIdx.x * gridDim.x + blockIdx.x] = sm->n_def[threadIdx.x];
      if (prof) { const long long t1 = clock64(); t_phase[0] += t1 - t0; t0 = t1; n_far += sm->n_def[0] + sm->n_def[1]; }
      bar_target += gridDim.x;
      grid_barrier(a.barrier, bar_target);
      if (prof) { const long long t1 = clock64(); t_phase[1] += t1 - t0; t0 = t1; }
      // ---- phase B: all warps of the grid drain the queue, one far query per warp ----
      if (warp < 2) {  // inclusive prefixes of the per-block counts (gridDim <= kIcpMaxBlocks): warp 0 small, warp 1 large
        int run = 0;
        for (int b0 = 0; b0 < (int)gridDim.x; b0 += 32) {
          const int b = b0 + lane;
          int c = b < (int)gridDim.x ? __ldcg(a.def_count + warp * gridDim.x + b) : 0;
          for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, c, o); if (lane >= o) c += t; }
          if (b < (int)gridDim.x) sm->prefix[warp][b] = run + c;
          run += __shfl_sync(0xffffffffu, c, 31);
        }
      }
      __syncthreads();
      if (blockIdx.x == 0 && threadIdx.x < 2) a.def_head[((pass + 1) & 1) * 2 + threadIdx.x] = 0;  // nobody touches the other parity before barrier 3
      // Groups claim far queries one at a time — whoever is free takes the next; a result does not depend on who computed
      // it. Large queries first, one per WARP; then the small ones, one per OCTET (64 dependent chains in flight per SM).
      {
        const int total_l = sm->prefix[1][gridDim.x - 1];
        int* head = a.def_head + (pass & 1) * 2 + 1;
        OctStack* stw = &sm->wstack[warp];
        LeafList* llw = &sm->leaves[warp];
        for (;;) {
          int e = 0;
          if (lane == 0) e = atomicAdd(head, 1);
          e = __shfl_sync(0xffffffffu, e, 0);
          if (e >= total_l) break;
          int bl = 0, br = (int)gridDim.x - 1;  // first block whose inclusive prefix exceeds e
          while (bl < br) { const int mid = (bl + br) >> 1; if (sm->prefix[1][mid] > e) br = mid; else bl = mid + 1; }
          const int j = e - (bl > 0 ? sm->prefix[1][bl - 1] : 0);
          const int slot = min(a.n_work, min(a.n_work, bl * chunk) + chunk) - 1 - j;
          const float4 q = __ldcg(a.def_q + slot);
          const int4 qm = __ldcg(a.def_m + slot);
          Nn1State nst;
          nst.d1 = q.w; nst.i1 = qm.y; nst.s2 = FLT_MAX;
          float r2 = 0.0f;
          const long long q0 = prof_any ? clock64() : 0;
          unsigned long long* cnt = (prof_any && pass < 64) ? (unsigned long long*)(a.phase_cycles + 16 + 64 * 8 + 64 + pass * 4) : nullptr;
          if (pass == 0) coop_nn1_far<32, true>(a.grid, fdir, stw, llw, q.x, q.y, q.z, a.max_d2_f, a.cert_gap, nst, &r2, cnt, qm.w);
          else coop_nn1_far<32, false>(a.grid, fdir, stw, llw, q.x, q.y, q.z, a.max_d2_f, a.cert_gap, nst, &r2, cnt, qm.w);
          if (prof_any && lane == 0 && pass < 64) {
            atomicMax((unsigned long long*)(a.phase_cycles + 16 + pass * 8 + 7), (unsigned long long)(clock64() - q0));
            atomicAdd((unsigned long long*)(a.phase_cycles + 16 + 64 * 8 + pass), 1ull);
          }
          if (lane == 0) a.def_res[slot] = make_float4(nst.d1, __int_as_float(nst.i1), nst.s2, r2);
          __syncwarp();
        }
      }
      if (prof) { const long long t1 = clock64(); t_phase[2] += t1 - t0; t0 = t1; }
      bar_target += gridDim.x;
      grid_barrier(a.barrier, bar_target);
      if (prof) { const long long t1 = clock64(); t_phase[3] += t1 - t0; t0 = t1; }
      // ---- this block's own far queries, in queue order (deterministic whoever searched them): merge the entries of a
      //      split query, gate, write neighbour / certificate / correspondence, accumulate the moments ----
      {
        const int n_def = sm->n_def[1];
        for (int base = 0; base < n_def; base += kIcpThreads) {
          const int j = base + (int)threadIdx.x;
          int m = -1;
          float d2 = 0.0f;
          float4 p = make_float4(0, 0, 0, 0);
          if (j < n_def) {
            const int qslot = hi - 1 - j;
            const int4 qm = a.def_m[qslot];
            const bool first = j == 0 || a.def_m[qslot + 1].x != qm.x;   // entries of one query are adjacent
            if (first) {
              p = a.def_q[qslot];
              Nn1State nst;
              nst.d1 = FLT_MAX; nst.i1 = 0x7fffffff; nst.s2 = FLT_MAX;
              float r2 = FLT_MAX;
              for (int k = 0; k < 8 && j + k < n_def; ++k) {
                if (k > 0 && a.def_m[qslot - k].x != qm.x) break;
                const float4 r = __ldcg(a.def_res + (qslot - k));
                const float rd1 = r.x, rs2 = r.z;
                const int ri1 = __float_as_int(r.y);
                r2 = fminf(r2, r.w);
                if (ri1 == nst.i1) { nst.s2 = fminf(nst.s2, rs2); continue; }   // the shared seed survived in several entries
                if (nb_less(rd1, ri1, nst.d1, nst.i1)) { nst.s2 = fminf(fminf(nst.s2, rs2), nst.d1); nst.d1 = rd1; nst.i1 = ri1; }
                else nst.s2 = fminf(fminf(nst.s2, rs2), rd1);
              }
              const int nn = nst.i1 == 0x7fffffff ? -1 : nst.i1;
              d2 = nst.d1;
              m = icp_gate(a, qm.x, qm.z, p, nn, d2);
              a.seed[qm.x] = nn; a.corr_match[qm.z] = m; a.corr_d2[qm.z] = d2;
              a.ref[qm.x] = make_float4(p.x, p.y, p.z, sqrtf(fminf(nst.s2, r2)));
            }
          }
          if (__ballot_sync(0xffffffffu, m >= 0) != 0u) {
            double v[16];
#pragma unroll
            for (int e = 0; e < 16; ++e) v[e] = 0.0;
            double dsum = 0.0;
            if (m >= 0) {
              const float4 t = __ldg(a.tgt_pts + m);
#pragma unroll
              for (int e = 0; e < 16; ++e) v[e] = moment_term(e, p, t, d2, morg);
              dsum = (double)d2;
            }
            int slot;
            const double w = warp_reduce16(v, lane, slot);
            dsum = warp_sum_d(dsum);
            if ((lane & 1) == 0) sm->red[warp][slot] += w;
            if (lane == 1) sm->red[warp][16] += dsum;
          }
        }
      }
      if (prof) { const long long t1 = clock64(); t_phase[4] += t1 - t0; t0 = t1; }
    } else {
      for (int s = wlo; s < whi; ++s) {  // one warp per source point
        const float4 p = a.cur_pts[s];
        const int orig = __float_as_int(p.w);
        float d2 = 0.0f;
        const int m = icp_correspond_shooting(a, st, s, orig, p, pass > 0, d2, tg_smem, sm->knn_buf[warp]);
        if (lane == 0) { a.corr_match[orig] = m; a.corr_d2[orig] = d2; }
        if (m >= 0 && lane < kIcpAcc) {
          const float4 t = tg_smem ? tg_smem[m] : __ldg(a.tgt_pts + m);
          sm->red[warp][lane] += moment_term(lane, p, t, d2, morg);
        }
        __syncwarp();
      }
      if (prof) { const long long t1 = clock64(); t_phase[0] += t1 - t0; t0 = t1; }
    }
    __syncthreads();
    double* my_partials = a.partials + ((size_t)(pass & 1) * gridDim.x + blockIdx.x) * kIcpAcc;
    if (threadIdx.x < kIcpAcc) {
      double sum = 0.0;
#pragma unroll
      for (int w = 0; w < kIcpWarps; ++w) sum += sm->red[w][threadIdx.x];
      my_partials[threadIdx.x] = sum;
    }
    bar_target += gridDim.x;
    grid_barrier(a.barrier, bar_target);
    if (prof) { const long long t1 = clock64(); t_phase[4] += t1 - t0; t0 = t1; }
    // ---- phase C: every block reduces all partials in the same order (warp per accumulator, lanes over blocks) ----
    for (int e = warp; e < kIcpAcc; e += kIcpWarps) {
      const double* base = a.partials + (size_t)(pass & 1) * gridDim.x * kIcpAcc;
      double sum = 0.0;
      for (int b0 = lane; b0 < (int)gridDim.x; b0 += 32 * 8) {   // 8 independent loads in flight, summed in block order
        double v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) { const int b = b0 + 32 * k; v[k] = b < (int)gridDim.x ? __ldcg(base + (size_t)b * kIcpAcc + e) : 0.0; }
#pragma unroll
        for (int k = 0; k < 8; ++k) sum += v[k];
      }
      sum = warp_sum_d(sum);
      if (lane == 0) sm->totals[e] = sum;
    }
    __syncthreads();
    if (warp == 0) {
      int stop = 0;
      n_corr = (int)sm->totals[0];
      if (n_corr < a.min_corr) {
        state = OPE_CONV_NO_CORRESPONDENCES; converged = 0; stop = 2;  // VP/impl/icp_mod.hpp:232-240
        if (lane == 0) sm->T_inc = mat4_identity();
      } else {
        // Umeyama prelude, one division per lane (same arithmetic as ope::umeyama_from_moments)
        const double n = sm->totals[0];
        double mean = 0.0;
        if (lane < 6) mean = sm->totals[1 + lane] / n;  // lanes 0-2: source mean, 3-5: target mean
        double ms[3], mt[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) { ms[k] = __shfl_sync(0xffffffffu, mean, k); mt[k] = __shfl_sync(0xffffffffu, mean, 3 + k); }
        float sg = 0.0f;
        if (lane < 9) {
          const int c = lane / 3, r = lane % 3;
          const double msc = c == 0 ? ms[0] : (c == 1 ? ms[1] : ms[2]);
          const double mtr = r == 0 ? mt[0] : (r == 1 ? mt[1] : mt[2]);
          sg = (float)(sm->totals[7 + lane] / n - mtr * msc);
        }
        float sigma[9];
#pragma unroll
        for (int k = 0; k < 9; ++k) sigma[k] = __shfl_sync(0xffffffffu, sg, k);
        if (lane == 0) {
          Mat4 T;
          const double msu[3] = {ms[0] + morg[0], ms[1] + morg[1], ms[2] + morg[2]};   // the moments are relative to morg
          const double mtu[3] = {mt[0] + morg[0], mt[1] + morg[1], mt[2] + morg[2]};
          umeyama_from_sigma_means(sigma, msu, mtu, T);
          sm->T_inc = T;
          final_t = mat4_mul(T, final_t);
          ++iterations;
          // DefaultConvergenceCriteria::hasConverged (SURVEY A.8)
          state = OPE_CONV_NOT_CONVERGED;
          int conv = 0;
          if (iterations >= a.max_iterations) {
            if (!a.fail_after_max) { state = OPE_CONV_ITERATIONS; conv = 1; }
            else { conv = 0; stop = 1; }
          } else {
            const double cos_angle = 0.5 * (double)(T(0, 0) + T(1, 1) + T(2, 2) - 1);
            const double translation_sqr = (double)(T(0, 3) * T(0, 3) + T(1, 3) * T(1, 3) + T(2, 3) * T(2, 3));
            int hit = 0, hit_state = 0;
            if (cos_angle >= a.rot_thr && translation_sqr <= a.trans_thr) { hit = 1; hit_state = OPE_CONV_TRANSFORM; }
            else {
              cur_mse = sm->totals[16] / (double)n_corr;
              if (fabs(cur_mse - prev_mse) < a.abs_mse_thr) { hit = 1; hit_state = OPE_CONV_ABS_MSE; }
              else if (fabs(cur_mse - prev_mse) / prev_mse < a.rel_mse_thr) { hit = 1; hit_state = OPE_CONV_REL_MSE; }
              else prev_mse = cur_mse;
            }
            if (hit) {
              if (similar < a.max_similar) ++similar;
              else { similar = 0; state = hit_state; conv = 1; }
            }
          }
          converged = conv;
          if (a.force_all && iterations < a.max_iterations) conv = 0;
          if (conv) stop = 1;
        }
      }
      if (lane == 0) sm->stop = stop;
    }
    __syncthreads();
    if (prof) { const long long t1 = clock64(); t_phase[5] += t1 - t0; t0 = t1; }
    // ---- transformCloud(input_transformed, transformation_), own points only ----
    const int stop = sm->stop;
    if (stop != 2) {
      const Mat4 T = sm->T_inc;
      if (!shooting) { for (int s = lo + (int)threadIdx.x; s < hi; s += kIcpThreads) icp_move(a, T, s); }
      else { for (int s = wlo + lane; s < whi; s += 32) icp_move(a, T, s); __syncwarp(); }
    }
    if (prof) {
      const long long t1 = clock64(); t_phase[6] += t1 - t0;
      if (pass < 64) for (int k = 0; k < 7; ++k) { a.phase_cycles[16 + pass * 8 + k] = t_phase[k] - t_prev[k]; t_prev[k] = t_phase[k]; }
    }
    if (stop) break;
  }
  if (prof) {
    for (int i = 0; i < 7; ++i) a.phase_cycles[i] = t_phase[i];
    a.phase_cycles[7] = n_far;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    ope_reg_result r;
    for (int i = 0; i < 16; ++i) r.T[i] = final_t.m[i];
    r.converged = converged; r.state = state; r.iterations = iterations; r.n_correspondences = n_corr;
    r.last_mse = cur_mse; r.best_error = 0.0; r.best_iteration = 0; r.reserved = 0;
    *a.result = r;
  }
}

// ================================================================ ICP, small clouds: one source point per THREAD ====
// The DetectAndLocalize fine stage (normal shooting, k = 20) works on ~2 k source points against a ~1.5 k point cluster. The
// kernel above gives every such query a whole warp and the whole GPU to one alignment; this one keeps the target in shared
// memory and gives every query ONE thread, so an alignment needs ceil(n / 256) blocks (8 SMs instead of 118) and a batch of
// independent frames (ope_pose_batch) fills the device with concurrent alignments.
//   per iteration and thread: bound = largest distance to the previous iteration's k neighbours (tight: they are still the k
//   nearest for almost every point) -> one pass over the target in shared memory (broadcast reads) collecting the points within
//   the bound into the thread's column of a shared slab -> all-against-all ranks of those ~k candidates ((d2, index) order, so
//   the list equals FLANN's) -> point-to-line distances of the k best in double, first minimum in list order -> rejectors ->
//   double moments, transpose-reduced per warp, summed per block, exchanged through a B-entry table and one grid barrier.
//   The rare query whose bound admits more than kSlabSlots points, and the first (unseeded) iteration, use the cooperative
//   warp_knn_smem for that query. Same results as icp_kernel (parity tests run both).
static constexpr int kSlabSlots = 32;
// A block keeps its alignment's target (points + group boxes) in shared memory next to 256 bytes of candidate slots per thread,
// so wider blocks share one target copy among more warps: 2 x 256 threads fit an SM where 3 x 128 do (16 resident warps instead
// of 12 of this latency-bound kernel). Up to 16 blocks: 4 096 source points.
static constexpr int kIcpSmallThreads = 256;
static constexpr int kIcpSmallMaxBlocks = 16;
// A thread's column of the candidate slab (entries THREADS apart) as a binary max-heap in (d2, index) order: v sinks from node i
// of a heap of n entries.
template <int THREADS>
__device__ __forceinline__ void heap_sift(float2* column, int i, float2 v, const int n) {
  for (;;) {
    const int l = 2 * i + 1;
    if (l >= n) break;
    float2 cv = column[l * THREADS];
    int pick = l;
    if (l + 1 < n) {
      const float2 cr = column[(l + 1) * THREADS];
      if (nb_less(cv.x, __float_as_int(cv.y), cr.x, __float_as_int(cr.y))) { cv = cr; pick = l + 1; }
    }
    if (!nb_less(v.x, __float_as_int(v.y), cv.x, __float_as_int(cv.y))) break;
    column[i * THREADS] = cv;
    i = pick;
  }
  column[i * THREADS] = v;
}

template <int THREADS>
struct IcpSmallSmem {
  double red[THREADS / 32][kIcpAcc];
  double totals[kIcpAcc];
  float2 knn_buf[THREADS / 32][kKnnBufCap + 32];   // warp_knn_smem_bounded scratch for the queries the thread-level scan hands over
  float4 wbox[THREADS / 32][2];                    // box around a warp's queries (.w of [0]: the widest bound among them, inflated)
  Mat4 T_inc;
  int stop;
};

// bid / nblk: this block's index among the nblk blocks of ITS alignment (the whole grid for a single alignment, one frame's share
// of a frame-spanning launch)
template <int THREADS>
__device__ __forceinline__ void icp_small_body(const IcpDev& a, const int bid, const int nblk) {
  constexpr int kIcpThreads = THREADS, kIcpWarps = THREADS / 32;   // shadow the wide kernel's constants inside this kernel
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double morg[3];   // origin of the moment accumulation: the target's first point (ope::umeyama_from_moments)
  { const float4 t0 = a.n_tgt > 0 ? __ldg(a.tgt_pts) : make_float4(0, 0, 0, 0); moment_origin(t0.x, t0.y, t0.z, morg[0], morg[1], morg[2]); }
  IcpSmallSmem<THREADS>* sm = reinterpret_cast<IcpSmallSmem<THREADS>*>(smem_raw);
  float4* tg = reinterpret_cast<float4*>(smem_raw + ((sizeof(IcpSmallSmem<THREADS>) + 15) & ~(size_t)15));
  const int n_tgt8 = (a.n_tgt + 7) & ~7, n_groups = n_tgt8 >> 3;   // the target in groups of 8 consecutive points, padded with +inf
  float4* blo = tg + n_tgt8;                                        // bounding box of every group (culling)
  float4* bhi = blo + n_groups;
  float2* slab = reinterpret_cast<float2*>(bhi + n_groups);         // [kSlabSlots][kIcpThreads]: column = thread
  const unsigned full = 0xffffffffu;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int s = bid * kIcpThreads + tid;    // this thread's point (sorted position)
  const bool in_range = s < a.n_work;
  const bool stale = a.variant == OPE_ICP_VARIANT_MODCORR;
  const int k = a.k_search < a.grid.n ? a.k_search : a.grid.n;
  auto col = [&](int slot) -> float2& { return slab[slot * kIcpThreads + tid]; };

  // input_transformed = guess applied to input (VP/impl/icp_mod.hpp:132-139), in sorted order; state lives in registers
  float4 p = make_float4(0, 0, 0, 0), nv = make_float4(0, 0, 0, 0);
  int orig = 0;
  if (in_range) {
    p = __ldg(a.src_sorted + s);
    orig = __float_as_int(p.w);
    if (a.src0_nrm) nv = __ldg(a.src0_nrm + orig);
    if (!mat4_is_identity(a.guess)) {
      float x, y, z;
      xform_point(a.guess, p.x, p.y, p.z, x, y, z);
      p.x = x; p.y = y; p.z = z;
      if (a.src0_nrm && finite3(nv.x, nv.y, nv.z)) { xform_normal(a.guess, nv.x, nv.y, nv.z, x, y, z); nv.x = x; nv.y = y; nv.z = z; }
    }
  }
  for (int j = tid; j < n_tgt8; j += kIcpThreads) tg[j] = j < a.n_tgt ? __ldg(a.tgt_pts + j) : make_float4(INFINITY, INFINITY, INFINITY, 0.0f);
  __syncthreads();
  // A down-sampled cluster arrives in voxel-key order (x fastest), so eight consecutive points are neighbours: their box is small
  // and most groups are farther from a query than its bound. Non-finite points never match and stay out of the boxes.
  for (int g = tid; g < n_groups; g += kIcpThreads) {
    float4 lo = make_float4(INFINITY, INFINITY, INFINITY, 0.0f), hi = make_float4(-INFINITY, -INFINITY, -INFINITY, 0.0f);
    for (int u = 0; u < 8; ++u) {
      const float4 t = tg[8 * g + u];
      if (!finite3(t.x, t.y, t.z)) continue;
      lo.x = fminf(lo.x, t.x); lo.y = fminf(lo.y, t.y); lo.z = fminf(lo.z, t.z);
      hi.x = fmaxf(hi.x, t.x); hi.y = fmaxf(hi.y, t.y); hi.z = fmaxf(hi.z, t.z);
    }
    blo[g] = lo; bhi[g] = hi;
  }
  __syncthreads();
  const bool ok = in_range && k > 0 && finite3(p.x, p.y, p.z);

  Mat4 final_t = a.guess;
  double prev_mse = DBL_MAX, cur_mse = DBL_MAX;
  int similar = 0, iterations = 0, state = OPE_CONV_NOT_CONVERGED, converged = 0, n_corr = 0;
  unsigned bar_target = 0;
  const bool prof = a.phase_cycles != nullptr && bid == 0 && tid == 0;
  long long t_phase[4] = {0, 0, 0, 0};

  // one query through the cooperative scan: the warp serves lane `q`'s point, the sorted result goes to that thread's column
  auto coop_query = [&](int q, float bound) {
    const float qx = __shfl_sync(full, p.x, q), qy = __shfl_sync(full, p.y, q), qz = __shfl_sync(full, p.z, q);
    float ld; int li;
    const int cnt = warp_knn_smem_bounded(tg, a.n_tgt, a.grid.n, true, qx, qy, qz, a.k_search, bound, sm->knn_buf[warp], ld, li);
    float2* c = slab + (warp * 32 + q);
    if (lane < kSlabSlots) c[lane * kIcpThreads] = lane < cnt ? make_float2(ld, __int_as_float(li)) : make_float2(FLT_MAX, __int_as_float(-1));
    return cnt;
  };

  for (int pass = 0;; ++pass) {
    long long t0 = prof ? clock64() : 0;
    int c = 0;           // entries in this thread's column
    bool have = false;   // the column already holds this iteration's k nearest
    bool seeded = pass > 0;
    if (pass == 0) {
      // Unseeded start: every eighth thread (a "leader") gets an exact cooperative search; its neighbours in Morton order are
      // spatially close, and ANY k distinct target points bound a query's k-th distance, so the other seven seed their bound
      // from the leader's list.
      const bool leader = (lane & 7) == 0;
      const unsigned lead = __ballot_sync(full, ok && leader);
      for (unsigned m = lead; m != 0u; m &= m - 1u) { const int q = __ffs(m) - 1; const int cnt = coop_query(q, FLT_MAX); if (lane == q) { c = cnt; have = true; } }
      __syncwarp();
      seeded = !leader && ((lead >> (lane & ~7)) & 1u);
    }
    float bound = FLT_MAX;
    if (ok && !have && seeded) {
      // the previous iteration's (pass 0: the leader's) k nearest, at this point's position, bound its k-th distance
      const float2* seed_col = slab + (pass == 0 ? (tid & ~7) : tid);
      float b = 0.0f;
      bool all = true;
#pragma unroll 4
      for (int j = 0; j < k; ++j) {
        const int idx = __float_as_int(seed_col[j * kIcpThreads].y);
        if (idx < 0) { all = false; continue; }
        const float4 t = tg[idx];
        b = fmaxf(b, dist2(p.x, p.y, p.z, t.x, t.y, t.z));
      }
      if (all) bound = b;
    }
    if (pass == 0) __syncwarp();   // the leaders' columns are read above, the others' columns are written below
    const bool scan = ok && !have && bound < FLT_MAX;
    int n_ins = 0;   // profile: calls of the overflow path
    bool heaped = false;                      // the column is full and ordered as a max-heap (see insert_full)
    float2 root = make_float2(0.0f, 0.0f);    // its root
    const long long ts0 = a.phase_cycles ? clock64() : 0;
    if (__any_sync(full, scan)) {
      // A full column (kSlabSlots entries) keeps the best kSlabSlots seen so far as a max-heap in (d2, index) order — root = slot 0
      // = the worst entry, cached in registers — and the bound shrinks to the root: log2(kSlabSlots) steps per replacement. Common
      // only in the first iterations (a seed from a neighbour's list, large increments), where it used to dominate the time.
      auto insert_full = [&](float d2, int j) {
        ++n_ins;
        if (!heaped) {
          for (int i = kSlabSlots / 2 - 1; i >= 0; --i) heap_sift<THREADS>(slab + tid, i, col(i), kSlabSlots);
          heaped = true;
          root = col(0);
          bound = root.x;   // every entry was admitted under a bound that has only shrunk to the largest entry since
        }
        if (nb_less(d2, j, root.x, __float_as_int(root.y))) {
          heap_sift<THREADS>(slab + tid, 0, make_float2(d2, __int_as_float(j)), kSlabSlots);
          root = col(0);
          bound = root.x;
        }
      };
      // The warp's 32 queries are neighbours on the Morton curve: the box around them, grown by the widest bound among them, is
      // tested against the group boxes by the warp together (one group per lane, 32 per step); only the groups that pass — a
      // third of them — reach the per-thread test below. Conservative comparisons throughout: a float box distance can only be
      // a rounding error above the float distance to a point inside the box.
      float wlx = scan ? p.x : INFINITY, wly = scan ? p.y : INFINITY, wlz = scan ? p.z : INFINITY;
      float whx = scan ? p.x : -INFINITY, why = scan ? p.y : -INFINITY, whz = scan ? p.z : -INFINITY;
      float wb = scan ? bound : 0.0f;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        wlx = fminf(wlx, __shfl_xor_sync(full, wlx, o)); wly = fminf(wly, __shfl_xor_sync(full, wly, o)); wlz = fminf(wlz, __shfl_xor_sync(full, wlz, o));
        whx = fmaxf(whx, __shfl_xor_sync(full, whx, o)); why = fmaxf(why, __shfl_xor_sync(full, why, o)); whz = fmaxf(whz, __shfl_xor_sync(full, whz, o));
        wb = fmaxf(wb, __shfl_xor_sync(full, wb, o));
      }
      if (lane == 0) { sm->wbox[warp][0] = make_float4(wlx, wly, wlz, wb * 1.0002f + 1e-30f); sm->wbox[warp][1] = make_float4(whx, why, whz, 0.0f); }
      __syncwarp();
      for (int g0 = 0; g0 < n_groups; g0 += 32) {
        bool near = false;
        if (g0 + lane < n_groups) {
          const float4 lo = blo[g0 + lane], hi = bhi[g0 + lane], wl = sm->wbox[warp][0], wh = sm->wbox[warp][1];
          const float ex = fmaxf(fmaxf(lo.x - wh.x, wl.x - hi.x), 0.0f), ey = fmaxf(fmaxf(lo.y - wh.y, wl.y - hi.y), 0.0f),
                      ez = fmaxf(fmaxf(lo.z - wh.z, wl.z - hi.z), 0.0f);
          near = ex * ex + ey * ey + ez * ez <= wl.w;
        }
        // eight targets per step: the loads (same address in every lane: broadcasts) and the distance arithmetic of a step are
        // independent of each other and of the slab stores, which only happen for the ~k hits of the whole scan
        for (unsigned cand = __ballot_sync(full, near); cand != 0u; cand &= cand - 1u) {
          const int g = g0 + __ffs(cand) - 1;
          const int j0 = 8 * g;
          bool mine = scan;
          if (mine) {   // squared distance to the group's box, conservatively compared (the float evaluation may round either way)
            const float4 lo = blo[g], hi = bhi[g];
            const float ex = fmaxf(fmaxf(lo.x - p.x, p.x - hi.x), 0.0f), ey = fmaxf(fmaxf(lo.y - p.y, p.y - hi.y), 0.0f),
                        ez = fmaxf(fmaxf(lo.z - p.z, p.z - hi.z), 0.0f);
            mine = ex * ex + ey * ey + ez * ez <= bound * 1.0001f + 1e-30f;
          }
          if (!mine) continue;
          float d2[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) { const float4 t = tg[j0 + u]; d2[u] = dist2(p.x, p.y, p.z, t.x, t.y, t.z); }
          unsigned hit = 0u;
#pragma unroll
          for (int u = 0; u < 8; ++u) hit |= (d2[u] <= bound ? 1u : 0u) << u;   // non-finite targets give inf / NaN: never a hit
          if (hit == 0u) continue;
          if (c + __popc(hit) <= kSlabSlots) {
#pragma unroll
            for (int u = 0; u < 8; ++u)   // predicated stores, no nested branches: the lanes of a warp hit at different u
              if ((hit >> u) & 1u) { col(c) = make_float2(d2[u], __int_as_float(j0 + u)); ++c; }
          } else {
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              const bool h = (hit >> u) & 1u;
              const bool room = c < kSlabSlots;
              if (h & room) col(c) = make_float2(d2[u], __int_as_float(j0 + u));
              if (h & !room) insert_full(d2[u], j0 + u);
              c += (h & room) ? 1 : 0;
            }
          }
        }
      }
    }
    // whoever could not be served above (no usable seed, or fewer than k points within the bound) gets a cooperative search
    const bool unserved = ok && !have && (!scan || c < k);
    const unsigned redo = __ballot_sync(full, unserved);
    if (a.phase_cycles && pass < 64) {
      unsigned long long* pc = (unsigned long long*)(a.phase_cycles + 16 + pass * 8);
      const unsigned long long dt = (unsigned long long)(clock64() - ts0);
      if (lane == 0) { atomicAdd(pc + 0, dt); atomicMax(pc + 1, dt); atomicAdd(pc + 5, 1ull); }
      if (n_ins > 0) { atomicAdd(pc + 2, (unsigned long long)n_ins); atomicAdd(pc + 3, 1ull); }
      if (ok) atomicAdd(pc + 4, (unsigned long long)c);
    }
    if (a.phase_cycles && bid == 0 && lane == 0 && pass > 0) atomicAdd((unsigned long long*)&a.phase_cycles[4], (unsigned long long)__popc(redo));
    if (a.phase_cycles && bid == 0 && ok && pass > 0) atomicAdd((unsigned long long*)&a.phase_cycles[5], (unsigned long long)c);
    for (unsigned m = redo; m != 0u; m &= m - 1u) {
      const int q = __ffs(m) - 1;
      const float bq = __shfl_sync(full, scan ? bound : FLT_MAX, q);
      const int cnt = coop_query(q, bq);
      if (lane == q) c = cnt;
    }
    __syncwarp();
    if (prof) { const long long t1 = clock64(); t_phase[0] += t1 - t0; t0 = t1; }
    // ---- ranks, normal shooting among the k best, compaction of the k best into slots [0, k) ----
    int match = -1;
    float d2m = 0.0f;
    if (ok && c > 0) {
      const float4 nr = stale ? __ldg(a.src0_nrm + orig) : nv;
      const double N0 = nr.x, N1 = nr.y, N2 = nr.z;
      double best = DBL_MAX;
      int best_idx = -1, first_idx = -1;
      float best_d2 = 0.0f, first_d2 = 0.0f;
      // The list order of the reference is ascending (d2, index). Nothing below needs the ranks themselves: the k best are what
      // remains after dropping the largest entry c - k times (c - k is 0 or 1 for almost every query), the nearest neighbour
      // is the minimum, and "first minimum in list order" is a tie-break by that same order.
      while (heaped && c > k) {   // pop the root: the last entry sinks from the top
        --c;
        if (c > 0) heap_sift<THREADS>(slab + tid, 0, col(c), c);
      }
      while (c > k) {
        int worst = 0;
        float2 wv = col(0);
        for (int e = 1; e < c; ++e) { const float2 o = col(e); if (nb_less(wv.x, __float_as_int(wv.y), o.x, __float_as_int(o.y))) { wv = o; worst = e; } }
        --c;
        if (worst != c) col(worst) = col(c);
      }
      float best_key = 0.0f;   // d2 of the current winner (its index is best_idx): the list-order key for ties
#pragma unroll 4
      for (int e = 0; e < c; ++e) {
        const float2 mine = col(e);
        const int mi = __float_as_int(mine.y);
        if (first_idx < 0 || nb_less(mine.x, mi, first_d2, first_idx)) { first_idx = mi; first_d2 = mine.x; }
        const float4 t = tg[mi];
        const float px = t.x - p.x, py = t.y - p.y, pz = t.z - p.z;
        const double V0 = px, V1 = py, V2 = pz;
        const double C0 = N1 * V2 - N2 * V1, C1 = N2 * V0 - N0 * V2, C2 = N0 * V1 - N1 * V0;
        const double dist = C0 * C0 + C1 * C1 + C2 * C2;
        if (dist < DBL_MAX && (dist < best || (dist == best && nb_less(mine.x, mi, best_key, best_idx)))) {
          best = dist; best_idx = mi; best_d2 = mine.x; best_key = mine.x;
        }
      }
      // the reference starts from min_index = 0: with no finite candidate it still reports neighbour 0 unless rejected below
      const int pick_idx = best_idx < 0 ? first_idx : best_idx;
      const float pick_d2 = best_idx < 0 ? first_d2 : best_d2;
      const double min_dist = best_idx < 0 ? DBL_MAX : best;
      if (!(min_dist > a.max_corr_dist)) { match = pick_idx; d2m = pick_d2; }   // sic (SURVEY A.8)
      // rejector chain (VP/impl/icp_mod.hpp:194-208) on register state
      for (int r = 0; r < a.n_rej && match >= 0; ++r) {
        const float4 sn = stale ? __ldg(a.src0_nrm + orig) : nv;
        double score;
        if (a.rej_kind[r] == OPE_REJ_SURFACE_NORMAL) {
          const float4 tn = __ldg(a.tgt_nrm + match);
          score = (double)((sn.x * tn.x) + (sn.y * tn.y) + (sn.z * tn.z));
        } else {
          const float4 sp = stale ? __ldg(a.src0_pts + orig) : p;
          const double sl = (double)sqrtf(sp.x * sp.x + sp.y * sp.y + sp.z * sp.z);
          score = (double)((sn.x * (-sp.x / sl)) + (sn.y * (-sp.y / sl)) + (sn.z * (-sp.z / sl)));
        }
        if (!(score > a.rej_thr[r])) match = -1;
      }
    }
    // slots [c, k) of a short list are invalid for the next bound
    if (ok) for (int j = (c < k ? c : k); j < k; ++j) col(j) = make_float2(FLT_MAX, __int_as_float(-1));
    if (in_range) { a.corr_match[orig] = match; a.corr_d2[orig] = d2m; }
    if (prof) { const long long t1 = clock64(); t_phase[1] += t1 - t0; t0 = t1; }
    // ---- moments: warp transpose reduction -> block -> table of B partials -> barrier ----
    {
      double v[16];
#pragma unroll
      for (int e = 0; e < 16; ++e) v[e] = 0.0;
      double dsum = 0.0;
      if (match >= 0) {
        const float4 t = tg[match];
#pragma unroll
        for (int e = 0; e < 16; ++e) v[e] = moment_term(e, p, t, d2m, morg);
        dsum = (double)d2m;
      }
      int slot;
      const double wsum = warp_reduce16(v, lane, slot);
      dsum = warp_sum_d(dsum);
      if ((lane & 1) == 0) sm->red[warp][slot] = wsum;
      if (lane == 1) sm->red[warp][16] = dsum;
    }
    __syncthreads();
    double* my_partials = a.partials + ((size_t)(pass & 1) * nblk + bid) * kIcpAcc;
    if (tid < kIcpAcc) {
      double sum = 0.0;
#pragma unroll
      for (int wv = 0; wv < kIcpWarps; ++wv) sum += sm->red[wv][tid];
      my_partials[tid] = sum;
    }
    if (nblk > 1) { bar_target += nblk; grid_barrier(a.barrier, bar_target); } else __syncthreads();
    if (tid < kIcpAcc) {
      const double* base = a.partials + (size_t)(pass & 1) * nblk * kIcpAcc;
      double sum = 0.0;
      for (int b0 = 0; b0 < nblk; b0 += 8) {   // 8 independent loads in flight, summed in block order
        double v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = b0 + u < nblk ? __ldcg(base + (size_t)(b0 + u) * kIcpAcc + tid) : 0.0;
#pragma unroll
        for (int u = 0; u < 8; ++u) sum += v[u];
      }
      sm->totals[tid] = sum;
    }
    __syncthreads();
    if (prof) { const long long t1 = clock64(); t_phase[2] += t1 - t0; t0 = t1; }
    // ---- Umeyama + DefaultConvergenceCriteria, replicated in every block (thread 0) ----
    if (tid == 0) {
      int stop = 0;
      n_corr = (int)sm->totals[0];
      if (n_corr < a.min_corr) {
        state = OPE_CONV_NO_CORRESPONDENCES; converged = 0; stop = 2;   // VP/impl/icp_mod.hpp:232-240
        sm->T_inc = mat4_identity();
      } else {
        Mat4 T;
        umeyama_from_moments(sm->totals, T, morg[0], morg[1], morg[2]);
        sm->T_inc = T;
        final_t = mat4_mul(T, final_t);
        ++iterations;
        state = OPE_CONV_NOT_CONVERGED;
        int conv = 0;
        if (iterations >= a.max_iterations) {
          if (!a.fail_after_max) { state = OPE_CONV_ITERATIONS; conv = 1; }
          else { conv = 0; stop = 1; }
        } else {
          const double cos_angle = 0.5 * (double)(T(0, 0) + T(1, 1) + T(2, 2) - 1);
          const double translation_sqr = (double)(T(0, 3) * T(0, 3) + T(1, 3) * T(1, 3) + T(2, 3) * T(2, 3));
          int hit = 0, hit_state = 0;
          if (cos_angle >= a.rot_thr && translation_sqr <= a.trans_thr) { hit = 1; hit_state = OPE_CONV_TRANSFORM; }
          else {
            cur_mse = sm->totals[16] / (double)n_corr;
            if (fabs(cur_mse - prev_mse) < a.abs_mse_thr) { hit = 1; hit_state = OPE_CONV_ABS_MSE; }
            else if (fabs(cur_mse - prev_mse) / prev_mse < a.rel_mse_thr) { hit = 1; hit_state = OPE_CONV_REL_MSE; }
            else prev_mse = cur_mse;
          }
          if (hit) {
            if (similar < a.max_similar) ++similar;
            else { similar = 0; state = hit_state; conv = 1; }
          }
        }
        converged = conv;
        if (a.force_all && iterations < a.max_iterations) conv = 0;
        if (conv) stop = 1;
      }
      sm->stop = stop;
    }
    __syncthreads();
    // ---- transformCloud(input_transformed, transformation_) on the registers ----
    const int stop = sm->stop;
    if (stop != 2 && in_range && finite3(p.x, p.y, p.z)) {
      const Mat4 T = sm->T_inc;
      float x, y, z;
      xform_point(T, p.x, p.y, p.z, x, y, z);
      p.x = x; p.y = y; p.z = z;
      if (a.src0_nrm && finite3(nv.x, nv.y, nv.z)) { xform_normal(T, nv.x, nv.y, nv.z, x, y, z); nv.x = x; nv.y = y; nv.z = z; }
    }
    if (prof) { const long long t1 = clock64(); t_phase[3] += t1 - t0; }
    if (stop) break;
  }
  if (prof) for (int i = 0; i < 4; ++i) a.phase_cycles[i] = t_phase[i];
  if (bid == 0 && tid == 0) {
    ope_reg_result r;
    for (int i = 0; i < 16; ++i) r.T[i] = final_t.m[i];
    r.converged = converged; r.state = state; r.iterations = iterations; r.n_correspondences = n_corr;
    r.last_mse = cur_mse; r.best_error = 0.0; r.best_iteration = 0; r.reserved = 0;
    *a.result = r;
  }
}

// Frame-spanning launch: every block takes a ticket and looks up (alignment, block-in-alignment) in a host-built map that lists
// the blocks alignment by alignment. Tickets are handed out in the order blocks START, so when a block spins on its alignment's
// barrier, every block it waits for either runs already or is next in line for the first free slot — which the alignments ahead
// of it release without waiting for anyone behind them: no deadlock, whatever the dispatch order of the hardware.
template <int THREADS>
__global__ void __launch_bounds__(THREADS, 512 / THREADS) icp_small_batch_kernel(const IcpDev* __restrict__ descs, const int2* __restrict__ map,
                                                                                unsigned* ticket) {
  __shared__ int s_ticket;
  __shared__ IcpDev s_desc;
  if (threadIdx.x == 0) s_ticket = (int)atomicAdd(ticket, 1u);
  __syncthreads();
  const int2 fb = map[s_ticket];
  for (int w = threadIdx.x; w < (int)(sizeof(IcpDev) / 4); w += THREADS) reinterpret_cast<int*>(&s_desc)[w] = reinterpret_cast<const int*>(descs + fb.x)[w];
  __syncthreads();
  icp_small_body<THREADS>(s_desc, fb.y, (s_desc.n_work + THREADS - 1) / THREADS);
}

// one estimation + rejection pass (no loop) on the clouds as given (cur_* = the caller's clouds, original order)
__global__ void __launch_bounds__(kIcpThreads, 1) correspond_once_kernel(IcpDev a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  IcpSmem* sm = reinterpret_cast<IcpSmem*>(smem_raw);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (a.estimator != OPE_EST_NORMAL_SHOOTING) {
    for (int base = blockIdx.x * kIcpThreads; base < a.n_src; base += gridDim.x * kIcpThreads) {
      const int i = base + (int)threadIdx.x;
      const bool in_range = i < a.n_src;
      float4 p = make_float4(0, 0, 0, 0);
      if (in_range) p = a.cur_pts[i];
      const bool ok = in_range && finite3(p.x, p.y, p.z);
      float d2 = 0.0f;
      const int nn = block_nn1<kIcpThreads>(a.grid, &sm->nn, ok, p.x, p.y, p.z, a.max_d2_f, -1, nullptr, d2);
      if (in_range) {
        const int m = ok ? icp_gate(a, i, i, p, nn, d2) : -1;
        a.corr_match[i] = m; a.corr_d2[i] = d2;
      }
    }
  } else {
    OctStack* st = &sm->wstack[warp];
    for (int i = blockIdx.x * kIcpWarps + warp; i < a.n_src; i += gridDim.x * kIcpWarps) {
      const float4 p = a.cur_pts[i];
      float d2 = 0.0f;
      const int m = icp_correspond_shooting(a, st, i, i, p, false, d2);
      if (lane == 0) { a.corr_match[i] = m; a.corr_d2[i] = d2; }
      __syncwarp();
    }
  }
}

// determineReciprocalCorrespondences, VP/impl/correspondence_estimation_mod.hpp:216-303: a pair (i, m) survives iff i is the
// nearest SOURCE point of target point m within the distance. gsrc indexes the CURRENT (transformed) source.
__global__ void __launch_bounds__(kIcpThreads, 1) reciprocal_filter_kernel(GridView gsrc, const float4* __restrict__ tgt_pts, int* match,
                                                                           int n, float max_d2_f, double max_corr_dist) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  IcpSmem* sm = reinterpret_cast<IcpSmem*>(smem_raw);
  for (int base = blockIdx.x * kIcpThreads; base < n; base += gridDim.x * kIcpThreads) {
    const int i = base + (int)threadIdx.x;
    const int m = i < n ? match[i] : -1;
    float4 q = make_float4(0, 0, 0, 0);
    if (m >= 0) q = __ldg(tgt_pts + m);
    const bool ok = m >= 0 && finite3(q.x, q.y, q.z);
    float d2 = 0.0f;
    const int back = block_nn1<kIcpThreads>(gsrc, &sm->nn, ok, q.x, q.y, q.z, max_d2_f, -1, nullptr, d2);
    if (m >= 0 && !(ok && back == i && !((double)d2 > max_corr_dist * max_corr_dist))) match[i] = -1;
  }
}

// The reference's fixed correspondences (VP/impl/correspondence_estimation_mod.hpp:150-165, VP/impl/icp_mod.hpp:209-225): pair j
// gets distance = squared distance * 1e10 and enters the list twice — in front, through the whole rejector chain (slot j), and
// at the end, through rejector 0 alone (slot F + j, only when rejectors exist). One small block.
__global__ void fixed_pairs_kernel(IcpDev a, const int* __restrict__ fq, const int* __restrict__ fm, int n_fixed, int front,
                                   int* __restrict__ is, int* __restrict__ it, float* __restrict__ d2) {
  for (int j = threadIdx.x; j < n_fixed; j += blockDim.x) {
    const int q = fq[j], m = fm[j];
    const float4 s = a.cur_pts[q], t = __ldg(a.tgt_pts + m);
    const float px = t.x - s.x, py = t.y - s.y, pz = t.z - s.z;
    const float dist = front ? (float)((double)(px * px + py * py + pz * pz) * 1e10) : d2[j];   // reciprocal mode: as the caller left it
    int keep_all = front ? m : -1, keep_first = a.n_rej > 0 ? m : -1;
    if (front) keep_all = icp_reject(a, q, q, s, m);
    if (a.n_rej > 0) {
      IcpDev one = a;
      one.n_rej = 1;
      keep_first = icp_reject(one, q, q, s, m);
    }
    is[j] = q; it[j] = keep_all; d2[j] = dist;
    is[n_fixed + j] = q; it[n_fixed + j] = keep_first; d2[n_fixed + j] = dist;
  }
}

// the first fixed pair (index into the list) whose source or target point is not finite, via atomicMin on *first_bad
__global__ void fixed_finite_kernel(const float4* __restrict__ src, const float4* __restrict__ tgt, const int* __restrict__ fq,
                                    const int* __restrict__ fm, int n_fixed, int* __restrict__ first_bad) {
  for (int j = threadIdx.x; j < n_fixed; j += blockDim.x) {
    const float4 s = __ldg(src + fq[j]), t = __ldg(tgt + fm[j]);
    if (!finite3(s.x, s.y, s.z) || !finite3(t.x, t.y, t.z)) atomicMin(first_bad, j);
  }
}

// raw Umeyama moments (+ pair count and the sum of the correspondence distances) of the pairs (src[is[i]], tgt[it[i]]), it[i] >= 0
static constexpr int kPairAcc = kMomentAcc + 1;
__global__ void pairs_moments_kernel(const float4* __restrict__ src, const float4* __restrict__ tgt, const int* __restrict__ is,
                                     const int* __restrict__ it, const float* __restrict__ d2, int n, double* __restrict__ partials) {
  __shared__ double smem[(kRedThreads / 32) * kPairAcc];
  double acc[kPairAcc];
  for (int a = 0; a < kPairAcc; ++a) acc[a] = 0.0;
  double o[3];
  { const float4 t0 = __ldg(tgt); moment_origin(t0.x, t0.y, t0.z, o[0], o[1], o[2]); }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int m = it[i];
    if (m < 0) continue;
    const float4 s = __ldg(src + (is ? is[i] : i));
    const float4 t = __ldg(tgt + m);
    const double sv[3] = {(double)s.x - o[0], (double)s.y - o[1], (double)s.z - o[2]};
    const double tv[3] = {(double)t.x - o[0], (double)t.y - o[1], (double)t.z - o[2]};
    acc[0] += 1.0;
    acc[1] += sv[0]; acc[2] += sv[1]; acc[3] += sv[2];
    acc[4] += tv[0]; acc[5] += tv[1]; acc[6] += tv[2];
    for (int c = 0; c < 3; ++c)
      for (int r = 0; r < 3; ++r) acc[7 + c * 3 + r] += tv[r] * sv[c];
    acc[kMomentAcc] += (double)d2[i];
  }
  block_reduce_store<kPairAcc>(acc, smem, partials + (size_t)blockIdx.x * kPairAcc);
}

// ============================================================================================ SAC-IA ====
// Every hypothesis is scored by the same stages, for a whole batch of frames (ope_pose_batch) or for the one frame of
// ope_sacia_align / ope_pose_estimate_final:
//   sacia_transform_batch_kernel  one THREAD per (frame, hypothesis): the 5-point Umeyama (double moments, as everywhere)
//   sacia_seed_batch_kernel       blockIdx.x = frame, blockIdx.y = a share of the cells: a kSeedG^3 grid around the frame's target;
//                                 every cell remembers the target point nearest to its centre. A query looks up its (clamped) cell and starts its search from that
//                                 point's distance: a bound within a cell size of the answer, so the box tests prune from the start
//   sacia_score_batch_kernel      blockIdx.x = frame, blockIdx.y = a few consecutive hypotheses: the frame's target (at most
//                                 kSaciaSmemMaxTargets points), its group boxes and the seed grid are staged in shared memory once
//                                 per block
//   sacia_kernel                  one frame whose target does not fit: one block per hypothesis, block_nn1 through the grid index
//   sacia_select_batch_kernel     first strictly-lower error wins, per frame
// Both scorers sum a hypothesis' terms as floats in point order in one thread (bit-exact with the reference's serial
// `error += ...`, so the first-lowest-error hypothesis is the same one), and only the DISTANCE of the nearest neighbour enters a
// term: ties need no index order.
static constexpr int kSaciaThreads = 256;
static constexpr int kSaciaMaxSamples = 16;
static constexpr int kSaciaSmemMaxTargets = 8192;   // 128 KB of the 227 KB shared memory

__global__ void __launch_bounds__(kSaciaThreads) sacia_kernel(SaciaBatch a, GridView grid, float* __restrict__ terms_all) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Nn1Smem<kSaciaThreads>* nn = reinterpret_cast<Nn1Smem<kSaciaThreads>*>(smem_raw);
  __shared__ Mat4 T;
  const int h = a.h_begin + blockIdx.x;
  if (threadIdx.x < 16) T.m[threadIdx.x] = __ldg(a.transforms + (size_t)h * 16 + threadIdx.x);
  __syncthreads();
  const Mat4 M = T;
  float* terms = terms_all + (size_t)blockIdx.x * a.ns;
  for (int base = 0; base < a.ns; base += kSaciaThreads) {
    const int i = base + (int)threadIdx.x;
    float x = 0, y = 0, z = 0;
    bool ok = false;
    if (i < a.ns) {
      const float4 p = __ldg(a.src + i);
      xform_point(M, p.x, p.y, p.z, x, y, z);
      ok = finite3(x, y, z);
    }
    float d2;
    const int idx = block_nn1<kSaciaThreads>(grid, nn, ok, x, y, z, a.threshold, -1, nullptr, d2);
    if (i < a.ns) terms[i] = (ok && idx >= 0 && d2 <= a.threshold) ? d2 / a.threshold : 1.0f;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float error = 0.0f;
    for (int i = 0; i < a.ns; ++i) error += terms[i];
    a.errors[h] = error;
  }
}
// squared distance from a query to an axis-aligned box (0 inside); an empty box (lo = +inf, hi = -inf) gives +inf
__device__ __forceinline__ float box_d2(const float4 lo, const float4 hi, float x, float y, float z) {
  const float ex = fmaxf(fmaxf(lo.x - x, x - hi.x), 0.0f), ey = fmaxf(fmaxf(lo.y - y, y - hi.y), 0.0f), ez = fmaxf(fmaxf(lo.z - z, z - hi.z), 0.0f);
  return ex * ex + ey * ey + ez * ez;
}
static constexpr int kSeedG = 12;
static constexpr int kSeedCells = kSeedG * kSeedG * kSeedG;
static_assert(kSaciaSmemMaxTargets <= 65536, "the seed grid stores target indices as unsigned short");
static constexpr int kSaciaHypPerBlock = 16;     // hypotheses per scoring block while the launch still fills the device
static constexpr int kSaciaScoreThreads = 128;   // points per early-exit check: most hypotheses are out after the first one

// The scoring kernel's work order of the source: along the Morton curve of its bounding box, so that the 32 points of a warp are
// neighbours (the coarse sample arrives in voxel-key order: rows across the whole model). .w carries the original index: the terms
// are stored — and finally summed — in the original order. One block per source (frame f's at out + f * out_stride); more than
// kSaciaOrderMax points keep their order.
static constexpr int kSaciaOrderMax = 4096;
__global__ void __launch_bounds__(kSaciaThreads) sacia_source_order_kernel(SaciaBatch a, int out_stride, float4* __restrict__ out_all) {
  __shared__ unsigned long long keys[kSaciaOrderMax];
  __shared__ float red[6][kSaciaThreads / 32];
  __shared__ float box[6];
  const int f = blockIdx.x;
  if (a.src_stride && !a.active[f]) return;
  const float4* src = a.src + (size_t)f * a.src_stride;
  const int n = a.src_counts ? a.src_counts[f] : a.ns;
  float4* out = out_all + (size_t)f * out_stride;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (n > kSaciaOrderMax) {
    for (int i = tid; i < n; i += kSaciaThreads) { float4 p = __ldg(src + i); p.w = __int_as_float(i); out[i] = p; }
    return;
  }
  float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int i = tid; i < n; i += kSaciaThreads) {
    const float4 p = __ldg(src + i);
    if (!finite3(p.x, p.y, p.z)) continue;
    lo[0] = fminf(lo[0], p.x); lo[1] = fminf(lo[1], p.y); lo[2] = fminf(lo[2], p.z);
    hi[0] = fmaxf(hi[0], p.x); hi[1] = fmaxf(hi[1], p.y); hi[2] = fmaxf(hi[2], p.z);
  }
  for (int o = 16; o > 0; o >>= 1)
    for (int d = 0; d < 3; ++d) { lo[d] = fminf(lo[d], __shfl_xor_sync(0xffffffffu, lo[d], o)); hi[d] = fmaxf(hi[d], __shfl_xor_sync(0xffffffffu, hi[d], o)); }
  if (lane == 0) for (int d = 0; d < 3; ++d) { red[d][warp] = lo[d]; red[3 + d][warp] = hi[d]; }
  __syncthreads();
  if (tid < 6) {
    float v = red[tid][0];
    for (int w = 1; w < kSaciaThreads / 32; ++w) v = tid < 3 ? fminf(v, red[tid][w]) : fmaxf(v, red[tid][w]);
    box[tid] = v;
  }
  __syncthreads();
  const float ext = fmaxf(fmaxf(box[3] - box[0], box[4] - box[1]), fmaxf(box[5] - box[2], 1e-9f));
  const float scale = 1023.0f / ext;
  int m2 = 1;
  while (m2 < n) m2 <<= 1;
  for (int i = tid; i < m2; i += kSaciaThreads) {
    unsigned long long k = ~0ull;
    if (i < n) {
      const float4 p = __ldg(src + i);
      unsigned code = 0x3fffffffu;   // non-finite points last
      if (finite3(p.x, p.y, p.z))
        code = morton3((unsigned)fminf(fmaxf((p.x - box[0]) * scale, 0.0f), 1023.0f), (unsigned)fminf(fmaxf((p.y - box[1]) * scale, 0.0f), 1023.0f),
                       (unsigned)fminf(fmaxf((p.z - box[2]) * scale, 0.0f), 1023.0f));
      k = ((unsigned long long)code << 32) | (unsigned)i;
    }
    keys[i] = k;
  }
  __syncthreads();
  for (int k2 = 2; k2 <= m2; k2 <<= 1)
    for (int j2 = k2 >> 1; j2 > 0; j2 >>= 1) {
      for (int i = tid; i < m2; i += kSaciaThreads) {
        const int l = i ^ j2;
        if (l > i) {
          const bool up = (i & k2) == 0;
          const unsigned long long ki = keys[i], kl = keys[l];
          if ((ki > kl) == up) { keys[i] = kl; keys[l] = ki; }
        }
      }
      __syncthreads();
    }
  for (int j = tid; j < n; j += kSaciaThreads) {
    const int from = (int)(unsigned)(keys[j] & 0xffffffffull);
    float4 p = __ldg(src + from);
    p.w = __int_as_float(from);
    out[j] = p;
  }
}

__global__ void __launch_bounds__(128) sacia_transform_batch_kernel(SaciaBatch a, int frames) {
  const int nh = a.h_end - a.h_begin;
  const int idx = blockIdx.x * 128 + threadIdx.x;
  if (idx >= frames * nh) return;
  const int f = idx / nh, h = a.h_begin + idx - f * nh;
  if (!a.active[f]) return;
  const float4* tgt = a.tgt + (size_t)f * a.stride;
  double acc[16];
  for (int i = 0; i < 16; ++i) acc[i] = 0.0;
  const int* samples = a.samples + ((size_t)f * a.H + h) * a.nr_samples;
  const int* picks = a.picks + ((size_t)f * a.H + h) * a.nr_samples;
  const int* knn = a.knn_idx + (size_t)f * a.ns * a.k_corr;
  const float4* src = a.src + (size_t)f * a.src_stride;
  for (int j = 0; j < a.nr_samples; ++j) {
    const int si = samples[j];
    int ti = knn[(size_t)si * a.k_corr + picks[j]];
    if (ti < 0) ti = knn[(size_t)si * a.k_corr];  // fewer than k target features
    const float4 sp = __ldg(src + si), tp = __ldg(tgt + ti);
    const double sv[3] = {sp.x, sp.y, sp.z}, tv[3] = {tp.x, tp.y, tp.z};
    acc[0] += 1.0;
    for (int k = 0; k < 3; ++k) { acc[1 + k] += sv[k]; acc[4 + k] += tv[k]; }
    for (int c = 0; c < 3; ++c)
      for (int r = 0; r < 3; ++r) acc[7 + c * 3 + r] += tv[r] * sv[c];
  }
  Mat4 M;
  umeyama_from_moments(acc, M);
  float* out = a.transforms + ((size_t)f * a.H + h) * 16;
  for (int i = 0; i < 16; ++i) out[i] = M.m[i];
}

__global__ void __launch_bounds__(kSaciaThreads) sacia_seed_batch_kernel(SaciaBatch a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float4* tg = reinterpret_cast<float4*>(smem_raw);
  __shared__ float red[6][kSaciaThreads / 32];
  __shared__ float box[6];
  const int f = blockIdx.x;
  if (!a.active[f]) return;
  const int nt = a.counts[f];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float4* scan = (a.tgt_scan ? a.tgt_scan : a.tgt) + (size_t)f * a.stride;
  float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int j = tid; j < nt; j += kSaciaThreads) {
    const float4 t = __ldg(scan + j);
    tg[j] = t;
    if (finite3(t.x, t.y, t.z)) {
      lo[0] = fminf(lo[0], t.x); lo[1] = fminf(lo[1], t.y); lo[2] = fminf(lo[2], t.z);
      hi[0] = fmaxf(hi[0], t.x); hi[1] = fmaxf(hi[1], t.y); hi[2] = fmaxf(hi[2], t.z);
    }
  }
  for (int o = 16; o > 0; o >>= 1)
    for (int d = 0; d < 3; ++d) { lo[d] = fminf(lo[d], __shfl_xor_sync(0xffffffffu, lo[d], o)); hi[d] = fmaxf(hi[d], __shfl_xor_sync(0xffffffffu, hi[d], o)); }
  if (lane == 0) for (int d = 0; d < 3; ++d) { red[d][warp] = lo[d]; red[3 + d][warp] = hi[d]; }
  __syncthreads();
  if (tid < 6) {
    float v = red[tid][0];
    for (int w = 1; w < kSaciaThreads / 32; ++w) v = tid < 3 ? fminf(v, red[tid][w]) : fmaxf(v, red[tid][w]);
    box[tid] = v;
  }
  __syncthreads();
  // a cubic grid over the bounding box grown by a quarter of its largest extent on every side (queries near the target, but
  // outside its box, still get a cell of their own; farther ones use the nearest border cell)
  float ext = fmaxf(fmaxf(box[3] - box[0], box[4] - box[1]), box[5] - box[2]);
  if (!(ext > 1e-6f) || !(ext < FLT_MAX)) ext = 1e-6f;
  const float cell = 1.5f * ext / (float)kSeedG;
  float org[3];
  for (int d = 0; d < 3; ++d) { org[d] = 0.5f * (box[d] + box[3 + d]) - 0.5f * cell * (float)kSeedG; if (!(fabsf(org[d]) < FLT_MAX)) org[d] = 0.0f; }
  if (tid == 0 && blockIdx.y == 0) { a.seed_geo[f] = make_float4(org[0], org[1], org[2], 1.0f / cell); a.best_bits[f] = 0x7f800000u; }   // +inf
  for (int c = (int)blockIdx.y * kSaciaThreads + tid; c < kSeedCells; c += (int)gridDim.y * kSaciaThreads) {
    const int cx = c % kSeedG, cy = (c / kSeedG) % kSeedG, cz = c / (kSeedG * kSeedG);
    const float x = org[0] + ((float)cx + 0.5f) * cell, y = org[1] + ((float)cy + 0.5f) * cell, z = org[2] + ((float)cz + 0.5f) * cell;
    float best = FLT_MAX;
    int arg = 0;
#pragma unroll 4
    for (int j = 0; j < nt; ++j) {
      const float4 t = tg[j];
      const float d2 = dist2(x, y, z, t.x, t.y, t.z);
      if (d2 < best) { best = d2; arg = j; }   // NaN / inf (non-finite targets) never wins
    }
    a.seed_tab[(size_t)f * kSeedCells + c] = (unsigned short)arg;
  }
}

__global__ void __launch_bounds__(kSaciaScoreThreads) sacia_score_batch_kernel(SaciaBatch a, int hyp_per_block) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  // blockIdx.x = frame (fastest): the hypothesis groups of one frame run one after the other, so the bound below is known early
  const int f = blockIdx.x;
  if (!a.active[f]) return;
  const int nt = a.counts[f];
  const int nt8 = (nt + 7) & ~7, n_groups = nt8 >> 3;
  float4* tg = reinterpret_cast<float4*>(smem_raw);
  float4* glo = tg + nt8;
  float4* ghi = glo + n_groups;
  float* terms = reinterpret_cast<float*>(ghi + n_groups);
  unsigned short* seed = reinterpret_cast<unsigned short*>(terms + a.ns);
  const int ns = a.src_counts ? a.src_counts[f] : a.ns;
  const float4* src_scan = a.src_scan + (a.src_stride ? (size_t)f * a.ns : 0);
  __shared__ Mat4 T;
  __shared__ float wpart[2][kSaciaScoreThreads / 32];
  __shared__ float s_best[2];
  const unsigned full = 0xffffffffu;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float4* scan = (a.tgt_scan ? a.tgt_scan : a.tgt) + (size_t)f * a.stride;   // a spatially sorted copy makes the boxes tight
  for (int j = tid; j < nt8; j += kSaciaScoreThreads) tg[j] = j < nt ? __ldg(scan + j) : make_float4(INFINITY, INFINITY, INFINITY, 0.0f);
  for (int c = tid; c < kSeedCells; c += kSaciaScoreThreads) seed[c] = a.seed_tab[(size_t)f * kSeedCells + c];
  const float4 geo = a.seed_geo[f];
  __syncthreads();
  // boxes of the groups of 8 consecutive target points
  for (int g = tid; g < n_groups; g += kSaciaScoreThreads) {
    float4 lo = make_float4(INFINITY, INFINITY, INFINITY, 0.0f), hi = make_float4(-INFINITY, -INFINITY, -INFINITY, 0.0f);
    for (int u = 0; u < 8; ++u) {
      const float4 t = tg[8 * g + u];
      if (!finite3(t.x, t.y, t.z)) continue;
      lo.x = fminf(lo.x, t.x); lo.y = fminf(lo.y, t.y); lo.z = fminf(lo.z, t.z);
      hi.x = fmaxf(hi.x, t.x); hi.y = fmaxf(hi.y, t.y); hi.z = fmaxf(hi.z, t.z);
    }
    glo[g] = lo; ghi[g] = hi;
  }
  unsigned* frame_best = a.best_bits + f;
  const int h_begin = a.h_begin + (int)blockIdx.y * hyp_per_block, h_end = min(a.h_end, h_begin + hyp_per_block);
  for (int h = h_begin; h < h_end; ++h) {
    // (this barrier also closes the previous hypothesis: thread 0's final sum has read the terms)
    if (tid < 16) T.m[tid] = __ldg(a.transforms + ((size_t)f * a.H + h) * 16 + tid);
    __syncthreads();
    const Mat4 M = T;
    // The error is the float sum of the terms IN POINT ORDER (bit-exact with the reference's serial `error += ...`), formed by one
    // thread — but only for a hypothesis that gets that far. The terms are >= 0, so the sum of any subset of them is a lower bound
    // of the total, and ANY summation order is within n * 2^-24 (relative) of the serial one: after every chunk of
    // kSaciaScoreThreads points the block adds the chunk up in parallel and compares that sum, shrunk by twice that bound, with the lowest
    // COMPLETE error any hypothesis of this frame has published so far. Once it is larger, the serial total would be larger too:
    // this hypothesis cannot be the first-lowest one and stops (its error is reported as +inf). Which hypotheses stop early
    // depends on timing; the winner, its error and its transform do not.
    float run = 0.0f;
    bool stop = false;
    int chunk = 0;
    const float shrink = 1.0f - 4.0f * (float)(ns + 32) * 5.97e-8f;   // twice the bound 2 n 2^-24 on the gap between two summation orders
    for (int base = 0; base < ns; base += kSaciaScoreThreads, ++chunk) {
      const int i = base + tid;
      float term = 0.0f;
      float x = 0.0f, y = 0.0f, z = 0.0f;
      bool search = false;
      int orig = 0;
      if (i < ns) {
        const float4 p = __ldg(src_scan + i);
        orig = __float_as_int(p.w);
        xform_point(M, p.x, p.y, p.z, x, y, z);
        term = 1.0f;
        search = finite3(x, y, z);
      }
      // only the DISTANCE of the nearest neighbour enters the score: ties need no index order
      float best = FLT_MAX;
      if (search) {
        const float fx = fminf(fmaxf((x - geo.x) * geo.w, 0.0f), (float)(kSeedG - 1)), fy = fminf(fmaxf((y - geo.y) * geo.w, 0.0f), (float)(kSeedG - 1)),
                    fz = fminf(fmaxf((z - geo.z) * geo.w, 0.0f), (float)(kSeedG - 1));
        const float4 t = tg[seed[((int)fz * kSeedG + (int)fy) * kSeedG + (int)fx]];
        const float d2 = dist2(x, y, z, t.x, t.y, t.z);
        if (d2 < best) best = d2;
      }
      // the box around the warp's 32 queries (consecutive model points: neighbours), grown by the widest bound among them, against
      // the group boxes, one group per lane; the groups that pass go through the per-thread test. Conservative comparisons: a
      // float box distance can only be a rounding error above the float distance to a point inside the box.
      float wlx = search ? x : INFINITY, wly = search ? y : INFINITY, wlz = search ? z : INFINITY;
      float whx = search ? x : -INFINITY, why = search ? y : -INFINITY, whz = search ? z : -INFINITY;
      float wb = search ? best : 0.0f;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        wlx = fminf(wlx, __shfl_xor_sync(full, wlx, o)); wly = fminf(wly, __shfl_xor_sync(full, wly, o)); wlz = fminf(wlz, __shfl_xor_sync(full, wlz, o));
        whx = fmaxf(whx, __shfl_xor_sync(full, whx, o)); why = fmaxf(why, __shfl_xor_sync(full, why, o)); whz = fmaxf(whz, __shfl_xor_sync(full, whz, o));
        wb = fmaxf(wb, __shfl_xor_sync(full, wb, o));
      }
      const float wlim = wb * 1.0002f + 1e-30f;
      for (int g0 = 0; g0 < n_groups; g0 += 32) {
        bool near = false;
        if (g0 + lane < n_groups) {
          const float4 lo = glo[g0 + lane], hi = ghi[g0 + lane];
          const float ex = fmaxf(fmaxf(lo.x - whx, wlx - hi.x), 0.0f), ey = fmaxf(fmaxf(lo.y - why, wly - hi.y), 0.0f),
                      ez = fmaxf(fmaxf(lo.z - whz, wlz - hi.z), 0.0f);
          near = ex * ex + ey * ey + ez * ez <= wlim;
        }
        for (unsigned cand = __ballot_sync(full, near); cand != 0u; cand &= cand - 1u) {
          const int g = g0 + __ffs(cand) - 1;
          if (!search || !(box_d2(glo[g], ghi[g], x, y, z) <= best * 1.0001f + 1e-30f)) continue;
          float d2[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) { const float4 t = tg[8 * g + u]; d2[u] = dist2(x, y, z, t.x, t.y, t.z); }
#pragma unroll
          for (int u = 0; u < 8; ++u) best = d2[u] < best ? d2[u] : best;   // NaN / inf (padding, non-finite targets) never wins
        }
      }
      if (search && best <= a.threshold) term = best / a.threshold;
      if (i < ns) terms[orig] = term;
      float part = term;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(full, part, o);
      const int par = chunk & 1;
      if (lane == 0) wpart[par][warp] = part;
      if (tid == 0) s_best[par] = __uint_as_float(*(volatile unsigned*)frame_best);
      __syncthreads();
#pragma unroll
      for (int w = 0; w < kSaciaScoreThreads / 32; ++w) run += wpart[par][w];
      if (a.early_exit && run * shrink > s_best[par]) { stop = true; break; }   // the same values in every thread
    }
    if (tid == 0) {
      float error = INFINITY;
      if (!stop) {
        error = 0.0f;
        for (int j = 0; j < ns; ++j) error += terms[j];
        atomicMin(frame_best, __float_as_uint(error));   // errors are >= 0: the bit pattern orders like the value
      }
      a.errors[(size_t)f * a.H + h] = error;
    }
  }
}
// first strictly-lower error wins, in hypothesis order (SURVEY A.6); one thread per frame
__global__ void sacia_select_batch_kernel(SaciaBatch a, int frames, ope_reg_result* __restrict__ out) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= frames || !a.active[f]) return;
  int best = -1;
  float lowest = 0.0f;
  for (int h = a.h_begin; h < a.h_end; ++h) {
    const float e = a.errors[(size_t)f * a.H + h];
    if (best < 0 || e < lowest) { lowest = e; best = h; }
  }
  ope_reg_result r;
  for (int i = 0; i < 16; ++i) r.T[i] = (best >= 0) ? a.transforms[((size_t)f * a.H + best) * 16 + i] : ((i % 5 == 0) ? 1.0f : 0.0f);
  r.converged = best >= 0; r.state = 0; r.iterations = a.H; r.n_correspondences = 0; r.last_mse = 0.0;
  r.best_error = lowest; r.best_iteration = best; r.reserved = 0;
  out[f] = r;
}
// getFitnessScore for every frame of a batch: one block per frame, the frame's target in shared memory, the transform from the
// frame's ICP result on the device
__global__ void __launch_bounds__(kNnThreads) fitness_smem_batch_kernel(const float4* __restrict__ tgt, const int* __restrict__ tgt_counts,
                                                                        const float4* __restrict__ src, const int* __restrict__ src_counts,
                                                                        int stride, const ope_reg_result* __restrict__ icp,
                                                                        const int* __restrict__ active, double* __restrict__ out) {
  extern __shared__ __align__(16) float4 tg_fit[];
  __shared__ double smem[(kNnThreads / 32) * 2];
  __shared__ double fin[2];
  const int f = blockIdx.x;
  if (!active[f]) return;
  const int nt = tgt_counts[f], n = src_counts[f];
  const int nt8 = (nt + 7) & ~7;
  const float4* tp = tgt + (size_t)f * stride;
  const float4* sp = src + (size_t)f * stride;
  for (int j = threadIdx.x; j < nt8; j += kNnThreads) tg_fit[j] = j < nt ? __ldg(tp + j) : make_float4(INFINITY, INFINITY, INFINITY, 0.0f);
  Mat4 T;
  for (int i = 0; i < 16; ++i) T.m[i] = icp[f].T[i];
  __syncthreads();
  double acc[2] = {0.0, 0.0};
  for (int base = 0; base < n; base += kNnThreads) {
    const int i = base + (int)threadIdx.x;
    float x = 0, y = 0, z = 0;
    bool ok = false;
    if (i < n) {
      const float4 p = __ldg(sp + i);
      xform_point(T, p.x, p.y, p.z, x, y, z);
      ok = finite3(x, y, z);
    }
    float best = INFINITY;
    if (ok) {
      for (int j0 = 0; j0 < nt8; j0 += 8) {
        float d2[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) { const float4 t = tg_fit[j0 + u]; d2[u] = dist2(x, y, z, t.x, t.y, t.z); }
#pragma unroll
        for (int u = 0; u < 8; ++u) if (d2[u] < best) best = d2[u];
      }
    }
    if (ok && best <= FLT_MAX) { acc[0] += (double)best; acc[1] += 1.0; }
  }
  block_reduce_store<2>(acc, smem, fin);
  if (threadIdx.x == 0) out[f] = fin[1] > 0 ? fin[0] / fin[1] : DBL_MAX;
}

// ================================================================================================ host ==
int transform_device(ope_ctx* ctx, const ope_cloud* in, const Mat4& T, ope_cloud* out) {
  if (in->n == 0) return OPE_OK;
  transform_kernel<<<div_up(in->n, 256), 256, 0, ctx->stream>>>(in->pts, in->normals, (int)in->n, T, out->pts, out->normals);
  return check_launch(ctx, "transform_kernel");
}

int umeyama_device(ope_ctx* ctx, const float4* src, const float4* tgt, const int* d_isrc, const int* d_itgt, size_t n,
                   float T[16]) {
  const int nb = umeyama_blocks(ctx, n);
  Scratch<double> partials(ctx);
  Scratch<float> out(ctx);
  OPE_TRY(partials.alloc((size_t)nb * kMomentAcc));
  OPE_TRY(out.alloc(16));
  moments_kernel<<<nb, kRedThreads, 0, ctx->stream>>>(src, tgt, d_isrc, d_itgt, (int)n, partials.p);
  OPE_TRY(check_launch(ctx, "moments_kernel"));
  umeyama_final_kernel<<<1, 32 * kMomentAcc, 0, ctx->stream>>>(partials.p, nb, out.p, tgt);
  OPE_TRY(check_launch(ctx, "umeyama_final_kernel"));
  void* h;
  OPE_TRY(read_back(ctx, out.p, 16 * sizeof(float), &h));
  std::memcpy(T, h, 16 * sizeof(float));
  return OPE_OK;
}

int umeyama_blocks(ope_ctx* ctx, size_t n) {
  return (int)std::min<size_t>(std::max<size_t>(1, (n + kRedThreads - 1) / kRedThreads), (size_t)ctx->sm_count * 4);
}
int track_commit_device(ope_ctx* ctx, const TrackCommit* d_commits, const TrackCommit* h_commits, int n, float* d_rigid) {
  if (n <= 0) return OPE_OK;
  int max_nb = 1;
  for (int i = 0; i < n; ++i) max_nb = std::max(max_nb, h_commits[i].nb);
  Scratch<double> partials(ctx);
  OPE_TRY(partials.alloc((size_t)n * max_nb * kMomentAcc));
  track_commit_kernel<<<dim3(max_nb, n), kRedThreads, 0, ctx->stream>>>(d_commits, partials.p);
  OPE_TRY(check_launch(ctx, "track_commit_kernel"));
  track_umeyama_final_kernel<<<n, 32 * kMomentAcc, 0, ctx->stream>>>(d_commits, partials.p, max_nb, d_rigid);
  return check_launch(ctx, "track_umeyama_final_kernel");
}

int fitness_device(ope_ctx* ctx, const ope_cloud* src, const ope_cloud* tgt, const Mat4& T, double max_range, double* out) {
  *out = DBL_MAX;
  if (src->n == 0) return OPE_OK;
  const int nb = (int)std::min<size_t>(std::max<size_t>(1, (src->n + kNnThreads - 1) / kNnThreads), (size_t)ctx->sm_count * 4);
  Scratch<double> partials(ctx), fin(ctx);
  OPE_TRY(partials.alloc((size_t)nb * 2));
  OPE_TRY(fin.alloc(2));
  const float mr = max_range >= (double)FLT_MAX ? FLT_MAX : (float)max_range;
  if (tgt->n <= (size_t)kFitSmemMax && !std::getenv("OPE_FITNESS_FORCE_GRID")) {
    const size_t bytes = ((tgt->n + 7) & ~(size_t)7) * sizeof(float4);
    OPE_TRY(dyn_smem(ctx, (const void*)fitness_smem_kernel, (size_t)kFitSmemMax * sizeof(float4)));
    fitness_smem_kernel<<<nb, kNnThreads, bytes, ctx->stream>>>(tgt->pts, (int)tgt->n, src->pts, (int)src->n, T, mr, partials.p);
    OPE_TRY(check_launch(ctx, "fitness_smem_kernel"));
  } else {
    OPE_TRY(cloud_bbox(ctx, const_cast<ope_cloud*>(tgt)));
    GridView g;
    OPE_TRY(cloud_grid(ctx, tgt, knn_cell_size(tgt, 1), &g));
    OPE_TRY(dyn_smem(ctx, (const void*)fitness_kernel, sizeof(Nn1Smem<kNnThreads>)));
    fitness_kernel<<<nb, kNnThreads, sizeof(Nn1Smem<kNnThreads>), ctx->stream>>>(g, src->pts, (int)src->n, T, mr, partials.p);
    OPE_TRY(check_launch(ctx, "fitness_kernel"));
  }
  sum_partials_kernel<<<1, 64, 0, ctx->stream>>>(partials.p, nb, 2, fin.p);
  OPE_TRY(check_launch(ctx, "sum_partials_kernel"));
  void* h;
  OPE_TRY(read_back(ctx, fin.p, 2 * sizeof(double), &h));
  const double* r = (const double*)h;
  *out = r[1] > 0 ? r[0] / r[1] : DBL_MAX;
  return OPE_OK;
}

// The parameter fields of every ICP path's descriptor: iterations, convergence thresholds and the rejector chain (checked)
static int icp_fill_params(ope_ctx* ctx, const ope_icp_params& prm, IcpDev* a) {
  if (prm.n_rejectors < 0 || prm.n_rejectors > OPE_MAX_REJECTORS) return fail(ctx, OPE_ERR_INVALID, "bad rejector count");
  for (int r = 0; r < prm.n_rejectors; ++r)
    if (prm.rejector_kind[r] != OPE_REJ_SURFACE_NORMAL && prm.rejector_kind[r] != OPE_REJ_SELF_OCCLUDED_NORMAL)
      return fail(ctx, OPE_ERR_UNSUPPORTED, "unknown correspondence rejector kind %d", prm.rejector_kind[r]);
  a->max_iterations = prm.max_iterations; a->min_corr = prm.min_number_correspondences;
  a->estimator = prm.estimator; a->k_search = prm.k_search; a->n_rej = prm.n_rejectors;
  a->transformation = prm.transformation; a->variant = prm.variant; a->force_all = prm.force_all_iterations;
  for (int r = 0; r < OPE_MAX_REJECTORS; ++r) { a->rej_kind[r] = prm.rejector_kind[r]; a->rej_thr[r] = prm.rejector_threshold[r]; }
  a->max_corr_dist = prm.max_correspondence_distance;
  const double m2 = prm.max_correspondence_distance * prm.max_correspondence_distance;
  a->max_d2_f = (m2 >= (double)FLT_MAX || !(m2 == m2)) ? FLT_MAX : (float)m2;
  a->rot_thr = 1.0 - prm.transformation_epsilon;
  a->trans_thr = prm.transformation_epsilon;
  a->rel_mse_thr = prm.euclidean_fitness_epsilon;
  a->abs_mse_thr = prm.mse_threshold_absolute;
  a->max_similar = prm.max_iterations_similar_transforms;
  a->fail_after_max = prm.failure_after_max_iterations;
  return OPE_OK;
}

static int icp_fill(ope_ctx* ctx, const ope_cloud* src, const ope_cloud* tgt, const ope_icp_params& prm, IcpDev* a,
                    bool allow_smem_target = false) {
  OPE_TRY(icp_fill_params(ctx, prm, a));
  const bool need_src_normals = prm.estimator == OPE_EST_NORMAL_SHOOTING || prm.n_rejectors > 0;
  bool need_tgt_normals = false;
  for (int r = 0; r < prm.n_rejectors; ++r)
    if (prm.rejector_kind[r] == OPE_REJ_SURFACE_NORMAL) need_tgt_normals = true;
  if (need_src_normals && !src->normals) return fail(ctx, OPE_ERR_INVALID, "estimator/rejector needs source normals");
  if (need_tgt_normals && !tgt->normals) return fail(ctx, OPE_ERR_INVALID, "rejector needs target normals");
  if (prm.use_reciprocal && prm.estimator != OPE_EST_NEAREST)
    return fail(ctx, OPE_ERR_UNSUPPORTED, "reciprocal correspondences are implemented for the nearest-neighbour estimator only");
  if (prm.transformation != OPE_TE_SVD && prm.transformation != OPE_TE_POINT_TO_PLANE_LLS && prm.transformation != OPE_TE_POINT_TO_PLANE)
    return fail(ctx, OPE_ERR_UNSUPPORTED, "unknown transformation estimator %d", prm.transformation);
  if (prm.transformation != OPE_TE_SVD && !tgt->normals) return fail(ctx, OPE_ERR_INVALID, "point-to-plane estimation needs target normals");
  if (prm.estimator == OPE_EST_NORMAL_SHOOTING && (prm.k_search < 1 || prm.k_search > 32))
    return fail(ctx, OPE_ERR_INVALID, "normal shooting k must be in [1, 32]");
  OPE_TRY(cloud_bbox(ctx, const_cast<ope_cloud*>(tgt)));
  const int kk = prm.estimator == OPE_EST_NORMAL_SHOOTING ? prm.k_search : 1;
  a->n_tgt = (int)tgt->n;
  const char* force_grid = std::getenv("OPE_ICP_FORCE_GRID");
  a->tgt_in_smem = (allow_smem_target && prm.estimator == OPE_EST_NORMAL_SHOOTING && tgt->n <= (size_t)kIcpSmemMaxTargets && !force_grid) ? 1 : 0;
  if (a->tgt_in_smem) {   // no spatial index needed: only the number of finite points (k is clamped to it)
    std::memset(&a->grid, 0, sizeof(a->grid));
    a->grid.n = tgt->n_finite;
  } else {
    OPE_TRY(cloud_grid(ctx, tgt, knn_cell_size(tgt, kk), &a->grid));
  }
  a->tgt_pts = tgt->pts; a->tgt_nrm = tgt->normals;
  a->src0_pts = src->pts; a->src0_nrm = src->normals;
  a->n_src = (int)src->n;
  return OPE_OK;
}

static void corr_to_host(const std::vector<int>& match, const std::vector<float>& d2, ope_correspondence* out, size_t* n) {
  size_t w = 0;
  for (size_t i = 0; i < match.size(); ++i)
    if (match[i] >= 0) out[w++] = ope_correspondence{(int32_t)i, match[i], d2[i]};
  if (n) *n = w;
}

static int icp_stepwise_device(ope_ctx* ctx, const ope_cloud* src, const ope_cloud* tgt, const ope_icp_params& prm, const Mat4& guess,
                               ope_reg_result* res, ope_correspondence* out_corr_host, ope_cloud** out_aligned,
                               ope_correspondence* fixed = nullptr, size_t n_fixed = 0);

// The thread-per-query ICP (icp_small_batch_kernel) takes normal shooting with SVD, k <= 32 and, per alignment, up to 4 096 finite
// source points against a target of up to 4 096 points in shared memory.
bool icp_small_applicable(const ope_icp_params& prm, size_t n_src, size_t n_tgt) {
  return prm.estimator == OPE_EST_NORMAL_SHOOTING && prm.transformation == OPE_TE_SVD && !prm.use_reciprocal && n_tgt > 0 &&
         n_tgt <= (size_t)kIcpSmemMaxTargets && n_src > 0 && n_src <= (size_t)kIcpSmallMaxBlocks * kIcpSmallThreads &&
         prm.k_search >= 1 && prm.k_search <= kSlabSlots;
}

// Runs the alignments descs[0, n) in one launch of icp_small_batch_kernel; the caller fills every descriptor but its partials
// and barrier, within icp_small_applicable. One alignment is a cooperative launch, so its blocks are co-resident whatever else
// runs on the device. More are ticketed (see the kernel), which counts on the residency bound checked below.
static int icp_small_launch(ope_ctx* ctx, IcpDev* descs, int n) {
  const bool trace = std::getenv("OPE_BATCH_TRACE") != nullptr;
  auto now = [] { return std::chrono::steady_clock::now(); };
  auto ms_since = [&](std::chrono::steady_clock::time_point t) { return std::chrono::duration<double, std::milli>(now() - t).count(); };
  const auto t_enter = now();
  auto smem_bytes = [](size_t n_tgt) {   // block state, the target in groups of 8 with a box per group, the candidate slab
    const size_t nt8 = (n_tgt + 7) & ~(size_t)7;
    return ((sizeof(IcpSmallSmem<kIcpSmallThreads>) + 15) & ~(size_t)15) + nt8 * sizeof(float4) + (nt8 / 8) * 2 * sizeof(float4) +
           (size_t)kSlabSlots * kIcpSmallThreads * sizeof(float2);
  };
  const void* kernel = (const void*)icp_small_batch_kernel<kIcpSmallThreads>;
  // A ticketed block spins on its alignment's barrier, and up to kMaxLanes lanes launch this kernel at once: each lane can park
  // all but one block of an alignment, and the device must still hold one more alignment whole. Counted at the largest target
  // the envelope admits, so the bound holds whatever the other lanes launch.
  const size_t smem_max = smem_bytes(kIcpSmemMaxTargets);
  OPE_TRY(dyn_smem(ctx, kernel, smem_max));
  int per_sm = 0;
  OPE_CUDA_TRY(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kIcpSmallThreads, smem_max));
  if (kMaxLanes * (kIcpSmallMaxBlocks - 1) + kIcpSmallMaxBlocks > per_sm * ctx->sm_count)
    return fail(ctx, OPE_ERR_CUDA, "icp_small_batch_kernel: %d resident blocks cannot hold %d lanes of %d-block alignments",
                per_sm * ctx->sm_count, kMaxLanes, kIcpSmallMaxBlocks);
  size_t max_nt = 0, total_blocks = 0;
  for (int i = 0; i < n; ++i) {
    max_nt = std::max(max_nt, (size_t)descs[i].n_tgt);
    total_blocks += div_up((size_t)descs[i].n_work, kIcpSmallThreads);
  }
  Scratch<double> partials(ctx);
  Scratch<unsigned> bars(ctx);
  Scratch<IcpDev> d_descs(ctx);
  Scratch<int2> d_map(ctx);
  OPE_TRY(partials.alloc(2 * total_blocks * kIcpAcc));
  OPE_TRY(bars.alloc((size_t)n + 1));   // the alignments' barriers, then the ticket counter
  OPE_TRY(d_descs.alloc((size_t)n)); OPE_TRY(d_map.alloc(total_blocks));
  OPE_CUDA_TRY(ctx, cudaMemsetAsync(bars.p, 0, ((size_t)n + 1) * sizeof(unsigned), ctx->stream));
  std::vector<int2> map;
  map.reserve(total_blocks);
  for (int i = 0; i < n; ++i) {
    descs[i].partials = partials.p + 2 * map.size() * kIcpAcc;
    descs[i].barrier = bars.p + i;
    for (int b = 0; b * kIcpSmallThreads < descs[i].n_work; ++b) map.push_back(make_int2(i, b));
  }
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_descs.p, descs, (size_t)n * sizeof(IcpDev), cudaMemcpyHostToDevice, ctx->stream));
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_map.p, map.data(), map.size() * sizeof(int2), cudaMemcpyHostToDevice, ctx->stream));
  const double t_prep = ms_since(t_enter);
  OPE_CUDA_TRY(ctx, ope::stream_sync(ctx));   // map and the caller's descs are gone or reused after the return
  if (trace) fprintf(stderr, "[ope batch] icp launch: host preparation %.3f ms, then %.3f ms until the stream had drained\n", t_prep, ms_since(t_enter) - t_prep);
  unsigned* ticket = bars.p + n;
  void* args[] = {(void*)&d_descs.p, (void*)&d_map.p, (void*)&ticket};
  const dim3 grid((unsigned)total_blocks), block(kIcpSmallThreads);
  const size_t smem = smem_bytes(max_nt);
  cudaEventRecord(ctx->kev[0][0], ctx->stream);
  const cudaError_t e = n == 1 ? cudaLaunchCooperativeKernel(kernel, grid, block, args, smem, ctx->stream)
                               : cudaLaunchKernel(kernel, grid, block, args, smem, ctx->stream);
  cudaEventRecord(ctx->kev[0][1], ctx->stream);
  ctx->kev_valid[0] = true;
  if (e != cudaSuccess) return fail(ctx, OPE_ERR_CUDA, "launch of icp_small_batch_kernel failed: %s", cudaGetErrorString(e));
  return check_launch(ctx, "icp_small_batch_kernel");
}

// icp_kernel on descriptor a (filled but for its search scratch, partials and barrier): one persistent cooperative launch, its
// grid (*blocks) sized by the query count and capped by co-residency and ctx->icp_max_blocks
static int icp_kernel_launch(ope_ctx* ctx, IcpDev a, int* blocks) {
  const bool shooting = a.estimator == OPE_EST_NORMAL_SHOOTING;
  const size_t nw = (size_t)a.n_work;
  const size_t smem_bytes = ((sizeof(IcpSmem) + 15) & ~(size_t)15) + (a.tgt_in_smem ? (size_t)a.n_tgt * sizeof(float4) : 0);
  Scratch<int> seed(ctx), dcount(ctx), dhead(ctx);
  Scratch<float4> defq(ctx), refs(ctx), defres(ctx);
  Scratch<int4> defm(ctx);
  Scratch<double> partials(ctx);
  Scratch<unsigned> bar(ctx);
  OPE_TRY(seed.alloc(shooting ? nw * (size_t)a.k_search : nw));
  if (!shooting) {
    OPE_TRY(defq.alloc(nw)); OPE_TRY(defm.alloc(nw)); OPE_TRY(refs.alloc(nw)); OPE_TRY(defres.alloc(nw));
  }
  OPE_TRY(bar.alloc(1));
  if (cudaMemsetAsync(bar.p, 0, sizeof(unsigned), ctx->stream) != cudaSuccess) return fail(ctx, OPE_ERR_CUDA, "memset failed");
  OPE_TRY(dyn_smem(ctx, (const void*)icp_kernel, smem_bytes));
  // cooperative grid: one point per thread (nearest) / per warp (normal shooting), capped by co-residency
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, icp_kernel, kIcpThreads, smem_bytes) != cudaSuccess)
    return fail(ctx, OPE_ERR_CUDA, "occupancy query failed");
  if (per_sm < 1) return fail(ctx, OPE_ERR_CUDA, "icp_kernel cannot be resident");
  int max_blocks = std::min(per_sm * ctx->sm_count, kIcpMaxBlocks);
  if (ctx->icp_max_blocks > 0) max_blocks = std::min(max_blocks, ctx->icp_max_blocks);
  const size_t want = shooting ? (nw + kIcpWarps - 1) / kIcpWarps : (nw + 127) / 128;
  *blocks = (int)std::min<size_t>(std::max<size_t>(1, want), (size_t)max_blocks);
  OPE_TRY(partials.alloc((size_t)2 * *blocks * kIcpAcc));
  OPE_TRY(dcount.alloc((size_t)2 * *blocks));
  OPE_TRY(dhead.alloc(4));
  if (cudaMemsetAsync(dhead.p, 0, 4 * sizeof(int), ctx->stream) != cudaSuccess) return fail(ctx, OPE_ERR_CUDA, "memset failed");
  a.seed = seed.p; a.def_q = defq.p; a.def_m = defm.p; a.def_count = dcount.p;
  a.ref = refs.p; a.def_head = dhead.p; a.def_res = defres.p;
  const char* g = std::getenv("OPE_ICP_CERT_GAP");  // in target-grid cells; 0 disables the certificates (every query searches)
  a.cert_gap = (g ? (float)std::atof(g) : 0.5f) * a.grid.h;
  const char* d = std::getenv("OPE_ICP_DFS_MAX");
  a.dfs_max = d ? std::atoi(d) : 0;   // measured: a single thread's traversal is a long dependent chain; the warp queue wins
  const char* sp_ = std::getenv("OPE_ICP_SPLIT_MIN");
  a.split_min = sp_ ? std::atoi(sp_) : kIcpSplitMin;
  a.partials = partials.p; a.barrier = bar.p;
  void* args[] = {(void*)&a};
  cudaEventRecord(ctx->kev[0][0], ctx->stream);
  cudaError_t e = cudaLaunchCooperativeKernel((const void*)icp_kernel, dim3(*blocks), dim3(kIcpThreads), args, smem_bytes, ctx->stream);
  cudaEventRecord(ctx->kev[0][1], ctx->stream);
  ctx->kev_valid[0] = true;
  if (e != cudaSuccess) return fail(ctx, OPE_ERR_CUDA, "cooperative launch of icp_kernel failed: %s", cudaGetErrorString(e));
  return check_launch(ctx, "icp_kernel");
}

int icp_device(ope_ctx* ctx, const ope_cloud* src, const ope_cloud* tgt, const ope_icp_params& prm, const Mat4& guess,
               ope_reg_result* res, ope_correspondence* out_corr_host, ope_cloud** out_aligned) {
  if (prm.transformation != OPE_TE_SVD || prm.use_reciprocal)
    return icp_stepwise_device(ctx, src, tgt, prm, guess, res, out_corr_host, out_aligned);
  IcpDev a;
  std::memset(&a, 0, sizeof(a));
  OPE_TRY(icp_fill(ctx, src, tgt, prm, &a, /*allow_smem_target=*/true));
  a.guess = guess;
  const size_t n = src->n;
  // the source in Morton order of its own (cached) grid: spatially coherent work order, finite points only
  GridView gsrc;
  std::memset(&gsrc, 0, sizeof(gsrc));
  if (n > 0) OPE_TRY(cloud_any_grid(ctx, src, &gsrc));
  a.src_sorted = gsrc.pts;
  a.n_work = gsrc.n;
  const size_t nw = (size_t)a.n_work;
  ope_cloud* work = nullptr;
  OPE_TRY(cloud_alloc(ctx, std::max<size_t>(n, 1), src->normals != nullptr, &work));
  work->n = n;
  a.cur_pts = work->pts; a.cur_nrm = work->normals;
  Scratch<int> match(ctx);
  Scratch<float> d2(ctx);
  Scratch<ope_reg_result> dres(ctx);
  int rc = match.alloc(n);
  if (rc == OPE_OK) rc = d2.alloc(n);
  if (rc == OPE_OK) rc = dres.alloc(1);
  if (rc == OPE_OK && n > 0 && cudaMemsetAsync(match.p, 0xff, n * sizeof(int), ctx->stream) != cudaSuccess) rc = fail(ctx, OPE_ERR_CUDA, "memset failed");
  if (rc == OPE_OK && n > 0 && cudaMemsetAsync(d2.p, 0, n * sizeof(float), ctx->stream) != cudaSuccess) rc = fail(ctx, OPE_ERR_CUDA, "memset failed");
  Scratch<long long> phases(ctx);
  const bool profile = std::getenv("OPE_PROFILE") != nullptr;
  const size_t n_prof = 16 + 64 * 8 + 64 + 64 * 4;
  if (rc == OPE_OK && profile) {
    rc = phases.alloc(n_prof); a.phase_cycles = phases.p;
    if (rc == OPE_OK) cudaMemsetAsync(phases.p, 0, n_prof * sizeof(long long), ctx->stream);
  }
  a.corr_match = match.p; a.corr_d2 = d2.p; a.result = dres.p;
  // Small clouds against a shared-memory target: one point per thread, a one-alignment run of the frame-spanning kernel.
  // It trades the latency of one alignment (the wide kernel spreads it over the whole device) for device time per alignment,
  // so it is what a batch of concurrent alignments wants (ope_pose_batch sets ctx->icp_prefer_small); OPE_ICP_SMALL=1/0 forces.
  const char* small_env = std::getenv("OPE_ICP_SMALL");
  const bool want_small = small_env ? std::atoi(small_env) != 0 : ctx->icp_prefer_small;
  const bool small = want_small && a.tgt_in_smem && icp_small_applicable(prm, nw, tgt->n);
  int blocks = (int)div_up(nw, kIcpSmallThreads);
  if (rc == OPE_OK) rc = small ? icp_small_launch(ctx, &a, 1) : icp_kernel_launch(ctx, a, &blocks);
  if (rc == OPE_OK) {
    void* h;
    rc = read_back(ctx, dres.p, sizeof(ope_reg_result), &h);
    if (rc == OPE_OK) std::memcpy(res, h, sizeof(ope_reg_result));
  }
  if (rc == OPE_OK && profile) {
    void* h;
    if (small) {
      if (read_back(ctx, phases.p, 6 * sizeof(long long), &h) == OPE_OK) {
        const long long* c = (const long long*)h;
        const double it = std::max(res->iterations, 1);
        if (std::getenv("OPE_PROFILE_ITER")) {
          std::vector<long long> all(n_prof);
          if (cudaMemcpy(all.data(), phases.p, n_prof * sizeof(long long), cudaMemcpyDeviceToHost) == cudaSuccess) {
            fprintf(stderr, "[ope profile] icp_small per iteration: mean warp scan cycles | slowest warp | overflow calls | threads overflowing | candidates per query\n");
            for (int p = 0; p < std::min(res->iterations, 64); ++p) {
              const long long* r = all.data() + 16 + p * 8;
              fprintf(stderr, "  it %2d: %7.0f %7lld %6lld %5lld %5.1f\n", p, (double)r[0] / (double)std::max<long long>(r[5], 1), r[1], r[2], r[3],
                      (double)r[4] / (double)std::max<size_t>(nw, 1));
            }
          }
        }
        fprintf(stderr, "[ope profile] icp_small_batch_kernel blocks=%d, block 0 cycles per iteration: search %.0f | rank+shoot+reject %.0f | moments+barrier %.0f | "
                "svd+transform %.0f | cooperative re-searches per iteration %.1f | candidates per query %.1f\n", blocks, c[0] / it, c[1] / it,
                c[2] / it, c[3] / it, c[4] / it, c[5] / it / kIcpSmallThreads);
      }
    } else if (read_back(ctx, phases.p, n_prof * sizeof(long long), &h) == OPE_OK) {
      const long long* c = (const long long*)h;
      const double it = std::max(res->iterations, 1);
      if (std::getenv("OPE_PROFILE_ITER")) {
        fprintf(stderr, "[ope profile] per iteration (block 0 cycles): A | bar1 | B | bar2 | far-moments+bar3 | C | xform | slowest far query (grid) | far queries (grid)\n");
        for (int p = 0; p < std::min(res->iterations, 64); ++p) {
          const long long* r = c + 16 + p * 8;
          const long long* k = c + 16 + 64 * 8 + 64 + p * 4;
          const double nq = (double)std::max<long long>(c[16 + 64 * 8 + p], 1);
          fprintf(stderr, "  it %2d: %7lld %7lld %7lld %7lld %7lld %7lld %6lld | %8lld | %6lld | per far query: %.1f pops %.1f leaves %.0f points %.1f flushes\n",
                  p, r[0], r[1], r[2], r[3], r[4], r[5], r[6], r[7], c[16 + 64 * 8 + p], k[0] / nq, k[1] / nq, k[2] / nq, k[3] / nq);
        }
      }
      fprintf(stderr, "[ope profile] icp_kernel blocks=%d, block 0 cycles per iteration: A fast path %.0f | barrier1 %.0f | B far queue %.0f | "
              "barrier2 %.0f | far moments + barrier3 %.0f | C partials+svd %.0f | transform %.0f | far queries of block 0: %.1f\n",
              blocks, c[0] / it, c[1] / it, c[2] / it, c[3] / it, c[4] / it, c[5] / it, c[6] / it, c[7] / it);
    }
  }
  if (rc == OPE_OK && out_corr_host && n > 0) {
    std::vector<int> hm(n);
    std::vector<float> hd(n);
    cudaError_t e = cudaMemcpyAsync(hm.data(), match.p, n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(hd.data(), d2.p, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = ope::stream_sync(ctx);
    if (e != cudaSuccess) rc = fail(ctx, OPE_ERR_CUDA, "correspondence download failed: %s", cudaGetErrorString(e));
    else corr_to_host(hm, hd, out_corr_host, nullptr);
  }
  if (rc == OPE_OK && out_aligned) {
    // output = *input_ transformed by the final transformation (VP/impl/icp_mod.hpp:269-271)
    Mat4 F;
    std::memcpy(F.m, res->T, sizeof(F.m));
    rc = transform_device(ctx, src, F, work);
    if (rc == OPE_OK) { *out_aligned = work; work = nullptr; }
  }
  if (work) ope_cloud_free(ctx, work);
  return rc;
}

// IterativeClosestPoint::computeTransformation (VP/impl/icp_mod.hpp:118-272) with a point-to-plane transformation estimator
// (BuildModel's getIcpNormal, BM/src/regmeshpcd.cpp:104-208; IterativeClosestPointWithNormals' default LLS, VP/icp_mod.h:352-357).
// The estimator is iterative itself (Levenberg-Marquardt: several reductions per ICP iteration, steered by 6x6 algebra on the
// host), so this loop is sequenced from the host: correspondences + rejectors (one launch), estimation (p2plane.cu), transform
// in place, DefaultConvergenceCriteria in double on the host. Everything the kernels read stays on the device; per step only
// the 28 reduced doubles come back.
// Umeyama over explicit pairs for the host-sequenced loop: double moments on the device, the 3x3 SVD on the host (same
// arithmetic as the fused kernel's lane 0: umeyama_from_moments is host/device code compiled without contraction)
static int svd_pairs_device(ope_ctx* ctx, const float4* src, const ope_cloud* tgt, const double origin[3], const int* d_is, const int* d_it,
                            const float* d_d2, size_t n, Mat4* T, int* n_pairs, double* sum_d2) {
  *T = mat4_identity(); *n_pairs = 0; *sum_d2 = 0.0;
  if (n == 0) return OPE_OK;
  const int nb = (int)std::min<size_t>(std::max<size_t>(1, (n + kRedThreads - 1) / kRedThreads), (size_t)ctx->sm_count * 4);
  Scratch<double> partials(ctx), out(ctx);
  OPE_TRY(partials.alloc((size_t)nb * kPairAcc));
  OPE_TRY(out.alloc(kPairAcc));
  pairs_moments_kernel<<<nb, kRedThreads, 0, ctx->stream>>>(src, tgt->pts, d_is, d_it, d_d2, (int)n, partials.p);
  OPE_TRY(check_launch(ctx, "pairs_moments_kernel"));
  sum_partials_kernel<<<1, 32 * kPairAcc, 0, ctx->stream>>>(partials.p, nb, kPairAcc, out.p);
  OPE_TRY(check_launch(ctx, "sum_partials_kernel"));
  void* h;
  OPE_TRY(read_back(ctx, out.p, kPairAcc * sizeof(double), &h));
  const double* acc = (const double*)h;
  *n_pairs = (int)acc[0];
  *sum_d2 = acc[kMomentAcc];
  if (*n_pairs > 0) umeyama_from_moments(acc, *T, origin[0], origin[1], origin[2]);
  return OPE_OK;
}

// The host-sequenced ICP loop: one launch for correspondences + rejectors, optional reciprocal filter and fixed pairs, the
// transformation estimate (SVD / point-to-plane LLS / LM), the transform, DefaultConvergenceCriteria on the host. Used whenever
// the fused kernel does not apply: point-to-plane estimators, reciprocal correspondences, fixed correspondences.
static int icp_stepwise_device(ope_ctx* ctx, const ope_cloud* src, const ope_cloud* tgt, const ope_icp_params& prm, const Mat4& guess,
                               ope_reg_result* res, ope_correspondence* out_corr_host, ope_cloud** out_aligned, ope_correspondence* fixed,
                               size_t n_fixed) {
  IcpDev a;
  std::memset(&a, 0, sizeof(a));
  OPE_TRY(icp_fill(ctx, src, tgt, prm, &a));
  const size_t n = src->n;
  const bool shooting = prm.estimator == OPE_EST_NORMAL_SHOOTING;
  // icp_modCorr.h has no setFixedCorrespondences. Normal shooting never puts the fixed pairs in front of its result (VP/impl/
  // correspondence_estimation_normal_shooting_weighted.hpp:81-100), but the loop still appends them after rejector 0 with the
  // caller's distances (VP/impl/icp_mod.hpp:209-225), as for the reciprocal estimator; without rejectors nothing is appended.
  if (prm.variant != OPE_ICP_VARIANT_MOD || (shooting && prm.n_rejectors == 0)) n_fixed = 0;
  const size_t F = n_fixed;
  for (size_t j = 0; j < F; ++j)
    if (fixed[j].index_query < 0 || (size_t)fixed[j].index_query >= n || fixed[j].index_match < 0 || (size_t)fixed[j].index_match >= tgt->n)
      return fail(ctx, OPE_ERR_INVALID, "fixed correspondence %zu out of range", j);
  ope_cloud *work = nullptr, *next = nullptr;   // ping-pong: transform_kernel reads through the read-only path
  struct Guard { ope_ctx* c; ope_cloud*& w; ~Guard() { if (w) ope_cloud_free(c, w); } } guard{ctx, work}, guard2{ctx, next};
  OPE_TRY(cloud_alloc(ctx, std::max<size_t>(n, 1), src->normals != nullptr, &work));
  OPE_TRY(cloud_alloc(ctx, std::max<size_t>(n, 1), src->normals != nullptr, &next));
  work->n = next->n = n;
  Mat4 final_t = guess;
  if (n > 0) OPE_TRY(transform_device(ctx, src, guess, work));   // identity guess: a plain copy
  // pair arrays: [0, F) fixed pairs through the whole rejector chain, [F, 2F) through rejector 0 alone, [2F, 2F + n) estimated
  Scratch<int> is(ctx), match(ctx), seed(ctx), fq(ctx), fm(ctx);
  Scratch<float> d2(ctx);
  OPE_TRY(match.alloc(n + 2 * F)); OPE_TRY(d2.alloc(n + 2 * F));
  OPE_TRY(seed.alloc(shooting ? n * (size_t)prm.k_search : n));
  std::vector<int> h_is, h_fq(F), h_fm(F);
  if (F) {
    OPE_TRY(is.alloc(n + 2 * F)); OPE_TRY(fq.alloc(F)); OPE_TRY(fm.alloc(F));
    h_is.resize(n + 2 * F);
    std::vector<float> h_fd(2 * F);
    for (size_t j = 0; j < F; ++j) { h_fq[j] = fixed[j].index_query; h_fm[j] = fixed[j].index_match; h_fd[j] = h_fd[F + j] = fixed[j].distance; }
    for (size_t i = 0; i < n; ++i) h_is[2 * F + i] = (int)i;
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(is.p, h_is.data(), (n + 2 * F) * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(fq.p, h_fq.data(), F * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(fm.p, h_fm.data(), F * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d2.p, h_fd.data(), 2 * F * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    // a pair naming a NaN / inf point has no defined result (its 1e10-scaled distance and the moments turn NaN): refused
    Scratch<int> bad(ctx);
    OPE_TRY(bad.alloc(1));
    OPE_CUDA_TRY(ctx, cudaMemsetAsync(bad.p, 0x7f, sizeof(int), ctx->stream));
    fixed_finite_kernel<<<1, 128, 0, ctx->stream>>>(src->pts, tgt->pts, fq.p, fm.p, (int)F, bad.p);
    OPE_TRY(check_launch(ctx, "fixed_finite_kernel"));
    void* h;
    OPE_TRY(read_back(ctx, bad.p, sizeof(int), &h));
    const int first_bad = *(const int*)h;
    if ((size_t)first_bad < F) return fail(ctx, OPE_ERR_INVALID, "fixed correspondence %d names a non-finite point", first_bad);
  }
  a.corr_match = match.p + 2 * F; a.corr_d2 = d2.p + 2 * F; a.seed = seed.p;
  OPE_TRY(dyn_smem(ctx, (const void*)correspond_once_kernel, sizeof(IcpSmem)));
  if (prm.use_reciprocal) OPE_TRY(dyn_smem(ctx, (const void*)reciprocal_filter_kernel, sizeof(IcpSmem)));
  const size_t want = shooting ? div_up(n, kIcpWarps) : div_up(n, kIcpThreads);
  const unsigned blocks = (unsigned)std::max<size_t>(1, std::min<size_t>(want, (size_t)ctx->sm_count * 4));
  double origin[3] = {0, 0, 0};
  if (prm.transformation == OPE_TE_SVD) {   // the moments are taken about the target's first point (see umeyama_from_moments)
    void* h;
    OPE_TRY(read_back(ctx, tgt->pts, sizeof(float4), &h));
    const float4 t0 = *(const float4*)h;
    moment_origin(t0.x, t0.y, t0.z, origin[0], origin[1], origin[2]);
  }
  int iterations = 0, state = OPE_CONV_NOT_CONVERGED, similar = 0, n_corr = 0;
  bool converged = false;
  double prev_mse = DBL_MAX, cur_mse = DBL_MAX;
  const double rot_thr = 1.0 - prm.transformation_epsilon, trans_thr = prm.transformation_epsilon;
  cudaEventRecord(ctx->kev[0][0], ctx->stream);
  do {
    a.cur_pts = work->pts; a.cur_nrm = work->normals;
    if (n > 0) {
      correspond_once_kernel<<<blocks, kIcpThreads, sizeof(IcpSmem), ctx->stream>>>(a);
      OPE_TRY(check_launch(ctx, "correspond_once_kernel"));
    }
    if (prm.use_reciprocal && n > 0) {   // a second index over the source as it stands in this iteration
      OPE_TRY(ope_cloud_invalidate(ctx, work));
      OPE_TRY(cloud_bbox(ctx, work));
      GridView gsrc;
      OPE_TRY(cloud_grid(ctx, work, knn_cell_size(work, 1), &gsrc));
      reciprocal_filter_kernel<<<blocks, kIcpThreads, sizeof(IcpSmem), ctx->stream>>>(gsrc, tgt->pts, a.corr_match, (int)n, a.max_d2_f,
                                                                                      a.max_corr_dist);
      OPE_TRY(check_launch(ctx, "reciprocal_filter_kernel"));
    }
    if (F) {
      // front = 0 (reciprocal, shooting): slots [0, F) stay -1, the tail keeps the caller's distances
      fixed_pairs_kernel<<<1, 128, 0, ctx->stream>>>(a, fq.p, fm.p, (int)F, (prm.use_reciprocal || shooting) ? 0 : 1, is.p, match.p, d2.p);
      OPE_TRY(check_launch(ctx, "fixed_pairs_kernel"));
    }
    Mat4 T = mat4_identity();
    double sum_d2 = 0.0;
    if (prm.transformation == OPE_TE_SVD)
      OPE_TRY(svd_pairs_device(ctx, work->pts, tgt, origin, F ? is.p : nullptr, match.p, d2.p, n + 2 * F, &T, &n_corr, &sum_d2));
    else
      OPE_TRY(point_to_plane_device(ctx, work->pts, tgt->pts, tgt->normals, F ? is.p : nullptr, match.p, d2.p, n + 2 * F, prm.transformation,
                                    &T, &n_corr, &sum_d2, nullptr));
    if (n_corr < prm.min_number_correspondences) {   // VP/impl/icp_mod.hpp:232-240
      state = OPE_CONV_NO_CORRESPONDENCES;
      converged = false;
      break;
    }
    if (n > 0) OPE_TRY(transform_device(ctx, work, T, next));   // transformCloud(*input_transformed, *input_transformed, transformation_)
    std::swap(work, next);
    final_t = mat4_mul(T, final_t);
    ++iterations;
    // DefaultConvergenceCriteria::hasConverged (VP/default_convergence_criteria_mod.h:64-282)
    state = OPE_CONV_NOT_CONVERGED;
    bool conv = false;
    auto similar_or_done = [&](int st) {
      if (similar < prm.max_iterations_similar_transforms) { ++similar; return false; }
      similar = 0; state = st; return true;
    };
    if (iterations >= prm.max_iterations) {
      if (!prm.failure_after_max_iterations) { state = OPE_CONV_ITERATIONS; conv = true; }
      else { converged = false; break; }
    } else {
      // float trace and float squared norm, widened afterwards: the arithmetic of Matrix4f expressions [UPSTREAM hasConverged]
      const double cos_angle = 0.5 * (double)(T(0, 0) + T(1, 1) + T(2, 2) - 1);
      const double tr2 = (double)(T(0, 3) * T(0, 3) + T(1, 3) * T(1, 3) + T(2, 3) * T(2, 3));
      if (cos_angle >= rot_thr && tr2 <= trans_thr) {
        conv = similar_or_done(OPE_CONV_TRANSFORM);
      } else {
        cur_mse = sum_d2 / (double)n_corr;
        if (std::fabs(cur_mse - prev_mse) < prm.mse_threshold_absolute) conv = similar_or_done(OPE_CONV_ABS_MSE);
        else if (std::fabs(cur_mse - prev_mse) / prev_mse < prm.euclidean_fitness_epsilon) conv = similar_or_done(OPE_CONV_REL_MSE);
        else prev_mse = cur_mse;
      }
    }
    converged = conv;
    if (prm.force_all_iterations && iterations < prm.max_iterations) converged = false;
  } while (!converged);
  cudaEventRecord(ctx->kev[0][1], ctx->stream);
  ctx->kev_valid[0] = true;
  std::memcpy(res->T, final_t.m, sizeof(final_t.m));
  res->converged = converged ? 1 : 0;
  res->state = state;
  res->iterations = iterations;
  res->n_correspondences = n_corr;
  res->last_mse = cur_mse;
  res->best_error = 0.0; res->best_iteration = 0; res->reserved = 0;
  if ((out_corr_host || F) && n + 2 * F > 0) {
    std::vector<int> hm(n + 2 * F);
    std::vector<float> hd(n + 2 * F);
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(hm.data(), match.p, (n + 2 * F) * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(hd.data(), d2.p, (n + 2 * F) * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    OPE_CUDA_TRY(ctx, ope::stream_sync(ctx));
    for (size_t j = 0; j < F; ++j) fixed[j].distance = hd[j];   // the loop rewrites the caller's list (it->distance = ...)
    if (out_corr_host) {   // the reference's order: fixed (whole chain), estimated, fixed again (rejector 0 alone)
      size_t w = 0;
      for (size_t j = 0; j < F; ++j) if (hm[j] >= 0) out_corr_host[w++] = ope_correspondence{h_fq[j], hm[j], hd[j]};
      for (size_t i = 0; i < n; ++i) if (hm[2 * F + i] >= 0) out_corr_host[w++] = ope_correspondence{(int32_t)i, hm[2 * F + i], hd[2 * F + i]};
      for (size_t j = 0; j < F; ++j) if (hm[F + j] >= 0) out_corr_host[w++] = ope_correspondence{h_fq[j], hm[F + j], hd[F + j]};
    }
  }
  if (out_aligned) {
    if (n > 0) OPE_TRY(transform_device(ctx, src, final_t, work));   // output = *input_ under the final transformation, :269-271
    *out_aligned = work;
    work = nullptr;
  }
  return OPE_OK;
}

// ---- the process-wide libc rand() stream, consumed in bulk ----------------------------------------------------------------
// SAC-IA draws ~4 000 numbers per alignment from rand(), and they must be THE numbers a loop over fresh PoseEstimators would get
// from the process's stream. glibc's rand() takes a lock per call (~25 ns); its generator itself (random_r.c: an additive
// feedback generator over 7 / 15 / 31 / 63 words, or an LCG for the 8-byte state) is three instructions. A session borrows the
// stream through the public API — initstate() hands back the live state array with the rear pointer's position encoded in front
// of it — advances it in place, and gives it back with setstate(), which resumes from exactly where the session stopped. A
// one-time self-test replays a few numbers against rand() itself (and rewinds); on any mismatch, or on another libc, every draw
// goes through rand().
class LibcRandSession {
 public:
  LibcRandSession() {
#if defined(__GLIBC__)
    if (!usable()) return;
    begin();
#endif
  }
  ~LibcRandSession() {
#if defined(__GLIBC__)
    if (state_) end();
#endif
  }
  LibcRandSession(const LibcRandSession&) = delete;
  LibcRandSession& operator=(const LibcRandSession&) = delete;
  inline int next() {
#if defined(__GLIBC__)
    if (state_) return step();
#endif
    return rand();
  }
  // [UPSTREAM ia_ransac.hpp getRandomIndex]: n * (rand() / (RAND_MAX + 1.0)), truncated. With RAND_MAX = 2^31 - 1 and 0 <= n <= 2^21
  // the double product n * r / 2^31 is exact (at most 52 significant bits), so its truncation is the integer (n * r) >> 31.
  inline int index(int n) {
    const int r = next();
#if RAND_MAX == 2147483647
    if (n >= 0 && n <= (1 << 21)) return (int)(((long long)n * (long long)r) >> 31);
#endif
    return (int)(n * (r / (RAND_MAX + 1.0)));
  }

 private:
#if defined(__GLIBC__)
  int32_t* word_ = nullptr;    // what initstate() returned: the word in front of the state array
  int32_t* state_ = nullptr;   // null: not borrowed, next() calls rand()
  int32_t *fptr_ = nullptr, *rptr_ = nullptr, *end_ = nullptr;
  int type_ = 0;

  bool begin() {
    static const int kDeg[5] = {0, 7, 15, 31, 63}, kSep[5] = {0, 3, 1, 3, 1};
    borrow_mutex().lock();   // one borrower at a time (concurrent drawers would interleave their numbers anyway)
    // the state libc runs on while its own is borrowed (nobody draws from it): seeded once, switched to with setstate() afterwards
    alignas(8) static char parked[128];
    static bool parked_ready = false;
    char* prev = parked_ready ? setstate(parked) : initstate(1u, parked, sizeof(parked));
    parked_ready = true;
    if (!prev) { borrow_mutex().unlock(); return false; }
    word_ = reinterpret_cast<int32_t*>(prev);
    type_ = word_[0] % 5;
    const int rear = word_[0] / 5;
    if (type_ < 0 || type_ > 4 || (type_ > 0 && (rear < 0 || rear >= kDeg[type_]))) {
      setstate(prev);
      word_ = nullptr;
      borrow_mutex().unlock();
      return false;
    }
    state_ = word_ + 1;
    if (type_ > 0) { rptr_ = state_ + rear; fptr_ = state_ + (rear + kSep[type_]) % kDeg[type_]; end_ = state_ + kDeg[type_]; }
    return true;
  }
  void end() {
    word_[0] = type_ == 0 ? 0 : (int32_t)(5 * (rptr_ - state_) + type_);
    setstate(reinterpret_cast<char*>(word_));
    state_ = nullptr;
    borrow_mutex().unlock();
  }
  static std::mutex& borrow_mutex() { static std::mutex m; return m; }
  inline int step() {
    if (type_ == 0) {
      const int32_t v = (int32_t)(((uint32_t)state_[0] * 1103515245u + 12345u) & 0x7fffffffu);
      state_[0] = v;
      return v;
    }
    const uint32_t v = (uint32_t)*fptr_ + (uint32_t)*rptr_;
    *fptr_ = (int32_t)v;
    ++fptr_;
    if (fptr_ >= end_) { fptr_ = state_; ++rptr_; }
    else { ++rptr_; if (rptr_ >= end_) rptr_ = state_; }
    return (int)(v >> 1);
  }
  // once per process: eight numbers drawn in a borrowed session against the same eight from rand(), the stream rewound after each
  // (libc ends up on its own state array, in its original state: nothing keeps pointing into this library)
  static bool usable() {
    static std::once_flag once;
    static bool ok = false;
    std::call_once(once, [] {
      if (const char* e = std::getenv("OPE_LIBC_RAND_FAST")) { if (std::atoi(e) == 0) return; }
      int32_t saved[65];   // header word + up to 63 state words
      int fast[8], slow[8];
      LibcRandSession probe(0);
      auto rewind = [&](size_t words) {   // borrowed: put the saved state back and return the array to libc
        std::memcpy(probe.word_, saved, words * sizeof(int32_t));
        probe.state_ = nullptr;
        setstate(reinterpret_cast<char*>(probe.word_));
        borrow_mutex().unlock();
      };
      if (!probe.begin()) return;
      const size_t words = probe.type_ == 0 ? 2 : (size_t)(probe.end_ - probe.state_) + 1;
      std::memcpy(saved, probe.word_, words * sizeof(int32_t));   // initstate() has just encoded the rear pointer in the header
      for (int i = 0; i < 8; ++i) fast[i] = probe.step();
      rewind(words);
      for (int i = 0; i < 8; ++i) slow[i] = rand();
      if (!probe.begin()) return;
      rewind(words);
      ok = std::memcmp(fast, slow, sizeof(fast)) == 0;
    });
    return ok;
  }
  explicit LibcRandSession(int) {}   // the self-test's probe: no borrowing in the constructor
#endif
};

// the smallest float s with sqrtf(s) >= m: `sqrtf(s) < m` (sqrtf is correctly rounded and monotone) is exactly `s < that`
static float sqrt_threshold(float m) {
  if (!(m > 0.0f)) return 0.0f;                      // nothing is closer than a non-positive (or NaN) distance
  float c = m * m;
  if (!(c < INFINITY)) return INFINITY;              // (a distance limit beyond sqrt(FLT_MAX): every finite distance is closer)
  while (c > 0.0f && std::sqrt(c) >= m) c = std::nextafter(c, 0.0f);
  while (std::sqrt(c) < m) c = std::nextafter(c, INFINITY);
  return c;
}

// selectSamples [UPSTREAM ia_ransac.hpp] on the host: it consumes libc rand() serially (SURVEY hard part 3)
static int draw_samples(LibcRandSession& rng, const float* src, size_t ns, size_t stride_f, int nr_samples, float& min_sample_distance,
                        int32_t* out) {
  if (nr_samples > (int)ns) return OPE_ERR_INVALID;
  int without = 0;
  const int max_without = (int)(3 * ns);
  int cnt = 0;
  float too_close = sqrt_threshold(min_sample_distance);   // squared-distance form of `distance < min_sample_distance`
  while (cnt < nr_samples) {
    const int si = rng.index((int)ns);
    bool valid = true;
    const float* a = src + (size_t)si * stride_f;
    for (int i = 0; i < cnt; ++i) {
      const float* b = src + (size_t)out[i] * stride_f;
      const float dx = a[0] - b[0], dy = a[1] - b[1], dz = a[2] - b[2];
      float s = dx * dx;     // (this file is compiled without contraction: three roundings, like the reference's float code)
      s = s + dy * dy;
      s = s + dz * dz;
      if (si == out[i] || s < too_close) { valid = false; break; }
    }
    if (valid) { out[cnt++] = si; without = 0; }
    else ++without;
    if (without >= max_without) { min_sample_distance *= 0.5f; too_close = sqrt_threshold(min_sample_distance); without = 0; }
  }
  return OPE_OK;
}

// dynamic shared memory of sacia_score_batch_kernel: the target padded to groups of 8, the group boxes, the terms, the seed grid
static size_t sacia_score_bytes(int max_nt, int ns) {
  const size_t nt8 = ((size_t)max_nt + 7) & ~(size_t)7;
  return (nt8 + 2 * (nt8 / 8)) * sizeof(float4) + (size_t)ns * sizeof(float) + (size_t)kSeedCells * sizeof(unsigned short);
}

int sacia_device(ope_ctx* ctx, const ope_cloud* src, const float* d_fsrc, const ope_cloud* tgt, const float* d_ftgt,
                 const ope_sacia_params& prm, const ope_rng_table* table, const float* host_src_xyz3, ope_reg_result* res,
                 float* out_errors_host) {
  const int H = prm.max_iterations, S = prm.nr_samples, K = prm.k_correspondences;
  if (H < 1 || S < 1 || S > kSaciaMaxSamples || K < 1 || K > 16) return fail(ctx, OPE_ERR_INVALID, "bad SAC-IA parameters");
  if (src->n == 0 || tgt->n == 0) return fail(ctx, OPE_ERR_EMPTY, "empty cloud");
  if ((size_t)S > src->n) return fail(ctx, OPE_ERR_INVALID, "The number of samples must not be greater than the number of points");
  int h0 = 0, h1 = H;
  if (prm.hypothesis_end > prm.hypothesis_begin) { h0 = std::min(H, std::max(0, prm.hypothesis_begin)); h1 = std::max(h0, std::min(H, prm.hypothesis_end)); }
  float final_msd = prm.min_sample_distance;
  // ---- decision table: replayed or drawn from libc rand() ----
  std::vector<int32_t> hs, hp;
  const int32_t *samples = nullptr, *picks = nullptr;
  if (table) {
    if (table->n_hypotheses < H || table->nr_samples != S) return fail(ctx, OPE_ERR_INVALID, "rng table shape mismatch");
    samples = table->samples; picks = table->picks;
  } else {
    std::vector<float> xyz;
    const float* hx = host_src_xyz3;
    if (!hx) {
      xyz.resize(3 * src->n);
      OPE_TRY(ope_cloud_download(ctx, src, xyz.data(), nullptr));
      hx = xyz.data();
    }
    hs.resize((size_t)H * S); hp.resize((size_t)H * S);
    float& msd = final_msd;
    LibcRandSession rng;
    for (int it = 0; it < H; ++it) {
      int rc = draw_samples(rng, hx, src->n, 3, S, msd, hs.data() + (size_t)it * S);
      if (rc != OPE_OK) return fail(ctx, rc, "selectSamples failed");
      for (int s = 0; s < S; ++s) hp[(size_t)it * S + s] = rng.index(K);
    }
    samples = hs.data(); picks = hp.data();
  }
  for (size_t i = 0; i < (size_t)H * S; ++i)
    if (samples[i] < 0 || (size_t)samples[i] >= src->n || picks[i] < 0 || picks[i] >= K)
      return fail(ctx, OPE_ERR_INVALID, "rng table entry out of range");
  // ---- device side: a one-frame run of the frame-spanning stages ----
  const size_t ns = src->n;
  Scratch<int> d_samples(ctx), d_picks(ctx), d_knn(ctx), d_frame(ctx);
  Scratch<float> d_errors(ctx), d_T(ctx), d_knn_d2(ctx);
  Scratch<ope_reg_result> d_res(ctx);
  OPE_TRY(d_samples.alloc((size_t)H * S)); OPE_TRY(d_picks.alloc((size_t)H * S));
  OPE_TRY(d_knn.alloc(ns * K)); OPE_TRY(d_knn_d2.alloc(ns * K));
  OPE_TRY(d_errors.alloc(H)); OPE_TRY(d_T.alloc((size_t)H * 16)); OPE_TRY(d_res.alloc(1)); OPE_TRY(d_frame.alloc(2));
  const int frame[2] = {(int)tgt->n, 1};   // counts[0], active[0]
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_samples.p, samples, (size_t)H * S * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_picks.p, picks, (size_t)H * S * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_frame.p, frame, sizeof(frame), cudaMemcpyHostToDevice, ctx->stream));
  OPE_CUDA_TRY(ctx, cudaMemsetAsync(d_errors.p, 0xff, (size_t)H * sizeof(float), ctx->stream));  // NaN = not evaluated
  // findSimilarFeatures for every source point at once (K6)
  OPE_TRY(feature_knn_device(ctx, d_ftgt, tgt->n, d_fsrc, ns, 33, K, d_knn.p, d_knn_d2.p));
  SaciaBatch a;
  std::memset(&a, 0, sizeof(a));
  a.src = src->pts; a.ns = (int)ns; a.tgt = tgt->pts; a.counts = d_frame.p; a.active = d_frame.p + 1;
  a.nr_samples = S; a.k_corr = K; a.H = H; a.h_begin = h0; a.h_end = h1;
  a.samples = d_samples.p; a.picks = d_picks.p; a.knn_idx = d_knn.p;
  a.threshold = (float)prm.max_correspondence_distance; a.errors = d_errors.p; a.transforms = d_T.p;
  a.early_exit = out_errors_host == nullptr;   // a hypothesis that stops early reports +inf: the caller gets every error exactly
  // the shared-memory scorer where the target and the source's terms fit, the grid index otherwise
  const char* force = std::getenv("OPE_SACIA_PATH");   // "grid" / "smem": force a path (tests); default: by size
  bool use_smem = tgt->n <= (size_t)kSaciaSmemMaxTargets && !(force && std::strcmp(force, "grid") == 0);
  if (use_smem) {
    int optin = 0;
    cudaFuncAttributes fa;
    OPE_CUDA_TRY(ctx, cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, ctx->device));
    OPE_CUDA_TRY(ctx, cudaFuncGetAttributes(&fa, (const void*)sacia_score_batch_kernel));
    use_smem = sacia_score_bytes((int)tgt->n, (int)ns) + fa.sharedSizeBytes <= (size_t)optin;
  }
  GridView grid;
  if (!use_smem) {
    OPE_TRY(cloud_bbox(ctx, const_cast<ope_cloud*>(tgt)));
    OPE_TRY(cloud_grid(ctx, tgt, knn_cell_size(tgt, 1), &grid));
  }
  OPE_TRY(sacia_batch_device(ctx, a, 1, (int)tgt->n, use_smem ? nullptr : &grid, d_res.p));
  void* h;
  OPE_TRY(read_back(ctx, d_res.p, sizeof(ope_reg_result), &h));
  std::memcpy(res, h, sizeof(ope_reg_result));
  res->last_mse = (double)final_msd;   // min_sample_distance_ as selectSamples left it (it halves the member and keeps it halved)
  if (out_errors_host) {
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(out_errors_host, d_errors.p, (size_t)H * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    OPE_CUDA_TRY(ctx, ope::stream_sync(ctx));
  }
  return OPE_OK;
}

// ---- the SAC-IA stages, for ope_pose_batch (batch.cu) and, with one frame, sacia_device ----------------------------------
int sacia_batch_device(ope_ctx* ctx, const SaciaBatch& a_in, int frames, int max_nt, const GridView* grid, ope_reg_result* d_results) {
  SaciaBatch a = a_in;
  if (frames <= 0 || a.H <= 0) return OPE_OK;
  if (a.nr_samples < 1 || a.nr_samples > kSaciaMaxSamples || a.k_corr < 1 || a.k_corr > 16) return fail(ctx, OPE_ERR_INVALID, "bad SAC-IA parameters");
  if (a.h_begin < 0 || a.h_end > a.H || a.h_begin > a.h_end) return fail(ctx, OPE_ERR_INVALID, "bad SAC-IA hypothesis range");
  if (grid && (frames != 1 || a.src_counts)) return fail(ctx, OPE_ERR_INVALID, "the grid SAC-IA scorer takes one frame");
  if (!grid && max_nt > kSaciaSmemMaxTargets) return fail(ctx, OPE_ERR_CAPACITY, "batched SAC-IA: target larger than the shared-memory path");
  { const char* e = std::getenv("OPE_SACIA_EARLY_EXIT"); if (e && std::atoi(e) == 0) a.early_exit = 0; }
  const int nh = a.h_end - a.h_begin;
  Scratch<unsigned short> seed_tab(ctx);
  Scratch<float4> seed_geo(ctx), src_scan(ctx);
  Scratch<unsigned> best_bits(ctx);
  Scratch<float> terms(ctx);
  if (nh > 0) {
    sacia_transform_batch_kernel<<<div_up((size_t)frames * nh, 128), 128, 0, ctx->stream>>>(a, frames);
    OPE_TRY(check_launch(ctx, "sacia_transform_batch_kernel"));
  }
  if (nh > 0 && grid) {
    OPE_TRY(terms.alloc((size_t)nh * a.ns));
    OPE_TRY(dyn_smem(ctx, (const void*)sacia_kernel, sizeof(Nn1Smem<kSaciaThreads>)));
    cudaEventRecord(ctx->kev[1][0], ctx->stream);
    sacia_kernel<<<nh, kSaciaThreads, sizeof(Nn1Smem<kSaciaThreads>), ctx->stream>>>(a, *grid, terms.p);
    cudaEventRecord(ctx->kev[1][1], ctx->stream);
    ctx->kev_valid[1] = true;
    OPE_TRY(check_launch(ctx, "sacia_kernel"));
  } else if (nh > 0) {
    OPE_TRY(seed_tab.alloc((size_t)frames * kSeedCells)); OPE_TRY(seed_geo.alloc((size_t)frames)); OPE_TRY(best_bits.alloc((size_t)frames));
    const int sources = a.src_stride ? frames : 1;
    OPE_TRY(src_scan.alloc((size_t)sources * a.ns));
    a.seed_tab = seed_tab.p; a.seed_geo = seed_geo.p; a.best_bits = best_bits.p; a.src_scan = src_scan.p;
    sacia_source_order_kernel<<<sources, kSaciaThreads, 0, ctx->stream>>>(a, a.ns, src_scan.p);
    OPE_TRY(check_launch(ctx, "sacia_source_order_kernel"));
    const size_t nt8 = ((size_t)max_nt + 7) & ~(size_t)7, bytes = sacia_score_bytes(max_nt, a.ns);
    // every block of a frame stages its target and finds the same box; a few frames split the cells over more blocks
    const unsigned seed_blocks = std::max(1u, std::min(div_up(kSeedCells, kSaciaThreads), (unsigned)(2 * ctx->sm_count / frames)));
    OPE_TRY(dyn_smem(ctx, (const void*)sacia_seed_batch_kernel, nt8 * sizeof(float4)));
    sacia_seed_batch_kernel<<<dim3(frames, seed_blocks), kSaciaThreads, nt8 * sizeof(float4), ctx->stream>>>(a);
    OPE_TRY(check_launch(ctx, "sacia_seed_batch_kernel"));
    // kSaciaHypPerBlock hypotheses per block while that still gives every SM two blocks, fewer for a few frames (the winner, its
    // error and its transform do not depend on how the hypotheses are grouped)
    int hyp_per_block = kSaciaHypPerBlock;
    while (hyp_per_block > 1 && (size_t)frames * div_up(nh, hyp_per_block) < 2 * (size_t)ctx->sm_count) hyp_per_block /= 2;
    OPE_TRY(dyn_smem(ctx, (const void*)sacia_score_batch_kernel, bytes));
    cudaEventRecord(ctx->kev[1][0], ctx->stream);
    sacia_score_batch_kernel<<<dim3(frames, div_up(nh, hyp_per_block)), kSaciaScoreThreads, bytes, ctx->stream>>>(a, hyp_per_block);
    cudaEventRecord(ctx->kev[1][1], ctx->stream);
    ctx->kev_valid[1] = true;
    OPE_TRY(check_launch(ctx, "sacia_score_batch_kernel"));
  }
  sacia_select_batch_kernel<<<div_up((size_t)frames, 128), 128, 0, ctx->stream>>>(a, frames, d_results);
  return check_launch(ctx, "sacia_select_batch_kernel");
}

int fitness_batch_device(ope_ctx* ctx, const float4* tgt, const int* tgt_counts, const float4* src, const int* src_counts, int stride, int frames,
                         int max_nt, const ope_reg_result* d_icp, const int* d_active, double* d_out) {
  if (frames <= 0) return OPE_OK;
  if (max_nt > kFitSmemMax) return fail(ctx, OPE_ERR_CAPACITY, "batched fitness: target larger than the shared-memory path");
  OPE_TRY(dyn_smem(ctx, (const void*)fitness_smem_batch_kernel, (size_t)kFitSmemMax * sizeof(float4)));
  const size_t bytes = (((size_t)max_nt + 7) & ~(size_t)7) * sizeof(float4);
  fitness_smem_batch_kernel<<<frames, kNnThreads, bytes, ctx->stream>>>(tgt, tgt_counts, src, src_counts, stride, d_icp, d_active, d_out);
  return check_launch(ctx, "fitness_smem_batch_kernel");
}

// ICP-with-normals (normal shooting, small clouds) for many independent alignments in ONE launch. frames[i]: clouds with normals,
// source points carrying their index in .w; results[i] on the device. Only alignments icp_small_applicable admits.
int icp_small_batch_device(ope_ctx* ctx, const ope_icp_params& prm, const IcpBatchFrame* frames, int n_frames, ope_reg_result* d_results) {
  if (n_frames <= 0) return OPE_OK;
  size_t total_src = 0;
  for (int i = 0; i < n_frames; ++i) {
    if (!icp_small_applicable(prm, (size_t)frames[i].n_src, (size_t)frames[i].n_tgt)) return fail(ctx, OPE_ERR_UNSUPPORTED, "alignment %d does not fit the small-cloud ICP kernel", i);
    total_src += (size_t)frames[i].n_src;
  }
  IcpDev common;
  std::memset(&common, 0, sizeof(common));
  OPE_TRY(icp_fill_params(ctx, prm, &common));
  common.tgt_in_smem = 1;
  common.guess = mat4_identity();
  Scratch<int> match(ctx);
  Scratch<float> d2(ctx);
  OPE_TRY(match.alloc(total_src)); OPE_TRY(d2.alloc(total_src));
  std::vector<IcpDev> descs((size_t)n_frames, common);
  size_t so = 0;
  for (int i = 0; i < n_frames; ++i) {
    IcpDev& a = descs[(size_t)i];
    const IcpBatchFrame& f = frames[i];
    a.grid.n = f.n_tgt;      // every target point is finite (it survived the sampling and the NaN-normal filter)
    a.n_tgt = f.n_tgt;
    a.tgt_pts = f.tgt_pts; a.tgt_nrm = f.tgt_nrm;
    a.src0_pts = f.src_pts; a.src0_nrm = f.src_nrm; a.src_sorted = f.src_pts;
    a.n_src = f.n_src; a.n_work = f.n_src;
    a.corr_match = match.p + so; a.corr_d2 = d2.p + so;
    a.result = d_results + i;
    so += (size_t)f.n_src;
  }
  return icp_small_launch(ctx, descs.data(), n_frames);
}

}  // namespace ope

// =========================================================================================== C ABI =====
using namespace ope;

extern "C" {

void ope_icp_params_default(ope_icp_params* p) {
  std::memset(p, 0, sizeof(*p));
  p->max_iterations = 10;                                // VP/registration_mod.h:102-130
  p->transformation_epsilon = 0.0;
  p->euclidean_fitness_epsilon = -DBL_MAX;
  p->max_correspondence_distance = std::sqrt(DBL_MAX);
  p->min_number_correspondences = 3;
  p->estimator = OPE_EST_NEAREST;
  p->k_search = 10;
  p->transformation = OPE_TE_SVD;
  p->variant = OPE_ICP_VARIANT_MOD;
  p->mse_threshold_absolute = 1e-12;                     // VP/default_convergence_criteria_mod.h:94-110
}
void ope_sacia_params_default(ope_sacia_params* p) {
  std::memset(p, 0, sizeof(*p));
  p->max_iterations = 10; p->nr_samples = 3; p->k_correspondences = 10; p->min_sample_distance = 0.0f;
  p->max_correspondence_distance = std::sqrt(DBL_MAX);
}
void ope_pose_params_default(ope_pose_params* p) {
  std::memset(p, 0, sizeof(*p));
  p->coarse_leaf = 0.01f; p->fine_leaf = 0.008f; p->normal_k = 30; p->fpfh_radius = 0.03f;
  ope_sacia_params_default(&p->sacia);
  p->sacia.max_iterations = 400; p->sacia.nr_samples = 5; p->sacia.k_correspondences = 5;
  p->sacia.min_sample_distance = 0.01f; p->sacia.max_correspondence_distance = 0.05;
  p->min_target_features = 10; p->min_target_points = 100;
  ope_icp_params_default(&p->icp);
  p->icp.max_iterations = 100; p->icp.transformation_epsilon = 1e-8; p->icp.euclidean_fitness_epsilon = 1e-8;
  p->icp.estimator = OPE_EST_NORMAL_SHOOTING; p->icp.k_search = 20;
  p->icp.n_rejectors = 2;
  p->icp.rejector_kind[0] = OPE_REJ_SURFACE_NORMAL; p->icp.rejector_threshold[0] = 0.7;
  p->icp.rejector_kind[1] = OPE_REJ_SELF_OCCLUDED_NORMAL; p->icp.rejector_threshold[1] = 0.6;
  p->icp.transformation = OPE_TE_SVD; p->icp.with_normals = 1;
  p->coarse_refit_threshold = 1e-4;
}

int ope_cloud_transform(ope_ctx* ctx, const ope_cloud* cloud, const float T[16], ope_cloud** out) {
  OPE_ENTER(ctx);
  if (!ctx || !cloud || !T || !out) return OPE_ERR_INVALID;
  ope_cloud* o = nullptr;
  OPE_TRY(cloud_alloc(ctx, cloud->n, cloud->normals != nullptr, &o));
  Mat4 M;
  std::memcpy(M.m, T, sizeof(M.m));
  int rc = transform_device(ctx, cloud, M, o);
  if (rc != OPE_OK) { ope_cloud_free(ctx, o); return rc; }
  OPE_CUDA_TRY(ctx, ope::stream_sync(ctx));
  *out = o;
  return OPE_OK;
}

int ope_umeyama(ope_ctx* ctx, const ope_cloud* src, const ope_cloud* tgt, const int32_t* isrc, const int32_t* itgt, size_t n,
                float T[16]) {
  OPE_ENTER(ctx);
  if (!ctx || !src || !tgt || !T || n == 0) return OPE_ERR_INVALID;
  if ((!isrc && n > src->n) || (!itgt && n > tgt->n)) return fail(ctx, OPE_ERR_INVALID, "n exceeds cloud size");
  Scratch<int> ds(ctx), dt(ctx);
  if (isrc) {
    for (size_t i = 0; i < n; ++i) if (isrc[i] < 0 || (size_t)isrc[i] >= src->n) return fail(ctx, OPE_ERR_INVALID, "source index out of range");
    OPE_TRY(ds.alloc(n));
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(ds.p, isrc, n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  }
  if (itgt) {
    for (size_t i = 0; i < n; ++i) if (itgt[i] < 0 || (size_t)itgt[i] >= tgt->n) return fail(ctx, OPE_ERR_INVALID, "target index out of range");
    OPE_TRY(dt.alloc(n));
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(dt.p, itgt, n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  }
  return umeyama_device(ctx, src->pts, tgt->pts, isrc ? ds.p : nullptr, itgt ? dt.p : nullptr, n, T);
}

int ope_point_to_plane(ope_ctx* ctx, const ope_cloud* src, const ope_cloud* tgt, const int32_t* isrc, const int32_t* itgt, size_t n,
                       int kind, float T[16], int32_t* lm_info) {
  OPE_ENTER(ctx);
  if (!ctx || !src || !tgt || !T) return OPE_ERR_INVALID;
  if (!tgt->normals) return fail(ctx, OPE_ERR_INVALID, "point-to-plane estimation needs target normals");
  if ((!isrc && n > src->n) || (!itgt && n > tgt->n)) return fail(ctx, OPE_ERR_INVALID, "n exceeds cloud size");
  Scratch<int> ds(ctx), dt(ctx);
  std::vector<int> ident;
  if (isrc) {
    for (size_t i = 0; i < n; ++i) if (isrc[i] < 0 || (size_t)isrc[i] >= src->n) return fail(ctx, OPE_ERR_INVALID, "source index out of range");
    OPE_TRY(ds.alloc(n));
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(ds.p, isrc, n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  }
  if (itgt) {
    for (size_t i = 0; i < n; ++i) if (itgt[i] < 0 || (size_t)itgt[i] >= tgt->n) return fail(ctx, OPE_ERR_INVALID, "target index out of range");
  } else {
    ident.resize(n);
    for (size_t i = 0; i < n; ++i) ident[i] = (int)i;
    itgt = ident.data();
  }
  OPE_TRY(dt.alloc(n));
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(dt.p, itgt, n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  Mat4 M;
  int rc = point_to_plane_device(ctx, src->pts, tgt->pts, tgt->normals, isrc ? ds.p : nullptr, dt.p, nullptr, n, kind, &M, nullptr, nullptr, lm_info);
  ope::stream_sync(ctx);   // the pageable index arrays must outlive their copies
  if (rc == OPE_OK) std::memcpy(T, M.m, sizeof(M.m));
  return rc;
}

int ope_fitness(ope_ctx* ctx, const ope_cloud* src, const ope_cloud* tgt, const float T[16], double max_range, double* out) {
  OPE_ENTER(ctx);
  if (!ctx || !src || !tgt || !T || !out) return OPE_ERR_INVALID;
  if (tgt->n == 0) return fail(ctx, OPE_ERR_EMPTY, "No input target dataset was given!");
  Mat4 M;
  std::memcpy(M.m, T, sizeof(M.m));
  return fitness_device(ctx, src, tgt, M, max_range, out);
}

int ope_correspondences(ope_ctx* ctx, const ope_cloud* src, const ope_cloud* tgt, const ope_icp_params* prm,
                        ope_correspondence* out, size_t* out_n) {
  OPE_ENTER(ctx);
  if (!ctx || !src || !tgt || !prm || !out || !out_n) return OPE_ERR_INVALID;
  *out_n = 0;
  if (tgt->n == 0) return fail(ctx, OPE_ERR_EMPTY, "No input target dataset was given!");
  if (src->n == 0) return OPE_OK;
  IcpDev a;
  std::memset(&a, 0, sizeof(a));
  OPE_TRY(icp_fill(ctx, src, tgt, *prm, &a));
  a.variant = OPE_ICP_VARIANT_MOD;
  a.cur_pts = src->pts; a.cur_nrm = src->normals;
  const size_t n = src->n;
  Scratch<int> match(ctx), seed(ctx);
  Scratch<float> d2(ctx);
  const bool shooting = prm->estimator == OPE_EST_NORMAL_SHOOTING;
  OPE_TRY(match.alloc(n)); OPE_TRY(d2.alloc(n));
  OPE_TRY(seed.alloc(shooting ? n * (size_t)prm->k_search : n));
  a.corr_match = match.p; a.corr_d2 = d2.p; a.seed = seed.p;
  OPE_TRY(dyn_smem(ctx, (const void*)correspond_once_kernel, sizeof(IcpSmem)));
  const size_t want = shooting ? div_up(n, kIcpWarps) : div_up(n, kIcpThreads);
  correspond_once_kernel<<<(unsigned)std::min<size_t>(want, (size_t)ctx->sm_count * 4), kIcpThreads, sizeof(IcpSmem), ctx->stream>>>(a);
  OPE_TRY(check_launch(ctx, "correspond_once_kernel"));
  if (prm->use_reciprocal) {   // determineReciprocalCorrespondences: the source's own (cached) index answers the way back
    OPE_TRY(cloud_bbox(ctx, const_cast<ope_cloud*>(src)));
    GridView gsrc;
    OPE_TRY(cloud_grid(ctx, src, knn_cell_size(src, 1), &gsrc));
    OPE_TRY(dyn_smem(ctx, (const void*)reciprocal_filter_kernel, sizeof(IcpSmem)));
    reciprocal_filter_kernel<<<(unsigned)std::min<size_t>(div_up(n, kIcpThreads), (size_t)ctx->sm_count * 4), kIcpThreads, sizeof(IcpSmem),
                               ctx->stream>>>(gsrc, tgt->pts, match.p, (int)n, a.max_d2_f, a.max_corr_dist);
    OPE_TRY(check_launch(ctx, "reciprocal_filter_kernel"));
  }
  std::vector<int> hm(n);
  std::vector<float> hd(n);
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(hm.data(), match.p, n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(hd.data(), d2.p, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  OPE_CUDA_TRY(ctx, ope::stream_sync(ctx));
  corr_to_host(hm, hd, out, out_n);
  return OPE_OK;
}

int ope_icp_align(ope_ctx* ctx, const ope_cloud* src, const ope_cloud* tgt, const ope_icp_params* prm, const float guess[16],
                  ope_reg_result* res, ope_correspondence* out_corr, ope_cloud** out_aligned) {
  OPE_ENTER(ctx);
  if (!ctx || !src || !prm || !res) return OPE_ERR_INVALID;
  Mat4 I = mat4_identity();
  std::memset(res, 0, sizeof(*res));
  std::memcpy(res->T, I.m, sizeof(I.m));
  if (out_aligned) *out_aligned = nullptr;
  // Registration::initCompute: no target -> PCL_ERROR + return, transforms stay identity (VP/impl/registration_mod.hpp:73-77)
  if (!tgt || tgt->n == 0) return fail(ctx, OPE_ERR_EMPTY, "No input target dataset was given!");
  Mat4 G = I;
  if (guess) std::memcpy(G.m, guess, sizeof(G.m));
  return icp_device(ctx, src, tgt, *prm, G, res, out_corr, out_aligned);
}

int ope_icp_align_fixed(ope_ctx* ctx, const ope_cloud* src, const ope_cloud* tgt, const ope_icp_params* prm, const float guess[16],
                        ope_correspondence* fixed, size_t n_fixed, ope_reg_result* res, ope_correspondence* out_corr, ope_cloud** out_aligned) {
  OPE_ENTER(ctx);
  if (!ctx || !src || !prm || !res || (n_fixed && !fixed)) return OPE_ERR_INVALID;
  if (n_fixed == 0) return ope_icp_align(ctx, src, tgt, prm, guess, res, out_corr, out_aligned);
  Mat4 I = mat4_identity();
  std::memset(res, 0, sizeof(*res));
  std::memcpy(res->T, I.m, sizeof(I.m));
  if (out_aligned) *out_aligned = nullptr;
  if (!tgt || tgt->n == 0) return fail(ctx, OPE_ERR_EMPTY, "No input target dataset was given!");
  Mat4 G = I;
  if (guess) std::memcpy(G.m, guess, sizeof(G.m));
  return icp_stepwise_device(ctx, src, tgt, *prm, G, res, out_corr, out_aligned, fixed, n_fixed);
}

int ope_sacia_draw(const float* src_xyz, size_t ns, size_t stride_bytes, int iterations, int nr_samples, int k_correspondences,
                   float* min_sample_distance, int32_t* samples, int32_t* picks) {
  if (!src_xyz || !samples || !picks || !min_sample_distance || stride_bytes % 4 != 0 || stride_bytes < 12) return OPE_ERR_INVALID;
  LibcRandSession rng;
  for (int it = 0; it < iterations; ++it) {
    int rc = draw_samples(rng, src_xyz, ns, stride_bytes / 4, nr_samples, *min_sample_distance, samples + (size_t)it * nr_samples);
    if (rc != OPE_OK) return rc;
    for (int s = 0; s < nr_samples; ++s) picks[(size_t)it * nr_samples + s] = rng.index(k_correspondences);
  }
  return OPE_OK;
}

int ope_sacia_align(ope_ctx* ctx, const ope_cloud* src, const float* fsrc, const ope_cloud* tgt, const float* ftgt,
                    const ope_sacia_params* prm, const ope_rng_table* table, ope_reg_result* res, float* out_errors) {
  OPE_ENTER(ctx);
  if (!ctx || !src || !fsrc || !tgt || !ftgt || !prm || !res) return OPE_ERR_INVALID;
  Mat4 I = mat4_identity();
  std::memset(res, 0, sizeof(*res));
  std::memcpy(res->T, I.m, sizeof(I.m));
  Scratch<float> dfs(ctx), dft(ctx);
  OPE_TRY(dfs.alloc(src->n * 33)); OPE_TRY(dft.alloc(tgt->n * 33));
  if (src->n) OPE_CUDA_TRY(ctx, cudaMemcpyAsync(dfs.p, fsrc, src->n * 33 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  if (tgt->n) OPE_CUDA_TRY(ctx, cudaMemcpyAsync(dft.p, ftgt, tgt->n * 33 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  return sacia_device(ctx, src, dfs.p, tgt, dft.p, *prm, table, nullptr, res, out_errors);
}

}  // extern "C"
