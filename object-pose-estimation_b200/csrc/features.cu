// features.cu — NormalEstimation (K4), SPFH/FPFH (K5) and the exact float32 feature-space k-NN (K6 ranking stage).
//
// Rooflines (DESIGN.md): normals read 16 B and write 16 B per point plus a k-neighbour gather that stays in
// L2; SPFH/FPFH move 428 B per point compulsory (16 pts + 16 normals + 132 SPFH write + 132 SPFH read +
// 132 FPFH write) plus an m-neighbour gather of 32 B (SPFH pass) / 136 B (FPFH pass) per neighbour from L2.
#include <algorithm>

#include <climits>
#include <cstdlib>
#include <vector>
#include <mutex>

#include "ope_host.cuh"
#include "ope_octet.cuh"

namespace ope {

// ------------------------------------------------------------------------------------------ normals ----
// One warp per point: exact k-NN on the cloud's own grid into the warp's register list (the point itself is neighbour 0),
// the neighbours' coordinates are fetched one per lane, then the covariance is summed sequentially in the sorted
// neighbour order (SURVEY A.4) from shuffles, eigen33, flip toward the viewpoint.
static constexpr int kNormThreads = 256;
__global__ void __launch_bounds__(kNormThreads) normals_kernel(GridView g, const float4* __restrict__ pts, int n, int k, float vpx,
                                                               float vpy, float vpz, float4* __restrict__ out) {
  __shared__ OctStack stacks[kNormThreads / 32];
  OctStack* st = &stacks[threadIdx.x >> 5];
  const int lane = threadIdx.x & 31;
  const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
  const float nan = __int_as_float(0x7fc00000);
  for (int i = wid; i < n; i += n_warps) {
    const float4 q = __ldg(pts + i);
    const bool ok = finite3(q.x, q.y, q.z);
    float ld;
    int li;
    const int cnt = warp_knn(g, st, ok, q.x, q.y, q.z, k, FLT_MAX, ld, li);
    float4 p = make_float4(0, 0, 0, 0);
    if (lane < cnt) p = __ldg(pts + li);
    float r[4] = {nan, nan, nan, nan};
    if (ok && cnt >= 3) {
      CovAccum acc;
      acc.reset();
      for (int j = 0; j < cnt; ++j)   // every lane sums the same sequence: uniform, no divergence
        acc.add(__shfl_sync(0xffffffffu, p.x, j), __shfl_sync(0xffffffffu, p.y, j), __shfl_sync(0xffffffffu, p.z, j));
      normal_from_accum(acc, cnt, q.x, q.y, q.z, vpx, vpy, vpz, r);
    }
    if (lane == 0) out[i] = make_float4(r[0], r[1], r[2], r[3]);
    __syncwarp();
  }
}

// Small clouds (a down-sampled model or cluster: 1-2 k points): no spatial index at all. Every block keeps the whole cloud in
// shared memory and its warps answer their queries by the exact brute-force warp scan (warp_knn_smem: same (d2, index) list as
// warp_knn, hence the same normals bit for bit). One launch instead of bounding box + grid build (six launches and a host
// round trip) + search; what a frame spends on normals falls from ~0.2 ms per cloud to the launch itself.
static constexpr int kNormSmemMax = 4096;
__device__ __forceinline__ void normals_smem_body(const float4* __restrict__ pts, int n, int k, float vpx, float vpy, float vpz,
                                                  float4* __restrict__ out) {
  extern __shared__ __align__(16) float4 tg_norm[];
  __shared__ float2 knn_buf[kNormThreads / 32][kKnnBufCap + 32];   // per-warp scratch of the two-pass exact search
  int fin = 0;
  for (int j = threadIdx.x; j < n; j += kNormThreads) {
    const float4 t = __ldg(pts + j);
    tg_norm[j] = t;
    fin += finite3(t.x, t.y, t.z) ? 1 : 0;
  }
  // number of finite points (nearestKSearch clamps k to it): every thread contributes its count
  __shared__ int s_fin;
  if (threadIdx.x == 0) s_fin = 0;
  __syncthreads();
  for (int o = 16; o > 0; o >>= 1) fin += __shfl_xor_sync(0xffffffffu, fin, o);
  if ((threadIdx.x & 31) == 0) atomicAdd(&s_fin, fin);
  __syncthreads();
  const int n_finite = s_fin;
  const int lane = threadIdx.x & 31;
  const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
  const float nan = __int_as_float(0x7fc00000);
  // The search is a warp's job (one query at a time); the covariance sums — serial over the neighbours in list order, like the
  // reference's — and the eigenvector are one THREAD's job. So a warp answers 32 queries, parks every neighbour list in shared
  // memory, and then each lane finishes one query: the serial part runs once per 32 queries instead of once per query with 31
  // lanes repeating it. Same operations in the same order per query: the same normals, bit for bit.
  __shared__ unsigned short nbr[kNormThreads / 32][32][34];   // [warp][slot][rank]; 34: lanes reading one rank hit 32 banks
  const int warp = threadIdx.x >> 5;
  for (int base = wid; base < n; base += 32 * n_warps) {
    int my_cnt = 0;
    bool my_ok = false;
    for (int slot = 0; slot < 32; ++slot) {
      const int i = base + slot * n_warps;
      if (i >= n) break;   // warp-uniform
      const float4 q = tg_norm[i];
      const bool ok = finite3(q.x, q.y, q.z);
      float ld;
      int li;
      const int cnt = warp_knn_smem_bounded(tg_norm, n, n_finite, ok, q.x, q.y, q.z, k, FLT_MAX, knn_buf[warp], ld, li);
      if (lane < cnt) nbr[warp][slot][lane] = (unsigned short)li;
      if (lane == slot) { my_cnt = cnt; my_ok = ok; }
    }
    __syncwarp();
    const int i = base + lane * n_warps;
    if (i < n) {
      float r[4] = {nan, nan, nan, nan};
      if (my_ok && my_cnt >= 3) {
        const float4 q = tg_norm[i];
        CovAccum acc;
        acc.reset();
        for (int j = 0; j < my_cnt; ++j) { const float4 p = tg_norm[nbr[warp][lane][j]]; acc.add(p.x, p.y, p.z); }
        normal_from_accum(acc, my_cnt, q.x, q.y, q.z, vpx, vpy, vpz, r);
      }
      out[i] = make_float4(r[0], r[1], r[2], r[3]);
    }
    __syncwarp();
  }
}
__global__ void __launch_bounds__(kNormThreads) normals_smem_kernel(const float4* __restrict__ pts, int n, int k, float vpx, float vpy,
                                                                    float vpz, float4* __restrict__ out) {
  normals_smem_body(pts, n, k, vpx, vpy, vpz, out);
}
// Frame-spanning launch (ope_pose_batch): blockIdx.y = cloud; cloud c has counts[c] points at pts + c * stride. Same body, so the
// same normals bit for bit as the single-cloud launch.
__global__ void __launch_bounds__(kNormThreads) normals_smem_batch_kernel(const float4* __restrict__ pts, const int* __restrict__ counts,
                                                                          int stride, int k, float vpx, float vpy, float vpz,
                                                                          float4* __restrict__ out) {
  const int n = counts[blockIdx.y];
  if (n <= 0 || (int)blockIdx.x * (kNormThreads / 32) >= n) return;   // more blocks than this cloud has points: nothing to do
  normals_smem_body(pts + (size_t)blockIdx.y * stride, n, k, vpx, vpy, vpz, out + (size_t)blockIdx.y * stride);
}

// k > 32 (warp_knn_list): the warp's list in shared memory, then lane 0 sums the covariance over it in list order — the same
// serial float chain as the kernels above, so pointNormal of the oracle is the reference for both. SMEM: the whole cloud in
// shared memory and the brute-force scan (clouds of up to kNormSmemMax points), otherwise the grid.
template <bool SMEM>
__global__ void __launch_bounds__(kNormThreads) normals_list_kernel(GridView g, const float4* __restrict__ pts, int n, int k, float vpx,
                                                                    float vpy, float vpz, float4* __restrict__ out) {
  extern __shared__ __align__(16) float4 tg_list[];
  __shared__ OctStack stacks[SMEM ? 1 : kNormThreads / 32];
  __shared__ KnnList lists[kNormThreads / 32];
  __shared__ int s_fin;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  KnnList* L = &lists[warp];
  int n_finite = 0;
  if (SMEM) {
    int fin = 0;
    for (int j = threadIdx.x; j < n; j += kNormThreads) {
      const float4 t = __ldg(pts + j);
      tg_list[j] = t;
      fin += finite3(t.x, t.y, t.z) ? 1 : 0;
    }
    if (threadIdx.x == 0) s_fin = 0;
    __syncthreads();
    for (int o = 16; o > 0; o >>= 1) fin += __shfl_xor_sync(0xffffffffu, fin, o);
    if (lane == 0) atomicAdd(&s_fin, fin);
    __syncthreads();
    n_finite = s_fin;
  }
  const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
  const float nan = __int_as_float(0x7fc00000);
  for (int i = wid; i < n; i += n_warps) {
    const float4 q = SMEM ? tg_list[i] : __ldg(pts + i);
    const bool ok = finite3(q.x, q.y, q.z);
    const int cnt = SMEM ? warp_knn_list_smem(tg_list, n, n_finite, L, ok, q.x, q.y, q.z, k)
                         : warp_knn_list(g, &stacks[SMEM ? 0 : warp], L, ok, q.x, q.y, q.z, k);
    if (lane == 0) {
      float r[4] = {nan, nan, nan, nan};
      if (ok && cnt >= 3) {
        CovAccum acc;
        acc.reset();
        for (int j = 0; j < cnt; ++j) {
          const int t = __float_as_int(L->e[j].y);
          const float4 p = SMEM ? tg_list[t] : __ldg(pts + t);
          acc.add(p.x, p.y, p.z);
        }
        normal_from_accum(acc, cnt, q.x, q.y, q.z, vpx, vpy, vpz, r);
      }
      out[i] = make_float4(r[0], r[1], r[2], r[3]);
    }
    __syncwarp();
  }
}

// ----------------------------------------------------------------------------------------- radius normals ----
// NormalEstimation::setRadiusSearch(r): the neighbours are the finite points with d2 < r2 (the query included), summed in
// ascending (d2, index) order. Neighbourhoods run from none to ~10^4 points, so:
//   count pass   one warp per query counts its neighbours (lanes stride over the grid's leaf ranges);
//   main pass    one block per query gathers its neighbours as 64-bit keys (d2 bits << 32 | index: d2 >= 0, so the key order is
//                the (d2, index) order) in any order, sorts them with a block-wide bitonic network, and thread 0 sums the
//                covariance over the sorted keys. A list of up to kRadSmemKeys keys lives in shared memory; a longer one in its
//                slice of a global scratch buffer, which the host fills by query tiles sized to a byte budget.
static constexpr int kRadThreads = 256;
static constexpr int kRadSmemKeys = 8192;   // 64 KB of shared memory per block
__global__ void radius_count_warp_kernel(GridView g, const float4* __restrict__ pts, int n, float r2, int* __restrict__ counts) {
  const int lane = threadIdx.x & 31;
  const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
  for (int i = wid; i < n; i += n_warps) {
    const float4 q = __ldg(pts + i);
    int cnt = 0;
    if (finite3(q.x, q.y, q.z))
      grid_radius_ranges(g, q.x, q.y, q.z, r2, 64, [&](int b, int e) {
        for (int j = b + lane; j < e; j += 32) {
          const float4 p = __ldg(g.pts + j);
          cnt += dist2(q.x, q.y, q.z, p.x, p.y, p.z) < r2 ? 1 : 0;
        }
      });
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (lane == 0) counts[i] = cnt;
  }
}

// Ascending sort of a[0, n) by the block: the bitonic network in its all-ascending form (each merge starts by comparing mirrored
// elements), so every comparator (i, j) has i < j and the positions >= n act as +inf that never move: no padding is stored.
__device__ __forceinline__ void block_bitonic_sort(unsigned long long* a, int n) {
  int N = 1;
  while (N < n) N <<= 1;
  for (int k = 2; k <= N; k <<= 1) {
    for (int s = k >> 1; s > 0; s >>= 1) {
      for (int t = threadIdx.x; t < N / 2; t += blockDim.x) {
        const int i = (t / s) * 2 * s + (t % s);
        const int j = (s == k >> 1) ? (i ^ (k - 1)) : i + s;
        if (j < n) {
          const unsigned long long x = a[i], y = a[j];
          if (y < x) { a[i] = y; a[j] = x; }
        }
      }
      __syncthreads();
    }
  }
}

// queries [q0, q1): counts from the count pass; a query with more than kRadSmemKeys neighbours keeps its keys at
// scratch + (big_off[i] - big_off[q0])
__global__ void __launch_bounds__(kRadThreads) normals_radius_kernel(GridView g, const float4* __restrict__ pts, int q0, int q1, float r2,
                                                                     const int* __restrict__ counts, const long long* __restrict__ big_off,
                                                                     unsigned long long* __restrict__ scratch, float vpx, float vpy,
                                                                     float vpz, float4* __restrict__ out) {
  extern __shared__ __align__(16) unsigned long long keys_smem[];
  __shared__ int s_fill;
  const float nan = __int_as_float(0x7fc00000);
  for (int i = q0 + blockIdx.x; i < q1; i += gridDim.x) {
    const int cnt = counts[i];
    const float4 q = __ldg(pts + i);
    if (cnt < 3) {   // also every non-finite query (count 0)
      if (threadIdx.x == 0) out[i] = make_float4(nan, nan, nan, nan);
      continue;
    }
    unsigned long long* keys = cnt <= kRadSmemKeys ? keys_smem : scratch + (big_off[i] - big_off[q0]);
    if (threadIdx.x == 0) s_fill = 0;
    __syncthreads();
    grid_radius_ranges(g, q.x, q.y, q.z, r2, 64, [&](int b, int e) {
      for (int j = b + (int)threadIdx.x; j < e; j += kRadThreads) {
        const float4 p = __ldg(g.pts + j);
        const float d2 = dist2(q.x, q.y, q.z, p.x, p.y, p.z);
        if (d2 < r2)
          keys[atomicAdd(&s_fill, 1)] = ((unsigned long long)__float_as_uint(d2) << 32) | (unsigned)__float_as_int(p.w);
      }
    });
    __syncthreads();
    block_bitonic_sort(keys, cnt);
    if (threadIdx.x == 0) {
      CovAccum acc;
      acc.reset();
      for (int j = 0; j < cnt; ++j) {
        const float4 p = __ldg(pts + (unsigned)keys[j]);
        acc.add(p.x, p.y, p.z);
      }
      float r[4];
      normal_from_accum(acc, cnt, q.x, q.y, q.z, vpx, vpy, vpz, r);
      out[i] = make_float4(r[0], r[1], r[2], r[3]);
    }
    __syncthreads();   // the keys are reused by the block's next query
  }
}

// ------------------------------------------------------------------------------------------- SPFH ------
// warp per point. Lanes stride over the candidate points of each grid row; every in-radius neighbour's three
// bin indices go to a per-warp shared-memory histogram of integer counts. Because every increment of one
// point's histogram is the same float (100/(m-1)), the reference's sequence of float additions depends only
// on the count, so the float bin value is rebuilt exactly by repeated addition afterwards.
static constexpr int kWarpsPerBlock = 8;

// SMEM = true (clouds of up to kFeatSmemMax points — a down-sampled model or cluster): no spatial index; the block keeps points
// and normals in shared memory and every warp tests all of them (ascending index, the oracle's order).
static constexpr int kFeatSmemMax = 2048;
template <bool SMEM>
__device__ __forceinline__ void spfh_body(const GridView& g, const float4* __restrict__ pts, const float4* __restrict__ nrm, int n, float r2,
                                          float* __restrict__ spfh) {
  extern __shared__ __align__(16) float4 sm_feat[];
  __shared__ int hist[kWarpsPerBlock][33];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int p_idx = blockIdx.x * kWarpsPerBlock + warp;
  if (SMEM) {
    for (int j = threadIdx.x; j < n; j += blockDim.x) { sm_feat[j] = __ldg(pts + j); sm_feat[n + j] = __ldg(nrm + j); }
    __syncthreads();
  }
  if (p_idx >= n) return;
  hist[warp][lane] = 0;
  if (lane == 0) hist[warp][32] = 0;
  __syncwarp();
  const float4 q = __ldg(pts + p_idx);
  int nb_count = 0;
  if (finite3(q.x, q.y, q.z)) {
    const float4 qn4 = __ldg(nrm + p_idx);
    const float qn[3] = {qn4.x, qn4.y, qn4.z};
    // the traversal is warp-uniform (one query per warp); lanes share each leaf range
    auto visit = [&](int b, int e) {
          for (int i = b + lane; i < e; i += 32) {
            const float4 c = SMEM ? sm_feat[i] : __ldg(g.pts + i);
            const float d2 = dist2(q.x, q.y, q.z, c.x, c.y, c.z);
            if (d2 < r2) {
              ++nb_count;
              const int j = SMEM ? i : __float_as_int(c.w);
              if (j != p_idx) {
                const float4 cn4 = SMEM ? sm_feat[n + j] : __ldg(nrm + j);
                const float cn[3] = {cn4.x, cn4.y, cn4.z};
                int h1, h2, h3;
                pair_feature_bins(q.x, q.y, q.z, qn, c.x, c.y, c.z, cn, h1, h2, h3);
                atomicAdd(&hist[warp][h1], 1);
                atomicAdd(&hist[warp][11 + h2], 1);
                atomicAdd(&hist[warp][22 + h3], 1);
              }
            }
          }
        };
    if (SMEM) visit(0, n); else grid_radius_ranges(g, q.x, q.y, q.z, r2, 64, visit);
  }
  for (int o = 16; o > 0; o >>= 1) nb_count += __shfl_xor_sync(0xffffffffu, nb_count, o);
  __syncwarp();
  const float incr = 100.0f / (float)(nb_count - 1);
  for (int b = lane; b < 33; b += 32) {
    const int c = hist[warp][b];
    float v = 0.0f;
    for (int t = 0; t < c; ++t) v += incr;
    spfh[(size_t)p_idx * 33 + b] = v;
  }
}
template <bool SMEM>
__global__ void spfh_kernel(GridView g, const float4* __restrict__ pts, const float4* __restrict__ nrm, int n, float r2,
                            float* __restrict__ spfh) {
  spfh_body<SMEM>(g, pts, nrm, n, r2, spfh);
}
// frame-spanning launch: blockIdx.y = cloud (points / normals at c * stride, histograms at c * stride * 33)
__global__ void spfh_batch_kernel(const float4* __restrict__ pts, const float4* __restrict__ nrm, const int* __restrict__ counts, int stride,
                                  float r2, float* __restrict__ spfh) {
  const int n = counts[blockIdx.y];
  if (n <= 0 || (int)blockIdx.x * kWarpsPerBlock >= n) return;
  GridView g;
  g.n = 0;
  const size_t o = (size_t)blockIdx.y * stride;
  spfh_body<true>(g, pts + o, nrm + o, n, r2, spfh + o * 33);
}

// ------------------------------------------------------------------------------------------- FPFH ------
// warp per point, lane = histogram bin (lane 0 also carries bin 32). Each leaf range is examined 32 candidates at a
// time (one per lane, coalesced float4 loads); the in-radius ones are then consumed in order, each as one coalesced
// 132-byte read of its SPFH row, weighted by 1/d2 and accumulated in float like the reference
// (weightPointSPFHSignature, SURVEY A.5). The three normalisation sums are carried in double.
template <bool SMEM>
__device__ __forceinline__ void fpfh_body(const GridView& g, const float4* __restrict__ pts, int n, float r2, const float* __restrict__ spfh,
                                          float* __restrict__ out) {
  extern __shared__ __align__(16) float4 sm_feat[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int p_idx = blockIdx.x * kWarpsPerBlock + warp;
  if (SMEM) {
    for (int j = threadIdx.x; j < n; j += blockDim.x) sm_feat[j] = __ldg(pts + j);
    __syncthreads();
  }
  if (p_idx >= n) return;
  const float4 q = __ldg(pts + p_idx);
  float acc = 0.0f, acc32 = 0.0f;
  double sum = 0.0, sum32 = 0.0;
  const bool ok = finite3(q.x, q.y, q.z);
  int found = 0;
  if (ok) {
    auto visit = [&](int b, int e) {
          for (int base = b; base < e; base += 32) {
            const int i = base + lane;
            float d2 = FLT_MAX;
            int j = -1;
            if (i < e) {
              const float4 c = SMEM ? sm_feat[i] : __ldg(g.pts + i);
              d2 = dist2(q.x, q.y, q.z, c.x, c.y, c.z);
              j = SMEM ? i : __float_as_int(c.w);
            }
            const bool inr = d2 < r2;
            const unsigned in_mask = __ballot_sync(0xffffffffu, inr);
            found += __popc(in_mask);
            unsigned use_mask = __ballot_sync(0xffffffffu, inr && d2 != 0.0f);
            while (use_mask) {
              const int src = __ffs(use_mask) - 1;
              use_mask &= use_mask - 1;
              const float dj = __shfl_sync(0xffffffffu, d2, src);
              const int jj = __shfl_sync(0xffffffffu, j, src);
              const float w = 1.0f / dj;
              const float* hrow = spfh + (size_t)jj * 33;
              const float val = __ldg(hrow + lane) * w;
              sum += val;
              acc += val;
              if (lane == 0) {
                const float v32 = __ldg(hrow + 32) * w;
                sum32 += v32;
                acc32 += v32;
              }
            }
          }
        };
    if (SMEM) visit(0, n); else grid_radius_ranges(g, q.x, q.y, q.z, r2, 64, visit);
  }
  // per-sub-histogram sums: bins 0-10 | 11-21 | 22-32
  const unsigned full = 0xffffffffu;
  double s1 = (lane <= 10) ? sum : 0.0, s2 = (lane >= 11 && lane <= 21) ? sum : 0.0, s3 = (lane >= 22) ? sum : 0.0;
  if (lane == 0) s3 += sum32;
  for (int o = 16; o > 0; o >>= 1) {
    s1 += __shfl_xor_sync(full, s1, o);
    s2 += __shfl_xor_sync(full, s2, o);
    s3 += __shfl_xor_sync(full, s3, o);
  }
  if (s1 != 0) s1 = 100.0 / s1;
  if (s2 != 0) s2 = 100.0 / s2;
  if (s3 != 0) s3 = 100.0 / s3;
  const float nan = __int_as_float(0x7fc00000);
  float* o = out + (size_t)p_idx * 33;
  if (!ok || found == 0) {
    o[lane] = nan;
    if (lane == 0) o[32] = nan;
    return;
  }
  const double sc = lane <= 10 ? s1 : (lane <= 21 ? s2 : s3);
  o[lane] = acc * (float)sc;
  if (lane == 0) o[32] = acc32 * (float)s3;
}
template <bool SMEM>
__global__ void fpfh_kernel(GridView g, const float4* __restrict__ pts, int n, float r2, const float* __restrict__ spfh,
                            float* __restrict__ out) {
  fpfh_body<SMEM>(g, pts, n, r2, spfh, out);
}
__global__ void fpfh_batch_kernel(const float4* __restrict__ pts, const int* __restrict__ counts, int stride, float r2,
                                  const float* __restrict__ spfh, float* __restrict__ out) {
  const int n = counts[blockIdx.y];
  if (n <= 0 || (int)blockIdx.x * kWarpsPerBlock >= n) return;
  GridView g;
  g.n = 0;
  const size_t o = (size_t)blockIdx.y * stride;
  fpfh_body<true>(g, pts + o, n, r2, spfh + o * 33, out + o * 33);
}

// ------------------------------------------------------------------------------- feature-space k-NN ----
// Exact float32 ranking: d = sum_c (q_c - t_c)^2 accumulated left to right (FLANN L2_Simple over 33 floats),
// ties on the smaller index. One thread per query; the block streams target tiles through shared memory
// (coalesced 16 KB tiles, every thread reads the same target row -> shared-memory broadcast). The target
// range is split over blockIdx.y so small query sets still fill the SMs; a merge kernel combines the splits.
static constexpr int kFkQueries = 128;   // threads per block = queries per block
static constexpr int kFkTile = 64;       // targets per shared-memory tile
static constexpr int kFkMaxDim = 64;
static constexpr int kFkMaxK = 16;

// blockIdx.z = frame: targets ftgt + z * stride * dim, counts[z] rows (counts null: nt rows); every frame answers the same nq
// queries (the rows qlist lists, null: 0 .. nq-1). Partial lists at ((z * nq + qi) * splits + y) * k; splits past a frame's end
// produce empty lists.
// frame f (blockIdx.z): targets ftgt + f * stride * dim (counts[f] rows, or nt), queries fqry + f * qstride * dim (qcounts[f] rows,
// or nq); qstride 0: every frame asks the same queries
__global__ void feature_knn_kernel(const float* __restrict__ ftgt, int nt, const int* __restrict__ counts, int stride,
                                   const float* __restrict__ fqry, int nq, int qstride, const int* __restrict__ qcounts, int dim, int k,
                                   int t_per_split, const int* __restrict__ qlist, int* __restrict__ part_idx, float* __restrict__ part_d2) {
  extern __shared__ float tile[];  // kFkTile * dim
  const int frame = blockIdx.z;
  if (counts) nt = counts[frame];
  const float* ft = ftgt + (size_t)frame * stride * dim;
  const float* fq = fqry + (size_t)frame * qstride * dim;
  const int nqf = qcounts ? qcounts[frame] : nq;
  const int qi = blockIdx.x * kFkQueries + threadIdx.x;   // position in the work list (nq entries)
  const int qsrc = (qi < nqf && qlist) ? qlist[qi] : qi;   // row of fq
  const int t_begin = blockIdx.y * t_per_split, t_end = min(nt, t_begin + t_per_split);
  float q[kFkMaxDim];
  if (qi < nqf)
    for (int c = 0; c < dim; ++c) q[c] = __ldg(fq + (size_t)qsrc * dim + c);
  float bd[kFkMaxK];
  int bi[kFkMaxK];
  int cnt = 0;
  for (int t0 = t_begin; t0 < t_end; t0 += kFkTile) {
    const int tn = min(kFkTile, t_end - t0);
    __syncthreads();
    for (int e = threadIdx.x; e < tn * dim; e += blockDim.x) tile[e] = __ldg(ft + (size_t)t0 * dim + e);
    __syncthreads();
    if (qi < nqf) {
      for (int t = 0; t < tn; ++t) {
        const float* f = tile + t * dim;
        float d = 0.0f;
        for (int c = 0; c < dim; ++c) { float df = q[c] - f[c]; d += df * df; }
        if (!isfinite(d)) continue;
        const int idx = t0 + t;
        if (cnt == k && !nb_less(d, idx, bd[k - 1], bi[k - 1])) continue;
        int j = cnt < k ? cnt : k - 1;
        while (j > 0 && nb_less(d, idx, bd[j - 1], bi[j - 1])) { bd[j] = bd[j - 1]; bi[j] = bi[j - 1]; --j; }
        bd[j] = d; bi[j] = idx;
        if (cnt < k) ++cnt;
      }
    }
  }
  if (qi < nqf) {
    const size_t o = (((size_t)frame * nq + qi) * gridDim.y + blockIdx.y) * k;
    for (int j = 0; j < k; ++j) { part_idx[o + j] = j < cnt ? bi[j] : -1; part_d2[o + j] = j < cnt ? bd[j] : INFINITY; }
  }
}
// one thread per (frame = blockIdx.y, query): the splits' lists merged into out_idx / out_d2 (optional) at row
// frame * nq + qlist[qi] (qlist null: qi)
__global__ void feature_knn_merge_kernel(const int* __restrict__ part_idx, const float* __restrict__ part_d2, int nq,
                                         const int* __restrict__ qcounts, int splits, int k, const int* __restrict__ qlist,
                                         int* __restrict__ out_idx, float* __restrict__ out_d2) {
  const int qi = blockIdx.x * blockDim.x + threadIdx.x;
  if (qi >= (qcounts ? qcounts[blockIdx.y] : nq)) return;
  const size_t row = (size_t)blockIdx.y * nq + qi;
  const size_t dst = (size_t)blockIdx.y * nq + (qlist ? qlist[qi] : qi);
  float bd[kFkMaxK];
  int bi[kFkMaxK];
  int cnt = 0;
  for (int s = 0; s < splits; ++s)
    for (int e = 0; e < k; ++e) {
      const size_t o = (row * splits + s) * k + e;
      const int idx = part_idx[o];
      if (idx < 0) break;
      const float d = part_d2[o];
      if (cnt == k && !nb_less(d, idx, bd[k - 1], bi[k - 1])) continue;
      int j = cnt < k ? cnt : k - 1;
      while (j > 0 && nb_less(d, idx, bd[j - 1], bi[j - 1])) { bd[j] = bd[j - 1]; bi[j] = bi[j - 1]; --j; }
      bd[j] = d; bi[j] = idx;
      if (cnt < k) ++cnt;
    }
  for (int j = 0; j < k; ++j) {
    out_idx[dst * k + j] = j < cnt ? bi[j] : -1;
    if (out_d2) out_d2[dst * k + j] = j < cnt ? bd[j] : INFINITY;
  }
}

// ------------------------------------------------------------------ removeNaNNormalsFromPointCloud ----
__global__ void finite_normal_flag_kernel(const float4* __restrict__ nrm, int n, int* __restrict__ flags) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float4 v = __ldg(nrm + i);
  flags[i] = finite3(v.x, v.y, v.z) ? 1 : 0;
}
__global__ void compact_cloud_kernel(const float4* __restrict__ pts, const float4* __restrict__ nrm, int n,
                                     const int* __restrict__ pos, float4* __restrict__ opts, float4* __restrict__ onrm) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (pos[i + 1] > pos[i]) { opts[pos[i]] = __ldg(pts + i); onrm[pos[i]] = __ldg(nrm + i); }
}

// ================================================================================================ host ==
int normals_device(ope_ctx* ctx, ope_cloud* cloud, int k, const float vp[3]) {
  static_assert(kKnnListMax == OPE_KNN_MAX_K, "the shared-memory list holds OPE_KNN_MAX_K entries");
  if (k < 1 || k > OPE_KNN_MAX_K) return fail(ctx, OPE_ERR_INVALID, "normal estimation k must be in [1, %d]", OPE_KNN_MAX_K);
  if (!cloud->normals) OPE_TRY(dalloc(ctx, &cloud->normals, cloud->n));
  if (cloud->n == 0) return OPE_OK;
  if (k > 32) {
    GridView g;
    std::memset(&g, 0, sizeof(g));
    if (cloud->n <= (size_t)kNormSmemMax && !std::getenv("OPE_NORMALS_FORCE_GRID")) {
      OPE_TRY(dyn_smem(ctx, (const void*)normals_list_kernel<true>, kNormSmemMax * sizeof(float4)));
      const unsigned blocks = (unsigned)std::min<size_t>(div_up(cloud->n * 32, kNormThreads), (size_t)ctx->sm_count * 2);
      normals_list_kernel<true><<<blocks, kNormThreads, cloud->n * sizeof(float4), ctx->stream>>>(g, cloud->pts, (int)cloud->n, k, vp[0],
                                                                                                   vp[1], vp[2], cloud->normals);
      return check_launch(ctx, "normals_list_kernel<smem>");
    }
    OPE_TRY(cloud_bbox(ctx, cloud));
    OPE_TRY(cloud_grid(ctx, cloud, knn_cell_size(cloud, k), &g));
    normals_list_kernel<false><<<(unsigned)std::min<size_t>(div_up(cloud->n * 32, kNormThreads), (size_t)ctx->sm_count * 8), kNormThreads, 0,
                                 ctx->stream>>>(g, cloud->pts, (int)cloud->n, k, vp[0], vp[1], vp[2], cloud->normals);
    return check_launch(ctx, "normals_list_kernel");
  }
  if (cloud->n <= (size_t)kNormSmemMax && !std::getenv("OPE_NORMALS_FORCE_GRID")) {
    const size_t bytes = cloud->n * sizeof(float4);
    OPE_TRY(dyn_smem(ctx, (const void*)normals_smem_kernel, kNormSmemMax * sizeof(float4)));
    const unsigned blocks = (unsigned)std::min<size_t>(div_up(cloud->n * 32, kNormThreads), (size_t)ctx->sm_count * 2);
    normals_smem_kernel<<<blocks, kNormThreads, bytes, ctx->stream>>>(cloud->pts, (int)cloud->n, k, vp[0], vp[1], vp[2], cloud->normals);
    return check_launch(ctx, "normals_smem_kernel");
  }
  OPE_TRY(cloud_bbox(ctx, cloud));
  GridView g;
  OPE_TRY(cloud_grid(ctx, cloud, knn_cell_size(cloud, k), &g));
  normals_kernel<<<(unsigned)std::min<size_t>(div_up(cloud->n * 32, kNormThreads), (size_t)ctx->sm_count * 8), kNormThreads, 0, ctx->stream>>>(g, cloud->pts, (int)cloud->n, k, vp[0], vp[1], vp[2],
                                                                 cloud->normals);
  return check_launch(ctx, "normals_kernel");
}

// Scratch budget of the lists longer than kRadSmemKeys: OPE_RADIUS_NORMALS_SCRATCH_BYTES (default 256 MiB). A query whose own list
// exceeds it still runs, alone in its tile.
static size_t radius_scratch_budget() {
  const char* e = std::getenv("OPE_RADIUS_NORMALS_SCRATCH_BYTES");
  const long long v = e ? std::atoll(e) : 0;
  return v > 0 ? (size_t)v : ((size_t)256 << 20);
}

int normals_radius_device(ope_ctx* ctx, ope_cloud* cloud, float radius, const float vp[3]) {
  if (!(radius > 0) || !std::isfinite(radius)) return fail(ctx, OPE_ERR_INVALID, "normal estimation radius must be positive and finite");
  if (!cloud->normals) OPE_TRY(dalloc(ctx, &cloud->normals, cloud->n));
  const size_t n = cloud->n;
  if (n == 0) return OPE_OK;
  if (n > (size_t)INT_MAX) return fail(ctx, OPE_ERR_INVALID, "radius normals: cloud larger than INT_MAX points");
  GridView g;
  OPE_TRY(cloud_grid(ctx, cloud, radius * 0.5f, &g));
  const float r2 = radius * radius;
  Scratch<int> cnt(ctx);
  OPE_TRY(cnt.alloc(n));
  radius_count_warp_kernel<<<(unsigned)std::min<size_t>(div_up(n * 32, kNormThreads), (size_t)ctx->sm_count * 8), kNormThreads, 0,
                             ctx->stream>>>(g, cloud->pts, (int)n, r2, cnt.p);
  OPE_TRY(check_launch(ctx, "radius_count_warp_kernel"));
  std::vector<int> h_cnt;
  OPE_TRY(download(ctx, cnt.p, n, h_cnt));
  // global slices of the long lists, then tiles of consecutive queries whose long lists fit the budget together
  std::vector<long long> off(n + 1, 0);
  for (size_t i = 0; i < n; ++i) off[i + 1] = off[i] + (h_cnt[i] > kRadSmemKeys ? h_cnt[i] : 0);
  const long long budget = (long long)(radius_scratch_budget() / sizeof(unsigned long long));
  std::vector<std::pair<int, int>> tiles;
  long long scratch_keys = 0;
  for (size_t q0 = 0; q0 < n;) {
    size_t q1 = q0 + 1;
    while (q1 < n && off[q1 + 1] - off[q0] <= budget) ++q1;
    tiles.emplace_back((int)q0, (int)q1);
    scratch_keys = std::max(scratch_keys, off[q1] - off[q0]);
    q0 = q1;
  }
  Scratch<long long> d_off(ctx);
  Scratch<unsigned long long> keys(ctx);
  if (off[n] > 0) {
    OPE_TRY(d_off.alloc(n + 1));
    OPE_TRY(keys.alloc((size_t)scratch_keys));
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_off.p, off.data(), (n + 1) * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
  }
  int max_smem = 0;
  for (size_t i = 0; i < n; ++i) if (h_cnt[i] <= kRadSmemKeys) max_smem = std::max(max_smem, h_cnt[i]);
  OPE_TRY(dyn_smem(ctx, (const void*)normals_radius_kernel, kRadSmemKeys * sizeof(unsigned long long)));
  for (const auto& t : tiles) {
    const unsigned blocks = (unsigned)std::min<size_t>((size_t)(t.second - t.first), (size_t)ctx->sm_count * 4);
    normals_radius_kernel<<<blocks, kRadThreads, (size_t)max_smem * sizeof(unsigned long long), ctx->stream>>>(
        g, cloud->pts, t.first, t.second, r2, cnt.p, d_off.p, keys.p, vp[0], vp[1], vp[2], cloud->normals);
    OPE_TRY(check_launch(ctx, "normals_radius_kernel"));   // the next tile reuses the scratch after this one, in stream order
  }
  return OPE_OK;
}

int fpfh_device(ope_ctx* ctx, const ope_cloud* cloud, float radius, float** d_fpfh, float** d_spfh_out) {
  *d_fpfh = nullptr;
  if (d_spfh_out) *d_spfh_out = nullptr;
  if (!cloud->normals) return fail(ctx, OPE_ERR_INVALID, "FPFH needs normals (setInputNormals)");
  const size_t n = cloud->n;
  float *spfh = nullptr, *fpfh = nullptr;
  OPE_TRY(dalloc(ctx, &spfh, n * 33));
  int rc = dalloc(ctx, &fpfh, n * 33);
  if (rc != OPE_OK) { dfree(ctx, spfh); return rc; }
  if (n > 0 && n <= (size_t)kFeatSmemMax && !std::getenv("OPE_FPFH_FORCE_GRID")) {
    // small cloud: both passes from shared memory, no spatial index (two launches instead of eight + a host round trip)
    const float r2 = radius * radius;
    const unsigned blocks = div_up(n, kWarpsPerBlock);
    GridView g;
    std::memset(&g, 0, sizeof(g));
    rc = dyn_smem(ctx, (const void*)spfh_kernel<true>, 2 * kFeatSmemMax * sizeof(float4));
    if (rc == OPE_OK) {
      spfh_kernel<true><<<blocks, kWarpsPerBlock * 32, 2 * n * sizeof(float4), ctx->stream>>>(g, cloud->pts, cloud->normals, (int)n, r2, spfh);
      rc = check_launch(ctx, "spfh_kernel<smem>");
    }
    if (rc == OPE_OK) {
      fpfh_kernel<true><<<blocks, kWarpsPerBlock * 32, n * sizeof(float4), ctx->stream>>>(g, cloud->pts, (int)n, r2, spfh, fpfh);
      rc = check_launch(ctx, "fpfh_kernel<smem>");
    }
  } else if (n > 0) {
    GridView g;
    rc = cloud_grid(ctx, cloud, radius * 0.5f, &g);
    if (rc == OPE_OK) {
      const float r2 = radius * radius;
      const unsigned blocks = div_up(n, kWarpsPerBlock);
      spfh_kernel<false><<<blocks, kWarpsPerBlock * 32, 0, ctx->stream>>>(g, cloud->pts, cloud->normals, (int)n, r2, spfh);
      rc = check_launch(ctx, "spfh_kernel");
      if (rc == OPE_OK) {
        fpfh_kernel<false><<<blocks, kWarpsPerBlock * 32, 0, ctx->stream>>>(g, cloud->pts, (int)n, r2, spfh, fpfh);
        rc = check_launch(ctx, "fpfh_kernel");
      }
    }
  }
  if (rc != OPE_OK) { dfree(ctx, spfh); dfree(ctx, fpfh); return rc; }
  *d_fpfh = fpfh;
  if (d_spfh_out) *d_spfh_out = spfh; else dfree(ctx, spfh);
  return OPE_OK;
}

int feature_knn_exact_device(ope_ctx* ctx, const float* d_ftgt, size_t nt, const float* d_fqry, size_t nq_all, int dim, int k,
                             const int* d_qlist, size_t n_list, int* d_idx, float* d_d2) {
  if (dim < 1 || dim > kFkMaxDim) return fail(ctx, OPE_ERR_INVALID, "feature dimension must be in [1, %d]", kFkMaxDim);
  if (k < 1 || k > kFkMaxK) return fail(ctx, OPE_ERR_INVALID, "feature k must be in [1, %d]", kFkMaxK);
  const size_t nq = d_qlist ? n_list : nq_all;
  if (nq == 0) return OPE_OK;
  const unsigned qblocks = div_up(nq, kFkQueries);
  // enough target splits to give every SM a block, at least one tile each
  int splits = (int)std::max<size_t>(1, std::min<size_t>((size_t)(2 * ctx->sm_count + qblocks - 1) / qblocks,
                                                         (nt + kFkTile - 1) / kFkTile));
  splits = std::min(splits, 1024);
  int t_per_split = (int)((nt + splits - 1) / std::max(splits, 1));
  t_per_split = std::max(kFkTile, (t_per_split + kFkTile - 1) / kFkTile * kFkTile);
  splits = (int)std::max<size_t>(1, (nt + t_per_split - 1) / t_per_split);
  Scratch<int> pi(ctx);
  Scratch<float> pd(ctx);
  OPE_TRY(pi.alloc(nq * splits * k));
  OPE_TRY(pd.alloc(nq * splits * k));
  dim3 grid(qblocks, splits);
  feature_knn_kernel<<<grid, kFkQueries, kFkTile * dim * sizeof(float), ctx->stream>>>(d_ftgt, (int)nt, nullptr, 0, d_fqry, (int)nq, 0,
                                                                                        nullptr, dim, k, t_per_split, d_qlist, pi.p, pd.p);
  OPE_TRY(check_launch(ctx, "feature_knn_kernel"));
  feature_knn_merge_kernel<<<div_up(nq, 128), 128, 0, ctx->stream>>>(pi.p, pd.p, (int)nq, nullptr, splits, k, d_qlist, d_idx, d_d2);
  return check_launch(ctx, "feature_knn_merge_kernel");
}

// tensor-core path (featgemm.cu) when the problem is large enough to pay for it, exact float32 kernel otherwise; both give
// the same indices and distances (the GEMM only nominates, the ranking is always the exact float32 one)
int feature_knn_device(ope_ctx* ctx, const float* d_ftgt, size_t nt, const float* d_fqry, size_t nq, int dim, int k,
                       int* d_idx, float* d_d2) {
  if (dim < 1 || dim > kFkMaxDim) return fail(ctx, OPE_ERR_INVALID, "feature dimension must be in [1, %d]", kFkMaxDim);
  if (k < 1 || k > kFkMaxK) return fail(ctx, OPE_ERR_INVALID, "feature k must be in [1, %d]", kFkMaxK);
  if (nq == 0) return OPE_OK;
  if (feature_knn_gemm_applicable(nt, nq, dim, k)) return feature_knn_gemm_device(ctx, d_ftgt, nt, d_fqry, nq, dim, k, d_idx, d_d2, nullptr);
  return feature_knn_exact_device(ctx, d_ftgt, nt, d_fqry, nq, dim, k, nullptr, 0, d_idx, d_d2);
}

// ---- frame-spanning launches for ope_pose_batch: `clouds` clouds of counts[c] <= max_n points at c * stride ----
int normals_smem_batch(ope_ctx* ctx, const float4* pts, const int* d_counts, int stride, int clouds, int max_n, int k, const float vp[3],
                       float4* out) {
  if (k < 1 || k > 32) return fail(ctx, OPE_ERR_INVALID, "normal estimation k must be in [1, 32]");
  if (max_n > kNormSmemMax) return fail(ctx, OPE_ERR_CAPACITY, "batched normals: cloud larger than the shared-memory path");
  if (clouds <= 0 || max_n <= 0) return OPE_OK;
  OPE_TRY(dyn_smem(ctx, (const void*)normals_smem_batch_kernel, kNormSmemMax * sizeof(float4)));
  // a few blocks per cloud: every block stages the whole cloud in shared memory, so more blocks mean more staging
  const unsigned bx = (unsigned)std::min<size_t>(div_up((size_t)max_n * 32, kNormThreads), 8);
  normals_smem_batch_kernel<<<dim3(bx, clouds), kNormThreads, (size_t)max_n * sizeof(float4), ctx->stream>>>(pts, d_counts, stride, k, vp[0],
                                                                                                           vp[1], vp[2], out);
  return check_launch(ctx, "normals_smem_batch_kernel");
}
int fpfh_smem_batch(ope_ctx* ctx, const float4* pts, const float4* nrm, const int* d_counts, int stride, int clouds, int max_n, float radius,
                    float* spfh, float* fpfh) {
  if (max_n > kFeatSmemMax) return fail(ctx, OPE_ERR_CAPACITY, "batched FPFH: cloud larger than the shared-memory path");
  if (clouds <= 0 || max_n <= 0) return OPE_OK;
  const float r2 = radius * radius;
  OPE_TRY(dyn_smem(ctx, (const void*)spfh_batch_kernel, 2 * kFeatSmemMax * sizeof(float4)));
  OPE_TRY(dyn_smem(ctx, (const void*)fpfh_batch_kernel, kFeatSmemMax * sizeof(float4)));
  const dim3 grid(div_up((size_t)max_n, kWarpsPerBlock), clouds);
  spfh_batch_kernel<<<grid, kWarpsPerBlock * 32, 2 * (size_t)max_n * sizeof(float4), ctx->stream>>>(pts, nrm, d_counts, stride, r2, spfh);
  OPE_TRY(check_launch(ctx, "spfh_batch_kernel"));
  fpfh_batch_kernel<<<grid, kWarpsPerBlock * 32, (size_t)max_n * sizeof(float4), ctx->stream>>>(pts, d_counts, stride, r2, spfh, fpfh);
  return check_launch(ctx, "fpfh_batch_kernel");
}
// k nearest target descriptors (frame f: ftgt + f * stride * dim, counts[f] rows) of each query descriptor of the frame
// (fqry + f * qstride * dim, d_qcounts[f] <= nq rows; qstride 0 and d_qcounts null: the same nq queries in every frame);
// frame f's answers at out_idx + f * nq * k
int feature_knn_batch(ope_ctx* ctx, const float* ftgt, const int* d_counts, int stride, int frames, int max_nt, const float* fqry, int nq,
                      int qstride, const int* d_qcounts, int dim, int k, int* out_idx) {
  if (dim < 1 || dim > kFkMaxDim) return fail(ctx, OPE_ERR_INVALID, "feature dimension must be in [1, %d]", kFkMaxDim);
  if (k < 1 || k > kFkMaxK) return fail(ctx, OPE_ERR_INVALID, "feature k must be in [1, %d]", kFkMaxK);
  if (frames <= 0 || nq <= 0) return OPE_OK;
  const unsigned qblocks = div_up((size_t)nq, kFkQueries);
  int splits = std::max(1, std::min(4, (max_nt + kFkTile - 1) / kFkTile));
  int t_per_split = (max_nt + splits - 1) / splits;
  t_per_split = std::max(kFkTile, (t_per_split + kFkTile - 1) / kFkTile * kFkTile);
  splits = std::max(1, (max_nt + t_per_split - 1) / t_per_split);
  Scratch<int> pi(ctx);
  Scratch<float> pd(ctx);
  OPE_TRY(pi.alloc((size_t)frames * nq * splits * k));
  OPE_TRY(pd.alloc((size_t)frames * nq * splits * k));
  feature_knn_kernel<<<dim3(qblocks, splits, frames), kFkQueries, kFkTile * dim * sizeof(float), ctx->stream>>>(
      ftgt, 0, d_counts, stride, fqry, nq, qstride, d_qcounts, dim, k, t_per_split, nullptr, pi.p, pd.p);
  OPE_TRY(check_launch(ctx, "feature_knn_kernel"));
  feature_knn_merge_kernel<<<dim3(div_up((size_t)nq, 128), frames), 128, 0, ctx->stream>>>(pi.p, pd.p, nq, d_qcounts, splits, k, nullptr,
                                                                                          out_idx, nullptr);
  return check_launch(ctx, "feature_knn_merge_kernel");
}

int remove_nan_normals_device(ope_ctx* ctx, ope_cloud** cloud) {
  ope_cloud* c = *cloud;
  if (!c->normals || c->n == 0) return OPE_OK;
  const size_t n = c->n;
  Scratch<int> flags(ctx);
  OPE_TRY(flags.alloc(n + 1));
  OPE_CUDA_TRY(ctx, cudaMemsetAsync(flags.p + n, 0, sizeof(int), ctx->stream));
  finite_normal_flag_kernel<<<div_up(n, 256), 256, 0, ctx->stream>>>(c->normals, (int)n, flags.p);
  OPE_TRY(check_launch(ctx, "finite_normal_flag_kernel"));
  OPE_TRY(exclusive_scan_i32(ctx, flags.p, n + 1));
  void* h;
  OPE_TRY(read_back(ctx, flags.p + n, sizeof(int), &h));
  const size_t m = (size_t) * (const int*)h;
  if (m == n) return OPE_OK;
  ope_cloud* o = nullptr;
  OPE_TRY(cloud_alloc(ctx, m, true, &o));
  compact_cloud_kernel<<<div_up(n, 256), 256, 0, ctx->stream>>>(c->pts, c->normals, (int)n, flags.p, o->pts, o->normals);
  int rc = check_launch(ctx, "compact_cloud_kernel");
  if (rc != OPE_OK) { ope_cloud_free(ctx, o); return rc; }
  ope_cloud_free(ctx, c);
  *cloud = o;
  return OPE_OK;
}

}  // namespace ope

// =========================================================================================== C ABI =====
using namespace ope;

extern "C" {

int ope_normals_knn(ope_ctx* ctx, ope_cloud* cloud, int k, const float viewpoint[3], float* out4) {
  OPE_ENTER(ctx);
  if (!ctx || !cloud) return OPE_ERR_INVALID;
  const float zero[3] = {0, 0, 0};
  OPE_TRY(normals_device(ctx, cloud, k, viewpoint ? viewpoint : zero));
  if (out4 && cloud->n)
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(out4, cloud->normals, cloud->n * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream));
  OPE_CUDA_TRY(ctx, ope::stream_sync(ctx));
  return OPE_OK;
}

int ope_normals_radius(ope_ctx* ctx, ope_cloud* cloud, float radius, const float viewpoint[3], float* out4) {
  OPE_ENTER(ctx);
  if (!ctx || !cloud) return OPE_ERR_INVALID;
  const float zero[3] = {0, 0, 0};
  OPE_TRY(normals_radius_device(ctx, cloud, radius, viewpoint ? viewpoint : zero));
  if (out4 && cloud->n)
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(out4, cloud->normals, cloud->n * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream));
  OPE_CUDA_TRY(ctx, ope::stream_sync(ctx));
  return OPE_OK;
}

int ope_fpfh(ope_ctx* ctx, const ope_cloud* cloud, float radius, float* out, float* out_spfh) {
  OPE_ENTER(ctx);
  if (!ctx || !cloud || !out || !(radius > 0)) return OPE_ERR_INVALID;
  float *f = nullptr, *s = nullptr;
  OPE_TRY(fpfh_device(ctx, cloud, radius, &f, &s));
  cudaError_t e = cudaSuccess;
  if (cloud->n) {
    e = cudaMemcpyAsync(out, f, cloud->n * 33 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && out_spfh)
      e = cudaMemcpyAsync(out_spfh, s, cloud->n * 33 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream);
  }
  if (e == cudaSuccess) e = ope::stream_sync(ctx);
  dfree(ctx, f); dfree(ctx, s);
  if (e != cudaSuccess) return fail(ctx, OPE_ERR_CUDA, "fpfh download failed: %s", cudaGetErrorString(e));
  return OPE_OK;
}

int ope_feature_knn(ope_ctx* ctx, const float* ftgt, size_t nt, const float* fqry, size_t nq, int dim, int k,
                    int32_t* out_idx, float* out_d2) {
  OPE_ENTER(ctx);
  if (!ctx || !ftgt || !fqry || !out_idx) return OPE_ERR_INVALID;
  Scratch<float> dt(ctx), dq(ctx), dd(ctx);
  Scratch<int> di(ctx);
  OPE_TRY(dt.alloc(nt * dim)); OPE_TRY(dq.alloc(nq * dim)); OPE_TRY(dd.alloc(nq * k)); OPE_TRY(di.alloc(nq * k));
  if (nt) OPE_CUDA_TRY(ctx, cudaMemcpyAsync(dt.p, ftgt, nt * dim * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  if (nq) OPE_CUDA_TRY(ctx, cudaMemcpyAsync(dq.p, fqry, nq * dim * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  OPE_TRY(feature_knn_device(ctx, dt.p, nt, dq.p, nq, dim, k, di.p, dd.p));
  if (nq) {
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(out_idx, di.p, nq * k * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    if (out_d2) OPE_CUDA_TRY(ctx, cudaMemcpyAsync(out_d2, dd.p, nq * k * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  }
  OPE_CUDA_TRY(ctx, ope::stream_sync(ctx));
  return OPE_OK;
}

}  // extern "C"
