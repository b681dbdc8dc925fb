// grid.cu — context, device clouds, the uniform-grid index (K2/K3) and the voxel down-samplers (K1).
//
// HBM layout: a cloud is one float4 array (x,y,z,1) [+ one float4 array of normals]; an index over it is
// `cell_start` (int32, ncells+1) plus the points counting-sorted by cell (float4, w = original index).
// All kernels here are HBM/L2-bound byte shuffles: float4 loads, one atomic per point, grid sizes a multiple
// of the SM count where the work is large enough to matter.
#include <algorithm>
#include <cmath>

#include "ope_host.cuh"
#include "ope_octet.cuh"

namespace ope {

static constexpr int kThreads = 256;
// Dense voxel tables (UniformSampling, VoxelGrid) cover a frame in windows of at most this many consecutive voxel indices, so
// their memory does not grow with the frame (2 GB of 64-bit keys for UniformSampling at most).
static constexpr int64_t kVoxelWindowCells = (int64_t)1 << 28;

// ============================================================================================ kernels ==
__device__ __forceinline__ int bin_coord(float v, float o, float inv, int min_b) {
  return (int)floorf((v - o) * inv) - min_b;
}
__device__ __forceinline__ int64_t bin_cell(const Binning& b, float x, float y, float z) {
  int cx = bin_coord(x, b.o[0], b.inv[0], b.min_b[0]);
  int cy = bin_coord(y, b.o[1], b.inv[1], b.min_b[1]);
  int cz = bin_coord(z, b.o[2], b.inv[2], b.min_b[2]);
  // clamp: rounding can put a point on the max face one cell out
  cx = min(max(cx, 0), b.dim[0] - 1);
  cy = min(max(cy, 0), b.dim[1] - 1);
  cz = min(max(cz, 0), b.dim[2] - 1);
  if (b.morton_bits > 0) return (int64_t)morton3((unsigned)cx, (unsigned)cy, (unsigned)cz);
  return ((int64_t)cz * b.dim[1] + cy) * b.dim[0] + cx;
}

// per-block min/max/count of finite points -> partials[block][8]
// partials[8 * block]; with `ticket` != nullptr the block that finishes last also folds the partials into `out` (one launch
// instead of two: min / max / count do not depend on the order) and re-arms the ticket for the next call on this context.
__global__ void bbox_partial_kernel(const float4* __restrict__ pts, int n, float* __restrict__ partials, unsigned* __restrict__ ticket = nullptr,
                                    float* __restrict__ out = nullptr) {
  float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
  int cnt = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    float4 p = __ldg(pts + i);
    if (finite3(p.x, p.y, p.z)) {
      mn[0] = fminf(mn[0], p.x); mn[1] = fminf(mn[1], p.y); mn[2] = fminf(mn[2], p.z);
      mx[0] = fmaxf(mx[0], p.x); mx[1] = fmaxf(mx[1], p.y); mx[2] = fmaxf(mx[2], p.z);
      ++cnt;
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    for (int d = 0; d < 3; ++d) {
      mn[d] = fminf(mn[d], __shfl_xor_sync(0xffffffffu, mn[d], o));
      mx[d] = fmaxf(mx[d], __shfl_xor_sync(0xffffffffu, mx[d], o));
    }
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  __shared__ float s[kThreads / 32][8];
  int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) {
    for (int d = 0; d < 3; ++d) { s[w][d] = mn[d]; s[w][3 + d] = mx[d]; }
    s[w][6] = __int_as_float(cnt);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int k = 1; k < kThreads / 32; ++k) {
      for (int d = 0; d < 3; ++d) { mn[d] = fminf(mn[d], s[k][d]); mx[d] = fmaxf(mx[d], s[k][3 + d]); }
      cnt += __float_as_int(s[k][6]);
    }
    float* o = partials + 8 * blockIdx.x;
    for (int d = 0; d < 3; ++d) { o[d] = mn[d]; o[3 + d] = mx[d]; }
    o[6] = __int_as_float(cnt);
  }
  if (!ticket) return;
  __shared__ int s_last;
  if (threadIdx.x == 0) {
    __threadfence();
    s_last = atomicAdd(ticket, 1u) == gridDim.x - 1 ? 1 : 0;
  }
  __syncthreads();
  if (!s_last || w != 0) return;
  __threadfence();
  float fmn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, fmx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
  int fc = 0;
  for (int b = l; b < (int)gridDim.x; b += 32) {
    const volatile float* p = partials + 8 * b;
    for (int d = 0; d < 3; ++d) { fmn[d] = fminf(fmn[d], p[d]); fmx[d] = fmaxf(fmx[d], p[3 + d]); }
    fc += __float_as_int(p[6]);
  }
  for (int o = 16; o > 0; o >>= 1) {
    for (int d = 0; d < 3; ++d) {
      fmn[d] = fminf(fmn[d], __shfl_xor_sync(0xffffffffu, fmn[d], o));
      fmx[d] = fmaxf(fmx[d], __shfl_xor_sync(0xffffffffu, fmx[d], o));
    }
    fc += __shfl_xor_sync(0xffffffffu, fc, o);
  }
  if (l == 0) {
    for (int d = 0; d < 3; ++d) { out[d] = fmn[d]; out[3 + d] = fmx[d]; }
    out[6] = __int_as_float(fc);
    *ticket = 0u;
  }
}
__global__ void bbox_final_kernel(const float* __restrict__ partials, int nblocks, float* __restrict__ out) {
  // one warp: lanes stride over the per-block partials, shuffle tree
  const int lane = threadIdx.x;
  float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
  int cnt = 0;
  for (int b = lane; b < nblocks; b += 32) {
    const float* p = partials + 8 * b;
    for (int d = 0; d < 3; ++d) { mn[d] = fminf(mn[d], p[d]); mx[d] = fmaxf(mx[d], p[3 + d]); }
    cnt += __float_as_int(p[6]);
  }
  for (int o = 16; o > 0; o >>= 1) {
    for (int d = 0; d < 3; ++d) {
      mn[d] = fminf(mn[d], __shfl_xor_sync(0xffffffffu, mn[d], o));
      mx[d] = fmaxf(mx[d], __shfl_xor_sync(0xffffffffu, mx[d], o));
    }
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  if (lane == 0) {
    for (int d = 0; d < 3; ++d) { out[d] = mn[d]; out[3 + d] = mx[d]; }
    out[6] = __int_as_float(cnt);
  }
}

// ---- exclusive scan (int32), 2048 items per block ----
static constexpr int kScanItems = 8;
__global__ void scan_block_kernel(int* __restrict__ data, size_t n, int* __restrict__ block_sums) {
  __shared__ int warp_sums[kThreads / 32];
  const size_t base = ((size_t)blockIdx.x * kThreads + threadIdx.x) * kScanItems;
  int v[kScanItems];
  int sum = 0;
#pragma unroll
  for (int j = 0; j < kScanItems; ++j) {
    v[j] = (base + j < n) ? data[base + j] : 0;
    sum += v[j];
  }
  int incl = sum;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) warp_sums[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int ws = lane < kThreads / 32 ? warp_sums[lane] : 0;
    int wi = ws;
    for (int o = 1; o < 32; o <<= 1) {
      int t = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= o) wi += t;
    }
    if (lane < kThreads / 32) warp_sums[lane] = wi - ws;  // exclusive
    if (lane == kThreads / 32 - 1 && block_sums) block_sums[blockIdx.x] = wi;
  }
  __syncthreads();
  int run = warp_sums[warp] + incl - sum;
#pragma unroll
  for (int j = 0; j < kScanItems; ++j) {
    if (base + j < n) data[base + j] = run;
    run += v[j];
  }
}
// Exclusive scan of up to a few 10^4 ints by ONE block in one launch (tiles of 4096 with a running carry): the cell tables of the
// small clouds of the frame path are this size, and a launch costs more than the scan.
static constexpr int kScan1Threads = 1024;
__global__ void __launch_bounds__(kScan1Threads) scan_single_kernel(int* __restrict__ data, int n) {
  __shared__ int warp_sums[kScan1Threads / 32];
  __shared__ int s_carry[2];   // double-buffered by tile parity: warp 0 writes the next carry while other warps still read this one
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_carry[0] = 0;
  __syncthreads();
  int par = 0;
  for (int tile = 0; tile < n; tile += kScan1Threads * 4, par ^= 1) {
    const int base = tile + threadIdx.x * 4;
    int v[4];
    int sum = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) { v[j] = base + j < n ? data[base + j] : 0; sum += v[j]; }
    int incl = sum;
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
    if (lane == 31) warp_sums[warp] = incl;
    __syncthreads();
    const int carry = s_carry[par];
    if (warp == 0) {
      const int ws = warp_sums[lane];
      int wi = ws;
      for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, wi, o); if (lane >= o) wi += t; }
      warp_sums[lane] = wi - ws;
      if (lane == 31) s_carry[par ^ 1] = carry + wi;
    }
    __syncthreads();
    int run = carry + warp_sums[warp] + incl - sum;
#pragma unroll
    for (int j = 0; j < 4; ++j) { if (base + j < n) data[base + j] = run; run += v[j]; }
    __syncthreads();
  }
}

__global__ void scan_add_kernel(int* __restrict__ data, size_t n, const int* __restrict__ block_offsets) {
  const size_t base = ((size_t)blockIdx.x * kThreads + threadIdx.x) * kScanItems;
  const int off = block_offsets[blockIdx.x];
#pragma unroll
  for (int j = 0; j < kScanItems; ++j)
    if (base + j < n) data[base + j] += off;
}

// ---- cell build ----
// The cell build covers the cells [c0, c0 + nwin) (a window of a voxel table, see kVoxelWindowCells; all cells of a search grid):
// points of other cells are skipped, counts1 / B / cell_start are indexed by cell - c0.
__global__ void cell_count_kernel(const float4* __restrict__ pts, int n, Binning bin, int64_t c0, int64_t nwin,
                                  int* __restrict__ counts1) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    float4 p = __ldg(pts + i);
    if (!finite3(p.x, p.y, p.z)) continue;
    const int64_t c = bin_cell(bin, p.x, p.y, p.z) - c0;
    if ((uint64_t)c < (uint64_t)nwin) atomicAdd(counts1 + c, 1);
  }
}
// B = cell_start base (see build_cells): after this kernel B[1+c] has advanced to the end of cell c.
__global__ void cell_scatter_kernel(const float4* __restrict__ pts, int n, Binning bin, int64_t c0, int64_t nwin, int* __restrict__ B,
                                    float4* __restrict__ sorted) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    float4 p = __ldg(pts + i);
    if (!finite3(p.x, p.y, p.z)) continue;
    const int64_t c = bin_cell(bin, p.x, p.y, p.z) - c0;
    if ((uint64_t)c >= (uint64_t)nwin) continue;
    int pos = atomicAdd(B + 1 + c, 1);
    sorted[pos] = make_float4(p.x, p.y, p.z, __int_as_float(i));
  }
}
// Order each cell's points by original index (deterministic traversal whatever order the atomics scattered them in): every point
// counts the points of its cell with a smaller index and goes to that rank in a second array. One thread per point, so a cell of a
// thousand points (a 5 cm clustering grid over a full-resolution frame) costs its points a thousand cached loads each instead of
// one thread a million moves.
__global__ void cell_rank_kernel(const float4* __restrict__ scattered, const int* __restrict__ cell_start, int64_t ncells, Binning bin,
                                 int64_t c0, float4* __restrict__ sorted) {
  const int total = cell_start[ncells];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const float4 v = scattered[i];
    const int c = (int)(bin_cell(bin, v.x, v.y, v.z) - c0);
    const int b = cell_start[c], e = cell_start[c + 1];
    const int key = __float_as_int(v.w);
    int rank = 0;
    for (int j = b; j < e; ++j) rank += __float_as_int(__ldg(&scattered[j].w)) < key ? 1 : 0;
    sorted[b + rank] = v;
  }
}

// ---- k-NN query kernels (ope_octet.cuh): k = 1 one query per thread (block_nn1), k > 1 one query per warp (warp_knn) ----
static constexpr int kKnnThreads = 256;
__global__ void __launch_bounds__(kKnnThreads) nn1_kernel(GridView g, const float4* __restrict__ qry, int nq,
                                                          int* __restrict__ out_idx, float* __restrict__ out_d2) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Nn1Smem<kKnnThreads>* nn = reinterpret_cast<Nn1Smem<kKnnThreads>*>(smem_raw);
  for (int base = blockIdx.x * kKnnThreads; base < nq; base += gridDim.x * kKnnThreads) {
    const int i = base + (int)threadIdx.x;
    float4 q = make_float4(0, 0, 0, 0);
    if (i < nq) q = __ldg(qry + i);
    const bool ok = i < nq && finite3(q.x, q.y, q.z);
    float d2;
    const int idx = block_nn1<kKnnThreads>(g, nn, ok, q.x, q.y, q.z, FLT_MAX, -1, nullptr, d2);
    if (i < nq) {
      out_idx[i] = ok ? idx : -1;
      if (out_d2) out_d2[i] = (ok && idx >= 0) ? d2 : INFINITY;
    }
  }
}
__global__ void __launch_bounds__(kKnnThreads) knn_kernel(GridView g, const float4* __restrict__ qry, int nq, int k,
                                                          int* __restrict__ out_idx, float* __restrict__ out_d2) {
  __shared__ OctStack stacks[kKnnThreads / 32];
  OctStack* st = &stacks[threadIdx.x >> 5];
  const int lane = threadIdx.x & 31;
  const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
  for (int i = wid; i < nq; i += n_warps) {
    const float4 q = __ldg(qry + i);
    const bool ok = finite3(q.x, q.y, q.z);
    float ld;
    int li;
    const int cnt = warp_knn(g, st, ok, q.x, q.y, q.z, k, FLT_MAX, ld, li);
    if (lane < k) {
      out_idx[(size_t)i * k + lane] = lane < cnt ? li : -1;
      if (out_d2) out_d2[(size_t)i * k + lane] = lane < cnt ? ld : INFINITY;
    }
    __syncwarp();
  }
}
// k > 32: the list in shared memory (warp_knn_list), written out with -1 / +inf padding past the count
__global__ void __launch_bounds__(kKnnThreads) knn_list_kernel(GridView g, const float4* __restrict__ qry, int nq, int k,
                                                               int* __restrict__ out_idx, float* __restrict__ out_d2) {
  __shared__ OctStack stacks[kKnnThreads / 32];
  __shared__ KnnList lists[kKnnThreads / 32];
  OctStack* st = &stacks[threadIdx.x >> 5];
  KnnList* L = &lists[threadIdx.x >> 5];
  const int lane = threadIdx.x & 31;
  const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
  for (int i = wid; i < nq; i += n_warps) {
    const float4 q = __ldg(qry + i);
    const int cnt = warp_knn_list(g, st, L, finite3(q.x, q.y, q.z), q.x, q.y, q.z, k);
    for (int j = lane; j < k; j += 32) {
      const float2 v = j < cnt ? L->e[j] : make_float2(INFINITY, __int_as_float(-1));
      out_idx[(size_t)i * k + j] = __float_as_int(v.y);
      if (out_d2) out_d2[(size_t)i * k + j] = v.x;
    }
    __syncwarp();
  }
}
__global__ void radius_count_kernel(GridView g, const float4* __restrict__ qry, int nq, float r2, int* __restrict__ counts) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nq) return;
  float4 q = __ldg(qry + i);
  int cnt = 0;
  if (finite3(q.x, q.y, q.z))
    grid_radius_visit(g, q.x, q.y, q.z, r2, [&](float, float, float, int, float) { ++cnt; });
  counts[i] = cnt;
}
__global__ void radius_fill_kernel(GridView g, const float4* __restrict__ qry, int nq, float r2, const int* __restrict__ offsets,
                                   int* __restrict__ out_idx, float* __restrict__ out_d2) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nq) return;
  float4 q = __ldg(qry + i);
  if (!finite3(q.x, q.y, q.z)) return;
  int w = offsets[i];
  grid_radius_visit(g, q.x, q.y, q.z, r2, [&](float, float, float, int idx, float d2) { out_idx[w] = idx; out_d2[w] = d2; ++w; });
}

// ---- pack / gather / UniformSampling / VoxelGrid ----
__global__ void gather_kernel(const float4* __restrict__ pts, const float4* __restrict__ nrm, const int* __restrict__ idx,
                              int n, float4* __restrict__ out_pts, float4* __restrict__ out_nrm) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int j = idx[i];
  out_pts[i] = __ldg(pts + j);
  if (nrm && out_nrm) out_nrm[i] = __ldg(nrm + j);
}

// UniformSampling first pass (SURVEY A.1): per voxel of the window [c0, c0 + nwin) keep argmin over (||p4 - ijk4||^2, index);
// keys is indexed by voxel - c0.
__global__ void uniform_key_kernel(const float4* __restrict__ pts, int n, Binning bin, int64_t c0, int64_t nwin,
                                   unsigned long long* __restrict__ keys) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    float4 p = __ldg(pts + i);
    if (!finite3(p.x, p.y, p.z)) continue;
    int ix = (int)floorf(p.x * bin.inv[0]), iy = (int)floorf(p.y * bin.inv[1]), iz = (int)floorf(p.z * bin.inv[2]);
    int64_t cell = ((int64_t)(iz - bin.min_b[2]) * bin.dim[1] + (iy - bin.min_b[1])) * bin.dim[0] + (ix - bin.min_b[0]) - c0;
    if ((uint64_t)cell >= (uint64_t)nwin) continue;
    float a = p.x - (float)ix, b = p.y - (float)iy, c = p.z - (float)iz;
    float d = a * a;
    d = d + b * b;
    d = d + c * c;
    d = d + 1.0f;  // 4th component of (p4 - ijk4): (1 - 0)^2
    unsigned long long key = ((unsigned long long)__float_as_uint(d) << 32) | (unsigned)i;
    atomicMin(keys + cell, key);
  }
}
__global__ void occupied_flag_u64_kernel(const unsigned long long* __restrict__ keys, int64_t ncells, int* __restrict__ flags) {
  for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < ncells; c += (int64_t)gridDim.x * blockDim.x)
    flags[c] = keys[c] != ~0ull ? 1 : 0;
}
__global__ void uniform_compact_kernel(const unsigned long long* __restrict__ keys, int64_t ncells,
                                       const int* __restrict__ pos, int* __restrict__ out_idx) {
  for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < ncells; c += (int64_t)gridDim.x * blockDim.x) {
    unsigned long long k = keys[c];
    if (k != ~0ull) out_idx[pos[c]] = (int)(unsigned)(k & 0xffffffffull);
  }
}
// Small voxel tables (a down-sampled model or cluster: a few thousand cells): flag, scan and compact in ONE launch by one block
// (tiles of 4096 cells with a running carry); out_idx receives the selected point indices in ascending voxel-key order, *count
// their number.
__global__ void __launch_bounds__(kScan1Threads) uniform_select_single_kernel(const unsigned long long* __restrict__ keys, int ncells,
                                                                              int* __restrict__ out_idx, int* __restrict__ count) {
  __shared__ int warp_sums[kScan1Threads / 32];
  __shared__ int s_carry[2];   // double-buffered by tile parity (see scan_single_kernel)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_carry[0] = 0;
  __syncthreads();
  int par = 0;
  for (int tile = 0; tile < ncells; tile += kScan1Threads * 4, par ^= 1) {
    const int base = tile + threadIdx.x * 4;
    unsigned long long k[4];
    int sum = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) { k[j] = base + j < ncells ? keys[base + j] : ~0ull; sum += k[j] != ~0ull ? 1 : 0; }
    int incl = sum;
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
    if (lane == 31) warp_sums[warp] = incl;
    __syncthreads();
    const int carry = s_carry[par];
    if (warp == 0) {
      const int ws = warp_sums[lane];
      int wi = ws;
      for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, wi, o); if (lane >= o) wi += t; }
      warp_sums[lane] = wi - ws;
      if (lane == 31) s_carry[par ^ 1] = carry + wi;
    }
    __syncthreads();
    int run = carry + warp_sums[warp] + incl - sum;
#pragma unroll
    for (int j = 0; j < 4; ++j) if (k[j] != ~0ull) out_idx[run++] = (int)(unsigned)(k[j] & 0xffffffffull);
    __syncthreads();
  }
  if (threadIdx.x == 0) *count = s_carry[par];
}

__global__ void occupied_flag_cells_kernel(const int* __restrict__ cell_start, int64_t ncells, int* __restrict__ flags) {
  for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < ncells; c += (int64_t)gridDim.x * blockDim.x)
    flags[c] = cell_start[c + 1] > cell_start[c] ? 1 : 0;
}
// VoxelGrid fourth pass (SURVEY A.2): float sums in ascending point index, divided by the count.
__global__ void voxel_centroid_kernel(const int* __restrict__ cell_start, int64_t ncells, const float4* __restrict__ sorted,
                                      const float* __restrict__ rgb, const int* __restrict__ pos, float* __restrict__ out_xyz,
                                      float* __restrict__ out_rgb) {
  for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < ncells; c += (int64_t)gridDim.x * blockDim.x) {
    const int b = cell_start[c], e = cell_start[c + 1];
    if (e <= b) continue;
    float s[6] = {0, 0, 0, 0, 0, 0};
    for (int i = b; i < e; ++i) {
      float4 p = sorted[i];
      s[0] += p.x; s[1] += p.y; s[2] += p.z;
      if (rgb) {
        unsigned u = __float_as_uint(rgb[__float_as_int(p.w)]);
        s[3] += (float)((u >> 16) & 0xff); s[4] += (float)((u >> 8) & 0xff); s[5] += (float)(u & 0xff);
      }
    }
    float cnt = (float)(e - b);
    for (int d = 0; d < 6; ++d) s[d] /= cnt;
    const int m = pos[c];
    out_xyz[3 * (size_t)m] = s[0]; out_xyz[3 * (size_t)m + 1] = s[1]; out_xyz[3 * (size_t)m + 2] = s[2];
    if (rgb && out_rgb) {
      int packed = ((int)s[3] << 16) | ((int)s[4] << 8) | (int)s[5];
      out_rgb[m] = __int_as_float(packed);
    }
  }
}

// ============================================================================================== host ===
static int grid_blocks(ope_ctx* ctx, size_t work) {
  size_t want = (work + kThreads - 1) / kThreads;
  size_t cap = (size_t)ctx->sm_count * 8;  // persistent-style cap: a multiple of the SM count
  if (want > cap) want = cap;
  return (int)std::max<size_t>(want, 1);
}

int cloud_alloc(ope_ctx* ctx, size_t n, bool with_normals, ope_cloud** out) {
  ope_cloud* c = new ope_cloud();
  c->ctx = ctx; c->n = n;
  int rc = dalloc(ctx, &c->pts, n);
  if (rc == OPE_OK && with_normals) rc = dalloc(ctx, &c->normals, n);
  if (rc != OPE_OK) { dfree(ctx, c->pts); delete c; return rc; }
  *out = c;
  return OPE_OK;
}

__global__ void content_hash_kernel(const float4* __restrict__ pts, int n, unsigned long long* __restrict__ out) {
  unsigned long long acc = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = __ldg(pts + i);
    unsigned long long a = ((unsigned long long)__float_as_uint(p.x) << 32) | __float_as_uint(p.y);
    unsigned long long b = ((unsigned long long)__float_as_uint(p.z) << 32) | (unsigned)i;
    a = (a ^ (b * 0x9fb21c651e98df25ull)) * 0xc2b2ae3d27d4eb4full;
    a ^= a >> 29;
    acc += a * 0x165667b19e3779f9ull;     // wrap-around sum: independent of the order the threads arrive in
  }
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, acc);
}

int cloud_content_hash(ope_ctx* ctx, const ope_cloud* c, unsigned long long* out) {
  *out = 0;
  if (c->n == 0) return OPE_OK;
  Scratch<unsigned long long> d(ctx);
  OPE_TRY(d.alloc(1));
  OPE_CUDA_TRY(ctx, cudaMemsetAsync(d.p, 0, sizeof(unsigned long long), ctx->stream));
  content_hash_kernel<<<std::min(grid_blocks(ctx, c->n), 592), kThreads, 0, ctx->stream>>>(c->pts, (int)c->n, d.p);
  OPE_TRY(check_launch(ctx, "content_hash_kernel"));
  void* h;
  OPE_TRY(read_back(ctx, d.p, sizeof(unsigned long long), &h));
  *out = *(const unsigned long long*)h ^ (unsigned long long)c->n;
  return OPE_OK;
}

int cloud_bbox(ope_ctx* ctx, ope_cloud* c) {
  if (c->bbox_valid) return OPE_OK;
  if (c->n == 0) {
    for (int d = 0; d < 6; ++d) c->bbox[d] = 0;
    c->n_finite = 0; c->bbox_valid = true;
    return OPE_OK;
  }
  const int nb = std::min(grid_blocks(ctx, c->n), 1024);
  Scratch<float> partials(ctx), fin(ctx);
  OPE_TRY(partials.alloc((size_t)nb * 8));
  OPE_TRY(fin.alloc(8));
  if (ctx->ticket) {
    bbox_partial_kernel<<<nb, kThreads, 0, ctx->stream>>>(c->pts, (int)c->n, partials.p, ctx->ticket, fin.p);
    OPE_TRY(check_launch(ctx, "bbox_partial_kernel"));
  } else {
    bbox_partial_kernel<<<nb, kThreads, 0, ctx->stream>>>(c->pts, (int)c->n, partials.p);
    OPE_TRY(check_launch(ctx, "bbox_partial_kernel"));
    bbox_final_kernel<<<1, 32, 0, ctx->stream>>>(partials.p, nb, fin.p);
    OPE_TRY(check_launch(ctx, "bbox_final_kernel"));
  }
  void* h;
  OPE_TRY(read_back(ctx, fin.p, 8 * sizeof(float), &h));
  const float* f = (const float*)h;
  for (int d = 0; d < 6; ++d) c->bbox[d] = f[d];
  int cnt; std::memcpy(&cnt, f + 6, 4);
  c->n_finite = cnt;
  c->bbox_valid = true;
  return OPE_OK;
}

int exclusive_scan_i32(ope_ctx* ctx, int* data, size_t n) {
  if (n == 0) return OPE_OK;
  const size_t per_block = (size_t)kThreads * kScanItems;
  const size_t nb = (n + per_block - 1) / per_block;
  if (nb > 1 && n <= 65536) {
    scan_single_kernel<<<1, kScan1Threads, 0, ctx->stream>>>(data, (int)n);
    return check_launch(ctx, "scan_single_kernel");
  }
  if (nb == 1) {
    scan_block_kernel<<<1, kThreads, 0, ctx->stream>>>(data, n, nullptr);
    return check_launch(ctx, "scan_block_kernel");
  }
  Scratch<int> sums(ctx);
  OPE_TRY(sums.alloc(nb));
  scan_block_kernel<<<(unsigned)nb, kThreads, 0, ctx->stream>>>(data, n, sums.p);
  OPE_TRY(check_launch(ctx, "scan_block_kernel"));
  OPE_TRY(exclusive_scan_i32(ctx, sums.p, nb));
  scan_add_kernel<<<(unsigned)nb, kThreads, 0, ctx->stream>>>(data, n, sums.p);
  return check_launch(ctx, "scan_add_kernel");
}

int build_cells(ope_ctx* ctx, const float4* pts, size_t n, const Binning& bin, int** cell_start, float4** sorted, int64_t c0,
                int64_t nwin) {
  const int64_t ncells = nwin >= 0 ? nwin : (int64_t)bin.dim[0] * bin.dim[1] * bin.dim[2] - c0;
  int* B = nullptr;
  float4* S = nullptr;
  OPE_TRY(dalloc(ctx, &B, (size_t)ncells + 2));
  int rc = dalloc(ctx, &S, n);
  if (rc != OPE_OK) { dfree(ctx, B); return rc; }
  auto bail = [&](int code) { dfree(ctx, B); dfree(ctx, S); return code; };
  cudaError_t e = cudaMemsetAsync(B, 0, ((size_t)ncells + 2) * sizeof(int), ctx->stream);
  if (e != cudaSuccess) return bail(fail(ctx, OPE_ERR_CUDA, "memset failed: %s", cudaGetErrorString(e)));
  if (n > 0) {
    cell_count_kernel<<<grid_blocks(ctx, n), kThreads, 0, ctx->stream>>>(pts, (int)n, bin, c0, ncells, B + 1);
    if ((rc = check_launch(ctx, "cell_count_kernel")) != OPE_OK) return bail(rc);
  }
  // exclusive scan over B[1 .. ncells+1]: B[1+c] = start of cell c, B[1+ncells] = total
  if ((rc = exclusive_scan_i32(ctx, B + 1, (size_t)ncells + 1)) != OPE_OK) return bail(rc);
  if (n > 0) {
    cell_scatter_kernel<<<grid_blocks(ctx, n), kThreads, 0, ctx->stream>>>(pts, (int)n, bin, c0, ncells, B, S);
    if ((rc = check_launch(ctx, "cell_scatter_kernel")) != OPE_OK) return bail(rc);
    // now B[c] = start of cell c for c in [0, ncells], B[0] = 0
    float4* R = nullptr;
    if ((rc = dalloc(ctx, &R, n)) != OPE_OK) return bail(rc);
    cell_rank_kernel<<<grid_blocks(ctx, n), kThreads, 0, ctx->stream>>>(S, B, ncells, bin, c0, R);
    rc = check_launch(ctx, "cell_rank_kernel");
    dfree(ctx, S);   // stream-ordered: released after the kernel
    S = R;
    if (rc != OPE_OK) return bail(rc);
  }
  *cell_start = B;
  *sorted = S;
  return OPE_OK;
}

float knn_cell_size(const ope_cloud* c, int k) {
  float ex[3];
  for (int d = 0; d < 3; ++d) ex[d] = std::max(c->bbox[3 + d] - c->bbox[d], 0.0f);
  float emax = std::max(ex[0], std::max(ex[1], ex[2]));
  if (!(emax > 0) || c->n_finite <= 0) return 1.0f;
  // surface-density heuristic: area proxy = sum of the three bbox face areas
  float lo = emax * 1e-3f;
  float a = std::max(ex[0], lo), b = std::max(ex[1], lo), cc = std::max(ex[2], lo);
  float area = a * b + b * cc + a * cc;
  float d1 = std::sqrt(area / (3.14159265f * (float)c->n_finite));
  float h = (k <= 1 ? 1.5f : 1.1f * std::sqrt((float)k)) * d1;
  return h;
}

// Search grid with cell edge close to h_wanted: 2^bits cells along the longest bbox axis (bits in [1, OPE_MAX_BITS]).
int cloud_grid(ope_ctx* ctx, const ope_cloud* cc, float h_wanted, GridView* out) {
  ope_cloud* c = const_cast<ope_cloud*>(cc);
  OPE_TRY(cloud_bbox(ctx, c));
  float emax = 0.0f;
  for (int d = 0; d < 3; ++d) emax = std::max(emax, c->bbox[3 + d] - c->bbox[d]);
  if (!(emax > 0) || !std::isfinite(emax)) emax = 1.0f;
  if (!(h_wanted > 0) || !std::isfinite(h_wanted)) h_wanted = emax;
  int bits = (int)std::ceil(std::log2(std::max(emax / h_wanted, 1.0f)));
  bits = std::min(std::max(bits, 1), OPE_MAX_BITS);
  // keep the start array (2^(3*bits) ints) proportionate to the cloud: at most ~64 codes per point, 9 bits only for >1M points
  while (bits > 1 && ((int64_t)1 << (3 * bits)) > std::max<int64_t>(64 * (int64_t)std::max(c->n_finite, 1), 4096)) --bits;
  for (auto& g : c->grids)
    if (g.bits == bits) { *out = g.view; return OPE_OK; }
  const float hh = emax * (1.0f + 1e-4f) / (float)(1 << bits);
  Binning bin;
  for (int d = 0; d < 3; ++d) { bin.o[d] = c->bbox[d]; bin.inv[d] = 1.0f / hh; bin.min_b[d] = 0; bin.dim[d] = 1 << bits; }
  bin.morton_bits = bits;
  GridEntry g;
  g.bits = bits;
  g.ncells = (int64_t)1 << (3 * bits);
  OPE_TRY(build_cells(ctx, c->pts, c->n, bin, &g.cell_start, &g.sorted));
  g.view.ox = bin.o[0]; g.view.oy = bin.o[1]; g.view.oz = bin.o[2];
  g.view.h = hh; g.view.inv_h = bin.inv[0];
  g.view.bits = bits;
  g.view.n = c->n_finite;
  g.view.start = g.cell_start;
  g.view.pts = g.sorted;
  c->grids.push_back(g);
  *out = g.view;
  return OPE_OK;
}

int cloud_any_grid(ope_ctx* ctx, const ope_cloud* c, GridView* out) {
  if (!c->grids.empty()) { *out = c->grids.front().view; return OPE_OK; }
  OPE_TRY(cloud_bbox(ctx, const_cast<ope_cloud*>(c)));
  return cloud_grid(ctx, c, knn_cell_size(c, 1), out);
}

int gather_cloud(ope_ctx* ctx, const ope_cloud* cloud, const int* d_idx, size_t n, ope_cloud** out) {
  ope_cloud* o = nullptr;
  OPE_TRY(cloud_alloc(ctx, n, cloud->normals != nullptr, &o));
  if (n > 0) {
    gather_kernel<<<div_up(n, kThreads), kThreads, 0, ctx->stream>>>(cloud->pts, cloud->normals, d_idx, (int)n, o->pts,
                                                                    o->normals);
    int rc = check_launch(ctx, "gather_kernel");
    if (rc != OPE_OK) { ope_cloud_free(ctx, o); return rc; }
  }
  *out = o;
  return OPE_OK;
}

// PCL voxel frame: min_b/max_b = floor(min*inv), div_b = max_b - min_b + 1
static int pcl_voxel_frame(ope_ctx* ctx, ope_cloud* c, const float leaf[3], Binning* bin, int64_t* ncells) {
  OPE_TRY(cloud_bbox(ctx, c));
  for (int d = 0; d < 3; ++d) {
    bin->o[d] = 0.0f;
    bin->inv[d] = 1.0f / leaf[d];
    volatile float lo = c->bbox[d] * bin->inv[d];
    volatile float hi = c->bbox[3 + d] * bin->inv[d];
    int min_b = (int)std::floor((float)lo), max_b = (int)std::floor((float)hi);
    bin->min_b[d] = min_b;
    int64_t dv = (int64_t)max_b - min_b + 1;
    if (dv > 0x7fffffff) return fail(ctx, OPE_ERR_GRID_TOO_LARGE, "voxel grid dimension overflows int32");
    bin->dim[d] = (int)dv;
  }
  bin->morton_bits = 0;
  *ncells = (int64_t)bin->dim[0] * bin->dim[1] * bin->dim[2];
  return OPE_OK;
}

int uniform_sample_device(ope_ctx* ctx, ope_cloud* cloud, float leaf, int** d_idx, size_t* out_n) {
  *d_idx = nullptr; *out_n = 0;
  OPE_TRY(cloud_bbox(ctx, cloud));
  if (cloud->n_finite == 0) return OPE_OK;
  Binning bin; int64_t ncells;
  float l3[3] = {leaf, leaf, leaf};
  OPE_TRY(pcl_voxel_frame(ctx, cloud, l3, &bin, &ncells));
  // PCL's UniformSampling numbers the voxels with an int: beyond INT_MAX voxels its result is undefined
  if (ncells > 0x7fffffffll)
    return fail(ctx, OPE_ERR_GRID_TOO_LARGE, "leaf size too small for the input: %lld voxels overflow the int voxel index",
                (long long)ncells);
  // the frame in windows of consecutive voxel indices, each selected in ascending voxel order: the windows concatenate in
  // ascending voxel order too. A table of at most 2^16 voxels is one window, selected in one launch.
  const int64_t win = std::min(ncells, kVoxelWindowCells);
  const bool single = ncells <= (1 << 16) && !std::getenv("OPE_UNIFORM_MULTI_PASS");
  Scratch<unsigned long long> keys(ctx);
  Scratch<int> flags(ctx);
  OPE_TRY(keys.alloc((size_t)win));
  if (!single) OPE_TRY(flags.alloc((size_t)win + 1));
  // the index buffer is sized for the worst case (every cell / every point occupied), plus the count of the one-launch select
  const size_t cap = std::min<size_t>((size_t)ncells, cloud->n);
  int* idx = nullptr;
  OPE_TRY(dalloc(ctx, &idx, cap + 1));
  auto bail = [&](int rc) { dfree(ctx, idx); return rc; };
  size_t m = 0;
  for (int64_t c0 = 0; c0 < ncells; c0 += win) {
    const int64_t nw = std::min(win, ncells - c0);
    cudaError_t e = cudaMemsetAsync(keys.p, 0xff, (size_t)nw * 8, ctx->stream);
    if (e != cudaSuccess) return bail(fail(ctx, OPE_ERR_CUDA, "memset failed: %s", cudaGetErrorString(e)));
    uniform_key_kernel<<<grid_blocks(ctx, cloud->n), kThreads, 0, ctx->stream>>>(cloud->pts, (int)cloud->n, bin, c0, nw, keys.p);
    int rc = check_launch(ctx, "uniform_key_kernel");
    void* h = nullptr;
    if (single) {
      if (rc == OPE_OK) {
        uniform_select_single_kernel<<<1, kScan1Threads, 0, ctx->stream>>>(keys.p, (int)nw, idx, idx + cap);
        rc = check_launch(ctx, "uniform_select_single_kernel");
      }
      if (rc == OPE_OK) rc = read_back(ctx, idx + cap, sizeof(int), &h);
      if (rc != OPE_OK) return bail(rc);
      m = (size_t) * (const int*)h;
      continue;
    }
    if (rc == OPE_OK && cudaMemsetAsync(flags.p + nw, 0, sizeof(int), ctx->stream) != cudaSuccess)
      rc = fail(ctx, OPE_ERR_CUDA, "memset failed");
    if (rc == OPE_OK) {
      occupied_flag_u64_kernel<<<grid_blocks(ctx, (size_t)nw), kThreads, 0, ctx->stream>>>(keys.p, nw, flags.p);
      rc = check_launch(ctx, "occupied_flag_u64_kernel");
    }
    if (rc == OPE_OK) rc = exclusive_scan_i32(ctx, flags.p, (size_t)nw + 1);
    if (rc == OPE_OK) rc = read_back(ctx, flags.p + nw, sizeof(int), &h);
    if (rc != OPE_OK) return bail(rc);
    const int mw = *(const int*)h;
    uniform_compact_kernel<<<grid_blocks(ctx, (size_t)nw), kThreads, 0, ctx->stream>>>(keys.p, nw, flags.p, idx + m);
    if ((rc = check_launch(ctx, "uniform_compact_kernel")) != OPE_OK) return bail(rc);
    m += (size_t)mw;
  }
  *d_idx = idx; *out_n = m;
  return OPE_OK;
}

}  // namespace ope

// =========================================================================================== C ABI =====
using namespace ope;

extern "C" {

const char* ope_version(void) { return "ope_cuda 0.1 sm_100a"; }

int ope_ctx_create(int device, void* stream, ope_ctx** out) {
  if (!out) return OPE_ERR_INVALID;
  *out = nullptr;
  // the frame-spanning batches run up to 8 lanes, each on its own stream, next to the caller's streams; the default of 8 hardware
  // work queues would make them share queues. Only effective when this is the process's first CUDA call; a host that
  // initialises CUDA earlier sets the variable itself (INTEGRATION.md).
  setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0);
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) {
    cudaGetLastError();
    return OPE_ERR_NO_DEVICE;  // no CPU fallback
  }
  if (cudaSetDevice(device) != cudaSuccess) return OPE_ERR_NO_DEVICE;
  ope_ctx* ctx = new ope_ctx();
  ctx->device = device;
  if (stream) { ctx->stream = (cudaStream_t)stream; ctx->owns_stream = false; }
  else {
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return OPE_ERR_CUDA; }
    ctx->owns_stream = true;
  }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->sm_count = prop.multiProcessorCount;
  {
    cudaMemPoolProps props;
    std::memset(&props, 0, sizeof(props));
    props.allocType = cudaMemAllocationTypePinned;
    props.handleTypes = cudaMemHandleTypeNone;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = device;
    uint64_t thr = ~0ull;   // keep everything cached: steady-state calls do not allocate
    if (cudaMemPoolCreate(&ctx->pool, &props) == cudaSuccess) cudaMemPoolSetAttribute(ctx->pool, cudaMemPoolAttrReleaseThreshold, &thr);
    else { cudaGetLastError(); ctx->pool = nullptr; }
    cudaMemPool_t dflt;
    if (!ctx->pool && cudaDeviceGetDefaultMemPool(&dflt, device) == cudaSuccess) cudaMemPoolSetAttribute(dflt, cudaMemPoolAttrReleaseThreshold, &thr);
  }
  ctx->pinned_bytes = 1 << 16;
  if (cudaHostAlloc(&ctx->pinned, ctx->pinned_bytes, cudaHostAllocDefault) != cudaSuccess) {
    if (ctx->owns_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return OPE_ERR_CUDA;
  }
  for (int w = 0; w < 3; ++w)
    for (int j = 0; j < 2; ++j) cudaEventCreate(&ctx->kev[w][j]);
  // a zeroed counter for "last block folds the partials" kernels (each such kernel re-arms it before it exits)
  if (cudaMalloc((void**)&ctx->ticket, sizeof(unsigned)) != cudaSuccess || cudaMemset(ctx->ticket, 0, sizeof(unsigned)) != cudaSuccess) {
    cudaGetLastError();
    ctx->ticket = nullptr;
  }
  *out = ctx;
  return OPE_OK;
}

double ope_ctx_last_kernel_ms(ope_ctx* ctx, int which) {
  OPE_ENTER(ctx);
  if (!ctx || which < 0 || which > 2 || !ctx->kev_valid[which]) return -1.0;
  float ms = 0;
  if (cudaEventSynchronize(ctx->kev[which][1]) != cudaSuccess) return -1.0;
  if (cudaEventElapsedTime(&ms, ctx->kev[which][0], ctx->kev[which][1]) != cudaSuccess) return -1.0;
  return (double)ms;
}

int ope_cloud_invalidate(ope_ctx* ctx, ope_cloud* c) {
  OPE_ENTER(ctx);
  if (!ctx || !c) return OPE_ERR_INVALID;
  for (auto& g : c->grids) { dfree(ctx, g.cell_start); dfree(ctx, g.sorted); }
  c->grids.clear();
  c->bbox_valid = false;
  return OPE_OK;
}

void ope_ctx_destroy(ope_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  ope::stream_sync(ctx);
  for (auto& e : ctx->model_cache) { if (e.sp) ope_cloud_free(ctx, e.sp); ope::dfree(ctx, e.fs); }
  if (ctx->batch_model.model) ope_cloud_free(ctx, ctx->batch_model.model);
  if (ctx->batch_model.sp) ope_cloud_free(ctx, ctx->batch_model.sp);
  ope::dfree(ctx, ctx->batch_model.fs);
  ctx->batch_model = BatchModelCache();
  ctx->model_cache.clear();
  for (int w = 0; w < 3; ++w)
    for (int j = 0; j < 2; ++j) if (ctx->kev[w][j]) cudaEventDestroy(ctx->kev[w][j]);
  if (ctx->pinned) cudaFreeHost(ctx->pinned);
  if (ctx->stage) cudaFreeHost(ctx->stage);
  if (ctx->sync_event) cudaEventDestroy(ctx->sync_event);
  if (ctx->ticket) cudaFree(ctx->ticket);
  for (ope_ctx* w : ctx->workers) ope_ctx_destroy(w);
  ctx->workers.clear();
  if (ctx->owns_stream) cudaStreamDestroy(ctx->stream);
  if (ctx->pool) cudaMemPoolDestroy(ctx->pool);   // allocations still held by live clouds keep their memory until freed
  delete ctx;
}

const char* ope_last_error(const ope_ctx* ctx) { return ctx ? ctx->error.c_str() : "no context"; }
int64_t ope_ctx_launch_count(const ope_ctx* ctx) {
  if (!ctx) return 0;
  int64_t n = ctx->launches;
  for (const ope_ctx* w : ctx->workers) n += w->launches;   // ope_pose_batch's worker contexts launch on behalf of this one
  return n;
}
int ope_ctx_feature_knn_stats(const ope_ctx* ctx, int64_t* gemm_queries, int64_t* fallbacks) {
  if (!ctx) return OPE_ERR_INVALID;
  if (gemm_queries) *gemm_queries = ctx->feature_knn_gemm_queries;
  if (fallbacks) *fallbacks = ctx->feature_knn_fallbacks;
  return OPE_OK;
}
int ope_ctx_model_cache_stats(const ope_ctx* ctx, int64_t* hits, int64_t* misses) {
  if (!ctx) return OPE_ERR_INVALID;
  if (hits) *hits = ctx->model_cache_hits;
  if (misses) *misses = ctx->model_cache_misses;
  return OPE_OK;
}
int ope_ctx_synchronize(ope_ctx* ctx) {
  OPE_ENTER(ctx);
  if (!ctx) return OPE_ERR_INVALID;
  OPE_CUDA_TRY(ctx, ope::stream_sync(ctx));
  return OPE_OK;
}

int ope_cloud_upload(ope_ctx* ctx, const void* pts, size_t n, size_t stride, size_t offset, const void* normals,
                     size_t nstride, size_t noffset, ope_cloud** out) {
  OPE_ENTER(ctx);
  if (!ctx || !out || (n > 0 && (!pts || stride < 12))) return OPE_ERR_INVALID;
  if (n > 0x7fffffffull) return fail(ctx, OPE_ERR_INVALID, "cloud too large");
  ope_cloud* c = nullptr;
  OPE_TRY(cloud_alloc(ctx, n, normals != nullptr, &c));
  if (n > 0) {
    // pack to float4 in the context's pinned staging arena, one async copy each
    void* stage = nullptr;
    const size_t bytes = n * sizeof(float4) * (normals ? 2 : 1);
    int rc = stage_reserve(ctx, bytes, &stage);
    if (rc != OPE_OK) { ope_cloud_free(ctx, c); return rc; }
    float4* hp = (float4*)stage;
    const char* b = (const char*)pts + offset;
    for (size_t i = 0; i < n; ++i) {
      float v[3];
      std::memcpy(v, b + i * stride, 12);
      hp[i] = make_float4(v[0], v[1], v[2], 1.0f);
    }
    cudaError_t e = cudaMemcpyAsync(c->pts, hp, n * sizeof(float4), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess && normals) {
      const char* nb = (const char*)normals + noffset;
      float4* hn = hp + n;
      for (size_t i = 0; i < n; ++i) {
        float v[4] = {0, 0, 0, 0};
        std::memcpy(v, nb + i * nstride, nstride >= 16 ? 16 : 12);
        hn[i] = make_float4(v[0], v[1], v[2], v[3]);
      }
      e = cudaMemcpyAsync(c->normals, hn, n * sizeof(float4), cudaMemcpyHostToDevice, ctx->stream);
    }
    if (e == cudaSuccess) e = ope::stream_sync(ctx);
    if (e != cudaSuccess) {
      ope_cloud_free(ctx, c);
      return fail(ctx, OPE_ERR_CUDA, "upload failed: %s", cudaGetErrorString(e));
    }
  }
  *out = c;
  return OPE_OK;
}

int ope_cloud_free(ope_ctx* ctx, ope_cloud* c) {
  OPE_ENTER(ctx);
  if (!c) return OPE_OK;
  if (!ctx) ctx = c->ctx;
  for (auto& g : c->grids) { dfree(ctx, g.cell_start); dfree(ctx, g.sorted); }
  dfree(ctx, c->pts);
  dfree(ctx, c->normals);
  delete c;
  return OPE_OK;
}

size_t ope_cloud_size(const ope_cloud* c) { return c ? c->n : 0; }
int ope_cloud_has_normals(const ope_cloud* c) { return c && c->normals ? 1 : 0; }

int ope_cloud_download(ope_ctx* ctx, const ope_cloud* c, float* xyz, float* normals4) {
  OPE_ENTER(ctx);
  if (!ctx || !c) return OPE_ERR_INVALID;
  if (c->n == 0) return OPE_OK;
  void* stage = nullptr;
  OPE_TRY(stage_reserve(ctx, c->n * sizeof(float4), &stage));
  const float4* h = (const float4*)stage;
  if (xyz) {
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(stage, c->pts, c->n * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream));
    OPE_CUDA_TRY(ctx, ope::stream_sync(ctx));
    for (size_t i = 0; i < c->n; ++i) { xyz[3 * i] = h[i].x; xyz[3 * i + 1] = h[i].y; xyz[3 * i + 2] = h[i].z; }
  }
  if (normals4) {
    if (!c->normals) return fail(ctx, OPE_ERR_INVALID, "cloud has no normals");
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(stage, c->normals, c->n * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream));
    OPE_CUDA_TRY(ctx, ope::stream_sync(ctx));
    std::memcpy(normals4, stage, c->n * sizeof(float4));
  }
  return OPE_OK;
}

int ope_cloud_select(ope_ctx* ctx, const ope_cloud* c, const int32_t* idx, size_t n, ope_cloud** out) {
  OPE_ENTER(ctx);
  if (!ctx || !c || !out || (n > 0 && !idx)) return OPE_ERR_INVALID;
  for (size_t i = 0; i < n; ++i)
    if (idx[i] < 0 || (size_t)idx[i] >= c->n) return fail(ctx, OPE_ERR_INVALID, "index out of range");
  Scratch<int> d(ctx);
  OPE_TRY(d.alloc(n));
  if (n) OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d.p, idx, n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  OPE_TRY(gather_cloud(ctx, c, d.p, n, out));
  OPE_CUDA_TRY(ctx, ope::stream_sync(ctx));
  return OPE_OK;
}

int ope_cloud_append(ope_ctx* ctx, ope_cloud* dst, const ope_cloud* src) {
  OPE_ENTER(ctx);
  if (!ctx || !dst || !src) return OPE_ERR_INVALID;
  if (src->n == 0) return OPE_OK;
  const size_t n = dst->n + src->n;
  const bool normals = dst->normals && src->normals;   // the concatenation keeps normals only when both sides carry them
  float4* pts = nullptr;
  float4* nrm = nullptr;
  OPE_TRY(dalloc(ctx, &pts, n));
  if (normals) { int rc = dalloc(ctx, &nrm, n); if (rc != OPE_OK) { dfree(ctx, pts); return rc; } }
  cudaError_t e = cudaSuccess;
  if (dst->n) e = cudaMemcpyAsync(pts, dst->pts, dst->n * sizeof(float4), cudaMemcpyDeviceToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(pts + dst->n, src->pts, src->n * sizeof(float4), cudaMemcpyDeviceToDevice, ctx->stream);
  if (e == cudaSuccess && normals && dst->n) e = cudaMemcpyAsync(nrm, dst->normals, dst->n * sizeof(float4), cudaMemcpyDeviceToDevice, ctx->stream);
  if (e == cudaSuccess && normals) e = cudaMemcpyAsync(nrm + dst->n, src->normals, src->n * sizeof(float4), cudaMemcpyDeviceToDevice, ctx->stream);
  if (e != cudaSuccess) { dfree(ctx, pts); dfree(ctx, nrm); return fail(ctx, OPE_ERR_CUDA, "device copy failed: %s", cudaGetErrorString(e)); }
  ope_cloud_invalidate(ctx, dst);
  dfree(ctx, dst->pts); dfree(ctx, dst->normals);
  dst->pts = pts; dst->normals = nrm; dst->n = n;
  return OPE_OK;
}

int ope_cloud_set_normals(ope_ctx* ctx, ope_cloud* c, const float* normals4) {
  OPE_ENTER(ctx);
  if (!ctx || !c || !normals4) return OPE_ERR_INVALID;
  if (!c->normals) OPE_TRY(dalloc(ctx, &c->normals, c->n));
  if (c->n) {
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(c->normals, normals4, c->n * sizeof(float4), cudaMemcpyHostToDevice, ctx->stream));
    OPE_CUDA_TRY(ctx, ope::stream_sync(ctx));
  }
  return OPE_OK;
}

static int knn_impl(ope_ctx* ctx, const ope_cloud* tgt, const float4* d_qry, size_t nq, int k, int32_t* out_idx, float* out_d2) {
  static_assert(kKnnListMax == OPE_KNN_MAX_K, "the shared-memory list holds OPE_KNN_MAX_K entries");
  if (k < 1 || k > OPE_KNN_MAX_K) return fail(ctx, OPE_ERR_INVALID, "k must be in [1, %d]", OPE_KNN_MAX_K);
  if (nq == 0) return OPE_OK;
  OPE_TRY(cloud_bbox(ctx, const_cast<ope_cloud*>(tgt)));
  GridView g;
  OPE_TRY(cloud_grid(ctx, tgt, knn_cell_size(tgt, k), &g));
  Scratch<int> di(ctx);
  Scratch<float> dd(ctx);
  OPE_TRY(di.alloc(nq * k));
  OPE_TRY(dd.alloc(nq * k));
  if (k == 1) {
    OPE_TRY(dyn_smem(ctx, (const void*)nn1_kernel, sizeof(Nn1Smem<kKnnThreads>)));
    nn1_kernel<<<(unsigned)std::min<size_t>(div_up(nq, kKnnThreads), (size_t)ctx->sm_count * 4), kKnnThreads,
                 sizeof(Nn1Smem<kKnnThreads>), ctx->stream>>>(g, d_qry, (int)nq, di.p, dd.p);
    OPE_TRY(check_launch(ctx, "nn1_kernel"));
  } else if (k > 32) {
    knn_list_kernel<<<(unsigned)std::min<size_t>(div_up(nq * 32, kKnnThreads), (size_t)ctx->sm_count * 8), kKnnThreads, 0,
                      ctx->stream>>>(g, d_qry, (int)nq, k, di.p, dd.p);
    OPE_TRY(check_launch(ctx, "knn_list_kernel"));
  } else {
    knn_kernel<<<(unsigned)std::min<size_t>(div_up(nq * 32, kKnnThreads), (size_t)ctx->sm_count * 8), kKnnThreads, 0,
                 ctx->stream>>>(g, d_qry, (int)nq, k, di.p, dd.p);
    OPE_TRY(check_launch(ctx, "knn_kernel"));
  }
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(out_idx, di.p, nq * k * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  if (out_d2) OPE_CUDA_TRY(ctx, cudaMemcpyAsync(out_d2, dd.p, nq * k * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  OPE_CUDA_TRY(ctx, ope::stream_sync(ctx));
  return OPE_OK;
}

int ope_knn_cloud(ope_ctx* ctx, const ope_cloud* tgt, const ope_cloud* qry, int k, int32_t* out_idx, float* out_d2) {
  OPE_ENTER(ctx);
  if (!ctx || !tgt || !qry || !out_idx) return OPE_ERR_INVALID;
  return knn_impl(ctx, tgt, qry->pts, qry->n, k, out_idx, out_d2);
}

int ope_knn(ope_ctx* ctx, const ope_cloud* tgt, const void* qry, size_t nq, size_t stride, size_t offset, int k,
            int32_t* out_idx, float* out_d2) {
  OPE_ENTER(ctx);
  if (!ctx || !tgt || !qry || !out_idx) return OPE_ERR_INVALID;
  ope_cloud* q = nullptr;
  OPE_TRY(ope_cloud_upload(ctx, qry, nq, stride, offset, nullptr, 0, 0, &q));
  int rc = knn_impl(ctx, tgt, q->pts, nq, k, out_idx, out_d2);
  ope_cloud_free(ctx, q);
  return rc;
}

int ope_radius_cloud(ope_ctx* ctx, const ope_cloud* tgt, const ope_cloud* qry, float radius, int64_t capacity,
                     int64_t* offsets, int32_t* out_idx, float* out_d2, int64_t* total) {
  OPE_ENTER(ctx);
  if (!ctx || !tgt || !qry || !total || !(radius > 0)) return OPE_ERR_INVALID;
  *total = 0;
  const size_t nq = qry->n;
  if (nq == 0) { if (offsets) offsets[0] = 0; return OPE_OK; }
  GridView g;
  OPE_TRY(cloud_grid(ctx, tgt, radius * 0.5f, &g));
  const float r2 = radius * radius;
  Scratch<int> cnt(ctx);
  OPE_TRY(cnt.alloc(nq + 1));
  OPE_CUDA_TRY(ctx, cudaMemsetAsync(cnt.p + nq, 0, sizeof(int), ctx->stream));
  radius_count_kernel<<<div_up(nq, 128), 128, 0, ctx->stream>>>(g, qry->pts, (int)nq, r2, cnt.p);
  OPE_TRY(check_launch(ctx, "radius_count_kernel"));
  OPE_TRY(exclusive_scan_i32(ctx, cnt.p, nq + 1));
  std::vector<int> off(nq + 1);
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(off.data(), cnt.p, (nq + 1) * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  OPE_CUDA_TRY(ctx, ope::stream_sync(ctx));
  *total = off[nq];
  if (offsets) for (size_t i = 0; i <= nq; ++i) offsets[i] = off[i];
  if (!out_idx || !out_d2) return OPE_OK;
  if (*total > capacity) return fail(ctx, OPE_ERR_CAPACITY, "radius result needs %lld entries", (long long)*total);
  if (*total == 0) return OPE_OK;
  Scratch<int> di(ctx);
  Scratch<float> dd(ctx);
  OPE_TRY(di.alloc((size_t)*total));
  OPE_TRY(dd.alloc((size_t)*total));
  radius_fill_kernel<<<div_up(nq, 128), 128, 0, ctx->stream>>>(g, qry->pts, (int)nq, r2, cnt.p, di.p, dd.p);
  OPE_TRY(check_launch(ctx, "radius_fill_kernel"));
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(out_idx, di.p, (size_t)*total * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(out_d2, dd.p, (size_t)*total * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  OPE_CUDA_TRY(ctx, ope::stream_sync(ctx));
  // canonical order of the API: ascending index per query (the device visits cells row by row)
  std::vector<std::pair<int, float>> tmp;
  for (size_t i = 0; i < nq; ++i) {
    const int b = off[i], e = off[i + 1];
    tmp.resize(e - b);
    for (int j = b; j < e; ++j) tmp[j - b] = {out_idx[j], out_d2[j]};
    std::sort(tmp.begin(), tmp.end());
    for (int j = b; j < e; ++j) { out_idx[j] = tmp[j - b].first; out_d2[j] = tmp[j - b].second; }
  }
  return OPE_OK;
}

int ope_uniform_sample(ope_ctx* ctx, const ope_cloud* cloud, float leaf, int32_t* out_idx, size_t* out_n) {
  OPE_ENTER(ctx);
  if (!ctx || !cloud || !out_idx || !out_n || !(leaf > 0)) return OPE_ERR_INVALID;
  int* d = nullptr;
  OPE_TRY(uniform_sample_device(ctx, const_cast<ope_cloud*>(cloud), leaf, &d, out_n));
  if (*out_n) {
    cudaError_t e = cudaMemcpyAsync(out_idx, d, *out_n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = ope::stream_sync(ctx);
    if (e != cudaSuccess) { dfree(ctx, d); return fail(ctx, OPE_ERR_CUDA, "download failed: %s", cudaGetErrorString(e)); }
  }
  dfree(ctx, d);
  return OPE_OK;
}

int ope_uniform_sample_cloud(ope_ctx* ctx, const ope_cloud* cloud, float leaf, ope_cloud** out) {
  OPE_ENTER(ctx);
  if (!ctx || !cloud || !out || !(leaf > 0)) return OPE_ERR_INVALID;
  int* d = nullptr; size_t m = 0;
  OPE_TRY(uniform_sample_device(ctx, const_cast<ope_cloud*>(cloud), leaf, &d, &m));
  int rc = gather_cloud(ctx, cloud, d, m, out);
  dfree(ctx, d);
  if (rc == OPE_OK) OPE_CUDA_TRY(ctx, ope::stream_sync(ctx));
  return rc;
}

int ope_voxel_grid(ope_ctx* ctx, const ope_cloud* cloud_c, const float* rgb, float lx, float ly, float lz, float* out_xyz,
                   float* out_rgb, size_t* out_n) {
  OPE_ENTER(ctx);
  if (!ctx || !cloud_c || !out_xyz || !out_n || !(lx > 0 && ly > 0 && lz > 0)) return OPE_ERR_INVALID;
  ope_cloud* cloud = const_cast<ope_cloud*>(cloud_c);
  *out_n = 0;
  OPE_TRY(cloud_bbox(ctx, cloud));
  if (cloud->n_finite == 0) return OPE_OK;
  float leaf[3] = {lx, ly, lz};
  // VoxelGrid::applyFilter overflow guard: (int64)((max-min)*inv)+1 per axis, product > INT_MAX -> refuse
  {
    int64_t prod = 1;
    for (int d = 0; d < 3; ++d) {
      volatile float inv = 1.0f / leaf[d];
      volatile float span = (cloud->bbox[3 + d] - cloud->bbox[d]) * inv;
      prod *= (int64_t)span + 1;
    }
    if (prod > 0x7fffffffll) return fail(ctx, OPE_ERR_GRID_TOO_LARGE, "Leaf size is too small for the input dataset");
  }
  Binning bin; int64_t ncells;
  OPE_TRY(pcl_voxel_frame(ctx, cloud, leaf, &bin, &ncells));
  // the frame in windows of consecutive voxel indices (see uniform_sample_device): centroids in ascending voxel order
  const int64_t win = std::min(ncells, kVoxelWindowCells);
  const size_t cap = std::min<size_t>((size_t)ncells, cloud->n);
  Scratch<int> flags(ctx);
  Scratch<float> drgb(ctx), oxyz(ctx), orgb(ctx);
  OPE_TRY(flags.alloc((size_t)win + 1));
  OPE_TRY(oxyz.alloc(cap * 3));
  OPE_TRY(orgb.alloc(cap));
  if (rgb) {
    OPE_TRY(drgb.alloc(cloud->n));
    if (cudaMemcpyAsync(drgb.p, rgb, cloud->n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess)
      return fail(ctx, OPE_ERR_CUDA, "rgb upload failed");
  }
  size_t m = 0;
  for (int64_t c0 = 0; c0 < ncells; c0 += win) {
    const int64_t nw = std::min(win, ncells - c0);
    int* cell_start = nullptr; float4* sorted = nullptr;
    OPE_TRY(build_cells(ctx, cloud->pts, cloud->n, bin, &cell_start, &sorted, c0, nw));
    auto done = [&](int code) { dfree(ctx, cell_start); dfree(ctx, sorted); return code; };
    cudaMemsetAsync(flags.p + nw, 0, sizeof(int), ctx->stream);
    occupied_flag_cells_kernel<<<grid_blocks(ctx, (size_t)nw), kThreads, 0, ctx->stream>>>(cell_start, nw, flags.p);
    int rc = check_launch(ctx, "occupied_flag_cells_kernel");
    if (rc == OPE_OK) rc = exclusive_scan_i32(ctx, flags.p, (size_t)nw + 1);
    void* h = nullptr;
    if (rc == OPE_OK) rc = read_back(ctx, flags.p + nw, sizeof(int), &h);
    if (rc != OPE_OK) return done(rc);
    const int mw = *(const int*)h;
    voxel_centroid_kernel<<<grid_blocks(ctx, (size_t)nw), kThreads, 0, ctx->stream>>>(
        cell_start, nw, sorted, rgb ? drgb.p : nullptr, flags.p, oxyz.p + 3 * m, orgb.p + m);
    if ((rc = done(check_launch(ctx, "voxel_centroid_kernel"))) != OPE_OK) return rc;
    m += (size_t)mw;
  }
  cudaError_t e = cudaMemcpyAsync(out_xyz, oxyz.p, m * 3 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess && rgb && out_rgb)
    e = cudaMemcpyAsync(out_rgb, orgb.p, m * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = ope::stream_sync(ctx);
  if (e != cudaSuccess) return fail(ctx, OPE_ERR_CUDA, "voxel grid download failed: %s", cudaGetErrorString(e));
  *out_n = m;
  return OPE_OK;
}

}  // extern "C"
