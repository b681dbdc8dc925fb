// ope_octet.cuh — device-side cooperative search over the implicit octree of ope_grid.cuh.
//
// Three building blocks, all exact (bit-identical to ope::grid_nn1 / ope::grid_knn: same float distances, same
// (d2, index) tie order, the same conservative bounds):
//
//  block_nn1   nearest neighbour, one query per THREAD. Each thread seeds its bound (the caller's previous match, or
//              nn1_probe) and tries ope::nn1_fast: the <= 8 cells/nodes the bound's ball touches, 16 independent `start`
//              loads and a few 16-byte point loads — two dependent L2 round trips. Queries whose candidate set is too large
//              (far from the indexed surface) are compacted into a shared-memory list and finished one per WARP with
//              large leaves (few dependent steps, wide pipelined point scans), so that a few slow queries never hold 31
//              finished lanes hostage.
//  coop_nn1    the pruned traversal with G lanes per query: at an internal node lane j tests child j (one 4-byte
//              `start` load + one box distance per lane, the sibling's load gives the range end by shuffle), at a leaf the
//              lanes test eight points per step. Starts from the ball's start nodes (ope::ball_nodes), nearest on top of a
//              small per-octet stack in shared memory.
//  warp_knn    exact k nearest (k <= 32), one query per WARP, the sorted result list held one entry per lane in
//              REGISTERS (insertion = ballot + shfl_up, no shared memory), leaves scanned 32 points per step, internal
//              nodes expanded by lanes 0..7.
#pragma once
#include "ope_grid.cuh"

namespace ope {

static constexpr int kOctStack = 72;   // >= 8 + 7 * OPE_MAX_BITS: initial push of <= 8 nodes, +7 net per expansion
static constexpr int kOctLeaf = 32;    // octet: nodes with at most this many points are scanned, 8 points per step
static constexpr int kWarpLeaf = 64;   // warp k-NN: ... 32 points per step
static constexpr int kFarLeaf = 256;   // deferred nearest-neighbour queries (a warp each): few dependent steps, wide scans

struct __align__(16) OctEntry {
  unsigned node;  // level << 27 | code
  float d2;       // conservative lower bound of the node's distance to the query
  int b, e;       // point range
};
struct OctStack { OctEntry s[kOctStack]; };

// A cooperative group of G lanes inside a warp (G = 8: octet, G = 32: warp)
template <int G>
struct Coop {
  unsigned sub;    // lane within the group
  unsigned gbase;  // first lane of the group within the warp
  unsigned mask;   // the group's lanes
  __device__ __forceinline__ Coop() {
    const unsigned lane = threadIdx.x & 31u;
    sub = lane & (unsigned)(G - 1);
    gbase = lane & ~(unsigned)(G - 1);
    mask = (G == 32) ? 0xffffffffu : (((1u << (G & 31)) - 1u) << gbase);
  }
};
using Octet = Coop<8>;

template <int G>
__device__ __forceinline__ float coop_min(const Coop<G>& o, float v) {
#pragma unroll
  for (int s = 1; s < G; s <<= 1) v = fminf(v, __shfl_xor_sync(o.mask, v, s));
  return v;
}

// Push the group's candidate nodes (lane j < 8 offers one when `pass`): all passing ones go on the stack, the nearest
// (ties: lower lane) on top. Returns the number pushed (group-uniform). Lanes >= 8 must call with pass = false.
template <int G>
__device__ __forceinline__ int coop_push(OctStack* st, const Coop<G>& o, int sp, bool pass, unsigned node, float d2, int b, int e) {
  const unsigned om = (__ballot_sync(o.mask, pass) >> o.gbase) & 0xffu;
  const int npass = __popc(om);
  if (npass == 0) return 0;
  float md = pass ? d2 : FLT_MAX;
  unsigned mi = o.sub;
#pragma unroll
  for (int s = 1; s < 8; s <<= 1) {   // the 8 offering lanes are an aligned group of 8: xor stays inside it
    const float od = __shfl_xor_sync(o.mask, md, s);
    const unsigned oi = __shfl_xor_sync(o.mask, mi, s);
    if (od < md || (od == md && oi < mi)) { md = od; mi = oi; }
  }
  if (G > 8) mi = __shfl_sync(o.mask, mi, 0);  // lanes >= 8 of a warp-sized group take lane 0's view
  if (pass) {
    const unsigned others = om & ~(1u << mi);
    const int pos = (o.sub == mi) ? sp + npass - 1 : sp + __popc(others & ((1u << o.sub) - 1u));
    OctEntry en;
    en.node = node; en.d2 = d2; en.b = b; en.e = e;
    st->s[pos] = en;
  }
  __syncwarp(o.mask);
  return npass;
}

// Start set of a (seeded) search: the ball's <= 8 nodes, lane j < 8 owns node j.
template <int G>
__device__ __forceinline__ int coop_push_ball(const GridView& g, OctStack* st, const Coop<G>& o, bool active, float ux, float uy,
                                              float uz, float bound) {
  bool pass = false;
  unsigned node = 0u;
  float d2 = FLT_MAX;
  int b = 0, e = 0;
  if (active && o.sub < 8u) {
    const BallNodes B = ball_nodes(g, ux, uy, uz, bound);
    unsigned code;
    if (ball_node(B, (int)o.sub, code)) {
      oct_node_range(g, B.L, code, b, e);
      if (e > b) {
        d2 = oct_node_d2(g, ux, uy, uz, B.L, code);
        pass = d2 <= bound;
        node = ((unsigned)B.L << 27) | code;
      }
    }
  }
  return coop_push(st, o, 0, pass, node, d2, b, e);
}

// Expand an internal node: lane j < 8 owns child j; children that are non-empty and within `bound` are pushed.
// `split` is group-uniform.
template <int G>
__device__ __forceinline__ int coop_expand(const GridView& g, OctStack* st, const Coop<G>& o, int sp, bool split, unsigned node, int e,
                                           float ux, float uy, float uz, float bound) {
  const int level = (int)(node >> 27);
  const unsigned code = node & 0x07ffffffu;
  const int cl = level - 1;
  const unsigned cc = (code << 3) | (o.sub & 7u);
  const bool mine = split && o.sub < 8u;
  int cb = 0;
  if (mine) cb = __ldg(g.start + ((size_t)cc << (3 * cl)));
  const int nb = __shfl_down_sync(o.mask, cb, 1, 8);
  const int ce = (o.sub == 7u) ? e : nb;
  float cd2 = FLT_MAX;
  bool pass = false;
  if (mine && ce > cb) {
    cd2 = oct_node_d2(g, ux, uy, uz, cl, cc);
    pass = cd2 <= bound;
  }
  return coop_push(st, o, sp, pass, ((unsigned)cl << 27) | cc, cd2, cb, ce);
}

// Exact nearest neighbour for the group's query (G lanes: 8 or 32), starting from st (a valid candidate or none).
// Nodes holding at most LEAF points are scanned G points per step (independent 16-byte loads), larger ones are expanded;
// everything within the scan radius nn1_scan_r2(best, max_d2, gap) is examined, so on return st holds the exact
// neighbour, the second-best distance, and *r2_out the squared radius the certificate may rely on (ope_grid.cuh).
// The lanes must call this together with the same arguments; every lane returns the same state.
template <int G, int LEAF>
__device__ __forceinline__ void coop_nn1(const GridView& g, OctStack* st_mem, const Coop<G>& o, bool active, float qx, float qy, float qz,
                                         float max_d2, float gap, Nn1State& st, float* r2_out) {
  const float ux = (qx - g.ox) * g.inv_h, uy = (qy - g.oy) * g.inv_h, uz = (qz - g.oz) * g.inv_h;
  float bound = nn1_scan_r2(st.d1, max_d2, gap);
  int sp = coop_push_ball(g, st_mem, o, active && g.n > 0, ux, uy, uz, bound);
  while (sp > 0) {
    --sp;
    const OctEntry en = st_mem->s[sp];
    __syncwarp(o.mask);  // every lane holds the popped entry before its slot can be overwritten
    bound = nn1_scan_r2(coop_min(o, st.d1), max_d2, gap);
    const bool live = en.d2 <= bound;
    const int level = (int)(en.node >> 27);
    const bool leaf = level == 0 || en.e - en.b <= LEAF;
    if (live && leaf) {
#pragma unroll 4
      for (int i = en.b + (int)o.sub; i < en.e; i += G) {
        const float4 p = __ldg(g.pts + i);
        nn1_offer(st, dist2(qx, qy, qz, p.x, p.y, p.z), __float_as_int(p.w));
      }
    }
    sp += coop_expand(g, st_mem, o, sp, live && !leaf, en.node, en.e, ux, uy, uz, bound);
  }
  // merge the lanes' states: best of the bests; second = the smallest of every lane's second and of the displaced bests
  float d1 = st.d1;
  int i1 = st.i1;
#pragma unroll
  for (int s = 1; s < G; s <<= 1) {
    const float od = __shfl_xor_sync(o.mask, d1, s);
    const int oi = __shfl_xor_sync(o.mask, i1, s);
    if (nb_less(od, oi, d1, i1)) { d1 = od; i1 = oi; }
  }
  float s2 = st.s2;
  if (st.i1 != i1) s2 = fminf(s2, st.d1);
  s2 = coop_min(o, s2);
  st.d1 = d1; st.i1 = i1; st.s2 = s2;
  if (r2_out) *r2_out = nn1_scan_r2(d1, max_d2, gap);
}
// plain form (no certificate): returns the index (INT_MAX: none), distance in best_d2
template <int G, int LEAF>
__device__ __forceinline__ int coop_nn1(const GridView& g, OctStack* st_mem, const Coop<G>& o, bool active, float qx, float qy, float qz,
                                        float max_d2, float& best_d2, int best_i) {
  Nn1State st;
  st.d1 = best_d2; st.i1 = best_i; st.s2 = FLT_MAX;
  coop_nn1<G, LEAF>(g, st_mem, o, active, qx, qy, qz, max_d2, 0.0f, st, nullptr);
  best_d2 = st.d1;
  return st.i1;
}

// ---- far queries: directory in shared memory, leaves collected then scanned wide ------------------------------
// A far query's traversal is a chain of dependent steps; with the `start` look-ups going to L2 (~300 cycles), a
// 5-shuffle bound update and a nearest-first argmin per step it costs ~850 cycles a step (ncu, profiles/). Here
//  * the upper levels of the implicit octree (levels >= dl: at most 4097 `start` entries, 16 KB) are cached in SHARED
//    memory once per persistent kernel, and nodes at level dl are never split, so the traversal itself touches no
//    global memory;
//  * leaves are only COLLECTED during the traversal and then scanned in batches (8 independent 16-byte loads per lane
//    in flight), the bound being refreshed per batch instead of per node;
//  * the nearest-first ordering of children is kept only for unseeded queries (ORDERED), whose bound must shrink.
static constexpr int kDirMaxLevels = 4;                       // directory covers the top 4 levels below the root
static constexpr int kDirEntries = (1 << (3 * kDirMaxLevels)) + 1;
static constexpr int kLeafCap = 96;                           // collected leaf ranges per warp
static constexpr int kFlushPts = 2048;                        // ... or this many points: scan, refresh the bound

struct FarDir {
  const int* sdir;  // shared memory: sdir[c] = start[c << (3 * dl)], c in [0, 2^(3 * (bits - dl))]
  int dl;           // lowest level the directory resolves
};
struct LeafList { int2 r[kLeafCap]; };   // point ranges [x, y) of the collected leaves

__device__ __forceinline__ int far_dir_level(const GridView& g) { return g.bits > kDirMaxLevels ? g.bits - kDirMaxLevels : 0; }
// block-cooperative load of the directory (call once, followed by __syncthreads)
__device__ __forceinline__ void far_dir_load(const GridView& g, int* sdir) {
  const int dl = far_dir_level(g);
  const int n = (1 << (3 * (g.bits - dl))) + 1;
  for (int c = threadIdx.x; c < n; c += blockDim.x) sdir[c] = g.n > 0 ? __ldg(g.start + ((size_t)c << (3 * dl))) : 0;
}
__device__ __forceinline__ void far_node_range(const GridView& g, const FarDir& D, int level, unsigned code, int& b, int& e) {
  if (level >= D.dl) {
    const int sh = 3 * (level - D.dl);
    b = D.sdir[(size_t)code << sh];
    e = D.sdir[(size_t)(code + 1u) << sh];
  } else {
    oct_node_range(g, level, code, b, e);
  }
}

// Exact nearest neighbour + certificate for the GROUP's query (G = 8 or 32 lanes, same arguments, same `st` on entry).
// Leaves are collected during the traversal and scanned in batches, the bound being refreshed per batch.
template <int G, bool ORDERED>
__device__ __forceinline__ void coop_nn1_far(const GridView& g, const FarDir& D, OctStack* stk, LeafList* LL, float qx, float qy, float qz,
                                             float max_d2, float gap, Nn1State& st, float* r2_out,
                                             unsigned long long* counters = nullptr /* [pops, leaves, points, flushes] */,
                                             int only_node = -1 /* >= 0: search only that start node (a split query) */) {
  const Coop<G> o;
  const int lane = (int)o.sub;
  const float ux = (qx - g.ox) * g.inv_h, uy = (qy - g.oy) * g.inv_h, uz = (qz - g.oz) * g.inv_h;
  float bound = nn1_scan_r2(st.d1, max_d2, gap);
  int sp = 0, nleaf = 0, leafpts = 0;
  // start set: the ball's <= 8 nodes
  {
    bool pass = false;
    unsigned node = 0u;
    float d2 = FLT_MAX;
    int b = 0, e = 0;
    if (g.n > 0 && lane < 8 && (only_node < 0 || lane == only_node)) {
      const BallNodes B = ball_nodes(g, ux, uy, uz, bound);
      unsigned code;
      if (ball_node(B, lane, code)) {
        far_node_range(g, D, B.L, code, b, e);
        if (e > b) {
          d2 = ball_node_d2(g, B, lane, ux, uy, uz);
          pass = d2 <= bound;
          node = ((unsigned)B.L << 27) | code;
        }
      }
    }
    sp = coop_push(stk, o, 0, pass, node, d2, b, e);
  }
  // every collected leaf is scanned with up to 8 loads per lane in flight (measured: flattening the leaves into one index
  // space costs more in look-ups than it saves in round trips)
  auto flush = [&]() {
    for (int r = 0; r < nleaf; ++r) {
      const int2 be = LL->r[r];
      for (int i0 = be.x + lane; i0 < be.y; i0 += G * 8) {
        float4 p[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) { const int i = i0 + G * k; p[k] = (i < be.y) ? __ldg(g.pts + i) : make_float4(0, 0, 0, 0); }
#pragma unroll
        for (int k = 0; k < 8; ++k)
          if (i0 + G * k < be.y) nn1_offer(st, dist2(qx, qy, qz, p[k].x, p[k].y, p[k].z), __float_as_int(p[k].w));
      }
    }
    if (counters && lane == 0) { atomicAdd(counters + 1, (unsigned long long)nleaf); atomicAdd(counters + 2, (unsigned long long)leafpts); atomicAdd(counters + 3, 1ull); }
    nleaf = 0; leafpts = 0;
    __syncwarp(o.mask);
    bound = nn1_scan_r2(coop_min(o, st.d1), max_d2, gap);
  };
  for (;;) {
    if (sp == 0) { if (nleaf > 0) flush(); break; }
    if (nleaf == kLeafCap || leafpts >= kFlushPts) flush();
    --sp;
    const OctEntry en = stk->s[sp];
    __syncwarp(o.mask);
    if (counters && lane == 0) atomicAdd(counters, 1ull);
    if (!(en.d2 <= bound)) continue;
    const int level = (int)(en.node >> 27);
    const int cnt = en.e - en.b;
    if (level <= D.dl || cnt <= kFarLeaf) {
      if (lane == 0) LL->r[nleaf] = make_int2(en.b, en.e);
      __syncwarp(o.mask);
      ++nleaf; leafpts += cnt;
      if (ORDERED && nleaf == 1 && sp > 0) flush();  // unseeded: the first (nearest) leaf tightens the bound for everything else
      continue;
    }
    // expand: lanes 0..7 own the children (level - 1 >= dl: resolved from shared memory)
    const unsigned code = en.node & 0x07ffffffu;
    const int cl = level - 1;
    const unsigned cc = (code << 3) | ((unsigned)lane & 7u);
    int cb = 0;
    if (lane < 8) cb = D.sdir[(size_t)cc << (3 * (cl - D.dl))];
    const int nb = __shfl_down_sync(o.mask, cb, 1, 8);
    const int ce = (lane == 7) ? en.e : nb;
    float cd2 = FLT_MAX;
    bool pass = false;
    if (lane < 8 && ce > cb) {
      cd2 = oct_node_d2(g, ux, uy, uz, cl, cc);
      pass = cd2 <= bound;
    }
    if (ORDERED) {
      sp += coop_push(stk, o, sp, pass, ((unsigned)cl << 27) | cc, cd2, cb, ce);
    } else {
      const unsigned om = (__ballot_sync(o.mask, pass) >> o.gbase) & 0xffu;
      if (pass) {
        OctEntry ne;
        ne.node = ((unsigned)cl << 27) | cc; ne.d2 = cd2; ne.b = cb; ne.e = ce;
        stk->s[sp + __popc(om & ((1u << lane) - 1u))] = ne;
      }
      sp += __popc(om);
      __syncwarp(o.mask);
    }
  }
  // merge the lanes' states
  float d1 = st.d1;
  int i1 = st.i1;
#pragma unroll
  for (int s = 1; s < G; s <<= 1) {
    const float od = __shfl_xor_sync(o.mask, d1, s);
    const int oi = __shfl_xor_sync(o.mask, i1, s);
    if (nb_less(od, oi, d1, i1)) { d1 = od; i1 = oi; }
  }
  float s2 = st.s2;
  if (st.i1 != i1) s2 = fminf(s2, st.d1);
  s2 = coop_min(o, s2);
  st.d1 = d1; st.i1 = i1; st.s2 = s2;
  if (r2_out) *r2_out = nn1_scan_r2(d1, max_d2, gap);
}

// ---- block_nn1 ----------------------------------------------------------------------------------------------
// Shared-memory workspace of one block of T threads (T a multiple of 32): deferred-query list, per-thread result
// slots, one stack per octet of the first kNn1Octets*8 threads.
template <int T>
struct Nn1Smem {
  static constexpr int kGroups = T / 32;   // deferred queries are finished one per warp
  int n_def;
  float4 def_q[T];   // x, y, z, seed d2
  int def_seed[T];   // seed index (INT_MAX: none)
  int def_tid[T];
  int res_i[T];
  float res_d[T];
  OctStack stacks[kGroups];
};

// One query per thread (active = false: none). seed_idx >= 0: index of an indexed point (seed_pts, original order) used
// as the initial bound. Returns the exact nearest neighbour's original index or -1 (nothing indexed) and its squared
// distance; only neighbours with d2 <= max_d2 matter (the caller rejects larger results). Contains __syncthreads():
// every thread of the block must call it.
template <int T>
__device__ __forceinline__ int block_nn1(const GridView& g, Nn1Smem<T>* sm, bool active, float qx, float qy, float qz, float max_d2,
                                         int seed_idx, const float4* __restrict__ seed_pts, float& d2_out,
                                         long long* prof = nullptr /* thread 0: [0] fast-phase cycles [1] deferred-phase cycles [2] deferred count */) {
  if (threadIdx.x == 0) sm->n_def = 0;
  __syncthreads();
  const long long pt0 = prof ? clock64() : 0;
  float best_d2 = FLT_MAX;
  int best_i = 0x7fffffff;
  bool deferred = false;
  active = active && g.n > 0;
  if (active) {
    const float ux = (qx - g.ox) * g.inv_h, uy = (qy - g.oy) * g.inv_h, uz = (qz - g.oz) * g.inv_h;
    if (seed_idx >= 0) {
      const float4 s = __ldg(seed_pts + seed_idx);
      best_d2 = dist2(qx, qy, qz, s.x, s.y, s.z);
      best_i = seed_idx;
    } else {
      nn1_probe(g, qx, qy, qz, ux, uy, uz, [&](int b, int e) {
        for (int i = b; i < e; ++i) {
          const float4 p = __ldg(g.pts + i);
          const float d2 = dist2(qx, qy, qz, p.x, p.y, p.z);
          const int idx = __float_as_int(p.w);
          if (nb_less(d2, idx, best_d2, best_i)) { best_d2 = d2; best_i = idx; }
        }
      });
    }
    if (!nn1_fast(g, qx, qy, qz, ux, uy, uz, max_d2, best_d2, best_i)) {
      deferred = true;
      const int slot = atomicAdd(&sm->n_def, 1);
      sm->def_q[slot] = make_float4(qx, qy, qz, best_d2);
      sm->def_seed[slot] = best_i;
      sm->def_tid[slot] = (int)threadIdx.x;
    }
  }
  __syncthreads();
  const int n_def = sm->n_def;
  const long long pt1 = prof ? clock64() : 0;
  if (n_def > 0) {
    const Coop<32> o;
    OctStack* st = &sm->stacks[threadIdx.x >> 5];
    for (int d = (int)(threadIdx.x >> 5); d < n_def; d += Nn1Smem<T>::kGroups) {
      const float4 q = sm->def_q[d];
      float bd = q.w;
      const int bi = coop_nn1<32, kFarLeaf>(g, st, o, true, q.x, q.y, q.z, max_d2, bd, sm->def_seed[d]);
      if (o.sub == 0u) { const int t = sm->def_tid[d]; sm->res_i[t] = bi; sm->res_d[t] = bd; }
    }
  }
  __syncthreads();
  if (prof) { const long long pt2 = clock64(); prof[0] += pt1 - pt0; prof[1] += pt2 - pt1; prof[2] += n_def; }
  if (deferred) { best_i = sm->res_i[threadIdx.x]; best_d2 = sm->res_d[threadIdx.x]; }
  d2_out = best_d2;
  return best_i == 0x7fffffff ? -1 : best_i;
}

// ---- warp_knn -----------------------------------------------------------------------------------------------
// Exact k nearest (k <= 32) for the warp's query. Result: lane j < count holds the j-th nearest (ld, li), ascending
// (d2, index); other lanes hold (FLT_MAX, INT_MAX). `init_bound`: only neighbours with d2 <= init_bound are wanted (an
// upper bound of the k-th distance, e.g. from the previous ICP iteration's list; FLT_MAX: none). All 32 lanes call
// with the same arguments. Returns the count (min(k, n) when init_bound is FLT_MAX).
__device__ __forceinline__ int warp_knn(const GridView& g, OctStack* st, bool active, float qx, float qy, float qz, int k,
                                        float init_bound, float& ld, int& li) {
  const Coop<32> o;
  const unsigned full = 0xffffffffu;
  const float ux = (qx - g.ox) * g.inv_h, uy = (qy - g.oy) * g.inv_h, uz = (qz - g.oz) * g.inv_h;
  if (k > g.n) k = g.n;
  ld = FLT_MAX; li = 0x7fffffff;
  int cnt = 0;
  if (!(active && g.n > 0 && k > 0)) return 0;
  const unsigned kmask = k >= 32 ? full : ((1u << k) - 1u);
  float kth_d = FLT_MAX;   // current k-th entry (valid when cnt == k)
  int kth_i = 0x7fffffff;
  int sp = coop_push_ball(g, st, o, true, ux, uy, uz, init_bound);
  while (sp > 0) {
    --sp;
    const OctEntry en = st->s[sp];
    __syncwarp();
    float bound = (cnt == k) ? fminf(kth_d, init_bound) : init_bound;
    const bool live = en.d2 <= bound;
    const int level = (int)(en.node >> 27);
    const bool leaf = level == 0 || en.e - en.b <= kWarpLeaf;
    if (live && leaf) {
      for (int base = en.b; base < en.e; base += 32) {
        const int i = base + (int)o.sub;
        float d2 = FLT_MAX;
        int idx = 0x7fffffff;
        if (i < en.e) {
          const float4 p = __ldg(g.pts + i);
          d2 = dist2(qx, qy, qz, p.x, p.y, p.z);
          idx = __float_as_int(p.w);
        }
        const bool cand = idx != 0x7fffffff && d2 <= init_bound && (cnt < k || nb_less(d2, idx, kth_d, kth_i));
        unsigned cm = __ballot_sync(full, cand);
        while (cm != 0u) {
          const int src = __ffs(cm) - 1;
          cm &= cm - 1u;
          const float cd = __shfl_sync(full, d2, src);
          const int ci = __shfl_sync(full, idx, src);
          if (cnt < k || nb_less(cd, ci, kth_d, kth_i)) {   // warp-uniform
            const int pos = __popc(__ballot_sync(full, nb_less(ld, li, cd, ci)) & kmask);
            const float ud = __shfl_up_sync(full, ld, 1);
            const int ui = __shfl_up_sync(full, li, 1);
            if ((int)o.sub > pos) { ld = ud; li = ui; }
            else if ((int)o.sub == pos) { ld = cd; li = ci; }
            if (cnt < k) ++cnt;
            if (cnt == k) { kth_d = __shfl_sync(full, ld, k - 1); kth_i = __shfl_sync(full, li, k - 1); }
          }
        }
      }
      bound = (cnt == k) ? fminf(kth_d, init_bound) : init_bound;
    }
    sp += coop_expand(g, st, o, sp, live && !leaf, en.node, en.e, ux, uy, uz, bound);
  }
  if ((int)o.sub >= cnt) { ld = FLT_MAX; li = 0x7fffffff; }
  return cnt;
}

// ---- warp_knn_smem ------------------------------------------------------------------------------------------
// Exact k nearest (k <= 32) of the warp's query among nt target points held in SHARED memory in their original order
// (small targets: a sampled cluster is ~1 500 points = 24 KB). No index and no dependent loads: 32 points per step,
// the same register list and (d2, index) order as warp_knn, so the results are identical. n_finite = number of finite
// target points (k is clamped to it, like KdTreeFLANN does).
__device__ __forceinline__ int warp_knn_smem(const float4* tg, int nt, int n_finite, bool active, float qx, float qy, float qz, int k,
                                             float init_bound, float& ld, int& li) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  if (k > n_finite) k = n_finite;
  ld = FLT_MAX; li = 0x7fffffff;
  int cnt = 0;
  if (!(active && k > 0)) return 0;
  const unsigned kmask = k >= 32 ? full : ((1u << k) - 1u);
  float kth_d = FLT_MAX;
  int kth_i = 0x7fffffff;
  for (int base = 0; base < nt; base += 32) {
    const int j = base + lane;
    float d2 = FLT_MAX;
    int idx = 0x7fffffff;
    if (j < nt) {
      const float4 t = tg[j];
      if (finite3(t.x, t.y, t.z)) { d2 = dist2(qx, qy, qz, t.x, t.y, t.z); idx = j; }
    }
    const bool cand = idx != 0x7fffffff && d2 <= init_bound && (cnt < k || nb_less(d2, idx, kth_d, kth_i));
    unsigned cm = __ballot_sync(full, cand);
    while (cm != 0u) {
      const int src = __ffs(cm) - 1;
      cm &= cm - 1u;
      const float cd = __shfl_sync(full, d2, src);
      const int ci = __shfl_sync(full, idx, src);
      if (cnt < k || nb_less(cd, ci, kth_d, kth_i)) {   // warp-uniform
        const int pos = __popc(__ballot_sync(full, nb_less(ld, li, cd, ci)) & kmask);
        const float ud = __shfl_up_sync(full, ld, 1);
        const int ui = __shfl_up_sync(full, li, 1);
        if (lane > pos) { ld = ud; li = ui; }
        else if (lane == pos) { ld = cd; li = ci; }
        if (cnt < k) ++cnt;
        if (cnt == k) { kth_d = __shfl_sync(full, ld, k - 1); kth_i = __shfl_sync(full, li, k - 1); }
      }
    }
  }
  if (lane >= cnt) { ld = FLT_MAX; li = 0x7fffffff; }
  return cnt;
}

// The same result when a TIGHT bound on the k-th distance is known (the ICP loop: the previous iteration's k neighbours at the
// query's new position), without the serial insertion chain: pass 1 compacts the few points within the bound into a per-warp
// shared buffer (ballot + popc, no dependency between steps except the running count), pass 2 ranks them all-against-all
// (broadcast reads) and scatters the k best into sorted order. (d2, index) pairs are distinct, so the ranks are a permutation
// and the list equals warp_knn_smem's exactly. buf: kKnnBufCap + 32 float2 entries owned by this warp. Falls back to the
// insertion scan when the bound admits more than kKnnBufCap points or fewer than k.
static constexpr int kKnnBufCap = 128;
__device__ __forceinline__ int warp_knn_smem_bounded(const float4* tg, int nt, int n_finite, bool active, float qx, float qy, float qz,
                                                     int k, float bound, float2* buf, float& ld, int& li) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  if (k > n_finite) k = n_finite;
  if (!(active && k > 0)) { ld = FLT_MAX; li = 0x7fffffff; return 0; }
  if (!(bound < FLT_MAX)) {
    // No bound given: make one. Every lane takes the minimum over its own stride of the target; the k lanes with the smallest
    // minima hold k DISTINCT points, so the k-th smallest of the 32 lane minima bounds the k-th distance (k <= 32). One extra
    // pass without any list maintenance, instead of ~k ln(n / k) serial insertions.
    float mn = FLT_MAX;
#pragma unroll 4
    for (int base = 0; base < nt; base += 32) {
      const int j = base + lane;
      if (j < nt) {
        const float4 t = tg[j];
        const float d2 = dist2(qx, qy, qz, t.x, t.y, t.z);
        if (finite3(t.x, t.y, t.z)) mn = fminf(mn, d2);
      }
    }
    int rank = 0;
#pragma unroll
    for (int o = 0; o < 32; ++o) {
      const float other = __shfl_sync(full, mn, o);
      rank += (other < mn || (other == mn && o < lane)) ? 1 : 0;
    }
    const unsigned holder = __ballot_sync(full, rank == k - 1);   // exactly one lane: the ranks are a permutation
    const float tau = __shfl_sync(full, mn, __ffs(holder) - 1);
    if (!(tau < FLT_MAX)) return warp_knn_smem(tg, nt, n_finite, active, qx, qy, qz, k, bound, ld, li);   // fewer than k lanes see a point
    bound = tau;
  }
  const unsigned lt = (1u << lane) - 1u;
  int c = 0;
#pragma unroll 4
  for (int base = 0; base < nt; base += 32) {
    const int j = base + lane;
    float d2 = FLT_MAX;
    bool cand = false;
    if (j < nt) {
      const float4 t = tg[j];
      d2 = dist2(qx, qy, qz, t.x, t.y, t.z);
      cand = finite3(t.x, t.y, t.z) && d2 <= bound;
    }
    const unsigned m = __ballot_sync(full, cand);
    if (cand) { const int pos = c + __popc(m & lt); if (pos < kKnnBufCap) buf[pos] = make_float2(d2, __int_as_float(j)); }
    c += __popc(m);
  }
  if (c > kKnnBufCap || c < k) return warp_knn_smem(tg, nt, n_finite, active, qx, qy, qz, k, bound, ld, li);
  __syncwarp();
  float2* sorted = buf + kKnnBufCap;
#pragma unroll
  for (int h = 0; h < kKnnBufCap / 32; ++h) {
    const int e = lane + 32 * h;
    if (e < c) {
      const float2 mine = buf[e];
      const int mi = __float_as_int(mine.y);
      int rank = 0;
      for (int t = 0; t < c; ++t) { const float2 o = buf[t]; rank += nb_less(o.x, __float_as_int(o.y), mine.x, mi) ? 1 : 0; }
      if (rank < 32) sorted[rank] = mine;
    }
  }
  __syncwarp();
  ld = FLT_MAX; li = 0x7fffffff;
  if (lane < k) { const float2 r = sorted[lane]; ld = r.x; li = __float_as_int(r.y); }
  __syncwarp();   // the buffer is reused by this warp's next query
  return k;
}

// ---- k nearest for 32 < k <= kKnnListMax: the sorted list in SHARED memory ---------------------------------------------
// One query per warp, as warp_knn, but the list no longer fits one entry per lane: it lives in the warp's KnnList, 8 B per entry
// (d2, index bits), ascending (d2, index). Candidates come 32 at a time (one per lane); the ones that beat the k-th entry are
// merged in one step: each ranks itself within the batch (shuffles) and within the list (binary search), each list entry counts
// the batch entries below it (binary search in the sorted batch), and every entry is written to its merged position. (d2, index)
// pairs are distinct, so the positions are a permutation and the list equals the one inserting the candidates one by one builds.
static constexpr int kKnnListMax = 256;   // OPE_KNN_MAX_K
struct KnnList {
  float2 e[kKnnListMax];   // the list
  float2 b[32];            // the sorted batch being merged
};

// Merge this lane's candidate (when `cand`) into L (cnt entries, at most k kept). All 32 lanes call; returns the new count.
__device__ __forceinline__ int knn_list_merge(KnnList* L, int cnt, int k, bool cand, float d2, int idx) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const unsigned cm = __ballot_sync(full, cand);
  if (cm == 0u) return cnt;
  const int nc = __popc(cm);
  int rb = 0;   // rank within the batch
#pragma unroll
  for (int o = 0; o < 32; ++o) {
    const float od = __shfl_sync(full, d2, o);
    const int oi = __shfl_sync(full, idx, o);
    rb += (((cm >> o) & 1u) && nb_less(od, oi, d2, idx)) ? 1 : 0;
  }
  int rl = 0;   // rank within the list
  if (cand) {
    int hi = cnt;
    while (rl < hi) {
      const int m = (rl + hi) >> 1;
      const float2 v = L->e[m];
      if (nb_less(v.x, __float_as_int(v.y), d2, idx)) rl = m + 1; else hi = m;
    }
    L->b[rb] = make_float2(d2, __int_as_float(idx));
  }
  __syncwarp();
  float2 keep[kKnnListMax / 32];
  int pos[kKnnListMax / 32];
#pragma unroll
  for (int t = 0; t < kKnnListMax / 32; ++t) {
    const int j = lane + 32 * t;
    pos[t] = k;   // not kept
    if (j < cnt) {
      keep[t] = L->e[j];
      const int vi = __float_as_int(keep[t].y);
      int lo = 0, hi = nc;
      while (lo < hi) {
        const int m = (lo + hi) >> 1;
        const float2 c = L->b[m];
        if (nb_less(c.x, __float_as_int(c.y), keep[t].x, vi)) lo = m + 1; else hi = m;
      }
      pos[t] = j + lo;
    }
  }
  __syncwarp();
#pragma unroll
  for (int t = 0; t < kKnnListMax / 32; ++t)
    if (pos[t] < k) L->e[pos[t]] = keep[t];
  if (cand && rb + rl < k) L->e[rb + rl] = make_float2(d2, __int_as_float(idx));
  __syncwarp();
  return min(cnt + nc, k);
}

// Exact k nearest (32 < k <= kKnnListMax) of the warp's query on the grid: warp_knn's traversal (nearest node first, nodes
// pruned by the current k-th distance), warp_knn's candidate rule, the list in L. Returns the count (min(k, g.n)); the
// entries L->e[0 .. count) are valid after the call.
__device__ __forceinline__ int warp_knn_list(const GridView& g, OctStack* st, KnnList* L, bool active, float qx, float qy, float qz, int k) {
  const Coop<32> o;
  const float ux = (qx - g.ox) * g.inv_h, uy = (qy - g.oy) * g.inv_h, uz = (qz - g.oz) * g.inv_h;
  if (k > g.n) k = g.n;
  int cnt = 0;
  if (!(active && g.n > 0 && k > 0)) return 0;
  float kth_d = FLT_MAX;
  int kth_i = 0x7fffffff;
  int sp = coop_push_ball(g, st, o, true, ux, uy, uz, FLT_MAX);
  while (sp > 0) {
    --sp;
    const OctEntry en = st->s[sp];
    __syncwarp();
    float bound = (cnt == k) ? kth_d : FLT_MAX;
    const bool live = en.d2 <= bound;
    const int level = (int)(en.node >> 27);
    const bool leaf = level == 0 || en.e - en.b <= kWarpLeaf;
    if (live && leaf) {
      for (int base = en.b; base < en.e; base += 32) {
        const int i = base + (int)o.sub;
        float d2 = FLT_MAX;
        int idx = 0x7fffffff;
        if (i < en.e) {
          const float4 p = __ldg(g.pts + i);
          d2 = dist2(qx, qy, qz, p.x, p.y, p.z);
          idx = __float_as_int(p.w);
        }
        const bool cand = idx != 0x7fffffff && d2 <= FLT_MAX && (cnt < k || nb_less(d2, idx, kth_d, kth_i));
        cnt = knn_list_merge(L, cnt, k, cand, d2, idx);
        if (cnt == k) { const float2 v = L->e[k - 1]; kth_d = v.x; kth_i = __float_as_int(v.y); }
      }
      bound = (cnt == k) ? kth_d : FLT_MAX;
    }
    sp += coop_expand(g, st, o, sp, live && !leaf, en.node, en.e, ux, uy, uz, bound);
  }
  return cnt;
}

// The same list among nt target points held in SHARED memory in their original order (warp_knn_smem's scan, n_finite = number
// of finite targets, k clamped to it): the same entries as warp_knn_list.
__device__ __forceinline__ int warp_knn_list_smem(const float4* tg, int nt, int n_finite, KnnList* L, bool active, float qx, float qy,
                                                  float qz, int k) {
  const int lane = threadIdx.x & 31;
  if (k > n_finite) k = n_finite;
  int cnt = 0;
  if (!(active && k > 0)) return 0;
  float kth_d = FLT_MAX;
  int kth_i = 0x7fffffff;
  for (int base = 0; base < nt; base += 32) {
    const int j = base + lane;
    float d2 = FLT_MAX;
    int idx = 0x7fffffff;
    if (j < nt) {
      const float4 t = tg[j];
      if (finite3(t.x, t.y, t.z)) { d2 = dist2(qx, qy, qz, t.x, t.y, t.z); idx = j; }
    }
    const bool cand = idx != 0x7fffffff && d2 <= FLT_MAX && (cnt < k || nb_less(d2, idx, kth_d, kth_i));
    cnt = knn_list_merge(L, cnt, k, cand, d2, idx);
    if (cnt == k) { const float2 v = L->e[k - 1]; kth_d = v.x; kth_i = __float_as_int(v.y); }
  }
  return cnt;
}

}  // namespace ope
