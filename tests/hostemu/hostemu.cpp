// tests/hostemu/hostemu.cpp — TEST INFRASTRUCTURE. Compiles the product's OPE_HD device functions
// (csrc/ope_device.cuh, csrc/ope_grid.cuh) with the HOST compiler so their per-query logic (ring search
// termination, tie order, eigen33, pair features, SVD) can be checked against the oracle without a GPU, and
// the host half of the point-to-plane estimators (csrc/ope_p2plane.h) against a serial accumulator.
// The grid is built serially here with the same binning formula as csrc/grid.cu. Never shipped, never loaded
// by the product.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>
using std::isfinite;
static long g_counts[4] = {0, 0, 0, 0};
#define OPE_COUNT(what) (g_counts[what]++)
#include "../../object-pose-estimation_b200/csrc/ope_grid.cuh"
#include "../../object-pose-estimation_b200/csrc/ope_p2plane.h"

using namespace ope;

namespace {
struct HostGrid {
  GridView v;
  std::vector<int> cell_start;
  std::vector<float4> sorted;
};

void build(const float* xyz, int n, float h_wanted, HostGrid& g) {
  float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
  int nf = 0;
  for (int i = 0; i < n; ++i) {
    const float* p = xyz + 3 * i;
    if (!finite3(p[0], p[1], p[2])) continue;
    ++nf;
    for (int d = 0; d < 3; ++d) { mn[d] = std::min(mn[d], p[d]); mx[d] = std::max(mx[d], p[d]); }
  }
  if (nf == 0) { mn[0] = mn[1] = mn[2] = mx[0] = mx[1] = mx[2] = 0; }
  float emax = std::max(mx[0] - mn[0], std::max(mx[1] - mn[1], mx[2] - mn[2]));
  if (!(emax > 0)) emax = 1.0f;
  int bits = (int)std::ceil(std::log2(std::max(emax / h_wanted, 1.0f)));
  bits = std::min(std::max(bits, 1), 8);
  const float hh = emax * (1.0f + 1e-4f) / (float)(1 << bits);
  const float inv = 1.0f / hh;
  g.v.ox = mn[0]; g.v.oy = mn[1]; g.v.oz = mn[2]; g.v.h = hh; g.v.inv_h = inv; g.v.bits = bits; g.v.n = nf;
  const size_t ncodes = (size_t)1 << (3 * bits);
  g.cell_start.assign(ncodes + 1, 0);
  for (int i = 0; i < n; ++i) { const float* p = xyz + 3 * i; if (finite3(p[0], p[1], p[2])) g.cell_start[grid_cell_code(g.v, p[0], p[1], p[2]) + 1]++; }
  for (size_t c = 0; c < ncodes; ++c) g.cell_start[c + 1] += g.cell_start[c];
  std::vector<int> cur(g.cell_start.begin(), g.cell_start.end() - 1);
  g.sorted.resize(nf);
  for (int i = 0; i < n; ++i) {  // ascending i => index-ordered within a cell
    const float* p = xyz + 3 * i;
    if (!finite3(p[0], p[1], p[2])) continue;
    g.sorted[cur[grid_cell_code(g.v, p[0], p[1], p[2])]++] = make_float4(p[0], p[1], p[2], i2f(i));
  }
  g.v.start = g.cell_start.data(); g.v.pts = g.sorted.data();
}

// the sums p2plane.cu's kernels reduce, taken pair after pair: what the device returns whenever the double sums are exact
struct SerialP2p {
  std::vector<float4> s, t, nr;
  double out[28];
  int jacobian(const Mat4 W[7], const float h[6], const double** r) {
    for (double& v : out) v = 0.0;
    for (size_t i = 0; i < s.size(); ++i) {
      const float f = plane_residual(W[0], s[i], t[i], nr[i]);
      double J[6];
      for (int j = 0; j < 6; ++j) J[j] = (double)((plane_residual(W[1 + j], s[i], t[i], nr[i]) - f) / h[j]);
      int e = 0;
      for (int a = 0; a < 6; ++a)
        for (int b = a; b < 6; ++b) out[e++] += J[a] * J[b];
      for (int a = 0; a < 6; ++a) out[21 + a] += J[a] * (double)f;
      out[27] += (double)f * (double)f;
    }
    *r = out;
    return 0;
  }
  int residual(const Mat4& W, const double** r) {
    out[0] = 0.0;
    for (size_t i = 0; i < s.size(); ++i) { const float f = plane_residual(W, s[i], t[i], nr[i]); out[0] += (double)f * (double)f; }
    *r = out;
    return 0;
  }
};

SerialP2p p2p_pairs(const float* s, const float* t, const float* n, int m) {
  SerialP2p a;
  for (int i = 0; i < m; ++i) {
    a.s.push_back(make_float4(s[3 * i], s[3 * i + 1], s[3 * i + 2], 1.0f));
    a.t.push_back(make_float4(t[3 * i], t[3 * i + 1], t[3 * i + 2], 1.0f));
    a.nr.push_back(make_float4(n[3 * i], n[3 * i + 1], n[3 * i + 2], 0.0f));
  }
  return a;
}
}  // namespace

extern "C" {
void emu_counts(long* out, int reset) { for (int i = 0; i < 4; ++i) { out[i] = g_counts[i]; if (reset) g_counts[i] = 0; } }

int emu_knn(const float* tgt, int nt, const float* qry, int nq, int k, float h, float max_d2, int* out_idx, float* out_d2) {
  HostGrid g;
  build(tgt, nt, h, g);
  for (int i = 0; i < nq; ++i) {
    const float* q = qry + 3 * i;
    float bd[32]; int bi[32]; int cnt = 0;
    if (k == 1) {
      float d2; int idx = grid_nn1(g.v, q[0], q[1], q[2], max_d2, d2);
      if (idx >= 0) { bd[0] = d2; bi[0] = idx; cnt = 1; }
    } else cnt = grid_knn<32>(g.v, q[0], q[1], q[2], k, bd, bi);
    for (int j = 0; j < k; ++j) { out_idx[i * k + j] = j < cnt ? bi[j] : -1; out_d2[i * k + j] = j < cnt ? bd[j] : INFINITY; }
  }
  return 0;
}

// nearest neighbour with a per-query seed index (-1 = none): the result must not depend on the seed
int emu_nn1_seeded(const float* tgt, int nt, const float* qry, int nq, const int* seeds, float h, float max_d2, int* out_idx,
                   float* out_d2) {
  HostGrid g;
  build(tgt, nt, h, g);
  std::vector<float4> orig(nt);
  for (int i = 0; i < nt; ++i) orig[i] = make_float4(tgt[3 * i], tgt[3 * i + 1], tgt[3 * i + 2], 1.0f);
  for (int i = 0; i < nq; ++i) {
    const float* q = qry + 3 * i;
    float d2;
    const int idx = grid_nn1(g.v, q[0], q[1], q[2], max_d2, d2, seeds[i], orig.data());
    out_idx[i] = idx; out_d2[i] = idx >= 0 ? d2 : INFINITY;
  }
  return 0;
}

// nearest neighbour + certificate radius (gap > 0): out_r2[i] = squared distance below which no OTHER point exists
int emu_nn1_cert(const float* tgt, int nt, const float* qry, int nq, const int* seeds, float h, float max_d2, float gap, int* out_idx,
                 float* out_d2, float* out_r2) {
  HostGrid g;
  build(tgt, nt, h, g);
  std::vector<float4> orig(nt);
  for (int i = 0; i < nt; ++i) orig[i] = make_float4(tgt[3 * i], tgt[3 * i + 1], tgt[3 * i + 2], 1.0f);
  for (int i = 0; i < nq; ++i) {
    const float* q = qry + 3 * i;
    float d2, r2;
    const int idx = grid_nn1(g.v, q[0], q[1], q[2], max_d2, d2, seeds ? seeds[i] : -1, orig.data(), gap, &r2);
    out_idx[i] = idx; out_d2[i] = idx >= 0 ? d2 : INFINITY; out_r2[i] = r2;
  }
  return 0;
}

// radius count via the pruned traversal
int emu_radius_count(const float* tgt, int nt, const float* qry, int nq, float radius, float h, int* counts) {
  HostGrid g;
  build(tgt, nt, h, g);
  const float r2 = radius * radius;
  for (int i = 0; i < nq; ++i) {
    const float* q = qry + 3 * i;
    int cnt = 0;
    grid_radius_visit(g.v, q[0], q[1], q[2], r2, [&](float, float, float, int, float) { ++cnt; });
    counts[i] = cnt;
  }
  return 0;
}

// normal of point q from an explicit neighbour list (indices into pts)
void emu_normal(const float* pts, const int* nn, int cnt, const float* q, const float* vp, float* out4) {
  CovAccum acc; acc.reset();
  for (int j = 0; j < cnt; ++j) acc.add(pts[3 * nn[j]], pts[3 * nn[j] + 1], pts[3 * nn[j] + 2]);
  normal_from_accum(acc, cnt, q[0], q[1], q[2], vp[0], vp[1], vp[2], out4);
}

void emu_pair_bins(const float* p1, const float* n1, const float* p2, const float* n2, int* h) {
  pair_feature_bins(p1[0], p1[1], p1[2], n1, p2[0], p2[1], p2[2], n2, h[0], h[1], h[2]);
}

void emu_umeyama_small(const float* s, const float* d, int n, float* T16) {
  Mat4 M; umeyama_small(s, d, n, M); std::memcpy(T16, M.m, 64);
}

void emu_umeyama_moments(const float* s, const float* d, int n, float* T16) {
  double acc[16]; for (int i = 0; i < 16; ++i) acc[i] = 0;
  for (int i = 0; i < n; ++i) {
    acc[0] += 1; for (int k = 0; k < 3; ++k) { acc[1 + k] += s[3 * i + k]; acc[4 + k] += d[3 * i + k]; }
    for (int c = 0; c < 3; ++c) for (int r = 0; r < 3; ++r) acc[7 + c * 3 + r] += (double)d[3 * i + r] * (double)s[3 * i + c];
  }
  Mat4 M; umeyama_from_moments(acc, M); std::memcpy(T16, M.m, 64);
}


// TransformationEstimationPointToPlane (LM) over the pairs (s[i], t[i], n[i]), xyz rows: p2plane.cu's host driver.
// info: (status, nfev, iterations); trace: (smallest Jacobian rank, smallest qrsolv nsing) the driver met.
int emu_p2p_lm(const float* s, const float* t, const float* n, int m, float* T16, int32_t* info, int32_t* trace) {
  SerialP2p acc = p2p_pairs(s, t, n, m);
  p2p::LmTrace tr;
  Mat4 T;
  const int rc = p2p::lm_estimate(acc, m, &T, info, &tr);
  std::memcpy(T16, T.m, 64);
  trace[0] = tr.min_rank; trace[1] = tr.min_nsing;
  return rc;
}

// TransformationEstimationPointToPlaneLLS: the device kernel's rows (non-finite ones skipped) + p2plane.cu's host solve.
// Returns whether the 6x6 system had no exactly zero pivot.
int emu_p2p_lls(const float* s, const float* t, const float* n, int m, float* T16) {
  SerialP2p a = p2p_pairs(s, t, n, m);
  double r[27];
  for (double& v : r) v = 0.0;
  for (int i = 0; i < m; ++i) {
    if (!finite3(a.s[i].x, a.s[i].y, a.s[i].z) || !finite3(a.t[i].x, a.t[i].y, a.t[i].z) || !finite3(a.nr[i].x, a.nr[i].y, a.nr[i].z)) continue;
    double v[6], d;
    plane_lls_row(a.s[i], a.t[i], a.nr[i], v, d);
    int e = 0;
    for (int p = 0; p < 6; ++p)
      for (int q = p; q < 6; ++q) r[e++] += v[p] * v[q];
    for (int p = 0; p < 6; ++p) r[21 + p] += v[p] * d;
  }
  bool solved;
  const Mat4 T = p2p::lls_transform(r, &solved);
  std::memcpy(T16, T.m, 64);
  return solved ? 1 : 0;
}

}  // extern "C"


// Exhaustive check of ope::div_by_const against the IEEE division over everything depth -> cloud can feed it: Z = raw / scale for
// every raw value, then (i - c) * Z / f for every row/column index of a `dim`-pixel axis. Returns the number of mismatches.
extern "C" long long emu_div_by_const_mismatches(float scale, float f, float c, int dim) {
  long long bad = 0;
  const float r_scale = 1.0f / scale, r_f = 1.0f / f;
  for (int raw = 0; raw <= 65535; ++raw) {
    const float z_ref = (float)raw / scale;
    const float z = ope::div_by_const((float)raw, scale, r_scale);
    if (z != z_ref) { ++bad; continue; }
    for (int i = 0; i < dim; ++i) {
      const float num = ((float)i - c) * z;
      if (ope::div_by_const(num, f, r_f) != num / f) ++bad;
    }
  }
  return bad;
}
