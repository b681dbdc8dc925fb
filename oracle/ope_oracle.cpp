// ope_oracle.cpp — TEST INFRASTRUCTURE: single-threaded CPU restatement of the reference's registration
// hot path (SURVEY section 8c, Appendix A). See ope_oracle.h for the contract and the "parity unpinned"
// note. Build: oracle/Makefile (g++ -O2 -ffp-contract=off, no -march=native, no fast-math).
//
// Nothing here is shipped or used by the product path (object-pose-estimation_b200/csrc).
#include "ope_oracle.h"

#include <algorithm>
#include <cfloat>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <map>
#include <vector>

#include "orc_kdtree.h"
#include "orc_linalg.h"
#include "orc_segment.h"
#include "orc_lm.h"

using orc::KdTree;
using orc::Mat4;
using orc::Neighbor;

namespace {

const float kNaN = std::numeric_limits<float>::quiet_NaN();

struct Clock {
  std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
  double lap() {
    auto t1 = std::chrono::steady_clock::now();
    double s = std::chrono::duration<double>(t1 - t0).count();
    t0 = t1;
    return s;
  }
};

inline const float* at(const float* base, size_t stride, size_t i) { return base + i * stride; }

// ---- A.1 UniformSampling ---------------------------------------------------------------------------
struct VoxelFrame {
  int min_b[3], max_b[3], div_b[3];
  int64_t mul[3];
  bool any = false;
};

VoxelFrame voxelFrame(const float* pts, size_t n, size_t stride, const float inv_leaf[3]) {
  VoxelFrame f;
  float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
  for (size_t i = 0; i < n; ++i) {
    const float* p = at(pts, stride, i);
    if (!orc::finite3(p)) continue;
    f.any = true;
    for (int d = 0; d < 3; ++d) { mn[d] = std::min(mn[d], p[d]); mx[d] = std::max(mx[d], p[d]); }
  }
  if (!f.any) return f;
  for (int d = 0; d < 3; ++d) {
    f.min_b[d] = (int)std::floor(mn[d] * inv_leaf[d]);
    f.max_b[d] = (int)std::floor(mx[d] * inv_leaf[d]);
    f.div_b[d] = f.max_b[d] - f.min_b[d] + 1;
  }
  f.mul[0] = 1; f.mul[1] = f.div_b[0]; f.mul[2] = (int64_t)f.div_b[0] * f.div_b[1];
  return f;
}

// ---- A.4 normals ------------------------------------------------------------------------------------
// computeMeanAndCovarianceMatrix (single pass, float) + solvePlaneParameters + flipNormalTowardsViewpoint.
bool pointNormal(const float* pts, size_t stride, const Neighbor* nn, int cnt, const float* query,
                 const float vp[3], float out[4]) {
  if (cnt < 3) return false;
  float accu[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  for (int j = 0; j < cnt; ++j) {
    const float* p = at(pts, stride, nn[j].idx);
    accu[0] += p[0] * p[0];
    accu[1] += p[0] * p[1];
    accu[2] += p[0] * p[2];
    accu[3] += p[1] * p[1];
    accu[4] += p[1] * p[2];
    accu[5] += p[2] * p[2];
    accu[6] += p[0];
    accu[7] += p[1];
    accu[8] += p[2];
  }
  float fc = (float)cnt;
  for (int i = 0; i < 9; ++i) accu[i] /= fc;
  float cov[9];
  cov[0] = accu[0] - accu[6] * accu[6];
  cov[1] = accu[1] - accu[6] * accu[7];
  cov[2] = accu[2] - accu[6] * accu[8];
  cov[4] = accu[3] - accu[7] * accu[7];
  cov[5] = accu[4] - accu[7] * accu[8];
  cov[8] = accu[5] - accu[8] * accu[8];
  cov[3] = cov[1]; cov[6] = cov[2]; cov[7] = cov[5];
  float ev, n[3];
  orc::eigen33(cov, ev, n);
  float eig_sum = cov[0] + cov[4] + cov[8];
  float curvature = (eig_sum != 0) ? std::fabs(ev / eig_sum) : 0.0f;
  float vx = vp[0] - query[0], vy = vp[1] - query[1], vz = vp[2] - query[2];
  float cos_theta = (vx * n[0] + vy * n[1] + vz * n[2]);
  if (cos_theta < 0) { n[0] *= -1; n[1] *= -1; n[2] *= -1; }
  out[0] = n[0]; out[1] = n[1]; out[2] = n[2]; out[3] = curvature;
  return true;
}

// ---- A.5 FPFH ---------------------------------------------------------------------------------------
// pcl::computePairFeatures (features/src/pfh.cpp). Returns false (with f1..f4 = 0) on the degenerate cases.
bool pairFeatures(const float* p1, const float* n1, const float* p2, const float* n2, float& f1, float& f2,
                  float& f3, float& f4) {
  float dp[3] = {p2[0] - p1[0], p2[1] - p1[1], p2[2] - p1[2]};
  f4 = std::sqrt(orc::dot3w0(dp, dp));
  if (f4 == 0.0f) { f1 = f2 = f3 = f4 = 0.0f; return false; }
  float a[3] = {n1[0], n1[1], n1[2]}, b[3] = {n2[0], n2[1], n2[2]};
  float angle1 = orc::dot3w0(a, dp) / f4;
  float angle2 = orc::dot3w0(b, dp) / f4;
  if (orc::acos_cr(std::fabs(angle1)) > orc::acos_cr(std::fabs(angle2))) {
    std::swap(a[0], b[0]); std::swap(a[1], b[1]); std::swap(a[2], b[2]);
    dp[0] *= -1; dp[1] *= -1; dp[2] *= -1;
    f3 = -angle2;
  } else {
    f3 = angle1;
  }
  float v[3];
  orc::cross3(dp, a, v);
  float v_norm = std::sqrt(orc::dot3w0(v, v));
  if (v_norm == 0.0f) { f1 = f2 = f3 = f4 = 0.0f; return false; }
  v[0] /= v_norm; v[1] /= v_norm; v[2] /= v_norm;
  float w[3];
  orc::cross3(a, v, w);
  f2 = orc::dot3w0(v, b);
  f1 = orc::atan2_cr(orc::dot3w0(w, b), orc::dot3w0(a, b));
  return true;
}

// computePointSPFHSignature: FPFHEstimation's own computePairFeatures wrapper returns true unconditionally
// [UPSTREAM features/impl/fpfh.hpp], so a degenerate pair is binned with f1 = f2 = f3 = 0.
void spfhPoint(const float* pts, size_t stride, const float* normals, int p_idx, const std::vector<Neighbor>& nn,
               float* hist /*33*/) {
  for (int b = 0; b < 33; ++b) hist[b] = 0.0f;
  const int nb = 11;
  const float d_pi = 1.0f / (2.0f * (float)M_PI);
  float hist_incr = 100.0f / (float)((long)nn.size() - 1);
  for (size_t j = 0; j < nn.size(); ++j) {
    int q = nn[j].idx;
    if (q == p_idx) continue;
    float f1, f2, f3, f4;
    pairFeatures(at(pts, stride, p_idx), normals + 4 * (size_t)p_idx, at(pts, stride, q), normals + 4 * (size_t)q, f1,
                 f2, f3, f4);
    int h = (int)std::floor(nb * ((f1 + M_PI) * d_pi));
    if (h < 0) h = 0;
    if (h >= nb) h = nb - 1;
    hist[h] += hist_incr;
    h = (int)std::floor(nb * ((f2 + 1.0) * 0.5));
    if (h < 0) h = 0;
    if (h >= nb) h = nb - 1;
    hist[11 + h] += hist_incr;
    h = (int)std::floor(nb * ((f3 + 1.0) * 0.5));
    if (h < 0) h = 0;
    if (h >= nb) h = nb - 1;
    hist[22 + h] += hist_incr;
  }
}

// weightPointSPFHSignature
void fpfhPoint(const float* spfh, const std::vector<Neighbor>& nn, float* out /*33*/) {
  double sum[3] = {0, 0, 0};
  for (int b = 0; b < 33; ++b) out[b] = 0.0f;
  for (size_t j = 0; j < nn.size(); ++j) {
    if (nn[j].d2 == 0) continue;
    float weight = 1.0f / nn[j].d2;
    const float* h = spfh + 33 * (size_t)nn[j].idx;
    for (int s = 0; s < 3; ++s)
      for (int b = 0; b < 11; ++b) {
        float val = h[11 * s + b] * weight;
        sum[s] += val;
        out[11 * s + b] += val;
      }
  }
  for (int s = 0; s < 3; ++s) {
    if (sum[s] != 0) sum[s] = 100.0 / sum[s];
    for (int b = 0; b < 11; ++b) out[11 * s + b] *= (float)sum[s];
  }
}

int computeSpfh(const float* pts, size_t n, size_t stride, const float* normals, float radius, const KdTree& tree,
                std::vector<float>& spfh) {
  spfh.assign(n * 33, 0.0f);
  std::vector<Neighbor> nn;
  float r2 = radius * radius;
  for (size_t i = 0; i < n; ++i) {
    if (!orc::finite3(at(pts, stride, i))) continue;
    tree.radius(at(pts, stride, i), r2, nn);
    if (nn.empty()) continue;
    spfhPoint(pts, stride, normals, (int)i, nn, &spfh[i * 33]);
  }
  return 0;
}

// ---- correspondences + rejectors --------------------------------------------------------------------
struct CloudView {
  const float* pts; size_t n; size_t stride; const float* normals;  // normals n*4 or null
  const float* p(size_t i) const { return pts + i * stride; }
  const float* nrm(size_t i) const { return normals + 4 * i; }
};

// `fixed` / `n_fixed`: the reference's own extension (setFixedCorrespondences, VP/icp_mod.h:267-281): pairs the caller pins.
// determineCorrespondences puts them in FRONT of the estimated ones with distance = squared distance * 1e10 and writes that
// distance back into the caller's list (VP/impl/correspondence_estimation_mod.hpp:134-161). The reciprocal variant
// (:216-303) ignores them: a pair (i, j) is kept iff j is i's nearest target point within the distance AND i is j's nearest
// SOURCE point within the distance (a second tree over the current source, rebuilt whenever the source moved).
void estimateCorrespondences(const CloudView& src, const CloudView& tgt, const KdTree& tgt_tree,
                             const float* est_src_normals, const ope_icp_params& prm,
                             std::vector<ope_correspondence>& out, ope_correspondence* fixed = nullptr, size_t n_fixed = 0) {
  out.clear();
  out.reserve(src.n + n_fixed);
  if (prm.estimator == OPE_EST_NEAREST) {
    double max_dist_sqr = prm.max_correspondence_distance * prm.max_correspondence_distance;
    Neighbor nn;
    if (prm.use_reciprocal) {
      KdTree src_tree; src_tree.build(src.pts, src.n, src.stride);
      Neighbor back;
      for (size_t i = 0; i < src.n; ++i) {
        if (tgt_tree.knn(src.p(i), 1, &nn) == 0) continue;
        if (nn.d2 > max_dist_sqr) continue;
        if (src_tree.knn(tgt.p(nn.idx), 1, &back) == 0) continue;
        if (back.d2 > max_dist_sqr || (int32_t)i != back.idx) continue;
        out.push_back(ope_correspondence{(int32_t)i, nn.idx, nn.d2});
      }
      return;
    }
    for (size_t f = 0; f < n_fixed; ++f) {
      const float* t = tgt.p(fixed[f].index_match);
      const float* q = src.p(fixed[f].index_query);
      float px = t[0] - q[0], py = t[1] - q[1], pz = t[2] - q[2];
      fixed[f].distance = (float)((px * px + py * py + pz * pz) * 1e10);   // float sum, double product, stored as float
      out.push_back(fixed[f]);
    }
    for (size_t i = 0; i < src.n; ++i) {
      // a non-finite query is skipped (FLANN would assert); the tree's answer to a NaN query has d2 = NaN, which the
      // `d2 > max` gate below would let through
      if (!orc::finite3(src.p(i))) continue;
      if (tgt_tree.knn(src.p(i), 1, &nn) == 0) continue;
      if (nn.d2 > max_dist_sqr) continue;
      out.push_back(ope_correspondence{(int32_t)i, nn.idx, nn.d2});
    }
  } else {
    int k = prm.k_search;
    std::vector<Neighbor> nn(std::max(k, 1));
    for (size_t i = 0; i < src.n; ++i) {
      int cnt = tgt_tree.knn(src.p(i), k, nn.data());
      if (cnt == 0) continue;
      double min_dist = std::numeric_limits<double>::max();
      int min_index = 0;
      const float* nr = est_src_normals + 4 * i;
      for (int j = 0; j < cnt; ++j) {
        const float* t = tgt.p(nn[j].idx);
        const float* s = src.p(i);
        float px = t[0] - s[0], py = t[1] - s[1], pz = t[2] - s[2];
        double N[3] = {nr[0], nr[1], nr[2]}, V[3] = {px, py, pz};
        double C[3] = {N[1] * V[2] - N[2] * V[1], N[2] * V[0] - N[0] * V[2], N[0] * V[1] - N[1] * V[0]};
        double dist = C[0] * C[0] + C[1] * C[1] + C[2] * C[2];
        if (dist < min_dist) { min_dist = dist; min_index = j; }
      }
      if (min_dist > prm.max_correspondence_distance) continue;  // sic: squared vs unsquared (SURVEY A.8)
      out.push_back(ope_correspondence{(int32_t)i, nn[min_index].idx, nn[min_index].d2});
    }
  }
}

bool rejectorKeeps(int kind, double thr, const ope_correspondence& c, const float* rs_pts, size_t rs_stride,
                   const float* rs_normals, const CloudView& tgt) {
  if (kind == OPE_REJ_SURFACE_NORMAL) {
    const float* a = rs_normals + 4 * (size_t)c.index_query;
    const float* b = tgt.nrm(c.index_match);
    double score = (double)((a[0] * b[0]) + (a[1] * b[1]) + (a[2] * b[2]));
    return score > thr;
  } else if (kind == OPE_REJ_SELF_OCCLUDED_NORMAL) {
    const float* a = rs_normals + 4 * (size_t)c.index_query;
    const float* p = rs_pts + rs_stride * (size_t)c.index_query;
    const double s = std::sqrt(p[0] * p[0] + p[1] * p[1] + p[2] * p[2]);  // float sqrt (std:: overload), widened
    double score = (double)((a[0] * (-p[0] / s)) + (a[1] * (-p[1] / s)) + (a[2] * (-p[2] / s)));
    return score > thr;
  }
  return true;
}

void applyRejectors(const ope_icp_params& prm, std::vector<ope_correspondence>& corr, const float* rs_pts,
                    size_t rs_stride, const float* rs_normals, const CloudView& tgt, int only_first = 0) {
  for (int r = 0; r < (only_first ? std::min(prm.n_rejectors, 1) : prm.n_rejectors) && r < OPE_MAX_REJECTORS; ++r) {
    size_t w = 0;
    for (size_t i = 0; i < corr.size(); ++i)
      if (rejectorKeeps(prm.rejector_kind[r], prm.rejector_threshold[r], corr[i], rs_pts, rs_stride, rs_normals, tgt))
        corr[w++] = corr[i];
    corr.resize(w);
  }
}

// TransformationEstimationPointToPlaneLLS [UPSTREAM transformation_estimation_point_to_plane_lls.hpp]
bool solve6(double A[36], double b[6], double x[6]) {
  for (int c = 0; c < 6; ++c) {
    int best = c; double bv = std::fabs(A[c * 6 + c]);
    for (int r = c + 1; r < 6; ++r) if (std::fabs(A[r * 6 + c]) > bv) { bv = std::fabs(A[r * 6 + c]); best = r; }
    if (bv == 0) return false;
    if (best != c) { for (int k = 0; k < 6; ++k) std::swap(A[c * 6 + k], A[best * 6 + k]); std::swap(b[c], b[best]); }
    for (int r = c + 1; r < 6; ++r) {
      double f = A[r * 6 + c] / A[c * 6 + c];
      for (int k = c; k < 6; ++k) A[r * 6 + k] -= f * A[c * 6 + k];
      b[r] -= f * b[c];
    }
  }
  for (int r = 5; r >= 0; --r) {
    double s = b[r];
    for (int k = r + 1; k < 6; ++k) s -= A[r * 6 + k] * x[k];
    x[r] = s / A[r * 6 + r];
  }
  return true;
}

void pointToPlaneLLS(const CloudView& src, const CloudView& tgt, const std::vector<ope_correspondence>& corr,
                     float T[16]) {
  double ATA[36], ATb[6];
  std::memset(ATA, 0, sizeof(ATA)); std::memset(ATb, 0, sizeof(ATb));
  for (const auto& c : corr) {
    const float* s = src.p(c.index_query); const float* d = tgt.p(c.index_match); const float* n = tgt.nrm(c.index_match);
    if (!orc::finite3(s) || !orc::finite3(d) || !orc::finite3(n)) continue;
    const float sx = s[0], sy = s[1], sz = s[2], dx = d[0], dy = d[1], dz = d[2], nx = n[0], ny = n[1], nz = n[2];
    double v[6] = {(double)(nz * sy - ny * sz), (double)(nx * sz - nz * sx), (double)(ny * sx - nx * sy), nx, ny, nz};
    double dd = nx * dx + ny * dy + nz * dz - nx * sx - ny * sy - nz * sz;
    for (int r = 0; r < 6; ++r) {
      for (int k = r; k < 6; ++k) ATA[r * 6 + k] += v[r] * v[k];
      ATb[r] += v[r] * dd;
    }
  }
  for (int r = 0; r < 6; ++r) for (int k = 0; k < r; ++k) ATA[r * 6 + k] = ATA[k * 6 + r];
  double x[6] = {0, 0, 0, 0, 0, 0};
  solve6(ATA, ATb, x);
  double alpha = x[0], beta = x[1], gamma = x[2];
  Mat4 M; std::memset(M.m, 0, sizeof(M.m));
  M(0, 0) = (float)(cos(gamma) * cos(beta));
  M(0, 1) = (float)(-sin(gamma) * cos(alpha) + cos(gamma) * sin(beta) * sin(alpha));
  M(0, 2) = (float)(sin(gamma) * sin(alpha) + cos(gamma) * sin(beta) * cos(alpha));
  M(1, 0) = (float)(sin(gamma) * cos(beta));
  M(1, 1) = (float)(cos(gamma) * cos(alpha) + sin(gamma) * sin(beta) * sin(alpha));
  M(1, 2) = (float)(-cos(gamma) * sin(alpha) + sin(gamma) * sin(beta) * cos(alpha));
  M(2, 0) = (float)(-sin(beta));
  M(2, 1) = (float)(cos(beta) * sin(alpha));
  M(2, 2) = (float)(cos(beta) * cos(alpha));
  M(0, 3) = (float)x[3]; M(1, 3) = (float)x[4]; M(2, 3) = (float)x[5]; M(3, 3) = 1.0f;
  std::memcpy(T, M.m, sizeof(M.m));
}

// WarpPointRigid6D::setParam [UPSTREAM registration/warp_point_rigid_6d.h]: x = (tx, ty, tz, qx, qy, qz); qw = sqrt(1 - |q|^2),
// q normalised, then Eigen's Quaternion::toRotationMatrix; everything in float.
void warpRigid6D(const float x[6], Mat4& M) {
  std::memset(M.m, 0, sizeof(M.m));
  M(0, 3) = x[0]; M(1, 3) = x[1]; M(2, 3) = x[2]; M(3, 3) = 1.0f;
  float qx = x[3], qy = x[4], qz = x[5];
  float qw = std::sqrt(1.0f - (((0.0f * 0.0f + qx * qx) + qy * qy) + qz * qz));
  const float nrm = std::sqrt(((qx * qx + qy * qy) + qz * qz) + qw * qw);
  qx /= nrm; qy /= nrm; qz /= nrm; qw /= nrm;
  const float tx = 2.0f * qx, ty = 2.0f * qy, tz = 2.0f * qz;
  const float twx = tx * qw, twy = ty * qw, twz = tz * qw;
  const float txx = tx * qx, txy = ty * qx, txz = tz * qx;
  const float tyy = ty * qy, tyz = tz * qy, tzz = tz * qz;
  M(0, 0) = 1.0f - (tyy + tzz); M(0, 1) = txy - twz; M(0, 2) = txz + twy;
  M(1, 0) = txy + twz; M(1, 1) = 1.0f - (txx + tzz); M(1, 2) = tyz - twx;
  M(2, 0) = txz - twy; M(2, 1) = tyz + twx; M(2, 2) = 1.0f - (txx + tyy);
}

// TransformationEstimationPointToPlane [UPSTREAM transformation_estimation_point_to_plane.h + transformation_estimation_lm.hpp],
// the estimator BuildModel plugs into IterativeClosestPointWithNormals (BM/src/regmeshpcd.cpp:162,193):
// residual_i = (warp(src_i) - tgt_i) . n_tgt_i, minimised over the 6 warp parameters by Eigen's Levenberg-Marquardt with a
// forward-difference Jacobian, starting from x = 0. Fewer than 4 pairs: PCL_ERROR and the identity; 4 or 5: lmMinimize refuses
// m < n (ImproperInputParameters) and x stays 0, the identity too.
orc::LmRoute g_lm_route = orc::LM_ROUTE_NORMAL_EQ;   // orc_lm_set_route(): the Householder route is a cross-check

void pointToPlaneLM(const CloudView& src, const CloudView& tgt, const std::vector<ope_correspondence>& corr, float T[16],
                    orc::LmStats* stats = nullptr) {
  Mat4 I = Mat4::identity();
  std::memcpy(T, I.m, sizeof(I.m));
  if (corr.size() < 4) return;
  auto functor = [&](const float* x, float* fvec) {
    Mat4 W;
    warpRigid6D(x, W);
    for (size_t i = 0; i < corr.size(); ++i) {
      const float* s = src.p(corr[i].index_query); const float* d = tgt.p(corr[i].index_match); const float* n = tgt.nrm(corr[i].index_match);
      float w[3];
      orc::xformPoint(W, s, w);
      // Vector4f (s - t).dot(n) with w = 0: Eigen's packet reduction, order per orc::redux4 (orc_linalg.h)
      const float p0 = (w[0] - d[0]) * n[0], p1 = (w[1] - d[1]) * n[1], p2 = (w[2] - d[2]) * n[2], p3 = 0.0f * 0.0f;
      fvec[i] = orc::redux4(p0, p1, p2, p3);
    }
  };
  float x[6] = {0, 0, 0, 0, 0, 0};
  orc::LmStats st = orc::lmMinimize(functor, (int)corr.size(), 6, x, g_lm_route);
  if (stats) *stats = st;
  Mat4 W;
  warpRigid6D(x, W);
  std::memcpy(T, W.m, sizeof(W.m));
}

void transformCloud(std::vector<float>& pts, std::vector<float>& normals, bool has_normals, const Mat4& T) {
  size_t n = pts.size() / 3;
  for (size_t i = 0; i < n; ++i) {
    float* p = &pts[3 * i];
    if (!orc::finite3(p)) continue;
    float o[3];
    orc::xformPoint(T, p, o);
    p[0] = o[0]; p[1] = o[1]; p[2] = o[2];
    if (has_normals) {
      float* q = &normals[4 * i];
      if (!orc::finite3(q)) continue;
      orc::xformNormal(T, q, o);
      q[0] = o[0]; q[1] = o[1]; q[2] = o[2];
    }
  }
}

double fitnessScore(const float* src, size_t ns, size_t sstride, const KdTree& tree, const Mat4& T, double max_range) {
  double fitness = 0.0;
  int nr = 0;
  Neighbor nn;
  for (size_t i = 0; i < ns; ++i) {
    float q[3];
    orc::xformPoint(T, at(src, sstride, i), q);
    if (tree.knn(q, 1, &nn) == 0) continue;
    if (nn.d2 <= max_range) { fitness += nn.d2; nr++; }
  }
  return nr > 0 ? fitness / nr : std::numeric_limits<double>::max();
}

// IterativeClosestPoint::computeTransformation, VP/impl/icp_mod.hpp:118-272 (variant switch: icp_modCorr.hpp).
int icpAlign(const CloudView& src, const CloudView& tgt, const KdTree& tgt_tree, const ope_icp_params& prm,
             const Mat4& guess, ope_reg_result* res, std::vector<ope_correspondence>& corr, ope_correspondence* fixed = nullptr,
             size_t n_fixed = 0) {
  const bool has_normals = src.normals != nullptr;
  std::vector<float> xp(src.n * 3), xn;
  for (size_t i = 0; i < src.n; ++i) std::memcpy(&xp[3 * i], src.p(i), 12);
  if (has_normals) xn.assign(src.normals, src.normals + 4 * src.n);
  int nr_iterations = 0;
  bool converged = false;
  Mat4 final_t = guess;
  if (!guess.isIdentity()) transformCloud(xp, xn, has_normals, guess);
  Mat4 transformation = Mat4::identity();
  // convergence criteria wiring, icp_mod.hpp:164-168
  double prev_mse = std::numeric_limits<double>::max(), cur_mse = std::numeric_limits<double>::max();
  const double rel_thr = prm.euclidean_fitness_epsilon;
  const double trans_thr = prm.transformation_epsilon;
  const double rot_thr = 1.0 - prm.transformation_epsilon;
  int similar = 0;
  int state = OPE_CONV_NOT_CONVERGED;
  do {
    CloudView cur{xp.data(), src.n, 3, has_normals ? xn.data() : nullptr};
    const bool stale = prm.variant == OPE_ICP_VARIANT_MODCORR;
    const float* est_normals = stale ? src.normals : cur.normals;
    const bool use_fixed = fixed && prm.variant == OPE_ICP_VARIANT_MOD;   // icp_modCorr.h has no setFixedCorrespondences
    estimateCorrespondences(cur, tgt, tgt_tree, est_normals, prm, corr, use_fixed ? fixed : nullptr, use_fixed ? n_fixed : 0);
    if (stale) applyRejectors(prm, corr, src.pts, src.stride, src.normals, tgt);
    else applyRejectors(prm, corr, cur.pts, 3, cur.normals, tgt);
    // "Apply the first rejector on the fixed correspondances" and append them (again), VP/impl/icp_mod.hpp:209-225
    if (use_fixed && prm.n_rejectors > 0) {
      std::vector<ope_correspondence> again(fixed, fixed + n_fixed);
      if (!again.empty()) applyRejectors(prm, again, cur.pts, 3, cur.normals, tgt, /*only_first=*/1);
      corr.insert(corr.end(), again.begin(), again.end());
    }
    if ((int)corr.size() < prm.min_number_correspondences) {
      state = OPE_CONV_NO_CORRESPONDENCES;
      converged = false;
      break;
    }
    if (prm.transformation == OPE_TE_POINT_TO_PLANE_LLS) {
      pointToPlaneLLS(cur, tgt, corr, transformation.m);
    } else if (prm.transformation == OPE_TE_POINT_TO_PLANE) {
      pointToPlaneLM(cur, tgt, corr, transformation.m);
    } else {
      orc::umeyama(corr.size(), [&](size_t i) { return cur.p(corr[i].index_query); },
                   [&](size_t i) { return tgt.p(corr[i].index_match); }, transformation.m, tgt.n > 0 ? tgt.p(0) : nullptr);
    }
    transformCloud(xp, xn, has_normals, transformation);
    final_t = orc::mul(transformation, final_t);
    ++nr_iterations;
    // DefaultConvergenceCriteria::hasConverged [UPSTREAM, PCL 1.7.2] (SURVEY A.8)
    state = OPE_CONV_NOT_CONVERGED;
    bool conv = false;
    auto similarOrDone = [&](int st) {
      if (similar < prm.max_iterations_similar_transforms) { ++similar; return false; }
      similar = 0; state = st; return true;
    };
    if (nr_iterations >= prm.max_iterations) {
      if (!prm.failure_after_max_iterations) { state = OPE_CONV_ITERATIONS; conv = true; }
      else { converged = false; break; }  // (upstream would spin forever; we stop unconverged)
    } else {
      double cos_angle = 0.5 * (transformation(0, 0) + transformation(1, 1) + transformation(2, 2) - 1);
      double translation_sqr = transformation(0, 3) * transformation(0, 3) + transformation(1, 3) * transformation(1, 3) +
                               transformation(2, 3) * transformation(2, 3);
      if (cos_angle >= rot_thr && translation_sqr <= trans_thr) {
        conv = similarOrDone(OPE_CONV_TRANSFORM);
      } else {
        double mse = 0;
        for (size_t i = 0; i < corr.size(); ++i) mse += corr[i].distance;
        mse /= double(corr.size());
        cur_mse = mse;
        if (std::fabs(cur_mse - prev_mse) < prm.mse_threshold_absolute) {
          conv = similarOrDone(OPE_CONV_ABS_MSE);
        } else if (std::fabs(cur_mse - prev_mse) / prev_mse < rel_thr) {
          conv = similarOrDone(OPE_CONV_REL_MSE);
        } else {
          prev_mse = cur_mse;
        }
      }
    }
    converged = conv;
    if (prm.force_all_iterations && nr_iterations < prm.max_iterations) converged = false;
  } while (!converged);
  std::memcpy(res->T, final_t.m, sizeof(final_t.m));
  res->converged = converged ? 1 : 0;
  res->state = state;
  res->iterations = nr_iterations;
  res->n_correspondences = (int32_t)corr.size();
  res->last_mse = cur_mse;
  res->best_error = 0; res->best_iteration = 0; res->reserved = 0;
  return OPE_OK;
}

// ---- A.6 SAC-IA --------------------------------------------------------------------------------------
inline int getRandomIndex(int n) { return (int)(n * (rand() / (RAND_MAX + 1.0))); }

int drawSamples(const float* src, size_t ns, size_t sstride, int nr_samples, float& min_sample_distance, int32_t* out) {
  if (nr_samples > (int)ns) return OPE_ERR_INVALID;
  int without = 0;
  const int max_without = (int)(3 * ns);
  int cnt = 0;
  while (cnt < nr_samples) {
    int si = getRandomIndex((int)ns);
    bool valid = true;
    for (int i = 0; i < cnt; ++i) {
      const float* a = at(src, sstride, si); const float* b = at(src, sstride, out[i]);
      float dx = a[0] - b[0], dy = a[1] - b[1], dz = a[2] - b[2];
      float dist = std::sqrt(dx * dx + dy * dy + dz * dz);  // pcl::euclideanDistance
      if (si == out[i] || dist < min_sample_distance) { valid = false; break; }
    }
    if (valid) { out[cnt++] = si; without = 0; }
    else ++without;
    if (without >= max_without) { min_sample_distance *= 0.5f; without = 0; }
  }
  return OPE_OK;
}

void featureKnn(const float* ftgt, size_t nt, const float* q, int dim, int k, Neighbor* out, int& cnt) {
  cnt = 0;
  for (size_t j = 0; j < nt; ++j) {
    const float* f = ftgt + j * (size_t)dim;
    float d = 0;
    bool fin = true;
    for (int c = 0; c < dim; ++c) { float t = q[c] - f[c]; d += t * t; }
    if (!std::isfinite(d)) fin = false;
    if (!fin) continue;
    Neighbor v{d, (int32_t)j};
    if (cnt < k) { out[cnt++] = v; std::push_heap(out, out + cnt); }
    else if (v < out[0]) { std::pop_heap(out, out + cnt); out[cnt - 1] = v; std::push_heap(out, out + cnt); }
  }
  std::sort(out, out + cnt);
}

float saciaError(const float* src, size_t ns, size_t sstride, const KdTree& tree, const Mat4& T, float threshold) {
  float error = 0;
  Neighbor nn;
  for (size_t i = 0; i < ns; ++i) {
    float q[3];
    orc::xformPoint(T, at(src, sstride, i), q);
    tree.knn(q, 1, &nn);
    float e = nn.d2;
    error += (e <= threshold) ? (e / threshold) : 1.0f;  // TruncatedError on the squared distance
  }
  return error;
}

int saciaAlign(const float* src, size_t ns, size_t sstride, const float* fsrc, const float* tgt, size_t nt,
               size_t tstride, const float* ftgt, const KdTree& tgt_tree, const ope_sacia_params& prm,
               const ope_rng_table* table, ope_reg_result* res, float* out_errors) {
  const int S = prm.nr_samples, K = prm.k_correspondences;
  std::vector<int32_t> samples(S), corr(S);
  std::vector<Neighbor> nn(std::max(K, 1));
  float min_sample_distance = prm.min_sample_distance;
  float lowest_error = 0;
  Mat4 final_t = Mat4::identity();
  bool converged = false;
  int best_it = -1;
  int h0 = 0, h1 = prm.max_iterations;
  if (prm.hypothesis_end > prm.hypothesis_begin) { h0 = prm.hypothesis_begin; h1 = std::min(prm.hypothesis_end, prm.max_iterations); }
  const float thr = (float)prm.max_correspondence_distance;
  for (int it = 0; it < prm.max_iterations; ++it) {
    int32_t picks[64];
    if (table) {
      for (int s = 0; s < S; ++s) { samples[s] = table->samples[it * S + s]; picks[s] = table->picks[it * S + s]; }
    } else {
      int rc = drawSamples(src, ns, sstride, S, min_sample_distance, samples.data());
      if (rc) return rc;
      for (int s = 0; s < S; ++s) picks[s] = getRandomIndex(K);
    }
    if (it < h0 || it >= h1) continue;
    for (int s = 0; s < S; ++s) {
      int cnt;
      featureKnn(ftgt, nt, fsrc + 33 * (size_t)samples[s], 33, K, nn.data(), cnt);
      corr[s] = nn[std::min(picks[s], cnt - 1)].idx;
    }
    Mat4 T;
    orc::umeyama((size_t)S, [&](size_t i) { return at(src, sstride, samples[i]); },
                 [&](size_t i) { return at(tgt, tstride, corr[i]); }, T.m);
    float error = saciaError(src, ns, sstride, tgt_tree, T, thr);
    if (out_errors) out_errors[it] = error;
    if (best_it < 0 || error < lowest_error) {
      lowest_error = error; final_t = T; converged = true; best_it = it;
    }
  }
  std::memcpy(res->T, final_t.m, sizeof(final_t.m));
  res->converged = converged; res->state = 0; res->iterations = prm.max_iterations; res->n_correspondences = 0;
  res->last_mse = 0; res->best_error = lowest_error; res->best_iteration = best_it; res->reserved = 0;
  return OPE_OK;
}

// ---- helpers used by the PoseEstimator restatement -----------------------------------------------------
void uniformSampleImpl(const float* pts, size_t n, size_t stride, float leaf, std::vector<int32_t>& out) {
  out.clear();
  float inv = 1.0f / leaf;
  float inv_leaf[3] = {inv, inv, inv};
  VoxelFrame f = voxelFrame(pts, n, stride, inv_leaf);
  if (!f.any) return;
  std::map<int64_t, int32_t> leaves;
  for (size_t i = 0; i < n; ++i) {
    const float* p = at(pts, stride, i);
    if (!orc::finite3(p)) continue;
    int ijk[3];
    for (int d = 0; d < 3; ++d) ijk[d] = (int)std::floor(p[d] * inv_leaf[d]);
    int64_t idx = (ijk[0] - f.min_b[0]) * f.mul[0] + (ijk[1] - f.min_b[1]) * f.mul[1] + (ijk[2] - f.min_b[2]) * f.mul[2];
    auto it = leaves.find(idx);
    if (it == leaves.end()) { leaves.emplace(idx, (int32_t)i); continue; }
    auto diff = [&](const float* q) {
      float a = q[0] - (float)ijk[0], b = q[1] - (float)ijk[1], c = q[2] - (float)ijk[2];
      // (pt - ijk.cast<float>()).squaredNorm() over 4 components, the 4th being (1 - 0)^2: left to right unless the cast
      // vectorises (Eigen >= 3.3), see orc::redux4 / orc::eigen_cast_vectorized (orc_linalg.h)
      if (orc::eigen_cast_vectorized()) return orc::redux4(a * a, b * b, c * c, 1.0f * 1.0f);
      float r = a * a; r = r + b * b; r = r + c * c; r = r + 1.0f;
      return r;
    };
    float diff_cur = diff(p), diff_prev = diff(at(pts, stride, it->second));
    if (diff_cur < diff_prev) it->second = (int32_t)i;
  }
  out.reserve(leaves.size());
  for (auto& kv : leaves) out.push_back(kv.second);
}

void normalsImpl(const float* pts, size_t n, size_t stride, int k, const float vp[3], const KdTree& tree, float* out) {
  std::vector<Neighbor> nn(std::max(k, 1));
  for (size_t i = 0; i < n; ++i) {
    float* o = out + 4 * i;
    const float* q = at(pts, stride, i);
    int cnt = orc::finite3(q) ? tree.knn(q, k, nn.data()) : 0;
    if (cnt == 0 || !pointNormal(pts, stride, nn.data(), cnt, q, vp, o)) o[0] = o[1] = o[2] = o[3] = kNaN;
  }
}

void fpfhImpl(const float* pts, size_t n, size_t stride, const float* normals, float radius, float* out) {
  KdTree tree; tree.build(pts, n, stride);
  std::vector<float> spfh;
  computeSpfh(pts, n, stride, normals, radius, tree, spfh);
  std::vector<Neighbor> nn;
  float r2 = radius * radius;
  for (size_t i = 0; i < n; ++i) {
    float* o = out + 33 * i;
    if (orc::finite3(at(pts, stride, i))) tree.radius(at(pts, stride, i), r2, nn); else nn.clear();
    if (nn.empty()) { for (int b = 0; b < 33; ++b) o[b] = kNaN; continue; }
    fpfhPoint(spfh.data(), nn, o);
  }
}

}  // namespace

// =====================================================================================================
extern "C" {

void orc_icp_params_default(ope_icp_params* p) {
  std::memset(p, 0, sizeof(*p));
  p->max_iterations = 10;
  p->transformation_epsilon = 0.0;
  p->euclidean_fitness_epsilon = -std::numeric_limits<double>::max();
  p->max_correspondence_distance = std::sqrt(std::numeric_limits<double>::max());
  p->min_number_correspondences = 3;
  p->estimator = OPE_EST_NEAREST;
  p->k_search = 10;
  p->transformation = OPE_TE_SVD;
  p->variant = OPE_ICP_VARIANT_MOD;
  p->mse_threshold_absolute = 1e-12;
}
void orc_sacia_params_default(ope_sacia_params* p) {
  std::memset(p, 0, sizeof(*p));
  p->max_iterations = 10; p->nr_samples = 3; p->k_correspondences = 10; p->min_sample_distance = 0.0f;
  p->max_correspondence_distance = std::sqrt(std::numeric_limits<double>::max());
}
void orc_pose_params_default(ope_pose_params* p) {
  std::memset(p, 0, sizeof(*p));
  p->coarse_leaf = 0.01f; p->fine_leaf = 0.008f; p->normal_k = 30; p->fpfh_radius = 0.03f;
  orc_sacia_params_default(&p->sacia);
  p->sacia.max_iterations = 400; p->sacia.nr_samples = 5; p->sacia.k_correspondences = 5;
  p->sacia.min_sample_distance = 0.01f; p->sacia.max_correspondence_distance = 0.05;
  p->min_target_features = 10; p->min_target_points = 100;
  orc_icp_params_default(&p->icp);
  p->icp.max_iterations = 100; p->icp.transformation_epsilon = 1e-8; p->icp.euclidean_fitness_epsilon = 1e-8;
  p->icp.estimator = OPE_EST_NORMAL_SHOOTING; p->icp.k_search = 20;
  p->icp.n_rejectors = 2;
  p->icp.rejector_kind[0] = OPE_REJ_SURFACE_NORMAL; p->icp.rejector_threshold[0] = 0.7;
  p->icp.rejector_kind[1] = OPE_REJ_SELF_OCCLUDED_NORMAL; p->icp.rejector_threshold[1] = 0.6;
  p->icp.transformation = OPE_TE_SVD; p->icp.with_normals = 1;
  p->coarse_refit_threshold = 1e-4;
}

int orc_knn(const float* tgt, size_t nt, size_t tstride, const float* qry, size_t nq, size_t qstride, int k, int brute,
            int32_t* out_idx, float* out_d2) {
  if (!tgt || !qry || k < 1 || !out_idx) return OPE_ERR_INVALID;
  std::vector<Neighbor> nn(k);
  KdTree tree;
  if (!brute) tree.build(tgt, nt, tstride);
  for (size_t i = 0; i < nq; ++i) {
    const float* q = at(qry, qstride, i);
    int cnt = 0;
    if (!brute) cnt = tree.knn(q, k, nn.data());
    else {
      for (size_t j = 0; j < nt; ++j) {
        const float* p = at(tgt, tstride, j);
        if (!orc::finite3(p)) continue;
        Neighbor v{orc::dist2(q, p), (int32_t)j};
        if (cnt < k) { nn[cnt++] = v; std::push_heap(nn.begin(), nn.begin() + cnt); }
        else if (v < nn[0]) { std::pop_heap(nn.begin(), nn.begin() + cnt); nn[cnt - 1] = v; std::push_heap(nn.begin(), nn.begin() + cnt); }
      }
      std::sort(nn.begin(), nn.begin() + cnt);
    }
    for (int j = 0; j < k; ++j) {
      out_idx[i * k + j] = j < cnt ? nn[j].idx : -1;
      if (out_d2) out_d2[i * k + j] = j < cnt ? nn[j].d2 : INFINITY;
    }
  }
  return OPE_OK;
}

int64_t orc_radius(const float* tgt, size_t nt, size_t tstride, const float* qry, size_t nq, size_t qstride, float radius,
                   int64_t capacity, int64_t* offsets, int32_t* out_idx, float* out_d2) {
  KdTree tree; tree.build(tgt, nt, tstride);
  std::vector<Neighbor> nn;
  int64_t total = 0;
  float r2 = radius * radius;
  for (size_t i = 0; i < nq; ++i) {
    if (offsets) offsets[i] = total;
    tree.radius(at(qry, qstride, i), r2, nn);
    for (auto& v : nn) {
      if (total < capacity) { if (out_idx) out_idx[total] = v.idx; if (out_d2) out_d2[total] = v.d2; }
      ++total;
    }
  }
  if (offsets) offsets[nq] = total;
  return total;
}

int orc_feature_knn(const float* ftgt, size_t nt, const float* fqry, size_t nq, int dim, int k, int32_t* out_idx,
                    float* out_d2) {
  if (!ftgt || !fqry || k < 1 || dim < 1) return OPE_ERR_INVALID;
  std::vector<Neighbor> nn(k);
  for (size_t i = 0; i < nq; ++i) {
    int cnt;
    featureKnn(ftgt, nt, fqry + i * (size_t)dim, dim, k, nn.data(), cnt);
    for (int j = 0; j < k; ++j) {
      out_idx[i * k + j] = j < cnt ? nn[j].idx : -1;
      if (out_d2) out_d2[i * k + j] = j < cnt ? nn[j].d2 : INFINITY;
    }
  }
  return OPE_OK;
}

int orc_uniform_sample(const float* pts, size_t n, size_t stride, float leaf, int32_t* out_idx, size_t* out_n) {
  if (!pts || !out_idx || !out_n || !(leaf > 0)) return OPE_ERR_INVALID;
  std::vector<int32_t> v;
  uniformSampleImpl(pts, n, stride, leaf, v);
  std::copy(v.begin(), v.end(), out_idx);
  *out_n = v.size();
  return OPE_OK;
}

int orc_voxel_grid(const float* pts, size_t n, size_t stride, const float* rgb, float lx, float ly, float lz,
                   float* out_xyz, float* out_rgb, size_t* out_n) {
  if (!pts || !out_xyz || !out_n || !(lx > 0 && ly > 0 && lz > 0)) return OPE_ERR_INVALID;
  float inv_leaf[3] = {1.0f / lx, 1.0f / ly, 1.0f / lz};
  // overflow guard + frame, as VoxelGrid::applyFilter
  float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
  bool any = false;
  for (size_t i = 0; i < n; ++i) {
    const float* p = at(pts, stride, i);
    if (!orc::finite3(p)) continue;
    any = true;
    for (int d = 0; d < 3; ++d) { mn[d] = std::min(mn[d], p[d]); mx[d] = std::max(mx[d], p[d]); }
  }
  *out_n = 0;
  if (!any) return OPE_OK;
  int64_t dxyz[3];
  for (int d = 0; d < 3; ++d) dxyz[d] = (int64_t)((mx[d] - mn[d]) * inv_leaf[d]) + 1;
  if (dxyz[0] * dxyz[1] * dxyz[2] > (int64_t)std::numeric_limits<int32_t>::max()) return OPE_ERR_GRID_TOO_LARGE;
  VoxelFrame f = voxelFrame(pts, n, stride, inv_leaf);
  std::vector<std::pair<uint32_t, int32_t>> iv;
  iv.reserve(n);
  for (size_t i = 0; i < n; ++i) {
    const float* p = at(pts, stride, i);
    if (!orc::finite3(p)) continue;
    int ijk[3];
    for (int d = 0; d < 3; ++d) ijk[d] = (int)(std::floor(p[d] * inv_leaf[d]) - (float)f.min_b[d]);
    int idx = ijk[0] * (int)f.mul[0] + ijk[1] * (int)f.mul[1] + ijk[2] * (int)f.mul[2];
    iv.emplace_back((uint32_t)idx, (int32_t)i);
  }
  std::stable_sort(iv.begin(), iv.end(), [](const auto& a, const auto& b) { return a.first < b.first; });
  size_t m = 0, first = 0;
  while (first < iv.size()) {
    size_t last = first + 1;
    while (last < iv.size() && iv[last].first == iv[first].first) ++last;
    float c[6] = {0, 0, 0, 0, 0, 0};
    for (size_t j = first; j < last; ++j) {
      const float* p = at(pts, stride, iv[j].second);
      c[0] += p[0]; c[1] += p[1]; c[2] += p[2];
      if (rgb) {
        uint32_t u; std::memcpy(&u, &rgb[iv[j].second], 4);
        c[3] += (float)((u >> 16) & 0xff); c[4] += (float)((u >> 8) & 0xff); c[5] += (float)(u & 0xff);
      }
    }
    float cnt = (float)(last - first);
    for (int d = 0; d < 6; ++d) c[d] /= cnt;
    out_xyz[3 * m] = c[0]; out_xyz[3 * m + 1] = c[1]; out_xyz[3 * m + 2] = c[2];
    if (rgb && out_rgb) {
      int packed = ((int)c[3] << 16) | ((int)c[4] << 8) | (int)c[5];
      std::memcpy(&out_rgb[m], &packed, 4);
    }
    ++m;
    first = last;
  }
  *out_n = m;
  return OPE_OK;
}

int orc_normals_knn(const float* pts, size_t n, size_t stride, int k, const float vp[3], float* out) {
  if (!pts || !out || k < 1) return OPE_ERR_INVALID;
  float zero[3] = {0, 0, 0};
  KdTree tree; tree.build(pts, n, stride);
  normalsImpl(pts, n, stride, k, vp ? vp : zero, tree, out);
  return OPE_OK;
}

int orc_fpfh(const float* pts, size_t n, size_t stride, const float* normals, float radius, float* out) {
  if (!pts || !normals || !out) return OPE_ERR_INVALID;
  fpfhImpl(pts, n, stride, normals, radius, out);
  return OPE_OK;
}

int orc_spfh(const float* pts, size_t n, size_t stride, const float* normals, float radius, float* out) {
  if (!pts || !normals || !out) return OPE_ERR_INVALID;
  KdTree tree; tree.build(pts, n, stride);
  std::vector<float> spfh;
  computeSpfh(pts, n, stride, normals, radius, tree, spfh);
  std::copy(spfh.begin(), spfh.end(), out);
  return OPE_OK;
}

int orc_umeyama(const float* src, size_t sstride, const float* tgt, size_t tstride, const int32_t* is, const int32_t* it,
                size_t n, float T[16]) {
  if (!src || !tgt || !T || n == 0) return OPE_ERR_INVALID;
  orc::umeyama(n, [&](size_t i) { return at(src, sstride, is ? is[i] : i); },
               [&](size_t i) { return at(tgt, tstride, it ? it[i] : i); }, T, at(tgt, tstride, 0));
  return OPE_OK;
}

// 0: normal equations with order-independent double sums (canonical); 1: Householder QR of the full Jacobian (cross-check)
void orc_lm_set_route(int householder) { g_lm_route = householder ? orc::LM_ROUTE_HOUSEHOLDER : orc::LM_ROUTE_NORMAL_EQ; }

// TransformationEstimationPointToPlane[LLS]::estimateRigidTransformation over explicit index pairs (kind = OPE_TE_*)
int orc_point_to_plane(const float* src, size_t ns, size_t sstride, const float* tgt, size_t nt, size_t tstride, const float* tgt_normals4,
                       const int32_t* is, const int32_t* it, size_t n, int kind, float T[16], int32_t* lm_info /* status, nfev, iterations */) {
  if (!src || !tgt || !tgt_normals4 || !T) return OPE_ERR_INVALID;
  CloudView s{src, ns, sstride, nullptr}, t{tgt, nt, tstride, tgt_normals4};
  std::vector<ope_correspondence> corr(n);
  for (size_t i = 0; i < n; ++i) corr[i] = ope_correspondence{is ? is[i] : (int32_t)i, it ? it[i] : (int32_t)i, 0.0f};
  if (kind == OPE_TE_POINT_TO_PLANE_LLS) pointToPlaneLLS(s, t, corr, T);
  else if (kind == OPE_TE_POINT_TO_PLANE) {
    orc::LmStats st;
    pointToPlaneLM(s, t, corr, T, &st);
    if (lm_info) { lm_info[0] = st.status; lm_info[1] = st.nfev; lm_info[2] = st.iterations; }
  } else return OPE_ERR_UNSUPPORTED;
  return OPE_OK;
}

// ---- SURVEY 8f-2 groundwork (ORACLE ONLY so far: the product has no segmentation stage yet) -------------------------------
// pcl::PassThrough::applyFilter for an unorganised cloud, non-negative limits [UPSTREAM filters/impl/passthrough.hpp], as
// ProcessingPcd::getPassThrough drives it (D&L/src/processingpcd.cpp:8-41): points with a non-finite coordinate are removed, a
// point is kept iff lo <= field <= hi. field: 0 = x, 1 = y, 2 = z. Writes the kept ORIGINAL indices in ascending order.
int64_t orc_pass_through(const float* pts, size_t n, size_t stride, int field, float lo, float hi, int32_t* out_idx) {
  if (!pts || !out_idx || field < 0 || field > 2) return -1;
  int64_t m = 0;
  for (size_t i = 0; i < n; ++i) {
    const float* p = at(pts, stride, i);
    if (!orc::finite3(p)) continue;
    const float v = p[field];
    if (v < lo || v > hi) continue;
    out_idx[m++] = (int32_t)i;
  }
  return m;
}

// pcl::extractEuclideanClusters [UPSTREAM segmentation/impl/extract_clusters.hpp] as ObjectSegmentationPlane::getClusters sets it
// up (D&L/src/objectsegmentationplane.cpp:74-90: tolerance 0.05, sizes 300 .. 1e5): region growing over radiusSearch (squared
// distance < tolerance^2, FLANN semantics), a component is kept iff min_size <= size <= max_size, its indices sorted ascending;
// clusters ordered by size descending (upstream uses an unstable sort: ties are canonicalised here by the smaller first index).
// labels[i] = cluster number (0 = largest) or -1; returns the number of clusters.
int orc_euclidean_clusters(const float* pts, size_t n, size_t stride, float tolerance, int min_size, int max_size, int32_t* labels) {
  if (!pts || !labels) return -1;
  for (size_t i = 0; i < n; ++i) labels[i] = -1;
  KdTree tree; tree.build(pts, n, stride);
  std::vector<char> processed(n, 0);
  std::vector<std::vector<int32_t>> clusters;
  std::vector<Neighbor> nn;
  const float r2 = tolerance * tolerance;
  for (size_t i = 0; i < n; ++i) {
    if (processed[i] || !orc::finite3(at(pts, stride, i))) continue;
    std::vector<int32_t> q{(int32_t)i};
    processed[i] = 1;
    for (size_t h = 0; h < q.size(); ++h) {
      tree.radius(at(pts, stride, q[h]), r2, nn);
      for (const auto& v : nn)
        if (!processed[v.idx]) { processed[v.idx] = 1; q.push_back(v.idx); }
    }
    if ((int)q.size() >= min_size && (int)q.size() <= max_size) { std::sort(q.begin(), q.end()); clusters.push_back(std::move(q)); }
  }
  std::sort(clusters.begin(), clusters.end(), [](const std::vector<int32_t>& a, const std::vector<int32_t>& b) {
    return a.size() != b.size() ? a.size() > b.size() : a[0] < b[0];
  });
  for (size_t c = 0; c < clusters.size(); ++c) for (int32_t i : clusters[c]) labels[i] = (int32_t)c;
  return (int)clusters.size();
}

void orc_segment_params_default(ope_segment_params* p) {
  std::memset(p, 0, sizeof(*p));
  p->distance_threshold = 0.01; p->max_iterations = 50; p->probability = 0.99; p->hull_margin = 0.1;
  p->cluster_tolerance = 0.05f; p->min_cluster_size = 300; p->max_cluster_size = 100000;
}

int orc_segment_objects_on_plane(const float* pts, size_t n, size_t stride, const ope_segment_params* prm, int32_t* labels, float plane1[4],
                                 float plane2[4], int32_t iters[2]) {
  if (!pts || !prm || !labels) return -1;
  for (size_t i = 0; i < n; ++i) labels[i] = OPE_SEG_OUTSIDE_PRISM;
  std::vector<int32_t> inl, prism;
  float c1[4], c2[4];
  int it1 = 0, it2 = 0;
  if (!orc::planeSegment(pts, n, stride, prm->distance_threshold, prm->max_iterations, prm->probability, c1, inl, &it1)) return -1;
  float rect[4][3];
  orc::hullRectangle(pts, stride, inl, c1, prm->hull_margin, rect);
  orc::prismSelect(pts, n, stride, rect, prism);
  // cloudObjWithPlane: the prism's points, compacted (:206-213)
  std::vector<float> sub(prism.size() * 3);
  for (size_t j = 0; j < prism.size(); ++j) std::memcpy(&sub[3 * j], at(pts, stride, (size_t)prism[j]), 12);
  std::vector<int32_t> inl2;
  if (!orc::planeSegment(sub.data(), prism.size(), 3, prm->distance_threshold, prm->max_iterations, prm->probability, c2, inl2, &it2)) return -1;
  for (int32_t j : prism) labels[j] = OPE_SEG_NO_CLUSTER;
  std::vector<char> is_plane(prism.size(), 0);
  for (int32_t j : inl2) { is_plane[(size_t)j] = 1; labels[prism[(size_t)j]] = OPE_SEG_PLANE; }
  std::vector<float> rest;
  std::vector<int32_t> rest_of;
  for (size_t j = 0; j < prism.size(); ++j)
    if (!is_plane[j]) { rest.insert(rest.end(), &sub[3 * j], &sub[3 * j] + 3); rest_of.push_back(prism[j]); }
  std::vector<int32_t> cl(std::max<size_t>(rest_of.size(), 1));
  const int k = orc_euclidean_clusters(rest.data(), rest_of.size(), 3, prm->cluster_tolerance, prm->min_cluster_size, prm->max_cluster_size, cl.data());
  for (size_t j = 0; j < rest_of.size(); ++j) labels[rest_of[j]] = cl[j] >= 0 ? cl[j] : OPE_SEG_NO_CLUSTER;
  if (plane1) std::memcpy(plane1, c1, 16);
  if (plane2) std::memcpy(plane2, c2, 16);
  if (iters) { iters[0] = it1; iters[1] = it2; }
  return k < 0 ? 0 : k;
}

// DataGrabber::rgbd2Pcl / depthToMeter (D&L/src/datagrabber.cpp:9-62,121-174), Kinect / Astra branch
int64_t orc_depth_to_cloud(const uint16_t* depth, int rows, int cols, float fx, float fy, float cx, float cy, float scale, float z_max,
                           float* out_xyz) {
  int64_t n = 0;
  for (int j = 0; j < cols; ++j)
    for (int i = 0; i < rows; ++i) {
      const float raw = (float)depth[(size_t)i * cols + j];
      float X = 0, Y = 0, Z = 0;
      if (!(raw <= 0.0f)) {
        Z = raw / scale;
        X = ((float)i - cx) * Z / fx;  // p_FeatX = row index (sic)
        Y = ((float)j - cy) * Z / fy;  // p_FeatY = column index (sic)
      }
      if (Z == 0 || Z > z_max) continue;
      out_xyz[3 * n] = Y;      // cloud.x = Y
      out_xyz[3 * n + 1] = X;  // cloud.y = X
      out_xyz[3 * n + 2] = Z;
      ++n;
    }
  return n;
}

int orc_transform(const float* pts, size_t n, size_t stride, const float* normals, const float T[16], float* out_pts,
                  float* out_normals) {
  Mat4 M; std::memcpy(M.m, T, sizeof(M.m));
  for (size_t i = 0; i < n; ++i) {
    orc::xformPoint(M, at(pts, stride, i), out_pts + 3 * i);
    if (normals && out_normals) {
      orc::xformNormal(M, normals + 4 * i, out_normals + 4 * i);
      out_normals[4 * i + 3] = normals[4 * i + 3];
    }
  }
  return OPE_OK;
}

int orc_fitness(const float* src, size_t ns, size_t sstride, const float* tgt, size_t nt, size_t tstride, const float T[16],
                double max_range, double* out) {
  if (!src || !tgt || !out) return OPE_ERR_INVALID;
  KdTree tree; tree.build(tgt, nt, tstride);
  Mat4 M; std::memcpy(M.m, T, sizeof(M.m));
  *out = fitnessScore(src, ns, sstride, tree, M, max_range);
  return OPE_OK;
}

int orc_correspondences(const float* src, size_t ns, size_t sstride, const float* src_normals, const float* tgt, size_t nt,
                        size_t tstride, const float* tgt_normals, const ope_icp_params* prm, ope_correspondence* out,
                        size_t* out_n) {
  if (!src || !tgt || !prm || !out || !out_n) return OPE_ERR_INVALID;
  KdTree tree; tree.build(tgt, nt, tstride);
  CloudView s{src, ns, sstride, src_normals}, t{tgt, nt, tstride, tgt_normals};
  std::vector<ope_correspondence> corr;
  estimateCorrespondences(s, t, tree, src_normals, *prm, corr);
  applyRejectors(*prm, corr, src, sstride, src_normals, t);
  std::copy(corr.begin(), corr.end(), out);
  *out_n = corr.size();
  return OPE_OK;
}

int orc_correspondences_fixed(const float* src, size_t ns, size_t sstride, const float* tgt, size_t nt, size_t tstride,
                              const ope_icp_params* prm, ope_correspondence* fixed, size_t n_fixed, ope_correspondence* out,
                              size_t* out_n) {
  if (!src || !tgt || !prm || !out || !out_n) return OPE_ERR_INVALID;
  KdTree tree; tree.build(tgt, nt, tstride);
  CloudView s{src, ns, sstride, nullptr}, t{tgt, nt, tstride, nullptr};
  std::vector<ope_correspondence> corr;
  estimateCorrespondences(s, t, tree, nullptr, *prm, corr, fixed, n_fixed);
  std::copy(corr.begin(), corr.end(), out);
  *out_n = corr.size();
  return OPE_OK;
}

int orc_icp(const float* src, size_t ns, size_t sstride, const float* src_normals, const float* tgt, size_t nt,
            size_t tstride, const float* tgt_normals, const ope_icp_params* prm, const float guess[16], ope_reg_result* res,
            ope_correspondence* out_corr) {
  return orc_icp_fixed(src, ns, sstride, src_normals, tgt, nt, tstride, tgt_normals, prm, guess, nullptr, 0, res, out_corr);
}

int orc_icp_fixed(const float* src, size_t ns, size_t sstride, const float* src_normals, const float* tgt, size_t nt,
                  size_t tstride, const float* tgt_normals, const ope_icp_params* prm, const float guess[16],
                  ope_correspondence* fixed, size_t n_fixed, ope_reg_result* res, ope_correspondence* out_corr) {
  if (!src || !prm || !res) return OPE_ERR_INVALID;
  Mat4 I = Mat4::identity();
  std::memcpy(res->T, I.m, sizeof(I.m));
  res->converged = 0; res->state = 0; res->iterations = 0; res->n_correspondences = 0; res->last_mse = 0;
  if (!tgt || nt == 0) return OPE_ERR_EMPTY;  // Registration::initCompute: PCL_ERROR + return
  KdTree tree; tree.build(tgt, nt, tstride);
  CloudView s{src, ns, sstride, src_normals}, t{tgt, nt, tstride, tgt_normals};
  Mat4 G = I;
  if (guess) std::memcpy(G.m, guess, sizeof(G.m));
  std::vector<ope_correspondence> corr;
  int rc = icpAlign(s, t, tree, *prm, G, res, corr, fixed, n_fixed);
  if (out_corr) std::copy(corr.begin(), corr.end(), out_corr);
  return rc;
}

void orc_srand(unsigned seed) { srand(seed); }

void orc_set_eigen_model(int redux_level, int cast_vectorized) {
  orc::eigen_redux_level() = redux_level;
  orc::eigen_cast_vectorized() = cast_vectorized != 0;
}

int orc_sacia_draw(const float* src, size_t ns, size_t sstride, int iterations, int nr_samples, int k_correspondences,
                   float* min_sample_distance, int32_t* samples, int32_t* picks) {
  if (!src || !samples || !picks || !min_sample_distance) return OPE_ERR_INVALID;
  for (int it = 0; it < iterations; ++it) {
    int rc = drawSamples(src, ns, sstride, nr_samples, *min_sample_distance, samples + (size_t)it * nr_samples);
    if (rc) return rc;
    for (int s = 0; s < nr_samples; ++s) picks[(size_t)it * nr_samples + s] = getRandomIndex(k_correspondences);
  }
  return OPE_OK;
}

int orc_sacia(const float* src, size_t ns, size_t sstride, const float* fsrc, const float* tgt, size_t nt, size_t tstride,
              const float* ftgt, const ope_sacia_params* prm, const ope_rng_table* table, ope_reg_result* res,
              float* out_errors) {
  if (!src || !fsrc || !tgt || !ftgt || !prm || !res) return OPE_ERR_INVALID;
  if (nt == 0 || ns == 0) return OPE_ERR_EMPTY;
  KdTree tree; tree.build(tgt, nt, tstride);
  return saciaAlign(src, ns, sstride, fsrc, tgt, nt, tstride, ftgt, tree, *prm, table, res, out_errors);
}

// ---- PoseEstimator ------------------------------------------------------------------------------------
struct orc_pose_estimator {
  ope_pose_params prm;
  int firstTimePose = 0;
  double fitnessScoreFine = 10;
  double alignedStrength = 0.0;
  std::vector<float> alignedSource;  // n*3
  std::vector<float> cloudModel;     // n*3
  double stage[8] = {0, 0, 0, 0, 0, 0, 0, 0};
};

orc_pose_estimator* orc_pose_create(const ope_pose_params* prm) {
  auto* pe = new orc_pose_estimator();
  if (prm) pe->prm = *prm; else orc_pose_params_default(&pe->prm);
  return pe;
}
void orc_pose_destroy(orc_pose_estimator* pe) { delete pe; }
void orc_pose_stage_seconds(const orc_pose_estimator* pe, double out[8]) { std::memcpy(out, pe->stage, sizeof(pe->stage)); }

namespace {
// subSampleAndCalculateNormals, D&L/src/poseestimator.cpp:131-158
void subSampleAndNormals(orc_pose_estimator* pe, const std::vector<float>& in, float leaf, std::vector<float>& pts,
                         std::vector<float>& normals) {
  Clock c;
  std::vector<int32_t> idx;
  uniformSampleImpl(in.data(), in.size() / 3, 3, leaf, idx);
  pts.resize(idx.size() * 3);
  for (size_t i = 0; i < idx.size(); ++i) std::memcpy(&pts[3 * i], &in[3 * (size_t)idx[i]], 12);
  pe->stage[0] += c.lap();
  normals.resize(idx.size() * 4);
  float vp[3] = {0, 0, 0};
  KdTree tree; tree.build(pts.data(), idx.size(), 3);
  normalsImpl(pts.data(), idx.size(), 3, pe->prm.normal_k, vp, tree, normals.data());
  pe->stage[1] += c.lap();
}

void removeNaN(std::vector<float>& pts) {
  size_t w = 0, n = pts.size() / 3;
  for (size_t i = 0; i < n; ++i)
    if (orc::finite3(&pts[3 * i])) { if (w != i) std::memcpy(&pts[3 * w], &pts[3 * i], 12); ++w; }
  pts.resize(3 * w);
}
void removeNaNNormals(std::vector<float>& pts, std::vector<float>& normals) {
  size_t w = 0, n = pts.size() / 3;
  for (size_t i = 0; i < n; ++i)
    if (orc::finite3(&normals[4 * i])) {
      if (w != i) { std::memcpy(&pts[3 * w], &pts[3 * i], 12); std::memcpy(&normals[4 * w], &normals[4 * i], 16); }
      ++w;
    }
  pts.resize(3 * w); normals.resize(4 * w);
}
void transformAll(const std::vector<float>& in, const Mat4& T, std::vector<float>& out) {
  out.resize(in.size());
  for (size_t i = 0; i < in.size() / 3; ++i) orc::xformPoint(T, &in[3 * i], &out[3 * i]);
}
}  // namespace

int orc_pose_estimate_final(orc_pose_estimator* pe, float* source, size_t ns, const float* target, size_t nt,
                            size_t tstride, const ope_rng_table* table, ope_pose_result* res) {
  if (!pe || !source || !res) return OPE_ERR_INVALID;
  Clock total;
  std::memset(pe->stage, 0, sizeof(pe->stage));
  std::memset(res, 0, sizeof(*res));
  const ope_pose_params& P = pe->prm;
  std::vector<float> p_source(source, source + 3 * ns);
  std::vector<float> p_target(3 * nt);
  for (size_t i = 0; i < nt; ++i) std::memcpy(&p_target[3 * i], at(target, tstride, i), 12);
  if (pe->firstTimePose == 0) pe->cloudModel = p_source;  // :386-388
  pe->firstTimePose++;
  Mat4 coarse = Mat4::identity(), fine = Mat4::identity();
  // ---- COARSE (estimateCoarsePose, :16-73) ----
  if (nt != 0 && pe->fitnessScoreFine > P.coarse_refit_threshold) {
    res->ran_coarse = 1;
    std::vector<float> sp, sn, tp, tn;
    subSampleAndNormals(pe, p_source, P.coarse_leaf, sp, sn);
    subSampleAndNormals(pe, p_target, P.coarse_leaf, tp, tn);
    Clock c;
    std::vector<float> sf(sp.size() / 3 * 33), tf(tp.size() / 3 * 33);
    fpfhImpl(sp.data(), sp.size() / 3, 3, sn.data(), P.fpfh_radius, sf.data());
    fpfhImpl(tp.data(), tp.size() / 3, 3, tn.data(), P.fpfh_radius, tf.data());
    pe->stage[2] += c.lap();
    res->n_src_coarse = (int32_t)(sp.size() / 3); res->n_tgt_coarse = (int32_t)(tp.size() / 3);
    if ((int)(tp.size() / 3) < P.min_target_features) {
      pe->alignedSource = p_source;  // :41
    } else {
      ope_reg_result rr;
      KdTree tree; tree.build(tp.data(), tp.size() / 3, 3);
      int rc = saciaAlign(sp.data(), sp.size() / 3, 3, sf.data(), tp.data(), tp.size() / 3, 3, tf.data(), tree, P.sacia,
                          table, &rr, nullptr);
      if (rc) return rc;
      pe->stage[3] += c.lap();
      std::memcpy(coarse.m, rr.T, sizeof(coarse.m));
      res->sacia_best_iteration = rr.best_iteration; res->sacia_best_error = rr.best_error;
      transformAll(p_source, coarse, pe->alignedSource);  // :67-70
      pe->stage[6] += c.lap();
    }
  }
  // ---- FINE (estimateFinePose, :161-379) ----
  if (nt != 0) {
    std::vector<float> srcc = pe->alignedSource, tgtc = p_target;
    removeNaN(srcc); removeNaN(tgtc);
    std::vector<float> sp, sn, tp, tn;
    subSampleAndNormals(pe, srcc, P.fine_leaf, sp, sn);
    subSampleAndNormals(pe, tgtc, P.fine_leaf, tp, tn);
    removeNaNNormals(sp, sn); removeNaNNormals(tp, tn);
    res->n_src_fine = (int32_t)(sp.size() / 3); res->n_tgt_fine = (int32_t)(tp.size() / 3);
    if ((int)(tp.size() / 3) >= P.min_target_points) {
      Clock c;
      KdTree tree; tree.build(tp.data(), tp.size() / 3, 3);
      CloudView s{sp.data(), sp.size() / 3, 3, sn.data()}, t{tp.data(), tp.size() / 3, 3, tn.data()};
      ope_reg_result rr;
      std::vector<ope_correspondence> corr;
      icpAlign(s, t, tree, P.icp, Mat4::identity(), &rr, corr);
      pe->stage[4] += c.lap();
      std::memcpy(fine.m, rr.T, sizeof(fine.m));
      pe->fitnessScoreFine = fitnessScore(sp.data(), sp.size() / 3, 3, tree, fine, std::numeric_limits<double>::max());
      pe->stage[5] += c.lap();
      std::vector<float> moved;
      transformAll(pe->alignedSource, fine, moved);  // :358-360
      pe->alignedSource.swap(moved);
      pe->alignedStrength = (double)rr.n_correspondences / (double)((long)(sp.size() / 3) + (long)(tp.size() / 3));  // VP/icp_mod.h:249-260
      res->icp_iterations = rr.iterations; res->icp_converged = rr.converged; res->icp_state = rr.state;
      pe->stage[6] += c.lap();
    }
  }
  Mat4 pose = orc::mul(coarse, fine);  // :421 (sic: coarse * fine)
  Mat4 rigid = Mat4::identity();
  {
    Clock c;
    size_t nm = pe->cloudModel.size() / 3;
    if (nm > 0 && nm <= ns)
      orc::umeyama(nm, [&](size_t i) { return &pe->cloudModel[3 * i]; }, [&](size_t i) { return &p_source[3 * i]; }, rigid.m, &p_source[0]);
    pe->stage[6] += c.lap();
  }
  Mat4 finalPose = orc::mul(rigid, pose);  // :439
  if (pe->alignedSource.size() == 3 * ns) std::memcpy(source, pe->alignedSource.data(), 12 * ns);  // :441
  std::memcpy(res->final_pose, finalPose.m, 64); std::memcpy(res->coarse_pose, coarse.m, 64);
  std::memcpy(res->fine_pose, fine.m, 64); std::memcpy(res->rigid_model_pose, rigid.m, 64);
  res->fitness = pe->fitnessScoreFine; res->align_strength = pe->alignedStrength;
  pe->stage[7] = total.lap();
  return OPE_OK;
}

}  // extern "C"
