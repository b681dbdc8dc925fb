// TEST INFRASTRUCTURE: the CPU reference of ope_normals_radius, pcl::NormalEstimation::compute with setRadiusSearch(radius).
// Built by tests/orc_radius.py with the oracle's flags (-O2, -ffp-contract=off, no fast-math) against the oracle's headers:
// orc::KdTree's radius set (d2 < radius^2, strict, the query included), sorted by (d2, index) — the order a sorted radius search
// gives, ties fixed by index — then computeMeanAndCovarianceMatrix (nine float sums, serial in that order), orc::eigen33 and the
// flip toward the viewpoint, as the oracle's pointNormal does for k-NN normals. NaN for a non-finite point or fewer than 3
// neighbours. out is n*4: nx, ny, nz, curvature.
#include <algorithm>
#include <cmath>
#include <cstddef>
#include <limits>
#include <vector>

#include "orc_kdtree.h"
#include "orc_linalg.h"

static bool point_normal(const float* pts, size_t stride, const std::vector<orc::Neighbor>& nn, const float* q, const float vp[3],
                         float out[4]) {
  const int cnt = (int)nn.size();
  if (cnt < 3) return false;
  float accu[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  for (int j = 0; j < cnt; ++j) {
    const float* p = pts + (size_t)nn[j].idx * stride;
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
  const float fc = (float)cnt;
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
  const float eig_sum = cov[0] + cov[4] + cov[8];
  const float curvature = (eig_sum != 0) ? std::fabs(ev / eig_sum) : 0.0f;
  const float vx = vp[0] - q[0], vy = vp[1] - q[1], vz = vp[2] - q[2];
  const float cos_theta = (vx * n[0] + vy * n[1] + vz * n[2]);
  if (cos_theta < 0) { n[0] *= -1; n[1] *= -1; n[2] *= -1; }
  out[0] = n[0]; out[1] = n[1]; out[2] = n[2]; out[3] = curvature;
  return true;
}

extern "C" int orc_normals_radius(const float* pts, size_t n, size_t stride, float radius, const float vp[3], float* out) {
  if (!pts || !out || !vp) return -1;
  const float nan = std::numeric_limits<float>::quiet_NaN();
  orc::KdTree tree;
  tree.build(pts, n, stride);
  const float r2 = radius * radius;
  std::vector<orc::Neighbor> nn;
  for (size_t i = 0; i < n; ++i) {
    float* o = out + 4 * i;
    const float* q = pts + i * stride;
    if (orc::finite3(q)) tree.radius(q, r2, nn); else nn.clear();
    std::sort(nn.begin(), nn.end());
    if (!point_normal(pts, stride, nn, q, vp, o)) o[0] = o[1] = o[2] = o[3] = nan;
  }
  return 0;
}
