// ope_p2plane.h — the host half of the point-to-plane estimators (p2plane.cu): the 6x6 algebra that turns the sums the device
// returns into a transform. Host code only, templated on where the sums come from, so that tests/hostemu compiles the same
// driver against a serial accumulator and holds it to the oracle without a GPU.
//   LLS: solve6 + PCL's constructTransformationMatrix on the 27 sums of A^T A and A^T b;
//   LM:  Eigen::LevenbergMarquardt::minimize (MINPACK lmdif) from the normal equations J^T J, J^T f of the forward-difference
//        Jacobian — the column-pivoted R of J = Q R is the pivoted Cholesky factor of J^T J and Q^T f = R^-T P^T J^T f, which is
//        algebraically what Eigen's ColPivHouseholderQR hands to lmpar/qrsolv (DESIGN.md section 2).
#pragma once
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdint>

#include "ope_device.cuh"

namespace ope {
namespace p2p {

constexpr int N6 = 6;
inline double norm6(const double* v) { double s = 0; for (int i = 0; i < N6; ++i) s += v[i] * v[i]; return std::sqrt(s); }

// WarpPointRigid6D::setParam [UPSTREAM warp_point_rigid_6d.h], float: translation, then q = (sqrt(1 - |v|^2), v) normalised
// and Eigen's Quaternion::toRotationMatrix
inline Mat4 warp_rigid_6d(const float x[6]) {
  Mat4 M;
  for (int i = 0; i < 16; ++i) M.m[i] = 0.0f;
  M(0, 3) = x[0]; M(1, 3) = x[1]; M(2, 3) = x[2]; M(3, 3) = 1.0f;
  volatile float qq = 0.0f * 0.0f + x[3] * x[3];
  qq = qq + x[4] * x[4];
  qq = qq + x[5] * x[5];
  float qw = std::sqrt(1.0f - qq);
  volatile float nn = x[3] * x[3] + x[4] * x[4];
  nn = nn + x[5] * x[5];
  nn = nn + qw * qw;
  const float nrm = std::sqrt((float)nn);
  const float qx = x[3] / nrm, qy = x[4] / nrm, qz = x[5] / nrm;
  qw = qw / nrm;
  const float tx = 2.0f * qx, ty = 2.0f * qy, tz = 2.0f * qz;
  const float twx = tx * qw, twy = ty * qw, twz = tz * qw;
  const float txx = tx * qx, txy = ty * qx, txz = tz * qx;
  const float tyy = ty * qy, tyz = tz * qy, tzz = tz * qz;
  M(0, 0) = 1.0f - (tyy + tzz); M(0, 1) = txy - twz; M(0, 2) = txz + twy;
  M(1, 0) = txy + twz; M(1, 1) = 1.0f - (txx + tzz); M(1, 2) = tyz - twx;
  M(2, 0) = txz - twy; M(2, 1) = tyz + twx; M(2, 2) = 1.0f - (txx + tyy);
  return M;
}

// P^T (J^T J) P = R^T R with the pivot rule of a column-pivoted QR (largest remaining column norm first, first on ties);
// qtf = R^-T P^T (J^T f). Returns the numerical rank by Eigen's ColPivHouseholderQR::rank() threshold (eps_float * 6 * |R00|).
inline int pivoted_factor(const double A[36], const double g[6], double R[36], int ipvt[6], double qtf[6]) {
  double W[36];
  for (int i = 0; i < 36; ++i) { W[i] = A[i]; R[i] = 0.0; }
  for (int j = 0; j < N6; ++j) ipvt[j] = j;
  for (int k = 0; k < N6; ++k) {
    int best = k;
    for (int j = k + 1; j < N6; ++j) if (W[j * N6 + j] > W[best * N6 + best]) best = j;
    if (best != k) {
      for (int i = 0; i < N6; ++i) std::swap(W[i * N6 + k], W[i * N6 + best]);
      for (int i = 0; i < N6; ++i) std::swap(W[k * N6 + i], W[best * N6 + i]);
      for (int i = 0; i < k; ++i) std::swap(R[i * N6 + k], R[i * N6 + best]);
      std::swap(ipvt[k], ipvt[best]);
    }
    const double piv = W[k * N6 + k];
    if (!(piv > 0.0)) break;   // the remaining columns are (numerically) in the span: their R rows stay zero
    const double rkk = std::sqrt(piv);
    R[k * N6 + k] = rkk;
    for (int j = k + 1; j < N6; ++j) R[k * N6 + j] = W[k * N6 + j] / rkk;
    for (int i = k + 1; i < N6; ++i)
      for (int j = k + 1; j < N6; ++j) W[i * N6 + j] -= R[k * N6 + i] * R[k * N6 + j];
  }
  int rank = 0;
  const double thr = std::fabs(R[0]) * (double)FLT_EPSILON * N6;
  for (int j = 0; j < N6; ++j) if (std::fabs(R[j * N6 + j]) > thr) ++rank;
  for (int j = 0; j < N6; ++j) {   // R^T y = P^T g
    if (R[j * N6 + j] == 0.0) { qtf[j] = 0.0; continue; }
    double s = g[ipvt[j]];
    for (int i = 0; i < j; ++i) s -= R[i * N6 + j] * qtf[i];
    qtf[j] = s / R[j * N6 + j];
  }
  return rank;
}

// MINPACK qrsolv: min ||R P^T x - qtb||^2 + ||D x||^2 by Givens rotations; S is left in the strict lower part of r and sdiag.
// Returns nsing, the number of leading non-zero diagonal entries of S (6 unless R P^T and D leave a direction free).
inline int qrsolv6(double* r, const int* ipvt, const double* diag, const double* qtb, double* x, double* sdiag) {
  double wa[N6];
  for (int j = 0; j < N6; ++j) {
    for (int i = j; i < N6; ++i) r[i * N6 + j] = r[j * N6 + i];
    x[j] = r[j * N6 + j];
    wa[j] = qtb[j];
  }
  for (int j = 0; j < N6; ++j) {
    const int l = ipvt[j];
    if (diag[l] != 0.0) {
      for (int k = j; k < N6; ++k) sdiag[k] = 0.0;
      sdiag[j] = diag[l];
      double qtbpj = 0.0;
      for (int k = j; k < N6; ++k) {
        if (sdiag[k] == 0.0) continue;
        double c, s;
        const double rkk = r[k * N6 + k];
        if (std::fabs(rkk) < std::fabs(sdiag[k])) {
          const double ct = rkk / sdiag[k];
          s = 0.5 / std::sqrt(0.25 + 0.25 * ct * ct);
          c = s * ct;
        } else {
          const double tg = sdiag[k] / rkk;
          c = 0.5 / std::sqrt(0.25 + 0.25 * tg * tg);
          s = c * tg;
        }
        r[k * N6 + k] = c * rkk + s * sdiag[k];
        const double t = c * wa[k] + s * qtbpj;
        qtbpj = -s * wa[k] + c * qtbpj;
        wa[k] = t;
        for (int i = k + 1; i < N6; ++i) {
          const double u = c * r[i * N6 + k] + s * sdiag[i];
          sdiag[i] = -s * r[i * N6 + k] + c * sdiag[i];
          r[i * N6 + k] = u;
        }
      }
    }
    sdiag[j] = r[j * N6 + j];
    r[j * N6 + j] = x[j];
  }
  int nsing = N6;
  for (int j = 0; j < N6; ++j) {
    if (sdiag[j] == 0.0 && nsing == N6) nsing = j;
    if (nsing < N6) wa[j] = 0.0;
  }
  for (int j = nsing - 1; j >= 0; --j) {
    double sum = 0.0;
    for (int i = j + 1; i < nsing; ++i) sum += r[i * N6 + j] * wa[i];
    wa[j] = (wa[j] - sum) / sdiag[j];
  }
  for (int j = 0; j < N6; ++j) x[ipvt[j]] = wa[j];
  return nsing;
}

// What the LM driver saw on its way, for tests: the smallest numerical rank of a Jacobian and the smallest nsing of qrsolv6
struct LmTrace { int min_rank = N6, min_nsing = N6; };

// Eigen lmpar2 / MINPACK lmpar: the damping parameter for the trust region ||D p|| <= delta and the step p
inline void lmpar6(const double* R, int rank, const int* ipvt, const double* diag, const double* qtb, double delta, double& par, double* x,
                   LmTrace* trace = nullptr) {
  const double dwarf = (double)FLT_MIN;
  double wa1[N6], wa2[N6], s[36], sdiag[N6];
  for (int j = 0; j < N6; ++j) wa1[j] = j < rank ? qtb[j] : 0.0;
  for (int j = rank - 1; j >= 0; --j) {
    double t = wa1[j];
    for (int i = j + 1; i < rank; ++i) t -= R[j * N6 + i] * wa1[i];
    wa1[j] = t / R[j * N6 + j];
  }
  for (int j = 0; j < N6; ++j) x[ipvt[j]] = wa1[j];
  int iter = 0;
  for (int j = 0; j < N6; ++j) wa2[j] = diag[j] * x[j];
  double dxnorm = norm6(wa2);
  double fp = dxnorm - delta;
  if (fp <= 0.1 * delta) { par = 0.0; return; }
  double parl = 0.0;
  if (rank == N6) {
    for (int j = 0; j < N6; ++j) { const int l = ipvt[j]; wa1[j] = diag[l] * (wa2[l] / dxnorm); }
    for (int j = 0; j < N6; ++j) {
      double sum = 0.0;
      for (int i = 0; i < j; ++i) sum += R[i * N6 + j] * wa1[i];
      wa1[j] = (wa1[j] - sum) / R[j * N6 + j];
    }
    const double t = norm6(wa1);
    parl = fp / delta / t / t;
  }
  for (int j = 0; j < N6; ++j) {
    double sum = 0.0;
    for (int i = 0; i <= j; ++i) sum += R[i * N6 + j] * qtb[i];
    wa1[j] = sum / diag[ipvt[j]];
  }
  const double gnorm = norm6(wa1);
  double paru = gnorm / delta;
  if (paru == 0.0) paru = dwarf / std::min(delta, 0.1);
  par = std::min(std::max(par, parl), paru);
  if (par == 0.0) par = gnorm / dxnorm;
  for (;;) {
    ++iter;
    if (par == 0.0) par = std::max(dwarf, 0.001 * paru);
    const double sq = std::sqrt(par);
    for (int j = 0; j < N6; ++j) wa1[j] = sq * diag[j];
    for (int i = 0; i < 36; ++i) s[i] = R[i];
    const int nsing = qrsolv6(s, ipvt, wa1, qtb, x, sdiag);
    if (trace) trace->min_nsing = std::min(trace->min_nsing, nsing);
    for (int j = 0; j < N6; ++j) wa2[j] = diag[j] * x[j];
    dxnorm = norm6(wa2);
    const double prev = fp;
    fp = dxnorm - delta;
    if (std::fabs(fp) <= 0.1 * delta || (parl == 0.0 && fp <= prev && prev < 0.0) || iter == 10) break;
    for (int j = 0; j < N6; ++j) { const int l = ipvt[j]; wa1[j] = diag[l] * (wa2[l] / dxnorm); }
    for (int j = 0; j < N6; ++j) {
      wa1[j] /= sdiag[j];
      const double t = wa1[j];
      for (int i = j + 1; i < N6; ++i) wa1[i] -= s[i * N6 + j] * t;
    }
    const double t = norm6(wa1);
    const double parc = fp / delta / t / t;
    if (fp > 0.0) parl = std::max(parl, par);
    if (fp < 0.0) paru = std::min(paru, par);
    par = std::max(parl, par + parc);
  }
}

// Eigen::LevenbergMarquardt::minimize with NumericalDiff<Forward> (defaults: factor 100, maxfev 400, ftol = xtol =
// sqrt(eps_float), gtol 0). Acc supplies the sums over the pairs, with f_i the residual of pair i under a warp:
//   int jacobian(const Mat4 W[7], const float h[6], const double** r): r[0..21) the upper triangle of J^T J row by row,
//       r[21..27) J^T f, r[27] f^T f, where f is taken under W[0] and column j of J is (f under W[1 + j] - f) / h[j] in float;
//   int residual(const Mat4& W, const double** r): r[0] = f^T f under W.
// Both return OPE_OK (0) or an error code, which is passed on. info: (status, function evaluations, iterations).
template <class Acc>
int lm_minimize(Acc& acc, float x[6], int32_t info[3], LmTrace* trace = nullptr) {
  const double factor = 100.0, ftol = (double)std::sqrt(FLT_EPSILON), xtol = ftol, gtol = 0.0, eps_mach = (double)FLT_EPSILON;
  const int maxfev = 400;
  const float eps = std::sqrt(FLT_EPSILON);
  int nfev = 1, iter = 1, status = -1;
  double fnorm = 0.0, par = 0.0, delta = 0.0, xnorm = 0.0, gnorm = 0.0;
  double diag[N6], colnorm[N6], R[36], qtf[N6], wa1[N6], wa3[N6], A[36], g[N6];
  int ipvt[N6];
  float xt[N6], h[N6];
  Mat4 W[7];
  bool have_fnorm = false;
  for (;;) {
    // Jacobian by forward differences: f(x) again plus one evaluation per parameter, fused into one pass
    W[0] = warp_rigid_6d(x);
    for (int j = 0; j < N6; ++j) {
      for (int k = 0; k < N6; ++k) xt[k] = x[k];
      float hj = eps * std::fabs(x[j]);
      if (hj == 0.0f) hj = eps;
      volatile float xj = x[j] + hj;
      xt[j] = xj;
      h[j] = hj;
      W[1 + j] = warp_rigid_6d(xt);
    }
    const double* r;
    if (const int rc = acc.jacobian(W, h, &r)) return rc;
    nfev += N6 + 1;
    {
      int e = 0;
      for (int i = 0; i < N6; ++i) for (int j = i; j < N6; ++j) { A[i * N6 + j] = A[j * N6 + i] = r[e++]; }
      for (int i = 0; i < N6; ++i) g[i] = r[21 + i];
      if (!have_fnorm) { fnorm = std::sqrt(r[27]); have_fnorm = true; }   // minimizeInit's evaluation of f(x0)
    }
    for (int j = 0; j < N6; ++j) colnorm[j] = std::sqrt(A[j * N6 + j]);
    const int rank = pivoted_factor(A, g, R, ipvt, qtf);
    if (trace) trace->min_rank = std::min(trace->min_rank, rank);
    if (iter == 1) {
      for (int j = 0; j < N6; ++j) diag[j] = colnorm[j] == 0.0 ? 1.0 : colnorm[j];
      for (int j = 0; j < N6; ++j) wa3[j] = diag[j] * (double)x[j];
      xnorm = norm6(wa3);
      delta = factor * xnorm;
      if (delta == 0.0) delta = factor;
    }
    gnorm = 0.0;
    if (fnorm != 0.0)
      for (int j = 0; j < N6; ++j)
        if (colnorm[ipvt[j]] != 0.0) {
          double s = 0.0;
          for (int i = 0; i <= j; ++i) s += R[i * N6 + j] * (qtf[i] / fnorm);
          gnorm = std::max(gnorm, std::fabs(s / colnorm[ipvt[j]]));
        }
    if (gnorm <= gtol) { status = 4; break; }
    for (int j = 0; j < N6; ++j) diag[j] = std::max(diag[j], colnorm[j]);
    double ratio = 0.0;
    do {
      lmpar6(R, rank, ipvt, diag, qtf, delta, par, wa1, trace);
      for (int j = 0; j < N6; ++j) { wa1[j] = -wa1[j]; xt[j] = (float)((double)x[j] + wa1[j]); wa3[j] = diag[j] * wa1[j]; }
      const double pnorm = norm6(wa3);
      if (iter == 1) delta = std::min(delta, pnorm);
      if (const int rc = acc.residual(warp_rigid_6d(xt), &r)) return rc;
      ++nfev;
      const double fnorm1 = std::sqrt(r[0]);
      double actred = -1.0;
      if (0.1 * fnorm1 < fnorm) actred = 1.0 - (fnorm1 / fnorm) * (fnorm1 / fnorm);
      for (int i = 0; i < N6; ++i) { double s = 0.0; for (int j = i; j < N6; ++j) s += R[i * N6 + j] * wa1[ipvt[j]]; wa3[i] = s; }
      const double t1 = norm6(wa3) / fnorm, t2 = std::sqrt(par) * pnorm / fnorm;
      const double temp1 = t1 * t1, temp2 = t2 * t2;
      const double prered = temp1 + temp2 / 0.5, dirder = -(temp1 + temp2);
      ratio = prered != 0.0 ? actred / prered : 0.0;
      if (ratio <= 0.25) {
        double temp = 0.5;
        if (actred < 0.0) temp = 0.5 * dirder / (dirder + 0.5 * actred);
        if (0.1 * fnorm1 >= fnorm || temp < 0.1) temp = 0.1;
        delta = temp * std::min(delta, pnorm / 0.1);
        par /= temp;
      } else if (!(par != 0.0 && ratio < 0.75)) {
        delta = pnorm / 0.5;
        par = 0.5 * par;
      }
      if (ratio >= 1e-4) {
        for (int j = 0; j < N6; ++j) { x[j] = xt[j]; wa3[j] = diag[j] * (double)x[j]; }
        xnorm = norm6(wa3);
        fnorm = fnorm1;
        ++iter;
      }
      const bool small_red = std::fabs(actred) <= ftol && prered <= ftol && 0.5 * ratio <= 1.0;
      if (small_red && delta <= xtol * xnorm) { status = 3; break; }
      if (small_red) { status = 1; break; }
      if (delta <= xtol * xnorm) { status = 2; break; }
      if (nfev >= maxfev) { status = 5; break; }
      if (std::fabs(actred) <= eps_mach && prered <= eps_mach && 0.5 * ratio <= 1.0) { status = 6; break; }
      if (delta <= eps_mach * xnorm) { status = 7; break; }
      if (gnorm <= eps_mach) { status = 8; break; }
    } while (ratio < 1e-4);
    if (status != -1) break;
  }
  if (info) { info[0] = status; info[1] = nfev; info[2] = iter; }
  return 0;
}

// TransformationEstimationPointToPlane::estimateRigidTransformation once the pairs are counted [UPSTREAM
// transformation_estimation_lm.hpp]: fewer than 4 pairs is a PCL_ERROR; with 4 or 5, Eigen's minimizeInit refuses m < n
// (ImproperInputParameters) before any evaluation. Both leave x = 0, so the result is the identity, and info stays (0, 0, 0).
template <class Acc>
int lm_estimate(Acc& acc, int pairs, Mat4* T, int32_t info[3], LmTrace* trace = nullptr) {
  *T = mat4_identity();
  if (info) info[0] = info[1] = info[2] = 0;
  if (pairs < N6) return 0;
  float x[6] = {0, 0, 0, 0, 0, 0};
  if (const int rc = lm_minimize(acc, x, info, trace)) return rc;
  *T = warp_rigid_6d(x);
  return 0;
}

// Gaussian elimination with partial pivoting. An exactly zero pivot column returns false and leaves x as it was.
inline bool solve6(double A[36], double b[6], double x[6]) {
  for (int c = 0; c < 6; ++c) {
    int best = c;
    double bv = std::fabs(A[c * 6 + c]);
    for (int r = c + 1; r < 6; ++r) if (std::fabs(A[r * 6 + c]) > bv) { bv = std::fabs(A[r * 6 + c]); best = r; }
    if (bv == 0) return false;
    if (best != c) { for (int k = 0; k < 6; ++k) std::swap(A[c * 6 + k], A[best * 6 + k]); std::swap(b[c], b[best]); }
    for (int r = c + 1; r < 6; ++r) {
      const double f = A[r * 6 + c] / A[c * 6 + c];
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

// TransformationEstimationPointToPlaneLLS from its sums: r[0..21) the upper triangle of A^T A row by row, r[21..27) A^T b.
// PCL solves x = ATA.inverse() * ATb; where A^T A is exactly singular that is not finite, and this returns the identity instead
// (x = 0, see ope_point_to_plane in ope_cuda.h). Then constructTransformationMatrix(alpha, beta, gamma, tx, ty, tz) [UPSTREAM],
// double trigonometry rounded once.
inline Mat4 lls_transform(const double* r, bool* solved = nullptr) {
  double A[36], b[6], x[6] = {0, 0, 0, 0, 0, 0};
  int e = 0;
  for (int i = 0; i < 6; ++i) for (int j = i; j < 6; ++j) { A[i * 6 + j] = A[j * 6 + i] = r[e++]; }
  for (int i = 0; i < 6; ++i) b[i] = r[21 + i];
  const bool ok = solve6(A, b, x);
  if (solved) *solved = ok;
  const double al = x[0], be = x[1], ga = x[2];
  Mat4 M = mat4_identity();
  M(0, 0) = (float)(cos(ga) * cos(be));
  M(0, 1) = (float)(-sin(ga) * cos(al) + cos(ga) * sin(be) * sin(al));
  M(0, 2) = (float)(sin(ga) * sin(al) + cos(ga) * sin(be) * cos(al));
  M(1, 0) = (float)(sin(ga) * cos(be));
  M(1, 1) = (float)(cos(ga) * cos(al) + sin(ga) * sin(be) * sin(al));
  M(1, 2) = (float)(-cos(ga) * sin(al) + sin(ga) * sin(be) * cos(al));
  M(2, 0) = (float)(-sin(be));
  M(2, 1) = (float)(cos(be) * sin(al));
  M(2, 2) = (float)(cos(be) * cos(al));
  M(0, 3) = (float)x[3]; M(1, 3) = (float)x[4]; M(2, 3) = (float)x[5];
  return M;
}

}  // namespace p2p
}  // namespace ope
