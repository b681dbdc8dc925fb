// orc_lm.h — TEST INFRASTRUCTURE (oracle). Levenberg-Marquardt as PCL's TransformationEstimationLM drives it:
// Eigen::LevenbergMarquardt<Eigen::NumericalDiff<Functor>, float>::minimize(x) [UPSTREAM Eigen
// unsupported/NonLinearOptimization: LevenbergMarquardt.h, lmpar.h (lmpar2), qrsolv.h; NumericalDiff.h, Forward mode],
// which is MINPACK lmdif with a column-pivoted Householder QR. Parameters are Eigen's defaults: factor = 100, maxfev = 400,
// ftol = xtol = sqrt(eps_float), gtol = 0, epsfcn = 0.
//
// Arithmetic (canonicalisation, see DESIGN.md §2): the residuals, the parameter vector and the forward-difference Jacobian
// entries are float exactly as in the reference; the linear algebra on them (QR, lmpar, norms) runs in double, because
// Eigen's float reductions over m rows depend on its vectorised summation order, which nothing else can reproduce.
// Two routes to the column-pivoted R and Q^T f of J = Q R:
//   LM_ROUTE_HOUSEHOLDER  factors the full m x n Jacobian by Householder reflections, as Eigen's ColPivHouseholderQR does;
//   LM_ROUTE_NORMAL_EQ    (default, the canonical one) accumulates J^T J and J^T f in double — sums that do not depend on
//                         the order of the rows to 1e-16 — and takes R as the pivoted Cholesky factor, Q^T f = R^-T P^T J^T f.
// Where every direction of the 6 parameters is well observed they take the same steps to the same pose (within 1e-6 rad /
// 1e-7 m; tests/test_oracle.py and tests/test_gpu_transform_estimation.py::test_lm_routes_envelope check that). Where a
// direction is unobservable (pairs on one plane: rotation about its normal) or nearly so (a sphere 30 m from the origin:
// rotation about its centre; the normal equations square cond(J)), the routes may take different steps and stop at
// different points along that direction with the same residual norm. The canonical route is the second one
// because an ICP loop around LM amplifies last-bit differences of one solve (the forward-difference Jacobian of float
// residuals is noisy and LM stops at sqrt(eps_float) tolerances), so the oracle and anything compared with it must agree on
// the sums to rounding, which only order-independent accumulation gives.
#ifndef ORC_LM_H_
#define ORC_LM_H_

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <vector>

namespace orc {

enum LmStatus {
  LM_NOT_STARTED = -2, LM_RUNNING = -1, LM_IMPROPER_INPUT = 0, LM_REL_REDUCTION_TOO_SMALL = 1, LM_REL_ERROR_TOO_SMALL = 2,
  LM_REL_ERROR_AND_REDUCTION_TOO_SMALL = 3, LM_COSINUS_TOO_SMALL = 4, LM_TOO_MANY_FEV = 5, LM_FTOL_TOO_SMALL = 6,
  LM_XTOL_TOO_SMALL = 7, LM_GTOL_TOO_SMALL = 8
};

enum LmRoute { LM_ROUTE_NORMAL_EQ = 0, LM_ROUTE_HOUSEHOLDER = 1 };

struct LmStats { int status = LM_NOT_STARTED, nfev = 0, iterations = 0; double fnorm = 0; };

namespace lm_detail {

inline double norm(const double* v, int n) { double s = 0; for (int i = 0; i < n; ++i) s += v[i] * v[i]; return std::sqrt(s); }

// qrsolv [MINPACK / Eigen qrsolv.h]: given the n x n upper triangle R (row-major r[i*n+j], j >= i; the strict lower part is
// scratch), the permutation ipvt, a diagonal d and Q^T b, solve min ||A x - b||^2 + ||D x||^2. sdiag receives the diagonal of
// the triangular factor S with S^T S = P^T (A^T A + D^2) P; its strict upper part is left in the strict LOWER part of r.
inline void qrsolv(int n, double* r, const int* ipvt, const double* diag, const double* qtb, double* x, double* sdiag) {
  std::vector<double> wa(n);
  for (int j = 0; j < n; ++j) {
    for (int i = j; i < n; ++i) r[i * n + j] = r[j * n + i];
    x[j] = r[j * n + j];
    wa[j] = qtb[j];
  }
  for (int j = 0; j < n; ++j) {
    const int l = ipvt[j];
    if (diag[l] != 0.0) {
      for (int k = j; k < n; ++k) sdiag[k] = 0.0;
      sdiag[j] = diag[l];
      double qtbpj = 0.0;
      for (int k = j; k < n; ++k) {
        if (sdiag[k] == 0.0) continue;
        double c, s;
        if (std::fabs(r[k * n + k]) < std::fabs(sdiag[k])) {
          const double cot = r[k * n + k] / sdiag[k];
          s = 0.5 / std::sqrt(0.25 + 0.25 * cot * cot);
          c = s * cot;
        } else {
          const double tn = sdiag[k] / r[k * n + k];
          c = 0.5 / std::sqrt(0.25 + 0.25 * tn * tn);
          s = c * tn;
        }
        r[k * n + k] = c * r[k * n + k] + s * sdiag[k];
        const double t = c * wa[k] + s * qtbpj;
        qtbpj = -s * wa[k] + c * qtbpj;
        wa[k] = t;
        for (int i = k + 1; i < n; ++i) {
          const double u = c * r[i * n + k] + s * sdiag[i];
          sdiag[i] = -s * r[i * n + k] + c * sdiag[i];
          r[i * n + k] = u;
        }
      }
    }
    sdiag[j] = r[j * n + j];
    r[j * n + j] = x[j];
  }
  int nsing = n;
  for (int j = 0; j < n; ++j) {
    if (sdiag[j] == 0.0 && nsing == n) nsing = j;
    if (nsing < n) wa[j] = 0.0;
  }
  for (int k = 1; k <= nsing; ++k) {
    const int j = nsing - k;
    double sum = 0.0;
    for (int i = j + 1; i < nsing; ++i) sum += r[i * n + j] * wa[i];
    wa[j] = (wa[j] - sum) / sdiag[j];
  }
  for (int j = 0; j < n; ++j) x[ipvt[j]] = wa[j];
}

// lmpar2 [Eigen lmpar.h]: the Levenberg-Marquardt parameter par and the step x with ||D x|| ~ delta
inline void lmpar(int n, const double* R, int rank, const int* ipvt, const double* diag, const double* qtb, double delta,
                  double& par, double* x) {
  const double dwarf = (double)FLT_MIN;
  std::vector<double> wa1(n), wa2(n), s(n * n), sdiag(n);
  for (int j = 0; j < n; ++j) wa1[j] = j < rank ? qtb[j] : 0.0;
  for (int j = rank - 1; j >= 0; --j) {   // R(0:rank,0:rank) z = qtb
    double t = wa1[j];
    for (int i = j + 1; i < rank; ++i) t -= R[j * n + i] * wa1[i];
    wa1[j] = t / R[j * n + j];
  }
  for (int j = 0; j < n; ++j) x[ipvt[j]] = wa1[j];
  int iter = 0;
  for (int j = 0; j < n; ++j) wa2[j] = diag[j] * x[j];
  double dxnorm = norm(wa2.data(), n);
  double fp = dxnorm - delta;
  if (fp <= 0.1 * delta) { par = 0.0; return; }
  double parl = 0.0;
  if (rank == n) {
    for (int j = 0; j < n; ++j) { const int l = ipvt[j]; wa1[j] = diag[l] * (wa2[l] / dxnorm); }
    for (int j = 0; j < n; ++j) {   // R^T z = wa1
      double sum = 0.0;
      for (int i = 0; i < j; ++i) sum += R[i * n + j] * wa1[i];
      wa1[j] = (wa1[j] - sum) / R[j * n + j];
    }
    const double t = norm(wa1.data(), n);
    parl = fp / delta / t / t;
  }
  for (int j = 0; j < n; ++j) {
    double sum = 0.0;
    for (int i = 0; i <= j; ++i) sum += R[i * n + j] * qtb[i];
    wa1[j] = sum / diag[ipvt[j]];
  }
  const double gnorm = norm(wa1.data(), n);
  double paru = gnorm / delta;
  if (paru == 0.0) paru = dwarf / std::min(delta, 0.1);
  par = std::max(par, parl);
  par = std::min(par, paru);
  if (par == 0.0) par = gnorm / dxnorm;
  for (;;) {
    ++iter;
    if (par == 0.0) par = std::max(dwarf, 0.001 * paru);
    const double sq = std::sqrt(par);
    for (int j = 0; j < n; ++j) wa1[j] = sq * diag[j];
    for (int i = 0; i < n * n; ++i) s[i] = R[i];
    qrsolv(n, s.data(), ipvt, wa1.data(), qtb, x, sdiag.data());
    for (int j = 0; j < n; ++j) wa2[j] = diag[j] * x[j];
    dxnorm = norm(wa2.data(), n);
    const double temp = fp;
    fp = dxnorm - delta;
    if (std::fabs(fp) <= 0.1 * delta || (parl == 0.0 && fp <= temp && temp < 0.0) || iter == 10) break;
    for (int j = 0; j < n; ++j) { const int l = ipvt[j]; wa1[j] = diag[l] * (wa2[l] / dxnorm); }
    for (int j = 0; j < n; ++j) {
      wa1[j] /= sdiag[j];
      const double t = wa1[j];
      for (int i = j + 1; i < n; ++i) wa1[i] -= s[i * n + j] * t;
    }
    const double t = norm(wa1.data(), n);
    const double parc = fp / delta / t / t;
    if (fp > 0.0) parl = std::max(parl, par);
    if (fp < 0.0) paru = std::min(paru, par);
    par = std::max(parl, par + parc);
  }
  if (iter == 0) par = 0.0;
}

// P^T A P = R^T R for the symmetric positive semi-definite A = J^T J with the pivot rule of a column-pivoted QR (largest
// remaining column norm first, the first one on ties); qtf = R^-T P^T g
inline void pivotedCholesky(int n, const double* A, const double* g, double* R, int* ipvt, double* qtf) {
  std::vector<double> W(A, A + n * n);
  std::fill(R, R + n * n, 0.0);
  for (int j = 0; j < n; ++j) ipvt[j] = j;
  for (int k = 0; k < n; ++k) {
    int best = k;
    for (int j = k + 1; j < n; ++j) if (W[j * n + j] > W[best * n + best]) best = j;
    if (best != k) {
      for (int i = 0; i < n; ++i) std::swap(W[i * n + k], W[i * n + best]);
      for (int i = 0; i < n; ++i) std::swap(W[k * n + i], W[best * n + i]);
      for (int i = 0; i < k; ++i) std::swap(R[i * n + k], R[i * n + best]);
      std::swap(ipvt[k], ipvt[best]);
    }
    const double piv = W[k * n + k];
    if (!(piv > 0.0)) break;
    const double rkk = std::sqrt(piv);
    R[k * n + k] = rkk;
    for (int j = k + 1; j < n; ++j) R[k * n + j] = W[k * n + j] / rkk;
    for (int i = k + 1; i < n; ++i)
      for (int j = k + 1; j < n; ++j) W[i * n + j] -= R[k * n + i] * R[k * n + j];
  }
  for (int j = 0; j < n; ++j) {
    if (R[j * n + j] == 0.0) { qtf[j] = 0.0; continue; }
    double s = g[ipvt[j]];
    for (int i = 0; i < j; ++i) s -= R[i * n + j] * qtf[i];
    qtf[j] = s / R[j * n + j];
  }
}

}  // namespace lm_detail

// F: void operator()(const float* x /* n */, float* fvec /* m */).
template <class F>
LmStats lmMinimize(F& functor, int m, int n, float* x, LmRoute route = LM_ROUTE_NORMAL_EQ) {
  using namespace lm_detail;
  LmStats st;
  const double factor = 100.0, ftol = (double)std::sqrt(FLT_EPSILON), xtol = ftol, gtol = 0.0, eps_mach = (double)FLT_EPSILON;
  const int maxfev = 400;
  if (n <= 0 || m < n) { st.status = LM_IMPROPER_INPUT; return st; }
  std::vector<float> fvec(m), f1(m), f2(m), xt(n);
  std::vector<double> J((size_t)m * n), R(n * n), qtf(n), wa1(n), wa2(n), wa3(n), diag(n), colnorm(n), q(m);
  std::vector<int> ipvt(n);
  functor(x, fvec.data());
  st.nfev = 1;
  auto fnorm_of = [&](const std::vector<float>& v) { double s = 0; for (int i = 0; i < m; ++i) s += (double)v[i] * (double)v[i]; return std::sqrt(s); };
  double fnorm = fnorm_of(fvec), par = 0.0, delta = 0.0, xnorm = 0.0, gnorm = 0.0;
  int iter = 1;
  for (;;) {   // minimizeOneStep
    // NumericalDiff::df, Forward: f(x) again, then one column per parameter
    const float eps = std::sqrt(FLT_EPSILON);
    functor(x, f1.data());
    st.nfev += 1;
    for (int j = 0; j < n; ++j) {
      for (int k = 0; k < n; ++k) xt[k] = x[k];
      float h = eps * std::fabs(x[j]);
      if (h == 0.0f) h = eps;
      xt[j] = x[j] + h;
      functor(xt.data(), f2.data());
      st.nfev += 1;
      for (int i = 0; i < m; ++i) J[(size_t)j * m + i] = (double)((f2[i] - f1[i]) / h);
    }
    for (int j = 0; j < n; ++j) colnorm[j] = norm(&J[(size_t)j * m], m);
    if (route == LM_ROUTE_NORMAL_EQ) {
      std::vector<double> A(n * n), g(n);
      for (int a = 0; a < n; ++a) {
        for (int b = a; b < n; ++b) {
          double s = 0;
          for (int i = 0; i < m; ++i) s += J[(size_t)a * m + i] * J[(size_t)b * m + i];
          A[a * n + b] = A[b * n + a] = s;
        }
        double s = 0;
        for (int i = 0; i < m; ++i) s += J[(size_t)a * m + i] * (double)fvec[i];
        g[a] = s;
        colnorm[a] = std::sqrt(A[a * n + a]);
      }
      pivotedCholesky(n, A.data(), g.data(), R.data(), ipvt.data(), qtf.data());
    } else {
    // column-pivoted Householder QR of J, applied to fvec as it goes
    for (int i = 0; i < m; ++i) q[i] = (double)fvec[i];
    for (int j = 0; j < n; ++j) ipvt[j] = j;
    std::fill(R.begin(), R.end(), 0.0);
    for (int k = 0; k < n; ++k) {
      int best = k; double bn = -1.0;
      for (int j = k; j < n; ++j) {
        double s = 0; for (int i = k; i < m; ++i) s += J[(size_t)j * m + i] * J[(size_t)j * m + i];
        if (s > bn) { bn = s; best = j; }
      }
      if (best != k) {
        for (int i = 0; i < m; ++i) std::swap(J[(size_t)k * m + i], J[(size_t)best * m + i]);
        std::swap(ipvt[k], ipvt[best]);
      }
      double* a = &J[(size_t)k * m];
      double tail = 0; for (int i = k + 1; i < m; ++i) tail += a[i] * a[i];
      const double c0 = a[k];
      double beta = std::sqrt(c0 * c0 + tail);
      if (tail == 0.0) { beta = c0; }       // nothing to reflect
      else {
        if (c0 >= 0) beta = -beta;
        const double tau = (beta - c0) / beta, inv = 1.0 / (c0 - beta);
        for (int i = k + 1; i < m; ++i) a[i] *= inv;   // essential part of v (v_k = 1)
        auto reflect = [&](double* y) {                // y -= tau * v (v . y)
          double d = y[k]; for (int i = k + 1; i < m; ++i) d += a[i] * y[i];
          d *= tau;
          y[k] -= d; for (int i = k + 1; i < m; ++i) y[i] -= d * a[i];
        };
        for (int j = k + 1; j < n; ++j) reflect(&J[(size_t)j * m]);
        reflect(q.data());
      }
      a[k] = beta;
    }
    for (int i = 0; i < n; ++i) for (int j = i; j < n; ++j) R[i * n + j] = J[(size_t)j * m + i];
    for (int j = 0; j < n; ++j) qtf[j] = q[j];
    }
    int rank = 0;
    { double mx = 0; for (int j = 0; j < n; ++j) mx = std::max(mx, std::fabs(R[j * n + j]));
      const double thr = mx * eps_mach * std::min(m, n);
      for (int j = 0; j < n; ++j) if (std::fabs(R[j * n + j]) > thr) ++rank; }
    if (iter == 1) {
      for (int j = 0; j < n; ++j) diag[j] = colnorm[j] == 0.0 ? 1.0 : colnorm[j];
      for (int j = 0; j < n; ++j) wa3[j] = diag[j] * (double)x[j];
      xnorm = norm(wa3.data(), n);
      delta = factor * xnorm;
      if (delta == 0.0) delta = factor;
    }
    gnorm = 0.0;
    if (fnorm != 0.0)
      for (int j = 0; j < n; ++j)
        if (colnorm[ipvt[j]] != 0.0) {
          double s = 0; for (int i = 0; i <= j; ++i) s += R[i * n + j] * (qtf[i] / fnorm);
          gnorm = std::max(gnorm, std::fabs(s / colnorm[ipvt[j]]));
        }
    if (gnorm <= gtol) { st.status = LM_COSINUS_TOO_SMALL; break; }
    for (int j = 0; j < n; ++j) diag[j] = std::max(diag[j], colnorm[j]);
    double ratio = 0.0;
    int status = LM_RUNNING;
    do {
      lmpar(n, R.data(), rank, ipvt.data(), diag.data(), qtf.data(), delta, par, wa1.data());
      for (int j = 0; j < n; ++j) { wa1[j] = -wa1[j]; xt[j] = (float)((double)x[j] + wa1[j]); wa3[j] = diag[j] * wa1[j]; }
      const double pnorm = norm(wa3.data(), n);
      if (iter == 1) delta = std::min(delta, pnorm);
      functor(xt.data(), f2.data());
      st.nfev += 1;
      const double fnorm1 = fnorm_of(f2);
      double actred = -1.0;
      if (0.1 * fnorm1 < fnorm) actred = 1.0 - (fnorm1 / fnorm) * (fnorm1 / fnorm);
      for (int i = 0; i < n; ++i) { double s = 0; for (int j = i; j < n; ++j) s += R[i * n + j] * wa1[ipvt[j]]; wa3[i] = s; }
      const double t1 = norm(wa3.data(), n) / fnorm, t2 = std::sqrt(par) * pnorm / fnorm;
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
        for (int j = 0; j < n; ++j) { x[j] = xt[j]; wa3[j] = diag[j] * (double)x[j]; }
        fvec.swap(f2);
        xnorm = norm(wa3.data(), n);
        fnorm = fnorm1;
        ++iter;
      }
      const bool small_red = std::fabs(actred) <= ftol && prered <= ftol && 0.5 * ratio <= 1.0;
      if (small_red && delta <= xtol * xnorm) { status = LM_REL_ERROR_AND_REDUCTION_TOO_SMALL; break; }
      if (small_red) { status = LM_REL_REDUCTION_TOO_SMALL; break; }
      if (delta <= xtol * xnorm) { status = LM_REL_ERROR_TOO_SMALL; break; }
      if (st.nfev >= maxfev) { status = LM_TOO_MANY_FEV; break; }
      if (std::fabs(actred) <= eps_mach && prered <= eps_mach && 0.5 * ratio <= 1.0) { status = LM_FTOL_TOO_SMALL; break; }
      if (delta <= eps_mach * xnorm) { status = LM_XTOL_TOO_SMALL; break; }
      if (gnorm <= eps_mach) { status = LM_GTOL_TOO_SMALL; break; }
    } while (ratio < 1e-4);
    if (status != LM_RUNNING) { st.status = status; break; }
  }
  st.iterations = iter;
  st.fnorm = fnorm;
  return st;
}

}  // namespace orc
#endif  // ORC_LM_H_
