// ope_device.cuh — device-side scalar math of the registration hot path (sm_100a).
//
// Everything is written as OPE_HD inline functions so the per-point logic can also be compiled by the
// host compiler inside tests/hostemu (logic checks without a GPU); the product only ever calls them from
// __global__ kernels. The whole library is compiled with -fmad=false and without fast-math: neighbour
// indices must be bit-exact against FLANN's L2_Simple ((dx*dx + dy*dy) + dz*dz, left to right, float32,
// no FMA — SURVEY "hard part 1").
#pragma once
#include <cfloat>
#include <cmath>
#include <cstdint>

#if defined(__CUDACC__)
#define OPE_HD __host__ __device__ __forceinline__
#include <cuda_runtime.h>
#else
#define OPE_HD inline
#ifndef OPE_HOST_FLOAT4
#define OPE_HOST_FLOAT4
struct float4 { float x, y, z, w; };
struct float3 { float x, y, z; };
static inline float4 make_float4(float x, float y, float z, float w) { return float4{x, y, z, w}; }
#endif
#endif

namespace ope {

// bit casts usable from host and device code
OPE_HD int f2i(float f) {
#if defined(__CUDA_ARCH__)
  return __float_as_int(f);
#else
  int i; __builtin_memcpy(&i, &f, 4); return i;
#endif
}
OPE_HD float i2f(int i) {
#if defined(__CUDA_ARCH__)
  return __int_as_float(i);
#else
  float f; __builtin_memcpy(&f, &i, 4); return f;
#endif
}

// ---- exact squared distance: FLANN L2_Simple order, no FMA (whole TU uses -fmad=false) ----------------
OPE_HD float dist2(float ax, float ay, float az, float bx, float by, float bz) {
  float dx = ax - bx, dy = ay - by, dz = az - bz;
  float r = dx * dx;
  r = r + dy * dy;
  r = r + dz * dz;
  return r;
}

// RN(a / d) for a launch constant d without the general division sequence: q = RN(a * RN(1/d)) is within a few ulp, and each
// Markstein step q <- RN(q + RN(a - q d) * RN(1/d)) (the residual is exact in an FMA) first makes it faithful, then correctly
// rounded. Valid away from overflow / underflow, which depth values in metres are. 5 instructions instead of ~15 and no slow
// path (depth.cu). tests/hostemu checks it exhaustively against the IEEE division for the ranges a depth image can produce.
OPE_HD float div_by_const(float a, float d, float rd) {
  float q = a * rd;
  float e = fmaf(-q, d, a);
  q = fmaf(e, rd, q);
  e = fmaf(-q, d, a);
  return fmaf(e, rd, q);
}

OPE_HD bool finite3(float x, float y, float z) { return isfinite(x) && isfinite(y) && isfinite(z); }

// (d2, idx) lexicographic "less": the canonical tie order of the oracle (SURVEY A.3).
OPE_HD bool nb_less(float d2a, int ia, float d2b, int ib) { return d2a < d2b || (d2a == d2b && ia < ib); }

// ---- 4x4 column-major (Eigen::Matrix4f) ------------------------------------------------------------------
struct Mat4 {
  float m[16];
  OPE_HD float& operator()(int r, int c) { return m[c * 4 + r]; }
  OPE_HD float operator()(int r, int c) const { return m[c * 4 + r]; }
};
OPE_HD Mat4 mat4_identity() {
  Mat4 I;
  for (int i = 0; i < 16; ++i) I.m[i] = 0.0f;
  I.m[0] = I.m[5] = I.m[10] = I.m[15] = 1.0f;
  return I;
}
OPE_HD bool mat4_is_identity(const Mat4& A) {
  for (int i = 0; i < 16; ++i)
    if (A.m[i] != ((i % 5 == 0) ? 1.0f : 0.0f)) return false;
  return true;
}
// C = A*B, each entry summed left to right in float (final_transformation_ = transformation_ * final_transformation_,
// VP/impl/icp_mod.hpp:249).
OPE_HD Mat4 mat4_mul(const Mat4& A, const Mat4& B) {
  Mat4 C;
  for (int c = 0; c < 4; ++c)
    for (int r = 0; r < 4; ++r) {
      float s = A(r, 0) * B(0, c);
      s = s + A(r, 1) * B(1, c);
      s = s + A(r, 2) * B(2, c);
      s = s + A(r, 3) * B(3, c);
      C(r, c) = s;
    }
  return C;
}
// pcl::transformPointCloud arithmetic ([UPSTREAM common/impl/transforms.hpp]; VP/impl/icp_mod.hpp:48-115).
OPE_HD void xform_point(const Mat4& T, float x, float y, float z, float& ox, float& oy, float& oz) {
  ox = T(0, 0) * x + T(0, 1) * y + T(0, 2) * z + T(0, 3);
  oy = T(1, 0) * x + T(1, 1) * y + T(1, 2) * z + T(1, 3);
  oz = T(2, 0) * x + T(2, 1) * y + T(2, 2) * z + T(2, 3);
}
OPE_HD void xform_normal(const Mat4& T, float x, float y, float z, float& ox, float& oy, float& oz) {
  ox = T(0, 0) * x + T(0, 1) * y + T(0, 2) * z;
  oy = T(1, 0) * x + T(1, 1) * y + T(1, 2) * z;
  oz = T(2, 0) * x + T(2, 1) * y + T(2, 2) * z;
}

// ---- float transcendental helpers ---------------------------------------------------------------------
// The reference calls glibc's float functions, which are correctly rounded in practice. CUDA's float
// versions are 1-2 ulp off, enough to flip an FPFH bin or a root ordering. Evaluating in double and rounding
// once reproduces glibc's result except in vanishing double-rounding cases; the op counts are tiny
// (3 per normal, 3 per point pair).
OPE_HD float atan2_f(float y, float x) { return (float)atan2((double)y, (double)x); }
OPE_HD float cos_f(float x) { return (float)cos((double)x); }
OPE_HD float sin_f(float x) { return (float)sin((double)x); }
OPE_HD float acos_f(float x) { return (float)acos((double)x); }

OPE_HD void cross3(const float a[3], const float b[3], float o[3]) {
  o[0] = a[1] * b[2] - a[2] * b[1];
  o[1] = a[2] * b[0] - a[0] * b[2];
  o[2] = a[0] * b[1] - a[1] * b[0];
}

// ---- pcl::eigen33 (smallest eigenpair of a symmetric 3x3), SURVEY A.4 ----------------------------------
OPE_HD void compute_roots2(float b, float c, float roots[3]) {
  roots[0] = 0.0f;
  float d = (float)((double)(b * b) - 4.0 * (double)c);
  if (d < 0.0f) d = 0.0f;
  float sd = sqrtf(d);
  roots[2] = 0.5f * (b + sd);
  roots[1] = 0.5f * (b - sd);
}

OPE_HD void swapf(float& a, float& b) { float t = a; a = b; b = t; }

OPE_HD void compute_roots(const float m[9], float roots[3]) {
  // symmetric: m[c*3+r]
  const float m00 = m[0], m01 = m[3], m02 = m[6], m11 = m[4], m12 = m[7], m22 = m[8];
  float c0 = m00 * m11 * m22 + 2.0f * m01 * m02 * m12 - m00 * m12 * m12 - m11 * m02 * m02 - m22 * m01 * m01;
  float c1 = m00 * m11 - m01 * m01 + m00 * m22 - m02 * m02 + m11 * m22 - m12 * m12;
  float c2 = m00 + m11 + m22;
  if (fabsf(c0) < FLT_EPSILON) {
    compute_roots2(c2, c1, roots);
    return;
  }
  const float s_inv3 = 1.0f / 3.0f;
  const float s_sqrt3 = sqrtf(3.0f);
  float c2_over_3 = c2 * s_inv3;
  float a_over_3 = (c1 - c2 * c2_over_3) * s_inv3;
  if (a_over_3 > 0.0f) a_over_3 = 0.0f;
  float half_b = 0.5f * (c0 + c2_over_3 * (2.0f * c2_over_3 * c2_over_3 - c1));
  float q = half_b * half_b + a_over_3 * a_over_3 * a_over_3;
  if (q > 0.0f) q = 0.0f;
  float rho = sqrtf(-a_over_3);
  float theta = atan2_f(sqrtf(-q), half_b) * s_inv3;
  float cos_theta = cos_f(theta);
  float sin_theta = sin_f(theta);
  roots[0] = c2_over_3 + 2.0f * rho * cos_theta;
  roots[1] = c2_over_3 - rho * (cos_theta + s_sqrt3 * sin_theta);
  roots[2] = c2_over_3 - rho * (cos_theta - s_sqrt3 * sin_theta);
  if (roots[0] >= roots[1]) swapf(roots[0], roots[1]);
  if (roots[1] >= roots[2]) {
    swapf(roots[1], roots[2]);
    if (roots[0] >= roots[1]) swapf(roots[0], roots[1]);
  }
  if (roots[0] <= 0.0f) compute_roots2(c2, c1, roots);
}

OPE_HD void eigen33(const float mat[9], float& eigenvalue, float evec[3]) {
  float scale = 0.0f;
  for (int i = 0; i < 9; ++i) scale = fmaxf(scale, fabsf(mat[i]));
  if (scale <= FLT_MIN) scale = 1.0f;
  float s[9];
  for (int i = 0; i < 9; ++i) s[i] = mat[i] / scale;
  float roots[3];
  compute_roots(s, roots);
  eigenvalue = roots[0] * scale;
  s[0] -= roots[0]; s[4] -= roots[0]; s[8] -= roots[0];
  float r0[3] = {s[0], s[3], s[6]}, r1[3] = {s[1], s[4], s[7]}, r2[3] = {s[2], s[5], s[8]};
  float v1[3], v2[3], v3[3];
  cross3(r0, r1, v1); cross3(r0, r2, v2); cross3(r1, r2, v3);
  float l1 = v1[0] * v1[0] + v1[1] * v1[1] + v1[2] * v1[2];
  float l2 = v2[0] * v2[0] + v2[1] * v2[1] + v2[2] * v2[2];
  float l3 = v3[0] * v3[0] + v3[1] * v3[1] + v3[2] * v3[2];
  float vx, vy, vz, l;
  if (l1 >= l2 && l1 >= l3) { vx = v1[0]; vy = v1[1]; vz = v1[2]; l = l1; }
  else if (l2 >= l1 && l2 >= l3) { vx = v2[0]; vy = v2[1]; vz = v2[2]; l = l2; }
  else { vx = v3[0]; vy = v3[1]; vz = v3[2]; l = l3; }
  float n = sqrtf(l);
  evec[0] = vx / n; evec[1] = vy / n; evec[2] = vz / n;
}

// ---- 3x3 SVD (one-sided Jacobi) and the Umeyama tail, SURVEY A.7 ---------------------------------------
template <typename T> OPE_HD T t_sqrt(T x);
template <> OPE_HD float t_sqrt<float>(float x) { return sqrtf(x); }
template <> OPE_HD double t_sqrt<double>(double x) { return sqrt(x); }
template <typename T> OPE_HD T t_abs(T x) { return x < 0 ? -x : x; }
template <typename T> struct t_consts;
template <> struct t_consts<float> {
  static OPE_HD float jac_eps() { return 4.76837158e-7f; }  // 2^-21: above the float rounding floor of the test
  static OPE_HD float tiny_rel() { return 1e-6f; }
  static OPE_HD float dummy_precision() { return 1e-5f; }
};
template <> struct t_consts<double> {
  static OPE_HD double jac_eps() { return 1e-15; }
  static OPE_HD double tiny_rel() { return 1e-13; }
  static OPE_HD double dummy_precision() { return 1e-12; }
};

// One-sided Jacobi rotation of the column pair (ap, aq) of A and the matching columns (vp, vq) of V. Returns whether it rotated.
// Every index is a compile-time constant after inlining, so A and V live in registers (a dynamically indexed local array
// would put the whole 3x3 state in local memory and make every access of this serial section an L1 round trip).
template <typename T>
OPE_HD bool svd3_rotate(T* ap, T* aq, T* vp, T* vq, T eps2) {
  const T alpha = ap[0] * ap[0] + ap[1] * ap[1] + ap[2] * ap[2];
  const T beta = aq[0] * aq[0] + aq[1] * aq[1] + aq[2] * aq[2];
  const T gamma = ap[0] * aq[0] + ap[1] * aq[1] + ap[2] * aq[2];
  if (gamma == 0 || gamma * gamma <= eps2 * (alpha * beta)) return false;  // sqrt-free relative test
  const T zeta = (beta - alpha) / (2 * gamma);
  const T t = (zeta >= 0 ? (T)1 : (T)-1) / (t_abs(zeta) + t_sqrt<T>(1 + zeta * zeta));
  const T c = 1 / t_sqrt<T>(1 + t * t);
  const T s = c * t;
#ifdef __CUDA_ARCH__
#pragma unroll
#endif
  for (int i = 0; i < 3; ++i) {
    const T x = ap[i], y = aq[i];
    ap[i] = c * x - s * y; aq[i] = s * x + c * y;
    const T vx = vp[i], vy = vq[i];
    vp[i] = c * vx - s * vy; vq[i] = s * vx + c * vy;
  }
  return true;
}
// exchange columns i and j (of A, V and the norms) when the later one is strictly larger
template <typename T>
OPE_HD void svd3_order(T* ni, T* nj, T* ai, T* aj, T* vi, T* vj) {
  if (*nj > *ni) {
    T t = *ni; *ni = *nj; *nj = t;
#ifdef __CUDA_ARCH__
#pragma unroll
#endif
    for (int k = 0; k < 3; ++k) { t = ai[k]; ai[k] = aj[k]; aj[k] = t; t = vi[k]; vi[k] = vj[k]; vj[k] = t; }
  }
}

template <typename T>
OPE_HD void svd3(const T Ain[9], T U[9], T S[3], T V[9]) {
  T A[9];
#ifdef __CUDA_ARCH__
#pragma unroll
#endif
  for (int i = 0; i < 9; ++i) { A[i] = Ain[i]; V[i] = 0; }
  V[0] = V[4] = V[8] = 1;
  const T eps2 = t_consts<T>::jac_eps() * t_consts<T>::jac_eps();
  for (int sweep = 0; sweep < 15; ++sweep) {
    bool rotated = svd3_rotate<T>(A + 0, A + 3, V + 0, V + 3, eps2);   // (p, q) = (0, 1), (0, 2), (1, 2)
    rotated = svd3_rotate<T>(A + 0, A + 6, V + 0, V + 6, eps2) || rotated;
    rotated = svd3_rotate<T>(A + 3, A + 6, V + 3, V + 6, eps2) || rotated;
    if (!rotated) break;
  }
  // singular values = column norms, sorted descending by the exchanges (0,1), (0,2), (1,2) (strict >: ties keep their order)
#ifdef __CUDA_ARCH__
#pragma unroll
#endif
  for (int j = 0; j < 3; ++j) S[j] = t_sqrt<T>(A[3 * j] * A[3 * j] + A[3 * j + 1] * A[3 * j + 1] + A[3 * j + 2] * A[3 * j + 2]);
  svd3_order<T>(S + 0, S + 1, A + 0, A + 3, V + 0, V + 3);
  svd3_order<T>(S + 0, S + 2, A + 0, A + 6, V + 0, V + 6);
  svd3_order<T>(S + 1, S + 2, A + 3, A + 6, V + 3, V + 6);
#ifdef __CUDA_ARCH__
#pragma unroll
#endif
  for (int i = 0; i < 9; ++i) U[i] = A[i];
  const T tiny = S[0] * t_consts<T>::tiny_rel();
  if (S[0] > 0) { U[0] /= S[0]; U[1] /= S[0]; U[2] /= S[0]; }
  else { U[0] = 1; U[1] = 0; U[2] = 0; }
  if (S[1] > tiny) { U[3] /= S[1]; U[4] /= S[1]; U[5] /= S[1]; }
  else {
    int k = 0;
    if (t_abs(U[1]) < t_abs(U[k == 0 ? 0 : 1])) k = 1;
    if (t_abs(U[2]) < t_abs(k == 0 ? U[0] : U[1])) k = 2;
    const T d = k == 0 ? U[0] : (k == 1 ? U[1] : U[2]);
    const T w0 = (k == 0 ? (T)1 : (T)0) - d * U[0], w1 = (k == 1 ? (T)1 : (T)0) - d * U[1], w2 = (k == 2 ? (T)1 : (T)0) - d * U[2];
    const T n = t_sqrt<T>(w0 * w0 + w1 * w1 + w2 * w2);
    U[3] = w0 / n; U[4] = w1 / n; U[5] = w2 / n;
  }
  if (S[2] > tiny) { U[6] /= S[2]; U[7] /= S[2]; U[8] /= S[2]; }
  else {
    U[6] = U[1] * U[5] - U[2] * U[4];
    U[7] = U[2] * U[3] - U[0] * U[5];
    U[8] = U[0] * U[4] - U[1] * U[3];
  }
}

template <typename T>
OPE_HD T det3(const T m[9]) {
  return m[0] * (m[4] * m[8] - m[7] * m[5]) - m[3] * (m[1] * m[8] - m[7] * m[2]) + m[6] * (m[1] * m[5] - m[4] * m[2]);
}

// sigma = 1/n * dst_demean * src_demean^T (col-major); Eigen::umeyama(with_scaling = false) incl. rank-2 branch.
template <typename T>
OPE_HD void umeyama_from_sigma(const T sigma[9], const T src_mean[3], const T dst_mean[3], Mat4& out) {
  T U[9], S[3], V[9];
  svd3<T>(sigma, U, S, V);
  T Sd[3] = {1, 1, 1};
  if (det3<T>(sigma) < 0) Sd[2] = -1;
  int rank = 0;
  const T prec = t_consts<T>::dummy_precision();
  for (int i = 0; i < 3; ++i)
    if (!(t_abs(S[i]) <= t_abs(S[0]) * prec)) ++rank;
  if (rank == 2) {
    if (det3<T>(U) * det3<T>(V) > 0) Sd[2] = 1;
    else Sd[2] = -1;
  }
  T R[9];
  for (int c = 0; c < 3; ++c)
    for (int r = 0; r < 3; ++r) {
      T s = U[0 * 3 + r] * Sd[0] * V[0 * 3 + c];
      s = s + U[1 * 3 + r] * Sd[1] * V[1 * 3 + c];
      s = s + U[2 * 3 + r] * Sd[2] * V[2 * 3 + c];
      R[c * 3 + r] = s;
    }
  for (int i = 0; i < 16; ++i) out.m[i] = 0.0f;
  out.m[15] = 1.0f;
  for (int c = 0; c < 3; ++c)
    for (int r = 0; r < 3; ++r) out.m[c * 4 + r] = (float)R[c * 3 + r];
  for (int r = 0; r < 3; ++r) {
    T rs = R[0 * 3 + r] * src_mean[0];
    rs = rs + R[1 * 3 + r] * src_mean[1];
    rs = rs + R[2 * 3 + r] * src_mean[2];
    out.m[12 + r] = (float)(dst_mean[r] - rs);
  }
}

// Umeyama from raw double moments (every Umeyama of the library: SAC-IA's 5 pairs, ICP, the dense model fit):
// acc = {n, Ss[3], St[3], Sts[9] (t_r*s_c at [c*3+r])}. Means and the cross-covariance are formed in double (the sums
// are order-independent to ~1e-16, so a parallel reduction and a serial loop agree after rounding), the 3x3 SVD runs in
// float like Eigen::JacobiSVD<Matrix3f> does in the reference, the translation is closed in double and rounded once.
// The part after the means and the float cross-covariance are known (split out so that a kernel can form them with one
// division per lane instead of fifteen in a row; the arithmetic is identical).
OPE_HD void umeyama_from_sigma_means(const float sigma[9], const double ms[3], const double mt[3], Mat4& out) {
  float U[9], S[3], V[9];
  svd3<float>(sigma, U, S, V);
  float Sd[3] = {1, 1, 1};
  if (det3<float>(sigma) < 0) Sd[2] = -1;
  int rank = 0;
  for (int i = 0; i < 3; ++i)
    if (!(t_abs(S[i]) <= t_abs(S[0]) * t_consts<float>::dummy_precision())) ++rank;
  if (rank == 2) Sd[2] = (det3<float>(U) * det3<float>(V) > 0) ? 1.0f : -1.0f;
  float R[9];
  for (int c = 0; c < 3; ++c)
    for (int r = 0; r < 3; ++r) {
      float s = U[0 * 3 + r] * Sd[0] * V[0 * 3 + c];
      s = s + U[1 * 3 + r] * Sd[1] * V[1 * 3 + c];
      s = s + U[2 * 3 + r] * Sd[2] * V[2 * 3 + c];
      R[c * 3 + r] = s;
    }
  for (int i = 0; i < 16; ++i) out.m[i] = 0.0f;
  out.m[15] = 1.0f;
  for (int c = 0; c < 3; ++c)
    for (int r = 0; r < 3; ++r) out.m[c * 4 + r] = R[c * 3 + r];
  for (int r = 0; r < 3; ++r) {
    double rs = (double)R[0 * 3 + r] * ms[0];
    rs = rs + (double)R[1 * 3 + r] * ms[1];
    rs = rs + (double)R[2 * 3 + r] * ms[2];
    out.m[12 + r] = (float)(mt[r] - rs);
  }
}
// acc: raw moments of the pairs RELATIVE TO `origin` (n, sum s', sum t', sum t' s'^T with s' = s - origin, t' = t - origin). The
// cross-covariance does not depend on the origin, but its float rounding does: sum t s^T / n - mu_t mu_s^T cancels ~3 digits for a
// 10 cm object at 1 m, which multiplies the 1e-16 summation-order noise of the double sums by 10^3 before the rounding to float;
// taken about a point of the cloud itself it cancels ~1 digit. The means are shifted back for the translation.
OPE_HD void umeyama_from_moments(const double* acc, Mat4& out, double ox = 0.0, double oy = 0.0, double oz = 0.0) {
  const double n = acc[0];
  double ms[3], mt[3];
  float sigma[9];
  for (int k = 0; k < 3; ++k) { ms[k] = acc[1 + k] / n; mt[k] = acc[4 + k] / n; }
  for (int c = 0; c < 3; ++c)
    for (int r = 0; r < 3; ++r) sigma[c * 3 + r] = (float)(acc[7 + c * 3 + r] / n - mt[r] * ms[c]);
  ms[0] += ox; ms[1] += oy; ms[2] += oz;
  mt[0] += ox; mt[1] += oy; mt[2] += oz;
  umeyama_from_sigma_means(sigma, ms, mt, out);
}
// the common origin of a moment accumulation: the first point of the TARGET cloud (0 when it is not finite)
OPE_HD void moment_origin(float x, float y, float z, double& ox, double& oy, double& oz) {
  const bool fin = isfinite(x) && isfinite(y) && isfinite(z);
  ox = fin ? (double)x : 0.0; oy = fin ? (double)y : 0.0; oz = fin ? (double)z : 0.0;
}

// Eigen::umeyama in float over a handful of pairs, sequential order (SAC-IA: 5 samples). s/d: n*3 arrays.
OPE_HD void umeyama_small(const float* s, const float* d, int n, Mat4& out) {
  const float one_over_n = 1.0f / (float)n;
  float sm[3] = {0, 0, 0}, dm[3] = {0, 0, 0};
  for (int i = 0; i < n; ++i)
    for (int k = 0; k < 3; ++k) { sm[k] += s[3 * i + k]; dm[k] += d[3 * i + k]; }
  for (int k = 0; k < 3; ++k) { sm[k] *= one_over_n; dm[k] *= one_over_n; }
  float sigma[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  for (int i = 0; i < n; ++i) {
    float sd[3] = {s[3 * i] - sm[0], s[3 * i + 1] - sm[1], s[3 * i + 2] - sm[2]};
    float dd[3] = {d[3 * i] - dm[0], d[3 * i + 1] - dm[1], d[3 * i + 2] - dm[2]};
    for (int c = 0; c < 3; ++c)
      for (int r = 0; r < 3; ++r) sigma[c * 3 + r] += dd[r] * sd[c];
  }
  for (int i = 0; i < 9; ++i) sigma[i] *= one_over_n;
  umeyama_from_sigma<float>(sigma, sm, dm, out);
}

// ---- pcl::computePairFeatures + the FPFH binning, SURVEY A.5 --------------------------------------------
// Returns the three bin indices (each in [0, 11)). Degenerate pairs are binned with f1 = f2 = f3 = 0 because
// FPFHEstimation's wrapper ignores the free function's return value.
// Eigen's 4-component dot of PCL's Vector4f map with w = 0, summed as (x + y) + (z + 0): the "+ 0" turns a -0 into +0, and the
// sign of a zero decides atan2(+-0, x) = +-pi (the first or the last f1 bin) and atan2(0, +-0)
OPE_HD float dot3w0(const float a[3], const float b[3]) { return (a[0] * b[0] + a[1] * b[1]) + (a[2] * b[2] + 0.0f); }
OPE_HD void pair_feature_bins(float p1x, float p1y, float p1z, const float n1[3], float p2x, float p2y, float p2z,
                              const float n2[3], int& h1, int& h2, int& h3) {
  float dp[3] = {p2x - p1x, p2y - p1y, p2z - p1z};
  float f1 = 0.0f, f2 = 0.0f, f3 = 0.0f;
  float f4 = sqrtf(dp[0] * dp[0] + dp[1] * dp[1] + dp[2] * dp[2]);
  if (f4 != 0.0f) {
    float a[3] = {n1[0], n1[1], n1[2]}, b[3] = {n2[0], n2[1], n2[2]};
    float angle1 = dot3w0(a, dp) / f4;
    float angle2 = dot3w0(b, dp) / f4;
    if (acos_f(fabsf(angle1)) > acos_f(fabsf(angle2))) {
      for (int k = 0; k < 3; ++k) { float t = a[k]; a[k] = b[k]; b[k] = t; dp[k] *= -1; }
      f3 = -angle2;
    } else {
      f3 = angle1;
    }
    float v[3];
    cross3(dp, a, v);
    float v_norm = sqrtf(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
    if (v_norm == 0.0f) {
      f1 = f2 = f3 = 0.0f;
    } else {
      v[0] /= v_norm; v[1] /= v_norm; v[2] /= v_norm;
      float w[3];
      cross3(a, v, w);
      f2 = dot3w0(v, b);
      f1 = atan2_f(dot3w0(w, b), dot3w0(a, b));
    }
  }
  const float d_pi = 1.0f / (2.0f * (float)3.14159265358979323846);
  h1 = (int)floor(11 * (((double)f1 + 3.14159265358979323846) * (double)d_pi));
  h2 = (int)floor(11 * (((double)f2 + 1.0) * 0.5));
  h3 = (int)floor(11 * (((double)f3 + 1.0) * 0.5));
  h1 = h1 < 0 ? 0 : (h1 > 10 ? 10 : h1);
  h2 = h2 < 0 ? 0 : (h2 > 10 ? 10 : h2);
  h3 = h3 < 0 ? 0 : (h3 > 10 ? 10 : h3);
}

// ---- normal from a sorted neighbour list: computeMeanAndCovarianceMatrix + solvePlaneParameters + flip ----
struct CovAccum {
  float a[9];
  OPE_HD void reset() { for (int i = 0; i < 9; ++i) a[i] = 0.0f; }
  OPE_HD void add(float x, float y, float z) {
    a[0] += x * x; a[1] += x * y; a[2] += x * z; a[3] += y * y; a[4] += y * z; a[5] += z * z;
    a[6] += x; a[7] += y; a[8] += z;
  }
};
OPE_HD void normal_from_accum(const CovAccum& in, int cnt, float qx, float qy, float qz, float vpx, float vpy, float vpz,
                              float out[4]) {
  float accu[9];
  float fc = (float)cnt;
  for (int i = 0; i < 9; ++i) accu[i] = in.a[i] / fc;
  float cov[9];
  cov[0] = accu[0] - accu[6] * accu[6];
  cov[1] = accu[1] - accu[6] * accu[7];
  cov[2] = accu[2] - accu[6] * accu[8];
  cov[4] = accu[3] - accu[7] * accu[7];
  cov[5] = accu[4] - accu[7] * accu[8];
  cov[8] = accu[5] - accu[8] * accu[8];
  cov[3] = cov[1]; cov[6] = cov[2]; cov[7] = cov[5];
  float ev, n[3];
  eigen33(cov, ev, n);
  float eig_sum = cov[0] + cov[4] + cov[8];
  float curvature = (eig_sum != 0) ? fabsf(ev / eig_sum) : 0.0f;
  float vx = vpx - qx, vy = vpy - qy, vz = vpz - qz;
  float cos_theta = (vx * n[0] + vy * n[1] + vz * n[2]);
  if (cos_theta < 0) { n[0] *= -1; n[1] *= -1; n[2] *= -1; }
  out[0] = n[0]; out[1] = n[1]; out[2] = n[2]; out[3] = curvature;
}

}  // namespace ope
