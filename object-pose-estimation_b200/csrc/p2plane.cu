// p2plane.cu — point-to-plane transformation estimation on the device (SURVEY 8a16 / 8f-4):
//   TransformationEstimationPointToPlaneLLS  [UPSTREAM transformation_estimation_point_to_plane_lls.hpp]
//       the default estimator of IterativeClosestPointWithNormals (VP/icp_mod.h:352-357): 6x6 normal equations, one pass;
//   TransformationEstimationPointToPlane     [UPSTREAM transformation_estimation_point_to_plane.h, ..._lm.hpp]
//       what BuildModel plugs in (BM/src/regmeshpcd.cpp:162,193): Eigen's Levenberg-Marquardt (MINPACK lmdif) over the
//       6-parameter rigid warp (WarpPointRigid6D) with a forward-difference Jacobian, residual (warp(s) - t) . n_t.
//
// Device side: ONE fused pass per Jacobian — every correspondence evaluates its residual under the 7 warps (x and x + h e_j)
// in float exactly as the reference's functor would, forms its Jacobian row (f(x + h e_j) - f(x)) / h in float, and the 21
// entries of J^T J, the 6 of J^T f and f^T f are accumulated in double (warp shuffles -> block -> one final warp per
// accumulator). The m x 6 Jacobian is never stored: 28 doubles come back to the host. A trial point costs one pass that
// returns f^T f. Host side (ope_p2plane.h): the lmdif driver works from those normal equations — the column-pivoted R of J = Q R
// is the pivoted Cholesky factor of J^T J and Q^T f = R^-T P^T J^T f — which is algebraically what Eigen's ColPivHouseholderQR
// hands to lmpar/qrsolv; the squared condition number matters only along (nearly) unobservable directions (DESIGN.md section 2).
// HBM-bound in principle (48 B per correspondence and pass), latency/launch bound at the sizes the apps use (1e3..1e5 pairs).
#include <cfloat>
#include <cmath>
#include <vector>

#include "ope_host.cuh"
#include "ope_p2plane.h"

namespace ope {

namespace {

constexpr int kP2pThreads = 256;
constexpr int kAccLls = 29;   // ATA upper triangle (21), ATb (6), pairs, sum of correspondence distances
constexpr int kAccJac = 30;   // J^T J upper triangle (21), J^T f (6), f^T f, pairs, sum of correspondence distances
constexpr int kAccF = 3;      // f^T f, pairs, sum of correspondence distances

struct P2pArgs {
  const float4* src;     // source points (by source index)
  const float4* tgt;     // target points
  const float4* tgt_n;   // target normals
  const int* is;         // n source indices or null (identity)
  const int* it;         // n target indices; < 0: no correspondence for this entry
  const float* d2;       // n correspondence distances or null
  int n;
  Mat4 W[7];             // warps: [0] at x, [1 + j] at x + h[j] e_j
  float h[6];
};

__device__ __forceinline__ double warp_sum(double v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <int NACC>
__device__ __forceinline__ void block_sum_store(double* acc, double* dst) {
  __shared__ double sm[(kP2pThreads / 32) * NACC];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int a = 0; a < NACC; ++a) acc[a] = warp_sum(acc[a]);
  if (lane == 0)
    for (int a = 0; a < NACC; ++a) sm[warp * NACC + a] = acc[a];
  __syncthreads();
  if (threadIdx.x < NACC) {
    double s = 0.0;
    for (int w = 0; w < kP2pThreads / 32; ++w) s += sm[w * NACC + threadIdx.x];
    dst[threadIdx.x] = s;
  }
}

// MODE 0: LLS normal equations; 1: LM residual norm at W[0]; 2: LM Jacobian normal equations at W[0..6]
template <int MODE>
__global__ void __launch_bounds__(kP2pThreads) p2p_accum_kernel(const P2pArgs a, double* __restrict__ partials) {
  constexpr int NACC = MODE == 0 ? kAccLls : (MODE == 1 ? kAccF : kAccJac);
  double acc[NACC];
#pragma unroll
  for (int e = 0; e < NACC; ++e) acc[e] = 0.0;
  for (int i = blockIdx.x * kP2pThreads + threadIdx.x; i < a.n; i += gridDim.x * kP2pThreads) {
    const int m = __ldg(a.it + i);
    if (m < 0) continue;
    const int si = a.is ? __ldg(a.is + i) : i;
    const float4 s = __ldg(a.src + si), t = __ldg(a.tgt + m), n = __ldg(a.tgt_n + m);
    acc[NACC - 2] += 1.0;
    if (a.d2) acc[NACC - 1] += (double)__ldg(a.d2 + i);
    if (MODE == 0) {
      if (!finite3(s.x, s.y, s.z) || !finite3(t.x, t.y, t.z) || !finite3(n.x, n.y, n.z)) continue;
      double v[6], d;
      plane_lls_row(s, t, n, v, d);
      int e = 0;
#pragma unroll
      for (int r = 0; r < 6; ++r)
#pragma unroll
        for (int c = r; c < 6; ++c) acc[e++] += v[r] * v[c];
#pragma unroll
      for (int r = 0; r < 6; ++r) acc[21 + r] += v[r] * d;
    } else if (MODE == 1) {
      const float f = plane_residual(a.W[0], s, t, n);
      acc[0] += (double)f * (double)f;
    } else {
      const float f = plane_residual(a.W[0], s, t, n);
      double J[6];
#pragma unroll
      for (int j = 0; j < 6; ++j) J[j] = (double)((plane_residual(a.W[1 + j], s, t, n) - f) / a.h[j]);
      int e = 0;
#pragma unroll
      for (int r = 0; r < 6; ++r)
#pragma unroll
        for (int c = r; c < 6; ++c) acc[e++] += J[r] * J[c];
#pragma unroll
      for (int r = 0; r < 6; ++r) acc[21 + r] += J[r] * (double)f;
      acc[27] += (double)f * (double)f;
    }
  }
  block_sum_store<NACC>(acc, partials + (size_t)blockIdx.x * NACC);
}

// one warp per accumulator, lanes stride over the blocks, fixed shuffle tree
__global__ void p2p_final_kernel(const double* __restrict__ partials, int nblocks, int nacc, double* __restrict__ out) {
  const int a = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (a >= nacc) return;
  double s = 0.0;
  for (int b = lane; b < nblocks; b += 32) s += partials[(size_t)b * nacc + a];
  s = warp_sum(s);
  if (lane == 0) out[a] = s;
}

// the sums of ope_p2plane.h's lm_minimize, reduced on the device
struct Accum {
  ope_ctx* ctx;
  P2pArgs a;
  Scratch<double> partials, out;
  int blocks = 1;
  explicit Accum(ope_ctx* c) : ctx(c), partials(c), out(c) {}
  int init() {
    blocks = (int)std::max<unsigned>(1u, std::min<unsigned>(div_up((size_t)std::max(a.n, 1), kP2pThreads), (unsigned)ctx->sm_count * 4u));
    OPE_TRY(partials.alloc((size_t)blocks * kAccJac));
    return out.alloc(kAccJac);
  }
  template <int MODE>
  int run(int nacc, const double** host) {
    p2p_accum_kernel<MODE><<<blocks, kP2pThreads, 0, ctx->stream>>>(a, partials.p);
    OPE_TRY(check_launch(ctx, "p2p_accum_kernel"));
    p2p_final_kernel<<<1, 32 * nacc, 0, ctx->stream>>>(partials.p, blocks, nacc, out.p);
    OPE_TRY(check_launch(ctx, "p2p_final_kernel"));
    void* h;
    OPE_TRY(read_back(ctx, out.p, (size_t)nacc * sizeof(double), &h));
    *host = (const double*)h;
    return OPE_OK;
  }
  int jacobian(const Mat4 W[7], const float h[6], const double** r) {
    for (int j = 0; j < 7; ++j) a.W[j] = W[j];
    for (int j = 0; j < 6; ++j) a.h[j] = h[j];
    return run<2>(kAccJac, r);
  }
  int residual(const Mat4& W, const double** r) {
    a.W[0] = W;
    return run<1>(kAccF, r);
  }
};

}  // namespace

// Estimate the rigid transform of the pairs (src[is[i]], tgt[it[i]]), it[i] >= 0, with the point-to-plane metric.
// kind = OPE_TE_POINT_TO_PLANE_LLS | OPE_TE_POINT_TO_PLANE. n_pairs / sum_d2 (sum of d2 over the pairs, for the ICP loop's MSE)
// and lm_info (status, nfev, iterations) may be null.
int point_to_plane_device(ope_ctx* ctx, const float4* src, const float4* tgt, const float4* tgt_n, const int* d_is, const int* d_it,
                          const float* d_d2, size_t n, int kind, Mat4* T, int* n_pairs, double* sum_d2, int32_t* lm_info) {
  *T = mat4_identity();
  if (n_pairs) *n_pairs = 0;
  if (sum_d2) *sum_d2 = 0.0;
  if (lm_info) lm_info[0] = lm_info[1] = lm_info[2] = 0;
  if (kind != OPE_TE_POINT_TO_PLANE_LLS && kind != OPE_TE_POINT_TO_PLANE) return fail(ctx, OPE_ERR_UNSUPPORTED, "unknown point-to-plane estimator %d", kind);
  if (!tgt_n) return fail(ctx, OPE_ERR_INVALID, "point-to-plane estimation needs target normals");
  if (n == 0) return OPE_OK;
  if (n > 0x7fffffffull) return fail(ctx, OPE_ERR_INVALID, "too many correspondences");
  Accum acc(ctx);
  acc.a.src = src; acc.a.tgt = tgt; acc.a.tgt_n = tgt_n; acc.a.is = d_is; acc.a.it = d_it; acc.a.d2 = d_d2; acc.a.n = (int)n;
  for (int j = 0; j < 7; ++j) acc.a.W[j] = mat4_identity();
  for (int j = 0; j < 6; ++j) acc.a.h[j] = 1.0f;
  OPE_TRY(acc.init());
  const double* r;
  if (kind == OPE_TE_POINT_TO_PLANE_LLS) {
    OPE_TRY(acc.run<0>(kAccLls, &r));
    if (n_pairs) *n_pairs = (int)r[27];
    if (sum_d2) *sum_d2 = r[28];
    *T = p2p::lls_transform(r);
    return OPE_OK;
  }
  // LM: the pair count first (fewer than 6 pairs: the identity, see p2p::lm_estimate)
  OPE_TRY(acc.run<1>(kAccF, &r));
  const int pairs = (int)r[1];
  if (n_pairs) *n_pairs = pairs;
  if (sum_d2) *sum_d2 = r[2];
  return p2p::lm_estimate(acc, pairs, T, lm_info);
}

}  // namespace ope
