// track.cu — ope_pose_tracker_step_batch: many independent trackers advanced by one frame each, the steady-state loop of
// PoseEstimator::estimateFinalPose (D&L/src/poseestimator.cpp:383-448) batched across sequences. The stages are the frame-spanning
// launches of ope_pose_batch (batch.cu) with a per-frame source:
//
//   target UniformSampling 1 cm + 8 mm, normals, FPFH      as ope_pose_batch
//   source UniformSampling 1 cm, normals, FPFH             re-coarse trackers (last fine fitness above the threshold), own source
//   SAC-IA decision tables                                 drawn in tracker order (a turnstile across the chunks), or replayed
//   feature k-NN, SAC-IA                                   per-frame source descriptors and points
//   fine stage                                             coarse(source) at 8 mm, or the tracker's alignedSource (tracking)
//   track_commit_kernel                                    new alignedSource, the copy that replaces the source, dense Umeyama
//
// Trackers outside the fast path's envelope (other parameters, empty or tiny targets, clouds beyond the shared-memory capacities)
// run ope_pose_estimate_final_device one at a time afterwards, with the table drawn for them at their turn.
#include <algorithm>
#include <atomic>
#include <cstring>
#include <set>
#include <thread>
#include <vector>

#include "ope_host.cuh"

namespace ope {
namespace {

template <typename T>
int download(ope_ctx* ctx, const T* d, size_t n, std::vector<T>& h) {
  h.resize(n);
  if (n == 0) return OPE_OK;
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(h.data(), d, n * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
  OPE_CUDA_TRY(ctx, stream_sync(ctx));
  return OPE_OK;
}

// one tracker of the call
struct Step {
  ope_pose_tracker* t;
  ope_cloud* src;                  // *sources[i]
  int fast = 0;                    // on the frame-spanning path
  int recoarse = 0;                // runs SAC-IA (fitness above the threshold)
  ope_cloud* model = nullptr;      // cloudModel after this call's first-call clone (owned by the call until committed)
  bool model_fresh = false;
  ope_cloud* new_aligned = nullptr;
  ope_cloud* new_source = nullptr;
  // the decision table: given, or drawn at the tracker's turn
  const ope_rng_table* table = nullptr;
  std::vector<int32_t> ds, dp;
  ope_rng_table drawn{};
  // filled in by the chunk when the tracker finished on the fast path
  int done = 0;
  double fitness = 0, strength = 0;
  ope_pose_result result;
};

struct Call {
  const ope_pose_params* P;
  Step* steps;
  const ope_frame_input* targets;
  bool draw;                                   // tables == NULL: draw from libc rand() in tracker order
  std::atomic<size_t> turn{0};                 // the chunk whose trackers draw next
  const std::atomic<int>* failed;
};

size_t target_size(const ope_frame_input& in) { return in.points ? in.n : (in.cloud ? ((const ope_cloud*)in.cloud)->n : 0); }

// Draws the table of a tracker that leaves the fast path, if the single call would draw one: the same tests as
// ope_pose_estimate_final_device, on the tracker's own parameters, through the single-frame sampling.
int draw_for_per_tracker(ope_ctx* c, Step& st, const ope_frame_input& in) {
  const ope_pose_params& P = st.t->prm;
  if (target_size(in) == 0 || !(st.t->fitnessScoreFine > P.coarse_refit_threshold)) return OPE_OK;
  auto sample_count = [&](ope_cloud* cl, int** idx, size_t* m) { return uniform_sample_device(c, cl, P.coarse_leaf, idx, m); };
  ope_cloud* tc = nullptr;
  if (in.points) OPE_TRY(ope_cloud_upload(c, in.points, in.n, in.stride, in.offset, nullptr, 0, 0, &tc));
  else {
    ope_cloud view = *(const ope_cloud*)in.cloud;
    view.normals = nullptr; view.grids.clear(); view.bbox_valid = false;
    OPE_TRY(cloud_alloc(c, view.n, false, &tc));
    OPE_CUDA_TRY(c, cudaMemcpyAsync(tc->pts, view.pts, view.n * sizeof(float4), cudaMemcpyDeviceToDevice, c->stream));
  }
  int* idx = nullptr;
  size_t m = 0;
  int rc = sample_count(tc, &idx, &m);
  dfree(c, idx);
  ope_cloud_free(c, tc);
  OPE_TRY(rc);
  if ((int)m < P.min_target_features) return OPE_OK;
  ope_cloud view = *st.src;   // the source sample (1 cm) whose coordinates selectSamples reads
  view.ctx = c; view.normals = nullptr; view.grids.clear(); view.bbox_valid = false;
  rc = sample_count(&view, &idx, &m);
  ope_cloud* sp = nullptr;
  if (rc == OPE_OK) rc = gather_cloud(c, &view, idx, m, &sp);
  dfree(c, idx);
  ope_cloud_invalidate(c, &view);   // whatever the view cached is this call's
  OPE_TRY(rc);
  const int H = P.sacia.max_iterations, S = P.sacia.nr_samples, K = P.sacia.k_correspondences;
  std::vector<float> xyz(3 * std::max<size_t>(m, 1));
  rc = ope_cloud_download(c, sp, xyz.data(), nullptr);
  ope_cloud_free(c, sp);
  OPE_TRY(rc);
  if (m == 0 || (size_t)S > m || H < 1 || S < 1) return OPE_OK;   // the single call fails before it draws
  st.ds.resize((size_t)H * S); st.dp.resize((size_t)H * S);
  float msd = P.sacia.min_sample_distance;
  OPE_TRY(ope_sacia_draw(xyz.data(), m, 12, H, S, K, &msd, st.ds.data(), st.dp.data()));
  st.drawn = ope_rng_table{H, S, st.ds.data(), st.dp.data()};
  st.table = &st.drawn;
  return OPE_OK;
}

// chunk k's turn to draw: wait() until the chunks before it have drawn, pass() to the next one; a chunk that leaves early still
// passes the turn on (after its own turn has come), so that no later chunk waits forever
struct Turn {
  Call& call; size_t k; bool passed = false;
  Turn(Call& c, size_t kk) : call(c), k(kk) {}
  void wait() { while (call.turn.load(std::memory_order_acquire) != k) sched_yield(); }
  void pass() { if (!passed) { call.turn.store(k + 1, std::memory_order_release); passed = true; } }
  ~Turn() { if (call.draw && !passed) { wait(); pass(); } }
};

int track_chunk(ope_ctx* ctx, Call& call, size_t f0, int B, size_t k) {
  const ope_pose_params& P = *call.P;
  const int H = P.sacia.max_iterations, S = P.sacia.nr_samples, K = P.sacia.k_correspondences;
  Step* st = call.steps + f0;
  Turn turn(call, k);
  // ---- targets: staged, sampled at 1 cm and 8 mm ----
  std::vector<int> h_off, h_cnt, h_active((size_t)B), h_re((size_t)B);
  for (int i = 0; i < B; ++i) h_active[(size_t)i] = st[i].fast;
  Scratch<float4> clusters(ctx), sampled(ctx), normals(ctx), compacted(ctx), cnormals(ctx);
  Scratch<const float4*> d_tsrc(ctx), d_ssrc(ctx);
  Scratch<int> d_cnt(ctx), d_scnt(ctx), d_active(ctx), d_re(ctx), d_counts(ctx), d_ccounts(ctx), d_flags(ctx), d_samples(ctx), d_picks(ctx), d_knn(ctx);
  Scratch<float> spfh(ctx), fpfh(ctx), sspfh(ctx), sfpfh(ctx), errors(ctx), transforms(ctx);
  Scratch<ope_reg_result> d_coarse(ctx);
  size_t total = 0;
  OPE_TRY(stage_frames(ctx, call.targets + f0, B, h_active, h_off, h_cnt, clusters, d_tsrc, &total));
  const size_t slab = (size_t)B * kBCap;
  OPE_TRY(sampled.alloc(3 * slab)); OPE_TRY(normals.alloc(3 * slab)); OPE_TRY(compacted.alloc(3 * slab)); OPE_TRY(cnormals.alloc(3 * slab));
  OPE_TRY(d_cnt.alloc(B)); OPE_TRY(d_scnt.alloc(B)); OPE_TRY(d_active.alloc(B)); OPE_TRY(d_re.alloc(B)); OPE_TRY(d_counts.alloc(3 * (size_t)B));
  OPE_TRY(d_ccounts.alloc(3 * (size_t)B)); OPE_TRY(d_flags.alloc(B)); OPE_TRY(d_ssrc.alloc(B)); OPE_TRY(d_coarse.alloc(B));
  std::vector<int> h_counts((size_t)2 * B, 0), h_scount((size_t)B, 0);
  if (!total) std::fill(h_active.begin(), h_active.end(), 0);
  if (total) {
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_cnt.p, h_cnt.data(), B * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_active.p, h_active.data(), B * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    OPE_CUDA_TRY(ctx, cudaMemsetAsync(d_flags.p, 0, B * sizeof(int), ctx->stream));
    OPE_CUDA_TRY(ctx, cudaMemsetAsync(d_counts.p, 0, 3 * (size_t)B * sizeof(int), ctx->stream));
    OPE_CUDA_TRY(ctx, cudaMemsetAsync(d_ccounts.p, 0, 3 * (size_t)B * sizeof(int), ctx->stream));
    BSampleArgs sa;
    std::memset(&sa, 0, sizeof(sa));
    sa.src = d_tsrc.p; sa.counts = d_cnt.p; sa.active = d_active.p; sa.flags = d_flags.p;
    sa.inv_leaf[0] = 1.0f / P.coarse_leaf; sa.inv_leaf[1] = 1.0f / P.fine_leaf;
    sa.cap[0] = kBFeatCap; sa.cap[1] = kBCap;
    sa.out[0] = sampled.p; sa.out[1] = sampled.p + slab;
    sa.out_counts[0] = d_counts.p; sa.out_counts[1] = d_counts.p + B;
    OPE_TRY(bsample_batch(ctx, sa, B, 2));
    // ---- re-coarse trackers: their own source sampled at 1 cm into slab [2] (the fine stage reuses the slab after SAC-IA) ----
    std::vector<const float4*> h_ssrc((size_t)B, nullptr);
    std::vector<int> h_sn((size_t)B, 0);
    for (int i = 0; i < B; ++i) {
      h_re[(size_t)i] = h_active[(size_t)i] && st[i].recoarse;
      h_ssrc[(size_t)i] = st[i].src->pts; h_sn[(size_t)i] = (int)st[i].src->n;
    }
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_ssrc.p, h_ssrc.data(), B * sizeof(const float4*), cudaMemcpyHostToDevice, ctx->stream));
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_scnt.p, h_sn.data(), B * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_re.p, h_re.data(), B * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    std::memset(&sa, 0, sizeof(sa));
    sa.src = d_ssrc.p; sa.counts = d_scnt.p; sa.active = d_re.p; sa.flags = d_flags.p;
    sa.inv_leaf[0] = 1.0f / P.coarse_leaf; sa.cap[0] = kBFeatCap; sa.out[0] = sampled.p + 2 * slab; sa.out_counts[0] = d_counts.p + 2 * (size_t)B;
    OPE_TRY(bsample_batch(ctx, sa, B, 1));
    std::vector<int> h_flags, h_all;
    OPE_TRY(download(ctx, d_counts.p, 3 * (size_t)B, h_all));
    OPE_TRY(download(ctx, d_flags.p, (size_t)B, h_flags));
    for (int i = 0; i < B; ++i) {
      h_counts[(size_t)i] = h_all[(size_t)i]; h_counts[(size_t)B + i] = h_all[(size_t)B + i]; h_scount[(size_t)i] = h_all[2 * (size_t)B + i];
      if (!h_active[(size_t)i]) continue;
      const int n1 = h_all[(size_t)i], n2 = h_all[(size_t)B + i], ns = h_all[2 * (size_t)B + i];
      // the envelope: the fine stage runs ICP, every cloud fits its shared-memory kernel; re-coarse trackers run SAC-IA as well
      bool ok = !h_flags[(size_t)i] && n2 >= std::max(P.min_target_points, 1) && n2 <= kBCap;
      if (st[i].recoarse) ok = ok && n1 >= std::max(P.min_target_features, 1) && n1 <= kBFeatCap && ns >= std::max(S, 1) && ns <= kBFeatCap;
      if (!ok) h_active[(size_t)i] = 0;
    }
  }
  int max_tp = 0, max_tp1 = 0, max_ns = 0, n_re = 0;
  for (int i = 0; i < B; ++i) {
    h_re[(size_t)i] = h_active[(size_t)i] && st[i].recoarse;
    if (!h_active[(size_t)i]) { h_counts[(size_t)i] = 0; h_counts[(size_t)B + i] = 0; h_scount[(size_t)i] = 0; continue; }
    if (!h_re[(size_t)i]) { h_counts[(size_t)i] = 0; h_scount[(size_t)i] = 0; }   // tracking: no coarse stage, no 1 cm samples
    max_tp = std::max(max_tp, std::max(h_counts[(size_t)i], h_counts[(size_t)B + i]));
    max_tp1 = std::max(max_tp1, h_counts[(size_t)i]);
    max_ns = std::max(max_ns, h_scount[(size_t)i]);
    n_re += h_re[(size_t)i];
  }
  // ---- decision tables, in tracker order: the serial loop's rand() stream ----
  if (call.draw) {
    std::vector<float4> hsp;
    if (n_re) OPE_TRY(download(ctx, (const float4*)(sampled.p + 2 * slab), slab, hsp));
    turn.wait();
    if (call.failed->load() != OPE_OK) return OPE_OK;
    for (int i = 0; i < B; ++i) {
      if (h_re[(size_t)i]) {
        float msd = P.sacia.min_sample_distance;   // min_sample_distance_ halves within one align() only
        st[i].ds.resize((size_t)H * S); st[i].dp.resize((size_t)H * S);
        OPE_TRY(ope_sacia_draw((const float*)(hsp.data() + (size_t)i * kBCap), (size_t)h_scount[(size_t)i], sizeof(float4), H, S, K, &msd,
                               st[i].ds.data(), st[i].dp.data()));
        st[i].drawn = ope_rng_table{H, S, st[i].ds.data(), st[i].dp.data()};
        st[i].table = &st[i].drawn;
      } else if (!h_active[(size_t)i]) {
        OPE_TRY(draw_for_per_tracker(ctx, st[i], call.targets[f0 + (size_t)i]));
      }
    }
    turn.pass();
  }
  if (!std::any_of(h_active.begin(), h_active.end(), [](int a) { return a != 0; })) return OPE_OK;
  const float vp[3] = {0, 0, 0};
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_active.p, h_active.data(), B * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_re.p, h_re.data(), B * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_counts.p, h_counts.data(), 2 * (size_t)B * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_counts.p + 2 * (size_t)B, h_scount.data(), (size_t)B * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  // ---- normals of tp1, tp2 and the source samples in one launch; FPFH of tp1 and of the source samples ----
  OPE_TRY(normals_smem_batch(ctx, sampled.p, d_counts.p, kBCap, 3 * B, std::max(max_tp, max_ns), P.normal_k, vp, normals.p));
  if (n_re) {
    OPE_TRY(spfh.alloc(slab * 33)); OPE_TRY(fpfh.alloc(slab * 33)); OPE_TRY(sspfh.alloc(slab * 33)); OPE_TRY(sfpfh.alloc(slab * 33));
    OPE_TRY(fpfh_smem_batch(ctx, sampled.p, normals.p, d_counts.p, kBCap, B, max_tp1, P.fpfh_radius, spfh.p, fpfh.p));
    OPE_TRY(fpfh_smem_batch(ctx, sampled.p + 2 * slab, normals.p + 2 * slab, d_counts.p + 2 * (size_t)B, kBCap, B, max_ns, P.fpfh_radius,
                            sspfh.p, sfpfh.p));
    // ---- findSimilarFeatures of every source point against its own target, SAC-IA with the frame's own source ----
    OPE_TRY(d_knn.alloc((size_t)B * max_ns * K));
    OPE_TRY(feature_knn_batch(ctx, fpfh.p, d_counts.p, kBCap, B, max_tp1, sfpfh.p, max_ns, kBCap, d_counts.p + 2 * (size_t)B, 33, K, d_knn.p));
    const size_t tb = (size_t)B * H * S;
    std::vector<int> hs(tb, 0), hp(tb, 0);
    for (int i = 0; i < B; ++i) {
      if (!h_re[(size_t)i]) continue;
      const ope_rng_table* tab = st[i].table;
      if (!tab || tab->n_hypotheses < H || tab->nr_samples != S || !tab->samples || !tab->picks)
        return fail(ctx, OPE_ERR_INVALID, "decision table of tracker %zu does not match the SAC-IA parameters", f0 + (size_t)i);
      for (size_t e = 0; e < (size_t)H * S; ++e) {
        const int s = tab->samples[e], p = tab->picks[e];
        if (s < 0 || s >= h_scount[(size_t)i] || p < 0 || p >= K) return fail(ctx, OPE_ERR_INVALID, "rng table entry out of range");
        hs[(size_t)i * H * S + e] = s; hp[(size_t)i * H * S + e] = p;
      }
    }
    OPE_TRY(d_samples.alloc(tb)); OPE_TRY(d_picks.alloc(tb));
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_samples.p, hs.data(), tb * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_picks.p, hp.data(), tb * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    OPE_TRY(errors.alloc((size_t)B * H)); OPE_TRY(transforms.alloc((size_t)B * H * 16));
    SaciaBatch sb;
    std::memset(&sb, 0, sizeof(sb));
    sb.src = sampled.p + 2 * slab; sb.ns = max_ns; sb.src_stride = kBCap; sb.src_counts = d_counts.p + 2 * (size_t)B;
    sb.tgt = sampled.p; sb.counts = d_counts.p; sb.stride = kBCap;
    sb.nr_samples = S; sb.k_corr = K; sb.H = H; sb.samples = d_samples.p; sb.picks = d_picks.p; sb.knn_idx = d_knn.p; sb.active = d_re.p;
    sb.h_begin = 0; sb.h_end = H; sb.early_exit = 1;
    sb.threshold = (float)P.sacia.max_correspondence_distance; sb.errors = errors.p; sb.transforms = transforms.p;
    OPE_TRY(sacia_batch_device(ctx, sb, B, max_tp1, nullptr, d_coarse.p));
    OPE_CUDA_TRY(ctx, stream_sync(ctx));   // hs / hp go out of scope
  }
  // ---- fine stage: coarse(source) for re-coarse trackers, the tracker's alignedSource for tracking ones ----
  {
    std::vector<const float4*> h_fsrc((size_t)B, nullptr);
    std::vector<int> h_fn((size_t)B, 0);
    for (int i = 0; i < B; ++i) {
      if (!h_active[(size_t)i]) continue;
      const ope_cloud* in = st[i].recoarse ? st[i].src : st[i].t->alignedSource;
      h_fsrc[(size_t)i] = in->pts; h_fn[(size_t)i] = (int)in->n;
    }
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_ssrc.p, h_fsrc.data(), B * sizeof(const float4*), cudaMemcpyHostToDevice, ctx->stream));
    OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_scnt.p, h_fn.data(), B * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    OPE_CUDA_TRY(ctx, stream_sync(ctx));
  }
  BSampleArgs sa;
  std::memset(&sa, 0, sizeof(sa));
  sa.src = d_ssrc.p; sa.counts = d_scnt.p; sa.xforms = d_coarse.p; sa.xform_on = d_re.p;
  BatchClouds bc{sampled.p, normals.p, compacted.p, cnormals.p, d_counts.p, d_ccounts.p, d_flags.p, d_active.p};
  std::vector<ope_reg_result> by_frame, h_coarse;
  std::vector<double> h_fit;
  std::vector<int> h_cc;
  OPE_TRY(fine_stage(ctx, P, B, bc, sa, h_active, by_frame, h_fit, h_cc, nullptr));
  if (!std::any_of(h_active.begin(), h_active.end(), [](int a) { return a != 0; })) return OPE_OK;
  OPE_TRY(download(ctx, d_coarse.p, (size_t)B, h_coarse));
  // ---- the commit: new alignedSource, the source's replacement, the dense Umeyama cloudModel -> source (:425-436) ----
  std::vector<TrackCommit> hc;
  std::vector<int> commit_of;
  for (int i = 0; i < B; ++i) {
    if (!h_active[(size_t)i]) continue;
    Step& s = st[i];
    TrackCommit c;
    std::memset(&c, 0, sizeof(c));
    const ope_cloud* in = s.recoarse ? s.src : s.t->alignedSource;
    c.in = in->pts; c.n_in = (int)in->n; c.pre = s.recoarse;
    Mat4 coarse = mat4_identity();
    if (s.recoarse) std::memcpy(coarse.m, h_coarse[(size_t)i].T, 64);
    std::memcpy(c.coarse, coarse.m, 64); std::memcpy(c.fine, by_frame[(size_t)i].T, 64);
    c.out_aligned = s.new_aligned->pts; c.out_source = s.new_source->pts;
    c.model = s.model->pts; c.src = s.src->pts;
    c.n_model = (s.model->n > 0 && s.model->n <= s.src->n) ? (int)s.model->n : 0;
    c.nb = umeyama_blocks(ctx, c.n_model ? (size_t)c.n_model : (size_t)c.n_in);
    hc.push_back(c);
    commit_of.push_back(i);
  }
  const int NC = (int)hc.size();
  Scratch<TrackCommit> d_commits(ctx);
  Scratch<float> d_rigid(ctx);
  OPE_TRY(d_commits.alloc(NC)); OPE_TRY(d_rigid.alloc((size_t)NC * 16));
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_commits.p, hc.data(), NC * sizeof(TrackCommit), cudaMemcpyHostToDevice, ctx->stream));
  OPE_TRY(track_commit_device(ctx, d_commits.p, hc.data(), NC, d_rigid.p));
  std::vector<float> h_rigid;
  OPE_TRY(download(ctx, d_rigid.p, (size_t)NC * 16, h_rigid));
  // ---- estimateFinalPose (:383-448): finalPose = rigidmodelPose * (coarse * fine) ----
  for (int j = 0; j < NC; ++j) {
    const int i = commit_of[(size_t)j];
    Step& s = st[i];
    ope_pose_result r;
    std::memset(&r, 0, sizeof(r));
    Mat4 coarse, fine, rigid = mat4_identity();
    std::memcpy(coarse.m, hc[(size_t)j].coarse, 64);
    std::memcpy(fine.m, by_frame[(size_t)i].T, 64);
    if (hc[(size_t)j].n_model) std::memcpy(rigid.m, h_rigid.data() + (size_t)j * 16, 64);
    const Mat4 final_pose = mat4_mul(rigid, mat4_mul(coarse, fine));
    std::memcpy(r.final_pose, final_pose.m, 64); std::memcpy(r.coarse_pose, coarse.m, 64);
    std::memcpy(r.fine_pose, fine.m, 64); std::memcpy(r.rigid_model_pose, rigid.m, 64);
    const int nsrc = h_cc[(size_t)B + i], nt = h_cc[(size_t)i];
    s.fitness = h_fit[(size_t)i];
    s.strength = (double)by_frame[(size_t)i].n_correspondences / (double)((long)nsrc + (long)nt);   // VP/icp_mod.h:249-260
    r.fitness = s.fitness; r.align_strength = s.strength;
    r.icp_iterations = by_frame[(size_t)i].iterations; r.icp_converged = by_frame[(size_t)i].converged; r.icp_state = by_frame[(size_t)i].state;
    r.n_src_fine = nsrc; r.n_tgt_fine = nt;
    if (s.recoarse) {
      r.ran_coarse = 1;
      r.n_src_coarse = h_scount[(size_t)i]; r.n_tgt_coarse = h_counts[(size_t)i];
      r.sacia_best_iteration = h_coarse[(size_t)i].best_iteration; r.sacia_best_error = h_coarse[(size_t)i].best_error;
    }
    s.done = 1;
    s.result = r;
  }
  return OPE_OK;
}

}  // namespace
}  // namespace ope

using namespace ope;

extern "C" int ope_pose_tracker_step_batch(ope_ctx* ctx, ope_pose_tracker* const* trackers, ope_cloud** sources, const ope_frame_input* targets,
                                           size_t n, const ope_rng_table* tables, ope_pose_result* results, int32_t* status) {
  OPE_ENTER(ctx);
  if (!ctx || (n && (!trackers || !sources || !targets || !results))) return OPE_ERR_INVALID;
  if (n == 0) return OPE_OK;
  {
    std::set<const void*> seen_t, seen_s;
    for (size_t i = 0; i < n; ++i) {
      if (!trackers[i] || trackers[i]->ctx != ctx) return fail(ctx, OPE_ERR_INVALID, "tracker %zu is missing or belongs to another context", i);
      if (!sources[i] || sources[i]->ctx != ctx) return fail(ctx, OPE_ERR_INVALID, "source %zu is missing or belongs to another context", i);
      if (!seen_t.insert(trackers[i]).second) return fail(ctx, OPE_ERR_INVALID, "tracker %zu is listed twice", i);
      if (!seen_s.insert(sources[i]).second) return fail(ctx, OPE_ERR_INVALID, "source %zu is listed twice", i);
      const ope_frame_input& in = targets[i];
      if (!in.points && in.cloud && ((const ope_cloud*)in.cloud)->ctx != ctx)
        return fail(ctx, OPE_ERR_INVALID, "target %zu belongs to another context", i);
    }
  }
  const ope_pose_params P = trackers[0]->prm;
  std::vector<Step> steps(n);
  struct Release {   // clouds allocated for trackers that did not finish on the fast path
    ope_ctx* ctx; std::vector<Step>& s;
    ~Release() {
      for (auto& x : s) {
        if (x.new_aligned) ope_cloud_free(ctx, x.new_aligned);
        if (x.new_source) ope_cloud_free(ctx, x.new_source);
        if (x.model_fresh && x.model) ope_cloud_free(ctx, x.model);
      }
    }
  } release{ctx, steps};
  const bool config_ok = icp_small_batch_applicable(P.icp, 1, 1) && P.icp.n_rejectors >= 0 && P.sacia.nr_samples >= 1 &&
                         P.sacia.max_iterations >= 1 && P.sacia.k_correspondences >= 1;
  for (size_t i = 0; i < n; ++i) {
    Step& s = steps[i];
    s.t = trackers[i]; s.src = sources[i];
    s.table = tables ? &tables[i] : nullptr;
    const bool same = std::memcmp(&s.t->prm, &P, sizeof(P)) == 0;
    s.recoarse = s.t->fitnessScoreFine > P.coarse_refit_threshold;
    const size_t nsrc = s.src->n;
    // tracking needs an alignedSource to refine; every tracker needs a target and a source the kernels can index
    s.fast = config_ok && same && target_size(targets[i]) > 0 && nsrc > 0 && nsrc <= 0x3fffffff &&
             (s.recoarse || (s.t->alignedSource && s.t->alignedSource->n > 0 && s.t->alignedSource->n <= 0x3fffffff));
    if (!s.fast) continue;
    // the clouds the commit writes: allocated here, on the tracker's context (the lanes only write into them)
    if (s.t->firstTimePose == 0) {
      OPE_TRY(cloud_alloc(ctx, nsrc, false, &s.model));
      s.model_fresh = true;
      OPE_CUDA_TRY(ctx, cudaMemcpyAsync(s.model->pts, s.src->pts, nsrc * sizeof(float4), cudaMemcpyDeviceToDevice, ctx->stream));
    } else {
      s.model = s.t->cloudModel;
      if (!s.model) { s.fast = 0; continue; }
    }
    const size_t n_out = s.recoarse ? nsrc : s.t->alignedSource->n;
    OPE_TRY(cloud_alloc(ctx, n_out, false, &s.new_aligned));
    OPE_TRY(cloud_alloc(ctx, n_out, false, &s.new_source));
  }
  OPE_TRY(ope_ctx_synchronize(ctx));   // the lanes read and write these clouds from their own streams
  std::atomic<int> failed{OPE_OK};
  Call call;
  call.P = &P; call.steps = steps.data(); call.targets = targets; call.draw = tables == nullptr; call.failed = &failed;
  const int lrc = run_chunks_on_lanes(ctx, n, nullptr, [&](ope_ctx* c, size_t f0, size_t nf, size_t k) {
    const int rc = track_chunk(c, call, f0, (int)nf, k);
    if (rc != OPE_OK) failed.store(rc);
    return rc;
  });
  OPE_TRY(lrc);
  // ---- commit the fast path's trackers (on this thread: the clouds belong to this context) ----
  for (size_t i = 0; i < n; ++i) {
    Step& s = steps[i];
    if (!s.done) continue;
    ope_pose_tracker* t = s.t;
    if (s.model_fresh) { if (t->cloudModel) ope_cloud_free(ctx, t->cloudModel); t->cloudModel = s.model; s.model_fresh = false; }
    t->firstTimePose++;
    if (t->alignedSource) ope_cloud_free(ctx, t->alignedSource);
    t->alignedSource = s.new_aligned; s.new_aligned = nullptr;
    t->fitnessScoreFine = s.fitness; t->alignedStrength = s.strength;
    ope_cloud_free(ctx, sources[i]);
    sources[i] = s.new_source; s.new_source = nullptr;
    results[i] = s.result;
    if (status) status[i] = OPE_OK;
  }
  // ---- the rest, one at a time, in tracker order, with the tables drawn at their turn ----
  int first = OPE_OK;
  std::string msg;
  for (size_t i = 0; i < n; ++i) {
    Step& s = steps[i];
    if (s.done) continue;
    const ope_frame_input& in = targets[i];
    ope_cloud* owned = nullptr;
    const ope_cloud* tgt = in.points ? nullptr : (const ope_cloud*)in.cloud;
    int rc = OPE_OK;
    if (in.points && in.n > 0) { rc = ope_cloud_upload(ctx, in.points, in.n, in.stride, in.offset, nullptr, 0, 0, &owned); tgt = owned; }
    if (rc == OPE_OK) rc = ope_pose_estimate_final_device(s.t, &sources[i], tgt, s.table, &results[i]);
    if (owned) ope_cloud_free(ctx, owned);
    if (status) status[i] = rc;
    if (rc != OPE_OK && first == OPE_OK) { first = rc; msg = ctx->error; }
  }
  OPE_CUDA_TRY(ctx, stream_sync(ctx));
  return first == OPE_OK ? OPE_OK : fail(ctx, first, "tracker step: %s", msg.c_str());
}
