// track.cu — ope_pose_tracker_step_batch: many independent trackers advanced by one frame each, the steady-state loop of
// PoseEstimator::estimateFinalPose (D&L/src/poseestimator.cpp:383-448) batched across sequences. A chunk of trackers runs through
// pose_chunk (batch.cu), the frame-spanning stages of ope_pose_batch, with a per-frame source:
//
//   target UniformSampling 1 cm + 8 mm, normals, FPFH      as ope_pose_batch
//   source UniformSampling 1 cm, normals, FPFH             re-coarse trackers (last fine fitness above the threshold), own source
//   feature k-NN, SAC-IA                                   per-frame source descriptors and points
//   SAC-IA decision tables (pose_chunk's table hook)       drawn in tracker order (a turnstile across the chunks), or the caller's
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
  PoseChunk ch;
  ch.targets = call.targets + f0; ch.first = f0;
  for (int i = 0; i < B; ++i) {   // SAC-IA on the tracker's own source; the fine stage on coarse(source), or on alignedSource (tracking)
    const ope_cloud* fine_in = !st[i].fast ? nullptr : st[i].recoarse ? st[i].src : st[i].t->alignedSource;
    ch.active.push_back(st[i].fast); ch.coarse.push_back(st[i].recoarse);
    ch.src_clouds.push_back(st[i].src->pts); ch.src_cloud_n.push_back((int)st[i].src->n);
    ch.fine_src.push_back(fine_in ? fine_in->pts : nullptr); ch.fine_n.push_back(fine_in ? (int)fine_in->n : 0);
  }
  // ---- decision tables, in tracker order: the serial loop's rand() stream ----
  auto tables = [&](PoseChunk& c) -> int {
    if (call.draw) {
      std::vector<float4> hsp;
      if (std::any_of(c.n_src_coarse.begin(), c.n_src_coarse.end(), [](int n) { return n > 0; }))   // a tracker runs SAC-IA
        OPE_TRY(download(ctx, c.src_samples, (size_t)B * kBCap, hsp));
      turn.wait();
      if (call.failed->load() != OPE_OK) { std::fill(c.active.begin(), c.active.end(), 0); return OPE_OK; }
      for (int i = 0; i < B; ++i) {
        if (c.active[(size_t)i] && st[i].recoarse) {
          float msd = P.sacia.min_sample_distance;   // min_sample_distance_ halves within one align() only
          st[i].ds.resize((size_t)H * S); st[i].dp.resize((size_t)H * S);
          OPE_TRY(ope_sacia_draw((const float*)(hsp.data() + (size_t)i * kBCap), (size_t)c.n_src_coarse[(size_t)i], sizeof(float4), H, S, K, &msd,
                                 st[i].ds.data(), st[i].dp.data()));
          st[i].drawn = ope_rng_table{H, S, st[i].ds.data(), st[i].dp.data()};
          st[i].table = &st[i].drawn;
        } else if (!c.active[(size_t)i]) {
          OPE_TRY(draw_for_per_tracker(ctx, st[i], call.targets[f0 + (size_t)i]));
        }
      }
      turn.pass();
    }
    for (int i = 0; i < B; ++i) c.tables[(size_t)i] = st[i].table;
    return OPE_OK;
  };
  OPE_TRY(pose_chunk(ctx, P, B, ch, tables));
  if (!std::any_of(ch.active.begin(), ch.active.end(), [](int a) { return a != 0; })) return OPE_OK;
  // ---- the commit: new alignedSource, the source's replacement, the dense Umeyama cloudModel -> source (:425-436) ----
  std::vector<TrackCommit> hc;
  std::vector<int> commit_of;
  for (int i = 0; i < B; ++i) {
    if (!ch.active[(size_t)i]) continue;
    Step& s = st[i];
    TrackCommit c;
    std::memset(&c, 0, sizeof(c));
    c.in = ch.fine_src[(size_t)i]; c.n_in = ch.fine_n[(size_t)i]; c.pre = s.recoarse;
    Mat4 coarse = mat4_identity();
    if (s.recoarse) std::memcpy(coarse.m, ch.coarse_res[(size_t)i].T, 64);
    std::memcpy(c.coarse, coarse.m, 64); std::memcpy(c.fine, ch.fine[(size_t)i].T, 64);
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
  for (int j = 0; j < NC; ++j) {
    Mat4 rigid = mat4_identity();
    if (hc[(size_t)j].n_model) std::memcpy(rigid.m, h_rigid.data() + (size_t)j * 16, 64);
    Step& s = st[commit_of[(size_t)j]];
    s.result = chunk_pose_result(ch, commit_of[(size_t)j], rigid);
    s.done = 1;
  }
  return OPE_OK;
}

}  // namespace
}  // namespace ope

using namespace ope;

namespace ope {

int step_batch_check(ope_ctx* ctx, ope_pose_tracker* const* trackers, ope_cloud* const* sources, const ope_frame_input* targets, size_t n) {
  std::set<const void*> seen_t, seen_s;
  for (size_t i = 0; i < n; ++i) {
    if (!trackers[i] || trackers[i]->ctx != ctx) return fail(ctx, OPE_ERR_INVALID, "tracker %zu is missing or belongs to another context", i);
    if (!sources[i] || sources[i]->ctx != ctx) return fail(ctx, OPE_ERR_INVALID, "source %zu is missing or belongs to another context", i);
    if (!seen_t.insert(trackers[i]).second) return fail(ctx, OPE_ERR_INVALID, "tracker %zu is listed twice", i);
    if (!seen_s.insert(sources[i]).second) return fail(ctx, OPE_ERR_INVALID, "source %zu is listed twice", i);
    if (!targets) continue;
    const ope_frame_input& in = targets[i];
    if (!in.points && in.cloud && ((const ope_cloud*)in.cloud)->ctx != ctx)
      return fail(ctx, OPE_ERR_INVALID, "target %zu belongs to another context", i);
  }
  return OPE_OK;
}

int tracker_step_batch(ope_ctx* ctx, ope_pose_tracker* const* trackers, ope_cloud** sources, const ope_frame_input* targets, size_t n,
                       const ope_rng_table* tables, ope_pose_result* results, int32_t* status) {
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
                         P.sacia.max_iterations >= 1 && P.sacia.k_correspondences >= 1 && P.normal_k <= 32;
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
    t->fitnessScoreFine = s.result.fitness; t->alignedStrength = s.result.align_strength;
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

}  // namespace ope

extern "C" int ope_pose_tracker_step_batch(ope_ctx* ctx, ope_pose_tracker* const* trackers, ope_cloud** sources, const ope_frame_input* targets,
                                           size_t n, const ope_rng_table* tables, ope_pose_result* results, int32_t* status) {
  OPE_ENTER(ctx);
  if (!ctx || (n && (!trackers || !sources || !targets || !results))) return OPE_ERR_INVALID;
  if (n == 0) return OPE_OK;
  OPE_TRY(step_batch_check(ctx, trackers, sources, targets, n));
  return tracker_step_batch(ctx, trackers, sources, targets, n, tables, results, status);
}
