// pipeline.cu — PoseEstimator::estimateFinalPose (D&L/src/poseestimator.cpp:383-448) sequenced on the device:
// UniformSampling -> NormalEstimation -> FPFH -> SAC-IA -> ICP-with-normals -> fitness -> dense Umeyama.
// Every stage is a call into the kernels of grid.cu / features.cu / registration.cu; only sizes, the 4x4s and the
// scores cross back to the host between stages.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <functional>
#include <memory>
#include <thread>
#include <sched.h>

#include "ope_host.cuh"

using namespace ope;


namespace {

bool model_cache_enabled() {
  const char* e = std::getenv("OPE_MODEL_CACHE");
  return !e || std::atoi(e) != 0;
}

int clone_cloud(ope_ctx* ctx, const ope_cloud* in, ope_cloud** out) {
  ope_cloud* o = nullptr;
  OPE_TRY(cloud_alloc(ctx, in->n, in->normals != nullptr, &o));
  cudaError_t e = cudaSuccess;
  if (in->n) {
    e = cudaMemcpyAsync(o->pts, in->pts, in->n * sizeof(float4), cudaMemcpyDeviceToDevice, ctx->stream);
    if (e == cudaSuccess && in->normals)
      e = cudaMemcpyAsync(o->normals, in->normals, in->n * sizeof(float4), cudaMemcpyDeviceToDevice, ctx->stream);
  }
  if (e != cudaSuccess) { ope_cloud_free(ctx, o); return fail(ctx, OPE_ERR_CUDA, "device copy failed: %s", cudaGetErrorString(e)); }
  *out = o;
  return OPE_OK;
}

struct StageTimer {
  ope_pose_tracker* t;
  explicit StageTimer(ope_pose_tracker* tr) : t(tr) { if (t->timing) cudaEventRecord(t->ev0, t->ctx->stream); }
  // closes the current interval into slot `s` and starts the next one
  void lap(int s) {
    if (!t->timing) return;
    cudaEventRecord(t->ev1, t->ctx->stream);
    cudaEventSynchronize(t->ev1);
    float ms = 0;
    cudaEventElapsedTime(&ms, t->ev0, t->ev1);
    t->stage_ms[s] += ms;
    std::swap(t->ev0, t->ev1);
  }
};

// subSampleAndCalculateNormals, D&L/src/poseestimator.cpp:131-158
int sub_sample_and_normals(ope_pose_tracker* t, StageTimer& tm, ope_cloud* in, float leaf, ope_cloud** out) {
  ope_ctx* ctx = t->ctx;
  int* d_idx = nullptr;
  size_t m = 0;
  OPE_TRY(uniform_sample_device(ctx, in, leaf, &d_idx, &m));
  ope_cloud* ds = nullptr;
  int rc = gather_cloud(ctx, in, d_idx, m, &ds);
  dfree(ctx, d_idx);
  if (rc != OPE_OK) return rc;
  dfree(ctx, ds->normals);  // the sub-sampled PointT cloud carries no normals
  ds->normals = nullptr;
  tm.lap(0);
  const float vp[3] = {0, 0, 0};
  rc = normals_device(ctx, ds, t->prm.normal_k, vp);
  if (rc != OPE_OK) { ope_cloud_free(ctx, ds); return rc; }
  tm.lap(1);
  *out = ds;
  return OPE_OK;
}

struct CloudGuard {
  ope_ctx* ctx;
  ope_cloud* c = nullptr;
  explicit CloudGuard(ope_ctx* x) : ctx(x) {}
  ~CloudGuard() { if (c) ope_cloud_free(ctx, c); }
};
struct DevGuard {
  ope_ctx* ctx;
  float* p = nullptr;
  explicit DevGuard(ope_ctx* x) : ctx(x) {}
  ~DevGuard() { dfree(ctx, p); }
};

}  // namespace

extern "C" {

int ope_pose_tracker_create(ope_ctx* ctx, const ope_pose_params* prm, ope_pose_tracker** out) {
  OPE_ENTER(ctx);
  if (!ctx || !out) return OPE_ERR_INVALID;
  ope_pose_tracker* t = new ope_pose_tracker();
  t->ctx = ctx;
  if (prm) t->prm = *prm; else ope_pose_params_default(&t->prm);
  if (cudaEventCreate(&t->ev0) != cudaSuccess || cudaEventCreate(&t->ev1) != cudaSuccess ||
      cudaEventCreate(&t->evt0) != cudaSuccess || cudaEventCreate(&t->evt1) != cudaSuccess) {
    delete t;
    return fail(ctx, OPE_ERR_CUDA, "event creation failed");
  }
  *out = t;
  return OPE_OK;
}

void ope_pose_tracker_destroy(ope_pose_tracker* t) {
  if (!t) return;
  if (t->alignedSource) ope_cloud_free(t->ctx, t->alignedSource);
  if (t->cloudModel) ope_cloud_free(t->ctx, t->cloudModel);
  cudaEventDestroy(t->ev0); cudaEventDestroy(t->ev1); cudaEventDestroy(t->evt0); cudaEventDestroy(t->evt1);
  delete t;
}

int ope_pose_stage_ms(const ope_pose_tracker* t, double out[8]) {
  if (!t || !out) return OPE_ERR_INVALID;
  std::memcpy(out, t->stage_ms, sizeof(t->stage_ms));
  return OPE_OK;
}

int ope_pose_estimate_final_device(ope_pose_tracker* t, ope_cloud** source, const ope_cloud* target,
                                   const ope_rng_table* table, ope_pose_result* res) {
  OPE_ENTER((t ? t->ctx : nullptr));
  if (!t || !source || !*source || !res) return OPE_ERR_INVALID;
  ope_ctx* ctx = t->ctx;
  const ope_pose_params& P = t->prm;
  std::memset(res, 0, sizeof(*res));
  std::memset(t->stage_ms, 0, sizeof(t->stage_ms));
  if (t->timing) cudaEventRecord(t->evt0, ctx->stream);
  StageTimer tm(t);
  ope_cloud* p_source = *source;
  const size_t nt = target ? target->n : 0;
  if (t->firstTimePose == 0) {  // :385-388
    if (t->cloudModel) { ope_cloud_free(ctx, t->cloudModel); t->cloudModel = nullptr; }
    OPE_TRY(clone_cloud(ctx, p_source, &t->cloudModel));
  }
  t->firstTimePose++;
  Mat4 coarse = mat4_identity(), fine = mat4_identity();

  // ---- COARSE: estimateCoarsePose, :16-73 ----
  if (nt != 0 && t->fitnessScoreFine > P.coarse_refit_threshold) {
    res->ran_coarse = 1;
    CloudGuard sp(ctx), tp(ctx);
    DevGuard fs(ctx), ft(ctx);
    // the model side is frame-invariant: with a cache attached (SURVEY 8f-3) the first call of a tracker reuses the model's
    // coarse sample, normals and descriptors instead of recomputing them as the reference does every frame (:34,116)
    bool cached = t->cache_sp && t->cache_fs && t->firstTimePose == 1 && t->cache_model_n == p_source->n;
    ope_cloud sp_view;
    const ope_cloud* spc = nullptr;
    const float* fsp = nullptr;
    // the context's own cache (every tracker of this context): an unchanged source cloud — same size, same content hash, same
    // parameters — keeps its coarse sample, normals and descriptors across frames and trackers. OPE_MODEL_CACHE=0 turns it off.
    ModelCacheEntry* hit = nullptr;
    unsigned long long src_hash = 0;
    const bool use_ctx_cache = !cached && model_cache_enabled();
    if (use_ctx_cache) {
      OPE_TRY(cloud_content_hash(ctx, p_source, &src_hash));
      for (auto& e : ctx->model_cache)
        if (e.hash == src_hash && e.n == p_source->n && e.leaf == P.coarse_leaf && e.k == P.normal_k && e.radius == P.fpfh_radius) hit = &e;
      if (hit) { hit->stamp = ++ctx->model_cache_clock; ctx->model_cache_hits++; } else ctx->model_cache_misses++;
      tm.lap(0);
    }
    if (cached || hit) {
      sp_view = cached ? *t->cache_sp : *hit->sp;      // shallow view: shared device arrays, private (empty) grid cache
      sp_view.ctx = ctx; sp_view.grids.clear();
      spc = &sp_view; fsp = cached ? t->cache_fs : hit->fs;
      cached = true;
    } else {
      OPE_TRY(sub_sample_and_normals(t, tm, p_source, P.coarse_leaf, &sp.c));
      spc = sp.c;
    }
    OPE_TRY(sub_sample_and_normals(t, tm, const_cast<ope_cloud*>(target), P.coarse_leaf, &tp.c));
    if (!cached) {
      OPE_TRY(fpfh_device(ctx, sp.c, P.fpfh_radius, &fs.p, nullptr));
      fsp = fs.p;
      if (use_ctx_cache) {   // hand the model side over to the cache (it owns the arrays from here on)
        ModelCacheEntry e;
        e.hash = src_hash; e.n = p_source->n; e.leaf = P.coarse_leaf; e.k = P.normal_k; e.radius = P.fpfh_radius;
        e.sp = sp.c; e.fs = fs.p; e.stamp = ++ctx->model_cache_clock;
        ope_cloud_invalidate(ctx, e.sp);
        sp.c = nullptr; fs.p = nullptr;
        if (ctx->model_cache.size() >= 4) {
          size_t old = 0;
          for (size_t i = 1; i < ctx->model_cache.size(); ++i) if (ctx->model_cache[i].stamp < ctx->model_cache[old].stamp) old = i;
          ope_cloud_free(ctx, ctx->model_cache[old].sp); dfree(ctx, ctx->model_cache[old].fs);
          ctx->model_cache[old] = e;
          hit = &ctx->model_cache[old];
        } else {
          ctx->model_cache.push_back(e);
          hit = &ctx->model_cache.back();
        }
        sp_view = *hit->sp; sp_view.ctx = ctx; sp_view.grids.clear();
        spc = &sp_view; fsp = hit->fs;
        cached = true;     // from here on the arrays are borrowed, exactly like a hit
      }
    }
    OPE_TRY(fpfh_device(ctx, tp.c, P.fpfh_radius, &ft.p, nullptr));
    tm.lap(2);
    res->n_src_coarse = (int32_t)spc->n; res->n_tgt_coarse = (int32_t)tp.c->n;
    // the tracker's state changes only once the stage has succeeded: a failing call leaves alignedSource as it was
    ope_cloud* fresh = nullptr;
    if ((int)tp.c->n < P.min_target_features) {
      OPE_TRY(clone_cloud(ctx, p_source, &fresh));  // :41
    } else {
      ope_reg_result rr;
      int src_rc = sacia_device(ctx, spc, fsp, tp.c, ft.p, P.sacia, table, nullptr, &rr, nullptr);
      if (cached) ope_cloud_invalidate(ctx, &sp_view);   // drop whatever index the view acquired
      OPE_TRY(src_rc);
      tm.lap(3);
      std::memcpy(coarse.m, rr.T, sizeof(coarse.m));
      res->sacia_best_iteration = rr.best_iteration; res->sacia_best_error = rr.best_error;
      OPE_TRY(cloud_alloc(ctx, p_source->n, false, &fresh));
      ope_cloud view = *p_source;  // transform points only
      view.normals = nullptr; view.grids.clear();
      const int trc = transform_device(ctx, &view, coarse, fresh);  // :67-70
      if (trc != OPE_OK) { ope_cloud_free(ctx, fresh); return trc; }
      tm.lap(6);
    }
    if (t->alignedSource) ope_cloud_free(ctx, t->alignedSource);
    t->alignedSource = fresh;
  }
  // ---- FINE: estimateFinePose, :161-379 ----
  if (nt != 0 && t->alignedSource) {
    CloudGuard sp(ctx), tp(ctx);
    OPE_TRY(sub_sample_and_normals(t, tm, t->alignedSource, P.fine_leaf, &sp.c));
    OPE_TRY(sub_sample_and_normals(t, tm, const_cast<ope_cloud*>(target), P.fine_leaf, &tp.c));
    OPE_TRY(remove_nan_normals_device(ctx, &sp.c));  // :215-216
    OPE_TRY(remove_nan_normals_device(ctx, &tp.c));
    tm.lap(1);
    res->n_src_fine = (int32_t)sp.c->n; res->n_tgt_fine = (int32_t)tp.c->n;
    if ((int)tp.c->n >= P.min_target_points) {  // :218-223
      ope_reg_result rr;
      OPE_TRY(icp_device(ctx, sp.c, tp.c, P.icp, mat4_identity(), &rr, nullptr, nullptr));
      tm.lap(4);
      std::memcpy(fine.m, rr.T, sizeof(fine.m));
      OPE_TRY(fitness_device(ctx, sp.c, tp.c, fine, DBL_MAX, &t->fitnessScoreFine));  // :354
      tm.lap(5);
      ope_cloud* moved = nullptr;
      OPE_TRY(cloud_alloc(ctx, t->alignedSource->n, false, &moved));
      int rc = transform_device(ctx, t->alignedSource, fine, moved);  // :358-360
      if (rc != OPE_OK) { ope_cloud_free(ctx, moved); return rc; }
      ope_cloud_free(ctx, t->alignedSource);
      t->alignedSource = moved;
      t->alignedStrength = (double)rr.n_correspondences / (double)((long)sp.c->n + (long)tp.c->n);  // VP/icp_mod.h:249-260
      res->icp_iterations = rr.iterations; res->icp_converged = rr.converged; res->icp_state = rr.state;
      tm.lap(6);
    }
  }
  const Mat4 pose = mat4_mul(coarse, fine);  // :421 (sic: coarse * fine)
  Mat4 rigid = mat4_identity();
  if (t->cloudModel && t->cloudModel->n > 0 && t->cloudModel->n <= p_source->n) {  // :425-436
    OPE_TRY(umeyama_device(ctx, t->cloudModel->pts, p_source->pts, nullptr, nullptr, t->cloudModel->n, rigid.m));
  }
  const Mat4 final_pose = mat4_mul(rigid, pose);  // :439
  {  // *p_sourceCloud = *alignedSource, :441 — before any alignment the member is an EMPTY cloud, and so becomes the source
    ope_cloud* copy = nullptr;
    if (t->alignedSource) OPE_TRY(clone_cloud(ctx, t->alignedSource, &copy));
    else OPE_TRY(cloud_alloc(ctx, 0, false, &copy));
    ope_cloud_free(ctx, p_source);
    *source = copy;
  }
  tm.lap(6);
  std::memcpy(res->final_pose, final_pose.m, 64); std::memcpy(res->coarse_pose, coarse.m, 64);
  std::memcpy(res->fine_pose, fine.m, 64); std::memcpy(res->rigid_model_pose, rigid.m, 64);
  res->fitness = t->fitnessScoreFine; res->align_strength = t->alignedStrength;
  if (t->timing) {
    cudaEventRecord(t->evt1, ctx->stream);
    cudaEventSynchronize(t->evt1);
    float ms = 0;
    cudaEventElapsedTime(&ms, t->evt0, t->evt1);
    t->stage_ms[7] = ms;
  }
  return OPE_OK;
}

}  // extern "C"

namespace ope {
// Runs run_chunk(lane context, first item, items, chunk index) over items [0, n) in chunks on a few lanes at once (OPE_BATCH_LANES,
// OPE_BATCH_CHUNK override the defaults below; chunk_items > 0 fixes the chunk size). Chunks are handed out in index order. A
// lane stops at the first failing chunk or when *stop is set; the return value is the first failure's code (its message in
// ctx->error). Every worker stream is idle on return.
int run_chunks_on_lanes(ope_ctx* ctx, size_t n, const std::atomic<int>* stop,
                        const std::function<int(ope_ctx*, size_t, size_t, size_t)>& run_chunk, size_t chunk_items) {
  // Chunks of frames run through the frame-spanning launches on a few LANES at once: lane 0 is this thread on this context,
  // the others are helper threads on worker contexts (own stream, own scratch pool). A lane's host work between its stages
  // (staging the clusters, copying decision tables, reading counts back) then overlaps the other lanes' kernels instead of
  // leaving the device idle; chunks are handed out in order, so the helper thread's tables arrive in the order they are needed.
  // Frames per chunk: at most two SM-sized waves of the one-block-per-frame kernels, and enough chunks for every lane to get
  // an equal share (a small batch is cut finer, so the device starts while the tables of the later frames are still drawn).
  const char* ce = std::getenv("OPE_BATCH_CHUNK");
  const char* le = std::getenv("OPE_BATCH_LANES");
  // lanes: one host thread each, plus the thread that draws the tables — as many as this process has cores for (its affinity
  // mask, shared with the other ranks of a torchrun-style launch on the same node), at most 8
  int cores = (int)std::thread::hardware_concurrency();
  {
    cpu_set_t set;
    CPU_ZERO(&set);
    if (sched_getaffinity(0, sizeof(set), &set) == 0 && CPU_COUNT(&set) > 0) cores = CPU_COUNT(&set);
    const char* lw = std::getenv("LOCAL_WORLD_SIZE");
    if (lw && std::atoi(lw) > 1) cores = std::max(1, cores / std::atoi(lw));
  }
  int lanes = std::max(1, std::min(le ? std::atoi(le) : std::max(2, cores - 1), 8));
  if (ctx->batch_timing) lanes = 1;   // per-stage device times are only meaningful when the stages do not share the device
  size_t chunk = chunk_items ? chunk_items : (size_t)std::max(1, ce ? std::atoi(ce) : 296);
  if (!ce && !chunk_items) {
    if (lanes > 1) {
      // measured (tools/bench_batch_lanes.py): many small chunks in flight beat few large ones — ~32 frames per chunk, every
      // lane the same number of chunks
      const size_t per_round = (size_t)lanes * 32;
      const size_t rounds = std::max<size_t>(1, (n + per_round / 2) / per_round);
      chunk = std::max<size_t>(std::min<size_t>(8, n), (n + rounds * lanes - 1) / (rounds * lanes));
    } else {
      const size_t rounds = std::max<size_t>(3, (n + 295) / 296);
      chunk = std::max<size_t>(std::min<size_t>(74, n), (n + rounds - 1) / rounds);
    }
  }
  const size_t n_chunks = (n + chunk - 1) / chunk;
  lanes = (int)std::min<size_t>((size_t)lanes, n_chunks);
  while ((int)ctx->workers.size() < lanes - 1) {
    ope_ctx* w = nullptr;
    const int rc = ope_ctx_create(ctx->device, nullptr, &w);
    if (rc != OPE_OK) return fail(ctx, rc, "worker context creation failed");
    ctx->workers.push_back(w);
  }
  if (lanes > 1) OPE_TRY(ope_ctx_synchronize(ctx));   // the other lanes read the model side from their own streams
  // How a lane waits for its stream: spinning is quickest but keeps a core (measured at 8 ranks x 4 cores: 31.3 k frames/s
  // spinning, 29.3 k sleeping); with fewer cores than lanes + the table thread the waits sleep on a blocking event instead
  // (OPE_BATCH_LANE_SYNC = spin | yield | block overrides)
  int wait_mode = lanes + 1 > cores ? 2 : 0;   // 0 spin, 1 poll + yield, 2 block
  if (const char* e = std::getenv("OPE_BATCH_LANE_SYNC")) wait_mode = std::strcmp(e, "block") == 0 ? 2 : std::strcmp(e, "yield") == 0 ? 1 : 0;
  struct WaitMode {   // applied to every lane's context for this call, the caller's own context gets its setting back
    ope_ctx* main; cudaEvent_t saved_event; bool saved_yield; cudaEvent_t mine = nullptr;
    explicit WaitMode(ope_ctx* c) : main(c), saved_event(c->sync_event), saved_yield(c->sync_yield) {}
    ~WaitMode() { main->sync_event = saved_event; main->sync_yield = saved_yield; if (mine) cudaEventDestroy(mine); }
  } wait_guard(ctx);
  if (lanes > 1) {
    for (int l = 0; l < lanes; ++l) {
      ope_ctx* c = l == 0 ? ctx : ctx->workers[(size_t)l - 1];
      if (l > 0 && c->sync_event) { cudaEventDestroy(c->sync_event); c->sync_event = nullptr; }
      cudaEvent_t ev = nullptr;
      if (wait_mode != 0 && cudaEventCreateWithFlags(&ev, (wait_mode == 2 ? cudaEventBlockingSync : 0) | cudaEventDisableTiming) != cudaSuccess) ev = nullptr;
      if (l == 0) wait_guard.mine = ev;
      c->sync_event = ev;
      c->sync_yield = wait_mode == 1 && ev;
    }
  }
  std::atomic<size_t> next_chunk{0};
  std::atomic<int> lane_rc{OPE_OK};
  std::mutex lane_mu;
  std::string lane_msg;
  auto run_lane = [&](ope_ctx* c) {
    ope::enter(c);
    for (;;) {
      const size_t f0 = next_chunk.fetch_add(1) * chunk;
      if (f0 >= n || lane_rc.load() != OPE_OK || (stop && stop->load() != OPE_OK)) break;
      const size_t nf = std::min(chunk, n - f0);
      const int rc = run_chunk(c, f0, nf, f0 / chunk);
      if (rc != OPE_OK) {
        std::lock_guard<std::mutex> lock(lane_mu);
        if (lane_rc.load() == OPE_OK) { lane_rc.store(rc); lane_msg = c->error; }
        break;
      }
    }
    if (c != ctx) stream_sync(c);
  };
  {
    std::vector<std::thread> lane_threads;
    struct JoinLanes { std::vector<std::thread>& t; ~JoinLanes() { for (auto& th : t) if (th.joinable()) th.join(); } } join_lanes{lane_threads};
    try {   // nothing may throw across the C ABI: without helper threads this thread takes every chunk
      for (int l = 1; l < lanes; ++l) lane_threads.emplace_back(run_lane, ctx->workers[(size_t)l - 1]);
    } catch (...) {
    }
    run_lane(ctx);
  }
  if (lane_rc.load() != OPE_OK) return fail(ctx, lane_rc.load(), "%s", lane_msg.c_str());
  return OPE_OK;
}

}  // namespace ope

extern "C" {

// ---- batched first-frame localisation (C5) ----------------------------------------------------------------------------------
namespace {

// A frame outside the frame-spanning launches' envelope, on context c: what a fresh PoseEstimator returns for it, with the
// model side (model, its 1 cm sample sp with normals, the FPFH fs of sp) borrowed from the batch.
int pose_one_frame(ope_ctx* c, const ope_pose_params& P, const ope_cloud* model, const ope_cloud* sp, const float* fs,
                   const ope_frame_input& in, const ope_rng_table* table, ope_pose_result* res) {
  // The frame's ICP runs next to the other lanes' chunks: the thread-per-query kernel where it applies (least device time per
  // alignment), and the cooperative icp_kernel's grid capped so that its blocks leave room for them. The cap is a constant:
  // the block count orders the kernel's sums, so a frame's result must not depend on the lanes. c may be the caller's context.
  struct IcpSettings {
    ope_ctx* c; bool prefer_small; int max_blocks;
    ~IcpSettings() { c->icp_prefer_small = prefer_small; c->icp_max_blocks = max_blocks; }
  } restore{c, c->icp_prefer_small, c->icp_max_blocks};
  c->icp_prefer_small = true;
  c->icp_max_blocks = std::max(8, c->sm_count / 8);
  ope_pose_tracker* t = nullptr;
  int rc = ope_pose_tracker_create(c, &P, &t);
  ope_cloud* src = nullptr;
  ope_cloud* tgt_owned = nullptr;
  const ope_cloud* tgt = nullptr;
  if (rc == OPE_OK) {
    t->timing = false;
    t->cache_sp = sp; t->cache_fs = fs; t->cache_model_n = model->n;
    rc = clone_cloud(c, model, &src);
  }
  if (rc == OPE_OK) {
    if (in.points) {
      if (in.n > 0) rc = ope_cloud_upload(c, in.points, in.n, in.stride, in.offset, nullptr, 0, 0, &tgt_owned);
      tgt = tgt_owned;
    } else if (in.cloud && ((const ope_cloud*)in.cloud)->n > 0) {
      // a private copy: the stages cache the bounding box and search grids IN the cloud they work on, and two frames may
      // name the same caller-owned cloud (or the caller may use it from its own context meanwhile)
      ope_cloud view = *(const ope_cloud*)in.cloud;
      view.normals = nullptr; view.grids.clear(); view.bbox_valid = false;
      rc = clone_cloud(c, &view, &tgt_owned);
      tgt = tgt_owned;
    }
  }
  if (rc == OPE_OK) rc = ope_pose_estimate_final_device(t, &src, tgt, table, res);
  if (src) ope_cloud_free(c, src);
  if (tgt_owned) ope_cloud_free(c, tgt_owned);
  if (t) ope_pose_tracker_destroy(t);
  return rc;
}

}  // namespace

int ope_pose_batch(ope_ctx* ctx, const ope_pose_params* prm, const float* model_xyz, size_t n_model, const ope_frame_input* frames,
                   size_t n_frames, const ope_rng_table* tables, int workers, ope_pose_result* results, int32_t* status) {
  OPE_ENTER(ctx);
  if (!ctx || !model_xyz || n_model == 0 || (!frames && n_frames) || !results) return OPE_ERR_INVALID;
  if (n_frames == 0) return OPE_OK;
  ope_pose_params P;
  if (prm) P = *prm; else ope_pose_params_default(&P);
  // ---- the frame-invariant model side, once (SURVEY 8f-3) — and kept across calls while the caller's model does not change ----
  struct Borrowed { ope_cloud* c = nullptr; } model, sp;
  struct BorrowedF { float* p = nullptr; } fs;
  Mat4 rigid = mat4_identity();
  {
    unsigned long long h = 0x9e3779b97f4a7c15ull;   // content hash of the host buffer (4-byte words)
    const uint32_t* w = (const uint32_t*)model_xyz;
    unsigned long long h2 = 0xc2b2ae3d27d4eb4full;
    const size_t words = n_model * 3;
    size_t i = 0;
    for (; i + 2 <= words; i += 2) {
      h = (h ^ w[i]) * 0x9fb21c651e98df25ull; h = (h << 29) | (h >> 35);
      h2 = (h2 ^ w[i + 1]) * 0x9fb21c651e98df25ull; h2 = (h2 << 31) | (h2 >> 33);
    }
    for (; i < words; ++i) { h = (h ^ w[i]) * 0x9fb21c651e98df25ull; h = (h << 29) | (h >> 35); }
    h ^= h2 * 3 + n_model;
    BatchModelCache& C = ctx->batch_model;
    const bool hit = model_cache_enabled() && C.model && C.hash == h && C.n == n_model && C.leaf == P.coarse_leaf && C.k == P.normal_k &&
                     C.radius == P.fpfh_radius;
    if (!hit) {
      if (C.model) ope_cloud_free(ctx, C.model);
      if (C.sp) ope_cloud_free(ctx, C.sp);
      dfree(ctx, C.fs);
      C = BatchModelCache();
      OPE_TRY(ope_cloud_upload(ctx, model_xyz, n_model, 12, 0, nullptr, 0, 0, &C.model));
      ope_pose_tracker tmp;
      tmp.ctx = ctx; tmp.prm = P; tmp.timing = false;
      StageTimer tm(&tmp);
      OPE_TRY(sub_sample_and_normals(&tmp, tm, C.model, P.coarse_leaf, &C.sp));
      OPE_TRY(fpfh_device(ctx, C.sp, P.fpfh_radius, &C.fs, nullptr));
      // the dense Umeyama of the pristine model onto the first frame's source — itself (:425-436)
      Mat4 R = mat4_identity();
      OPE_TRY(umeyama_device(ctx, C.model->pts, C.model->pts, nullptr, nullptr, C.model->n, R.m));
      std::memcpy(C.rigid, R.m, sizeof(C.rigid));
      C.hash = h; C.n = n_model; C.leaf = P.coarse_leaf; C.k = P.normal_k; C.radius = P.fpfh_radius;
    }
    model.c = C.model; sp.c = C.sp; fs.p = C.fs;
    std::memcpy(rigid.m, C.rigid, sizeof(C.rigid));
  }
  // ---- SAC-IA decision tables: replayed, or drawn here in frame order from libc rand() ----
  // Drawing is inherently serial (one process-wide rand() stream, consumed exactly as a loop over fresh PoseEstimators would) and
  // costs ~0.1 ms per frame on the host, so a helper thread draws ahead while the device works: `tables_ready` counts the frames
  // whose table is complete, the chunk loop waits for the ones it needs right before it uploads them.
  std::vector<int32_t> draw_s, draw_p;
  std::vector<ope_rng_table> drawn;
  std::atomic<size_t> tables_ready{n_frames};
  std::atomic<int> draw_rc{OPE_OK};
  std::thread drawer;
  struct JoinDrawer { std::thread& t; ~JoinDrawer() { if (t.joinable()) t.join(); } } join_drawer{drawer};
  if (!tables) {
    const int H = P.sacia.max_iterations, S = P.sacia.nr_samples, K = P.sacia.k_correspondences;
    if (H < 1 || S < 1 || K < 1) return fail(ctx, OPE_ERR_INVALID, "bad SAC-IA parameters");
    auto xyz = std::make_shared<std::vector<float>>(3 * std::max<size_t>(sp.c->n, 1));
    OPE_TRY(ope_cloud_download(ctx, sp.c, xyz->data(), nullptr));
    draw_s.resize(n_frames * (size_t)H * S); draw_p.resize(n_frames * (size_t)H * S);
    drawn.resize(n_frames);
    tables_ready.store(0);
    const size_t n_sp = sp.c->n;
    const float msd0 = P.sacia.min_sample_distance;
    auto draw_all = [&, xyz, H, S, K, n_sp, msd0]() {
      for (size_t f = 0; f < n_frames; ++f) {
        float msd = msd0;   // min_sample_distance_ halves within one align() only
        int32_t* s = draw_s.data() + f * (size_t)H * S;
        int32_t* p = draw_p.data() + f * (size_t)H * S;
        const int rc = ope_sacia_draw(xyz->data(), n_sp, 12, H, S, K, &msd, s, p);
        if (rc != OPE_OK) { draw_rc.store(rc); tables_ready.store(n_frames); return; }
        drawn[f] = ope_rng_table{H, S, s, p};
        tables_ready.store(f + 1, std::memory_order_release);
      }
    };
    try { drawer = std::thread(draw_all); } catch (...) { draw_all(); }   // no thread available: draw here, as before
    tables = drawn.data();
  }
  // ---- frame-spanning launches (batch.cu): one launch per stage for a whole chunk of frames; the frames outside their envelope
  // (tiny / empty / oversized clusters, or every frame when the ICP parameters are outside it) are collected for a second pass ----
  // normal_k above 32 is outside the frame-spanning normal kernel: every frame then runs on the per-frame path
  const bool fast = icp_small_batch_applicable(P.icp, 1, 1) && P.icp.n_rejectors >= 0 && P.normal_k <= 32;
  std::mutex frame_mu;
  std::vector<size_t> rest;
  int lrc = run_chunks_on_lanes(ctx, n_frames, &draw_rc, [&](ope_ctx* c, size_t f0, size_t nf, size_t) -> int {
    PoseChunk ch;   // every frame's SAC-IA source is the model's cached 1 cm sample, its fine source the model under the coarse pose
    ch.targets = frames + f0; ch.first = f0; ch.active.assign(nf, fast ? 1 : 0);
    ch.src_pts = sp.c->pts; ch.src_fpfh = fs.p; ch.src_n = (int)sp.c->n;
    ch.fine_src.assign(nf, model.c->pts); ch.fine_n.assign(nf, (int)model.c->n);
    OPE_TRY(pose_chunk(c, P, (int)nf, ch, [&](PoseChunk& k) -> int {
      // the tables of this chunk may still be on their way (drawn by the helper thread while the device worked)
      while (tables_ready.load(std::memory_order_acquire) < f0 + nf) sched_yield();
      for (size_t i = 0; i < nf; ++i) k.tables[i] = tables + f0 + i;
      return OPE_OK;
    }));
    for (size_t i = 0; i < nf; ++i) {
      const size_t f = f0 + i;
      if (ch.active[i]) {
        results[f] = chunk_pose_result(ch, (int)i, rigid);
        if (status) status[f] = OPE_OK;
        continue;
      }
      std::lock_guard<std::mutex> lock(frame_mu);
      rest.push_back(f);
    }
    return OPE_OK;
  });
  if (lrc != OPE_OK) {
    if (draw_rc.load() != OPE_OK) tables_ready.store(n_frames);
    return lrc;
  }
  if (drawer.joinable()) drawer.join();
  if (draw_rc.load() != OPE_OK) return fail(ctx, draw_rc.load(), "selectSamples failed");
  // ---- the collected frames through the per-frame path, one frame per chunk on the same lanes ----
  std::sort(rest.begin(), rest.end());
  size_t failed_frame = n_frames;   // the lowest frame that failed on the per-frame path, its code and message
  int failed_rc = OPE_OK;
  std::string failed_msg;
  lrc = run_chunks_on_lanes(ctx, rest.size(), nullptr, [&](ope_ctx* c, size_t i0, size_t, size_t) -> int {
    const size_t f = rest[i0];
    // a frame's failure is its own: the other frames of the batch go on
    const int rc = pose_one_frame(c, P, model.c, sp.c, fs.p, frames[f], tables + f, &results[f]);
    if (status) status[f] = rc;
    if (rc != OPE_OK) {
      std::lock_guard<std::mutex> lock(frame_mu);
      if (f < failed_frame) { failed_frame = f; failed_rc = rc; failed_msg = c->error; }
    }
    return OPE_OK;
  }, 1);
  if (lrc != OPE_OK) return lrc;
  if (failed_rc != OPE_OK) return fail(ctx, failed_rc, "frame %zu: %s", failed_frame, failed_msg.c_str());
  return OPE_OK;
}

// RegMeshPcd::registerPointClouds, BM/src/regmeshpcd.cpp:210-271 — the whole chain on the device
int ope_register_point_clouds(ope_ctx* ctx, const ope_frame_input* views, size_t n_views, const ope_icp_params* prm, int normal_k,
                              ope_reg_result* pair_results, ope_cloud** merged) {
  OPE_ENTER(ctx);
  if (!ctx || !views || n_views == 0 || !prm || !merged) return OPE_ERR_INVALID;
  auto load = [&](const ope_frame_input& v, ope_cloud** out) -> int {
    if (v.points) return ope_cloud_upload(ctx, v.points, v.n, v.stride, v.offset, nullptr, 0, 0, out);
    if (!v.cloud) return fail(ctx, OPE_ERR_INVALID, "view without points");
    ope_cloud view = *(const ope_cloud*)v.cloud;     // private copy without normals: normals are recomputed per pair (:74-90)
    view.normals = nullptr; view.grids.clear();
    return clone_cloud(ctx, &view, out);
  };
  CloudGuard cur(ctx);
  OPE_TRY(load(views[0], &cur.c));   // cloudTemp = cloudVector[0], :226
  const float vp[3] = {0, 0, 0};
  for (size_t i = 0; i + 1 < n_views; ++i) {
    CloudGuard tgt(ctx), moved(ctx);
    OPE_TRY(load(views[i + 1], &tgt.c));
    ope_reg_result rr;
    std::memset(&rr, 0, sizeof(rr));
    for (int j = 0; j < 16; ++j) rr.T[j] = (j % 5 == 0) ? 1.f : 0.f;
    if (cur.c->n > 0 && tgt.c->n > 0) {
      ope_cloud_invalidate(ctx, cur.c);
      OPE_TRY(normals_device(ctx, cur.c, normal_k, vp));   // normEst on the (growing) source and on the view, :82-90
      OPE_TRY(normals_device(ctx, tgt.c, normal_k, vp));
      OPE_TRY(icp_device(ctx, cur.c, tgt.c, *prm, mat4_identity(), &rr, nullptr, nullptr));   // :166-199
    }
    if (pair_results) pair_results[i] = rr;
    Mat4 M;
    std::memcpy(M.m, rr.T, sizeof(M.m));
    OPE_TRY(cloud_alloc(ctx, cur.c->n, false, &moved.c));
    ope_cloud view = *cur.c;           // pcl::transformPointCloud(*p_cloudSource, *cloudAligned, T): points only, :204
    view.normals = nullptr; view.grids.clear();
    OPE_TRY(transform_device(ctx, &view, M, moved.c));
    dfree(ctx, tgt.c->normals); tgt.c->normals = nullptr;
    OPE_TRY(ope_cloud_append(ctx, moved.c, tgt.c));   // *cloudAlignedIcp += *cloudTarget, :254
    std::swap(cur.c, moved.c);                       // *cloudTemp = *cloudAlignedIcp, :258
  }
  OPE_CUDA_TRY(ctx, stream_sync(ctx));
  *merged = cur.c;
  cur.c = nullptr;
  return OPE_OK;
}

// per-stage device time of the frame-spanning launches of ope_pose_batch since the last reset (enable < 0: just read)
int ope_pose_batch_stage_ms(ope_ctx* ctx, int enable, double out[12]) {
  if (!ctx) return OPE_ERR_INVALID;
  if (out) std::memcpy(out, ctx->batch_stage_ms, 12 * sizeof(double));
  if (enable >= 0) { ctx->batch_timing = enable != 0; std::memset(ctx->batch_stage_ms, 0, sizeof(ctx->batch_stage_ms)); }
  return OPE_OK;
}

int ope_pose_estimate_final(ope_pose_tracker* t, float* source_xyz, size_t ns, const void* target, size_t nt, size_t tstride,
                            size_t toffset, const ope_rng_table* table, ope_pose_result* res) {
  OPE_ENTER((t ? t->ctx : nullptr));
  if (!t || !source_xyz || !res) return OPE_ERR_INVALID;
  ope_ctx* ctx = t->ctx;
  ope_cloud* src = nullptr;
  OPE_TRY(ope_cloud_upload(ctx, source_xyz, ns, 12, 0, nullptr, 0, 0, &src));
  CloudGuard tg(ctx);
  if (nt > 0) {
    int rc = ope_cloud_upload(ctx, target, nt, tstride, toffset, nullptr, 0, 0, &tg.c);
    if (rc != OPE_OK) { ope_cloud_free(ctx, src); return rc; }
  }
  int rc = ope_pose_estimate_final_device(t, &src, tg.c, table, res);
  if (rc == OPE_OK && src->n == ns) rc = ope_cloud_download(ctx, src, source_xyz, nullptr);
  ope_cloud_free(ctx, src);
  return rc;
}

}  // extern "C"
