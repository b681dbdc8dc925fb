// scene_track.cu — ope_scene_track_step: the cluster choice of the reference's online loop (D&L/src/rosinterface.cpp:243-327,
// SURVEY 3.1 and A.0) joined to the batched tracker step, for every camera of a scene batch at once:
//
//   centroid_chain_kernel          compute3DCentroid of every tracking camera's source and of its frame's clusters, one launch
//   gate (host)                    one read-back; the first cluster in rank order whose centroid is inside the gate
//   rounds                         round r: scene_cut_kernel cuts the round's clusters, then ONE tracker step (tracker_step_batch,
//                                  the body of ope_pose_tracker_step_batch) over the round's tracking steps and acquisition tries
//   commit (host)                  an accepted try's tracker state and source are swapped into the caller's tracker
//
// The call is defined as a serial loop of public calls (include/ope_cuda.h); running each round as one step batch keeps libc
// rand() consumption in that loop's order, since the step batch draws in tracker order.
#include <chrono>
#include <climits>
#include <cmath>
#include <cstring>
#include <limits>
#include <vector>

#include "ope_host.cuh"

namespace ope {
namespace {

// one centroid: the points of pts[0 .. n) whose label is `want` (labels null: every point), finite ones only
struct CentroidJob { const float4* pts; const int* labels; int n; int want; };

// One warp per job. The warp walks the points in index order, kDepth x 32 at a time: a ballot per 32 selects the finite points
// carrying the wanted label, the batch goes to the warp's slice of shared memory, and every lane adds the selected points in index
// order into three float chains: the serial sums of compute3DCentroid bit for bit (-fmad=false, round-to-nearest adds). The next
// batch's global loads are issued before the chain runs, so the 256 adds of a batch (about 1 000 cycles) cover the memory latency,
// and the broadcast loads from shared memory do not depend on the chain. out[j] = (sum / count per axis, count as int bits).
constexpr int kCentroidThreads = 256;
constexpr int kDepth = 8;
__global__ void __launch_bounds__(kCentroidThreads) centroid_chain_kernel(const CentroidJob* __restrict__ jobs, int n_jobs,
                                                                           float4* __restrict__ out) {
  __shared__ float4 tiles[kCentroidThreads / 32][kDepth * 32];
  const int j = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (j >= n_jobs) return;
  float4* tile = tiles[threadIdx.x >> 5];
  const CentroidJob c = jobs[j];
  float4 p[kDepth];
  bool keep[kDepth];
  auto fetch = [&](int base) {
#pragma unroll
    for (int d = 0; d < kDepth; ++d) {
      const int i = base + d * 32 + lane;
      keep[d] = false;
      p[d] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      if (i < c.n) {
        p[d] = c.pts[i];
        keep[d] = isfinite(p[d].x) && isfinite(p[d].y) && isfinite(p[d].z) && (!c.labels || c.labels[i] == c.want);
      }
    }
  };
  float sx = 0.0f, sy = 0.0f, sz = 0.0f;
  int count = 0;
  fetch(0);
  for (int t0 = 0; t0 < c.n; t0 += kDepth * 32) {
    unsigned m[kDepth];
#pragma unroll
    for (int d = 0; d < kDepth; ++d) {
      m[d] = __ballot_sync(0xffffffffu, keep[d]);
      count += __popc(m[d]);
      tile[d * 32 + lane] = p[d];
    }
    __syncwarp();
    fetch(t0 + kDepth * 32);   // the next batch, in flight during the chain
#pragma unroll
    for (int d = 0; d < kDepth; ++d) {
      const float4* q = tile + d * 32;
      if (m[d] == 0xffffffffu) {
#pragma unroll
        for (int k = 0; k < 32; ++k) { sx = __fadd_rn(sx, q[k].x); sy = __fadd_rn(sy, q[k].y); sz = __fadd_rn(sz, q[k].z); }
      } else {
        for (unsigned b = m[d]; b; b &= b - 1) {   // warp-uniform: the selected points in ascending order
          const float4 v = q[__ffs(b) - 1];
          sx = __fadd_rn(sx, v.x); sy = __fadd_rn(sy, v.y); sz = __fadd_rn(sz, v.z);
        }
      }
    }
    __syncwarp();
  }
  if (lane == 0) {
    const float f = (float)(unsigned)count;
    out[j] = count ? make_float4(__fdiv_rn(sx, f), __fdiv_rn(sy, f), __fdiv_rn(sz, f), __int_as_float(count))
                   : make_float4(0.0f, 0.0f, 0.0f, __int_as_float(0));
  }
}

// every job's centroid, in job order, on the host
int centroids_device(ope_ctx* ctx, const std::vector<CentroidJob>& jobs, std::vector<float4>& out) {
  out.clear();
  if (jobs.empty()) return OPE_OK;
  const int n = (int)jobs.size();
  Scratch<CentroidJob> d_jobs(ctx);
  Scratch<float4> d_out(ctx);
  OPE_TRY(d_jobs.alloc(jobs.size())); OPE_TRY(d_out.alloc(jobs.size()));
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_jobs.p, jobs.data(), jobs.size() * sizeof(CentroidJob), cudaMemcpyHostToDevice, ctx->stream));
  centroid_chain_kernel<<<div_up((size_t)n * 32, kCentroidThreads), kCentroidThreads, 0, ctx->stream>>>(d_jobs.p, n, d_out.p);
  OPE_TRY(check_launch(ctx, "centroid_chain_kernel"));
  return download(ctx, d_out.p, jobs.size(), out);
}

// the centroid jobs of frame F's clusters in rank order (one job, the whole cloud, when there is no plane)
void cluster_jobs(const ope_scene_batch::Frame& F, std::vector<CentroidJob>& jobs) {
  if (F.status != OPE_OK) return;
  if (F.info.n_clusters < 0) { jobs.push_back(CentroidJob{F.pts, nullptr, F.info.n_cropped, INT_MIN}); return; }
  for (int k = 0; k < F.info.n_clusters; ++k) jobs.push_back(CentroidJob{F.pts, F.labels, F.info.n_cropped, k});
}

int candidates(const ope_scene_batch::Frame& F) { return F.status != OPE_OK ? 0 : F.info.n_clusters < 0 ? 1 : F.info.n_clusters; }

bool accepted(const ope_track_params& tp, const ope_pose_result& r) { return r.fitness < tp.accept_fitness || r.align_strength > tp.accept_strength; }

// one camera of the call
struct Cam {
  bool searching = false;        // acquisition: tries left
  bool reacq = false;            // came to acquisition through a failed gate
  int limit = 0;                 // tries this call may make
  int chosen = -1;               // tracking: the cluster inside the gate
  const ope_cloud* model = nullptr;   // acquisition: the pristine model
};

// a temporary tracker and its source: one acquisition try
struct Try {
  size_t cam = 0;
  ope_pose_tracker* t = nullptr;
  ope_cloud* src = nullptr;
};

double ms_since(std::chrono::steady_clock::time_point t0) {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
}

}  // namespace
}  // namespace ope

using namespace ope;

extern "C" {

void ope_track_params_default(ope_track_params* p) {
  if (!p) return;
  p->accept_fitness = 1e-4;     // rosinterface.cpp acceptance (SURVEY A.0)
  p->accept_strength = 0.4;
  p->gate = 0.05f;              // 5 cm between the cluster's and the model's centroids (rosinterface.cpp:269-273)
  p->max_tries = 0;
  p->reacquire = 1;
}

int ope_cloud_centroid(ope_ctx* ctx, const ope_cloud* cloud, float c[3], int32_t* n_used) {
  OPE_ENTER(ctx);
  if (!ctx || !cloud || !c || cloud->ctx != ctx || cloud->n > (size_t)INT_MAX) return OPE_ERR_INVALID;
  std::vector<float4> h;
  OPE_TRY(centroids_device(ctx, {CentroidJob{cloud->pts, nullptr, (int)cloud->n, INT_MIN}}, h));
  c[0] = h[0].x; c[1] = h[0].y; c[2] = h[0].z;
  if (n_used) std::memcpy(n_used, &h[0].w, sizeof(int32_t));
  return OPE_OK;
}

int ope_scene_batch_centroids(const ope_scene_batch* s, size_t frame, float* xyz, int32_t* n_out) {
  if (!s || frame >= s->frames.size() || !n_out) return OPE_ERR_INVALID;
  ope_ctx* ctx = s->ctx;
  OPE_ENTER(ctx);
  std::vector<CentroidJob> jobs;
  cluster_jobs(s->frames[frame], jobs);
  if (!jobs.empty() && !xyz) return OPE_ERR_INVALID;
  std::vector<float4> h;
  OPE_TRY(centroids_device(ctx, jobs, h));
  for (size_t k = 0; k < h.size(); ++k) { xyz[3 * k] = h[k].x; xyz[3 * k + 1] = h[k].y; xyz[3 * k + 2] = h[k].z; }
  *n_out = (int32_t)h.size();
  return OPE_OK;
}

int ope_scene_track_phase_ms(const ope_ctx* ctx, double* out, int cap, int32_t* n_out) {
  if (!ctx) return OPE_ERR_INVALID;
  const std::vector<double>& v = ctx->track_phase_ms;
  for (int i = 0; out && i < cap && i < (int)v.size(); ++i) out[i] = v[(size_t)i];
  if (n_out) *n_out = (int32_t)v.size();
  return OPE_OK;
}

int ope_scene_track_step(const ope_scene_batch* s, const ope_track_params* tp, ope_pose_tracker* const* trackers, ope_cloud** sources,
                         size_t n, ope_pose_result* results, ope_track_choice* choice, int32_t* status) {
  if (!s) return OPE_ERR_INVALID;
  ope_ctx* ctx = s->ctx;
  OPE_ENTER(ctx);
  if (n != s->frames.size()) return fail(ctx, OPE_ERR_INVALID, "%zu cameras for a scene batch of %zu frames", n, s->frames.size());
  if (n && (!trackers || !sources || !results || !choice)) return OPE_ERR_INVALID;
  if (n == 0) return OPE_OK;
  OPE_TRY(step_batch_check(ctx, trackers, sources, nullptr, n));
  for (size_t i = 0; i < n; ++i)
    if (sources[i]->n > (size_t)INT_MAX) return fail(ctx, OPE_ERR_INVALID, "source %zu has more than INT_MAX points", i);
  ope_track_params TP;
  if (tp) TP = *tp; else ope_track_params_default(&TP);
  ctx->track_phase_ms.assign(2, 0.0);
  std::vector<int32_t> code(n, OPE_OK);   // status[i]
  const float nan = std::numeric_limits<float>::quiet_NaN();

  // ---- branches; centroids of every tracking camera's source and of its frame's clusters, one launch, one read-back ----
  auto t0 = std::chrono::steady_clock::now();
  std::vector<Cam> cams(n);
  std::vector<CentroidJob> jobs;
  std::vector<size_t> job0(n, 0);
  for (size_t i = 0; i < n; ++i) {
    const ope_scene_batch::Frame& F = s->frames[i];
    std::memset(&results[i], 0, sizeof(results[i]));
    choice[i] = ope_track_choice{OPE_TRACK_NOT_FOUND, -1, 0, nan};
    if (F.status != OPE_OK) {
      choice[i].mode = OPE_TRACK_NO_SCENE;
      code[i] = F.status;
      continue;
    }
    if (trackers[i]->firstTimePose == 0) { cams[i].searching = true; continue; }
    job0[i] = jobs.size();
    jobs.push_back(CentroidJob{sources[i]->pts, nullptr, (int)sources[i]->n, INT_MIN});
    cluster_jobs(F, jobs);
  }
  std::vector<float4> cen;
  OPE_TRY(centroids_device(ctx, jobs, cen));
  for (size_t i = 0; i < n; ++i) {
    Cam& c = cams[i];
    if (choice[i].mode == OPE_TRACK_NO_SCENE || c.searching) continue;
    const float4 m = cen[job0[i]];
    const int K = candidates(s->frames[i]);
    float nearest = nan;
    for (int k = 0; k < K; ++k) {
      const float4 q = cen[job0[i] + 1 + (size_t)k];
      const float dx = q.x - m.x, dy = q.y - m.y, dz = q.z - m.z;
      const float d = sqrtf((dx * dx + dy * dy) + dz * dz);   // float, no contraction (-ffp-contract=off)
      if (!(d >= nearest)) nearest = d;
      if (d < TP.gate) { c.chosen = k; choice[i].gate_distance = d; break; }
    }
    if (c.chosen >= 0) { choice[i].mode = OPE_TRACK_TRACKED; choice[i].cluster = c.chosen; continue; }
    choice[i].gate_distance = nearest;
    if (TP.reacquire) { c.searching = true; c.reacq = true; }
    else choice[i].mode = OPE_TRACK_LOST;
  }
  for (size_t i = 0; i < n; ++i) {
    Cam& c = cams[i];
    if (!c.searching) continue;
    const int K = candidates(s->frames[i]);
    c.limit = TP.max_tries > 0 ? std::min(K, (int)TP.max_tries) : K;
    c.model = trackers[i]->cloudModel ? trackers[i]->cloudModel : sources[i];
    c.searching = c.limit > 0;
  }
  ctx->track_phase_ms[0] = ms_since(t0);

  // ---- rounds: round r = the tracking steps (r == 0) and the rank-r tries, in camera order, as one tracker step ----
  std::vector<Try> tries;   // this round's temporaries
  struct Release {
    ope_ctx* ctx; std::vector<Try>& v;
    void operator()() {
      for (Try& x : v) { if (x.t) ope_pose_tracker_destroy(x.t); if (x.src) ope_cloud_free(ctx, x.src); }
      v.clear();
    }
    ~Release() { (*this)(); }
  } release{ctx, tries};
  double commit_ms = 0;
  for (int r = 0;; ++r) {
    t0 = std::chrono::steady_clock::now();
    std::vector<ope_pose_tracker*> ts;
    std::vector<ope_cloud*> ss;
    std::vector<size_t> cam_of;
    std::vector<int> try_of, rank_of;
    for (size_t i = 0; i < n; ++i) {
      Cam& c = cams[i];
      if (r == 0 && c.chosen >= 0) {
        ts.push_back(trackers[i]); ss.push_back(sources[i]); cam_of.push_back(i); try_of.push_back(-1); rank_of.push_back(c.chosen);
      } else if (c.searching) {
        Try x;
        x.cam = i;
        OPE_TRY(ope_pose_tracker_create(ctx, &trackers[i]->prm, &x.t));
        tries.push_back(x);
        OPE_TRY(cloud_alloc(ctx, c.model->n, false, &tries.back().src));
        OPE_CUDA_TRY(ctx, cudaMemcpyAsync(tries.back().src->pts, c.model->pts, c.model->n * sizeof(float4), cudaMemcpyDeviceToDevice,
                                          ctx->stream));
        ts.push_back(x.t); ss.push_back(tries.back().src); cam_of.push_back(i); try_of.push_back((int)tries.size() - 1); rank_of.push_back(r);
      }
    }
    if (ts.empty()) break;
    const size_t m = ts.size();
    // the round's targets: cluster rank_of[j] of frame cam_of[j] (the whole cropped cloud without a plane), as ope_scene_pose_batch cuts
    std::vector<SceneCut> cuts;
    std::vector<size_t> off(m, 0), cnt(m, 0);
    size_t total = 0;
    for (size_t j = 0; j < m; ++j) {
      const ope_scene_batch::Frame& F = s->frames[cam_of[j]];
      SceneCut cut{F.pts, F.labels, F.info.n_cropped, INT_MIN, (long long)total};
      if (F.info.n_clusters >= 0) { cut.want = rank_of[j]; cnt[j] = (size_t)F.sizes[(size_t)rank_of[j]]; }
      else cnt[j] = (size_t)F.info.n_cropped;
      off[j] = total;
      total += cnt[j];
      if (cnt[j]) cuts.push_back(cut);
    }
    Scratch<float4> buf(ctx);
    Scratch<SceneCut> d_cuts(ctx);
    OPE_TRY(buf.alloc(total)); OPE_TRY(d_cuts.alloc(cuts.size()));
    if (!cuts.empty()) {
      OPE_CUDA_TRY(ctx, cudaMemcpyAsync(d_cuts.p, cuts.data(), cuts.size() * sizeof(SceneCut), cudaMemcpyHostToDevice, ctx->stream));
      OPE_TRY(scene_cut_device(ctx, d_cuts.p, (int)cuts.size(), buf.p));
    }
    std::vector<ope_cloud> views(m);
    std::vector<ope_frame_input> inputs(m);
    for (size_t j = 0; j < m; ++j) {
      inputs[j] = ope_frame_input{nullptr, 0, 0, 0, nullptr};
      if (!cnt[j]) continue;
      views[j].ctx = ctx; views[j].n = cnt[j]; views[j].pts = buf.p + off[j];
      inputs[j].cloud = &views[j];
    }
    std::vector<ope_pose_result> res(m);
    std::vector<int32_t> st(m, 1);   // 1: not reached (the step stopped as a whole)
    const int rc = tracker_step_batch(ctx, ts.data(), ss.data(), inputs.data(), m, nullptr, res.data(), st.data());
    for (size_t j = 0; j < m; ++j)
      if (rc != OPE_OK && st[j] == 1) return rc;
    for (size_t j = 0; j < m; ++j) {   // the step replaced the sources it advanced
      if (try_of[j] < 0) sources[cam_of[j]] = ss[j];
      else tries[(size_t)try_of[j]].src = ss[j];
    }
    ctx->track_phase_ms.push_back(ms_since(t0));
    // ---- outcomes; an accepted try's state and source go to the caller's tracker (on this thread: the clouds are this context's) ----
    t0 = std::chrono::steady_clock::now();
    for (size_t j = 0; j < m; ++j) {
      const size_t i = cam_of[j];
      Cam& c = cams[i];
      results[i] = res[j];
      code[i] = st[j];
      if (try_of[j] < 0) continue;   // a tracking step: TRACKED whatever its code
      choice[i].tries++;
      if (st[j] == OPE_OK && accepted(TP, res[j])) {
        Try& x = tries[(size_t)try_of[j]];
        ope_pose_tracker* t = trackers[i];
        std::swap(t->firstTimePose, x.t->firstTimePose);
        std::swap(t->fitnessScoreFine, x.t->fitnessScoreFine);
        std::swap(t->alignedStrength, x.t->alignedStrength);
        std::swap(t->alignedSource, x.t->alignedSource);
        std::swap(t->cloudModel, x.t->cloudModel);
        std::swap(sources[i], x.src);   // the temporary now holds the caller's old state and source: released with it
        choice[i].mode = c.reacq ? OPE_TRACK_REACQUIRED : OPE_TRACK_ACQUIRED;
        choice[i].cluster = r;
        c.searching = false;
      } else if (r + 1 >= c.limit) {
        c.searching = false;       // NOT_FOUND
      }
    }
    release();
    commit_ms += ms_since(t0);
  }
  ctx->track_phase_ms[1] = commit_ms;
  if (status) std::memcpy(status, code.data(), n * sizeof(int32_t));
  for (size_t i = 0; i < n; ++i) {
    if (code[i] == OPE_OK) continue;
    if (choice[i].mode == OPE_TRACK_NO_SCENE) return fail(ctx, code[i], "camera %zu: the frame's scene failed", i);
    const std::string msg = ctx->error;
    return fail(ctx, code[i], "camera %zu: %s", i, msg.c_str());
  }
  return OPE_OK;
}

}  // extern "C"
