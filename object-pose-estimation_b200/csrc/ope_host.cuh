// ope_host.cuh — host-side internals of libope_cuda.so: context, device clouds, cached grids, scratch memory.
#pragma once
#include <cuda_runtime.h>
#include <sched.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <functional>
#include <map>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "../../include/ope_cuda.h"
#include "ope_grid.cuh"

struct ope_cloud;
// SURVEY 8f-3: the frame-invariant model side of the coarse stage (1 cm sample + normals, FPFH descriptors), keyed by the
// content of the full-resolution source cloud it was computed from and by the parameters that shape it
struct ModelCacheEntry {
  unsigned long long hash = 0;
  size_t n = 0;
  float leaf = 0, radius = 0;
  int k = 0;
  ope_cloud* sp = nullptr;   // owned
  float* fs = nullptr;       // owned (device, sp->n * 33)
  unsigned long long stamp = 0;
};

// ope_pose_batch: the device copy of the model it was last called with and everything frame-invariant computed from it
struct BatchModelCache {
  unsigned long long hash = 0;   // of the caller's host buffer
  size_t n = 0;
  float leaf = 0, radius = 0;
  int k = 0;
  ope_cloud* model = nullptr;    // owned: full-resolution model
  ope_cloud* sp = nullptr;       // owned: its coarse sample with normals
  float* fs = nullptr;           // owned: FPFH of sp
  float rigid[16];               // dense Umeyama of the model onto itself
};

struct ope_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool owns_stream = false;
  cudaMemPool_t pool = nullptr;   // this context's own stream-ordered pool: allocations of concurrent contexts (the lanes of
                                  // the frame-spanning batches) never wait on each other's frees
  int sm_count = 148;
  int64_t launches = 0;
  std::string error;
  void* pinned = nullptr;      // small pinned staging buffer for scalar read-backs
  size_t pinned_bytes = 0;
  void* stage = nullptr;       // grow-only pinned staging arena for cloud uploads / downloads (host <-> device at PCIe speed)
  size_t stage_bytes = 0;
  cudaEvent_t kev[3][2] = {{nullptr, nullptr}, {nullptr, nullptr}, {nullptr, nullptr}};  // [which][begin/end] around the dominant kernels
  bool kev_valid[3] = {false, false, false};
  std::vector<ope_ctx*> workers;  // run_chunks_on_lanes: the helper lanes' contexts (own stream, pool, staging), kept warm between calls
  cudaEvent_t sync_event = nullptr;  // set: waits sleep on this cudaEventBlockingSync event instead of spinning in cudaStreamSynchronize
                                     // (lanes beyond the host's core count)
  unsigned* ticket = nullptr;        // device counter, zero between kernels (see bbox_partial_kernel)
  bool sync_yield = false;           // with sync_event: poll it and sched_yield() between polls instead of sleeping
  // both set only by pose_one_frame (pipeline.cu) for the duration of one ope_pose_batch frame outside the frame-spanning launches
  bool icp_prefer_small = false;  // small clouds: prefer the thread-per-query ICP kernel (least device time per alignment)
  int icp_max_blocks = 0;      // > 0: cap of the cooperative icp_kernel grid (the frame shares the SMs with the other lanes)
  int64_t feature_knn_gemm_queries = 0;  // queries answered through the tcgen05 distance GEMM ...
  int64_t feature_knn_fallbacks = 0;     // ... of which the exact kernel had to re-answer (candidate set not provably complete)
  bool batch_timing = false;             // ope_pose_batch: per-stage CUDA-event laps of the frame-spanning launches
  double batch_stage_ms[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  BatchModelCache batch_model;
  std::vector<ModelCacheEntry> model_cache;   // at most 4 entries, least recently used replaced (pipeline.cu)
  unsigned long long model_cache_clock = 0;
  int64_t model_cache_hits = 0, model_cache_misses = 0;
  std::vector<double> track_phase_ms;   // ope_scene_track_step's last call: gate, commit, round 0, 1, ... (host wall ms)
};

// PoseEstimator (D&L/include/poseestimator.h): the state one tracker carries from frame to frame
struct ope_pose_tracker {
  ope_ctx* ctx = nullptr;
  ope_pose_params prm;
  int firstTimePose = 0;           // D&L/include/poseestimator.h:50-53
  double fitnessScoreFine = 10;
  double alignedStrength = 0.0;
  ope_cloud* alignedSource = nullptr;
  ope_cloud* cloudModel = nullptr;
  double stage_ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  bool timing = true;              // per-stage CUDA-event laps (each lap synchronises); the batch path turns them off
  // frame-invariant model side of the coarse stage (SURVEY 8f-3): the 1 cm sample of the pristine model with its normals,
  // and its FPFH descriptors. Not owned. Used by the first call of this tracker only (the source IS the model then).
  const ope_cloud* cache_sp = nullptr;
  const float* cache_fs = nullptr;
  size_t cache_model_n = 0;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, evt0 = nullptr, evt1 = nullptr;
};

// How points are binned into cells: c = (int)floorf((p - o) * inv) - min_b, per axis.
//  * search grids: o = bbox min, inv = 1/h, min_b = 0
//  * PCL voxel frames (UniformSampling / VoxelGrid, SURVEY A.1/A.2): o = 0, inv = 1/leaf, min_b = floor(min*inv)
struct Binning {
  float o[3];
  float inv[3];
  int min_b[3];
  int dim[3];
  int morton_bits;  // > 0: cells are numbered by the Morton code of (cx,cy,cz) (search grids); 0: x-fastest linear index
};

struct GridEntry {
  int bits = 0;
  ope::GridView view{};
  int* cell_start = nullptr;
  float4* sorted = nullptr;
  int64_t ncells = 0;
};

struct ope_cloud {
  ope_ctx* ctx = nullptr;
  size_t n = 0;
  float4* pts = nullptr;       // x, y, z, 1
  float4* normals = nullptr;   // nx, ny, nz, curvature (optional)
  bool bbox_valid = false;
  float bbox[6];               // min xyz, max xyz over finite points
  int n_finite = 0;
  std::vector<GridEntry> grids;
};

// ope_scene_batch_create's result: the cropped clouds and labels of every frame, resident on the device (segment.cu)
struct ope_scene_batch {
  ope_ctx* ctx = nullptr;
  struct Frame {
    const float4* pts = nullptr;   // n_cropped points (device, inside one of `blocks`)
    const int* labels = nullptr;   // n_cropped labels (device)
    ope_scene_frame info{};
    int status = OPE_OK;
    std::vector<int> sizes;        // point count of cluster 0, 1, ...
  };
  std::vector<Frame> frames;
  std::vector<void*> blocks;       // device allocations, one pair per chunk
};

namespace ope {

inline int fail(ope_ctx* ctx, int code, const char* fmt, ...) {
  if (ctx) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    ctx->error = buf;
  }
  return code;
}

#define OPE_CUDA_TRY(ctx, expr)                                                                       \
  do {                                                                                                \
    cudaError_t e__ = (expr);                                                                         \
    if (e__ != cudaSuccess)                                                                           \
      return ope::fail((ctx), OPE_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

#define OPE_TRY(expr)            \
  do {                           \
    int rc__ = (expr);           \
    if (rc__ != OPE_OK) return rc__; \
  } while (0)

// stream-ordered scratch allocation (cudaMallocAsync pool, release threshold = keep everything cached)
template <typename T>
inline int dalloc(ope_ctx* ctx, T** p, size_t count) {
  *p = nullptr;
  if (count == 0) count = 1;
  if (ctx->pool) OPE_CUDA_TRY(ctx, cudaMallocFromPoolAsync((void**)p, count * sizeof(T), ctx->pool, ctx->stream));
  else OPE_CUDA_TRY(ctx, cudaMallocAsync((void**)p, count * sizeof(T), ctx->stream));
  return OPE_OK;
}
template <typename T>
inline void dfree(ope_ctx* ctx, T* p) {
  if (p) cudaFreeAsync((void*)p, ctx->stream);
}
// RAII scratch buffer
template <typename T>
struct Scratch {
  ope_ctx* ctx;
  T* p = nullptr;
  explicit Scratch(ope_ctx* c) : ctx(c) {}
  ~Scratch() { dfree(ctx, p); }
  int alloc(size_t count) { return dalloc(ctx, &p, count); }
  Scratch(const Scratch&) = delete;
  Scratch& operator=(const Scratch&) = delete;
};

// wait for everything queued on the context's stream
inline cudaError_t stream_sync(ope_ctx* ctx) {
  if (!ctx->sync_event) return cudaStreamSynchronize(ctx->stream);
  cudaError_t e = cudaEventRecord(ctx->sync_event, ctx->stream);
  if (e != cudaSuccess) return e;
  if (!ctx->sync_yield) return cudaEventSynchronize(ctx->sync_event);
  while ((e = cudaEventQuery(ctx->sync_event)) == cudaErrorNotReady) sched_yield();   // poll, but hand the core to the other workers
  return e;
}

inline int check_launch(ope_ctx* ctx, const char* what) {
  ctx->launches++;
  cudaError_t e = cudaPeekAtLastError();
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(ctx, OPE_ERR_CUDA, "launch of %s failed: %s", what, cudaGetErrorString(e));
  }
  return OPE_OK;
}

// copy n elements from device to a host vector and wait
template <typename T>
int download(ope_ctx* ctx, const T* d, size_t n, std::vector<T>& h) {
  h.resize(n);
  if (n == 0) return OPE_OK;
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(h.data(), d, n * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
  OPE_CUDA_TRY(ctx, stream_sync(ctx));
  return OPE_OK;
}

// copy `bytes` from device to the pinned staging buffer and wait; returns the host pointer
inline int read_back(ope_ctx* ctx, const void* dsrc, size_t bytes, void** host) {
  if (bytes > ctx->pinned_bytes) return fail(ctx, OPE_ERR_INVALID, "read_back larger than staging buffer");
  OPE_CUDA_TRY(ctx, cudaMemcpyAsync(ctx->pinned, dsrc, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  OPE_CUDA_TRY(ctx, stream_sync(ctx));
  *host = ctx->pinned;
  return OPE_OK;
}

// Entry guard of every extern "C" function that takes a context: the calling host thread's current device becomes the
// context's device (a process may hold contexts on several GPUs; launches and attribute calls go to the CURRENT device).
inline void enter(const ope_ctx* ctx) {
  if (!ctx) return;
  int d = -1;
  if (cudaGetDevice(&d) != cudaSuccess || d != ctx->device) cudaSetDevice(ctx->device);
}
#define OPE_ENTER(ctx) ope::enter(ctx)

// Opt a kernel in to `bytes` of dynamic shared memory (B200: up to 227 KB per block). The opt-in is a property of the
// (device, function) pair, shared by every stream and host thread of the process (ope_pose_batch runs several contexts
// concurrently): only ever raise it, under a lock, per device.
inline int dyn_smem(ope_ctx* ctx, const void* fn, size_t bytes) {
  static std::mutex mu;
  static std::map<std::pair<int, const void*>, size_t> granted;
  std::lock_guard<std::mutex> lock(mu);
  size_t& have = granted[std::make_pair(ctx->device, fn)];
  if (bytes > have) {
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return fail(ctx, OPE_ERR_CUDA, "shared memory opt-in of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
    have = bytes;
  }
  return OPE_OK;
}

inline unsigned div_up(size_t a, size_t b) { return (unsigned)((a + b - 1) / b); }

// pinned staging arena of at least `bytes` (grow-only; the previous contents are not preserved)
inline int stage_reserve(ope_ctx* ctx, size_t bytes, void** out) {
  if (bytes > ctx->stage_bytes) {
    if (ctx->stage) cudaFreeHost(ctx->stage);
    ctx->stage = nullptr; ctx->stage_bytes = 0;
    size_t want = bytes + bytes / 4 + (1 << 16);
    if (cudaHostAlloc(&ctx->stage, want, cudaHostAllocDefault) != cudaSuccess) {
      cudaGetLastError();
      return fail(ctx, OPE_ERR_CUDA, "pinned staging allocation of %zu bytes failed", want);
    }
    ctx->stage_bytes = want;
  }
  *out = ctx->stage;
  return OPE_OK;
}

// ---- implemented in grid.cu ----
int cloud_alloc(ope_ctx* ctx, size_t n, bool with_normals, ope_cloud** out);
int cloud_bbox(ope_ctx* ctx, ope_cloud* c);
// cached search grid with cell edge ~h (adjusted to respect the cell cap)
int cloud_grid(ope_ctx* ctx, const ope_cloud* c, float h, GridView* out);
// any cached search grid of the cloud (builds the default nearest-neighbour grid when there is none): used for the
// Morton work order of a source cloud
int cloud_any_grid(ope_ctx* ctx, const ope_cloud* c, GridView* out);
// suggested cell edge for k-NN queries against this cloud (surface-density heuristic)
float knn_cell_size(const ope_cloud* c, int k);
int exclusive_scan_i32(ope_ctx* ctx, int* data, size_t n);
// build cell_start (ncells+1) and the cell-sorted, index-ordered point array for an arbitrary binning, over its cells
// [c0, c0 + nwin) (nwin < 0: to the last cell; cell_start is indexed by cell - c0); points of other cells are left out
int build_cells(ope_ctx* ctx, const float4* pts, size_t n, const Binning& bin, int** cell_start, float4** sorted, int64_t c0 = 0,
                int64_t nwin = -1);
// device-side versions used by the pipeline
int uniform_sample_device(ope_ctx* ctx, ope_cloud* cloud, float leaf, int** d_idx, size_t* out_n);
int gather_cloud(ope_ctx* ctx, const ope_cloud* cloud, const int* d_idx, size_t n, ope_cloud** out);
// 64-bit content hash of a device cloud's points (order-sensitive), for the model-side cache
int cloud_content_hash(ope_ctx* ctx, const ope_cloud* cloud, unsigned long long* out);

// ---- features.cu ----
int normals_device(ope_ctx* ctx, ope_cloud* cloud, int k, const float vp[3]);
// NormalEstimation with setRadiusSearch(radius): neighbours d2 < radius^2, summed in (d2, index) order (features.cu)
int normals_radius_device(ope_ctx* ctx, ope_cloud* cloud, float radius, const float vp[3]);
int fpfh_device(ope_ctx* ctx, const ope_cloud* cloud, float radius, float** d_fpfh, float** d_spfh_or_null);
int feature_knn_device(ope_ctx* ctx, const float* d_ftgt, size_t nt, const float* d_fqry, size_t nq, int dim, int k,
                       int* d_idx, float* d_d2);
// exact float32 kernel; d_qlist (n_list entries) restricts it to those queries, nullptr = all nq
int feature_knn_exact_device(ope_ctx* ctx, const float* d_ftgt, size_t nt, const float* d_fqry, size_t nq, int dim, int k,
                             const int* d_qlist, size_t n_list, int* d_idx, float* d_d2);
// ---- featgemm.cu: tcgen05 / TMA distance GEMM + exact re-rank ----
bool feature_knn_gemm_applicable(size_t nt, size_t nq, int dim, int k);
int feature_knn_gemm_device(ope_ctx* ctx, const float* d_ftgt, size_t nt, const float* d_fqry, size_t nq, int dim, int k, int* d_idx,
                            float* d_d2, int* n_fallback);
int remove_nan_normals_device(ope_ctx* ctx, ope_cloud** cloud);

// ---- registration.cu ----
int transform_device(ope_ctx* ctx, const ope_cloud* in, const Mat4& T, ope_cloud* out);
int umeyama_device(ope_ctx* ctx, const float4* src, const float4* tgt, const int* d_isrc, const int* d_itgt, size_t n,
                   float T[16]);
int fitness_device(ope_ctx* ctx, const ope_cloud* src, const ope_cloud* tgt, const Mat4& T, double max_range, double* out);
int icp_device(ope_ctx* ctx, const ope_cloud* src, const ope_cloud* tgt, const ope_icp_params& prm, const Mat4& guess,
               ope_reg_result* res, ope_correspondence* out_corr_host, ope_cloud** out_aligned);
int sacia_device(ope_ctx* ctx, const ope_cloud* src, const float* d_fsrc, const ope_cloud* tgt, const float* d_ftgt,
                 const ope_sacia_params& prm, const ope_rng_table* table, const float* host_src_xyz3, ope_reg_result* res,
                 float* out_errors_host);


// ---- frame-spanning launches (ope_pose_batch, batch.cu): clouds of counts[c] points at c * stride ----
struct SaciaBatch {
  const float4* src; int ns;                               // frame f's source: src + f * src_stride, src_counts[f] <= ns points
  int src_stride; const int* src_counts;                   // (src_stride 0, src_counts null: one source of ns points for every frame)
  const float4* tgt; const int* counts; int stride;        // frame f: tgt + f * stride, counts[f] points
  const float4* tgt_scan;                                  // the same points in any order (null: tgt): what the distance scan reads
  int nr_samples, k_corr, H;
  int h_begin, h_end;                                      // the hypotheses scored: [h_begin, h_end) of 0 .. H-1
  const int* samples; const int* picks;                    // frame f: + f * H * nr_samples
  const int* knn_idx;                                      // frame f: + f * ns * k_corr
  const int* active;                                       // per frame: 0 = skip
  float threshold;
  float* errors;                                           // frames * H (+inf: stopped early, cannot be the winner)
  float* transforms;                                       // frames * H * 16
  int early_exit;                                          // 1: the shared-memory scorer may stop a hypothesis whose partial error
                                                           // already exceeds the frame's lowest complete one (OPE_SACIA_EARLY_EXIT=0: never)
  unsigned* best_bits;                                     // set by sacia_batch_device: per frame, float bits of the lowest complete error
  unsigned short* seed_tab; float4* seed_geo;              // set by sacia_batch_device: per frame, the seed grid of the distance search
  const float4* src_scan;                                  // set by sacia_batch_device: the source in scoring order, .w = original index
};
struct IcpBatchFrame { const float4* src_pts; const float4* src_nrm; int n_src; const float4* tgt_pts; const float4* tgt_nrm; int n_tgt; };
int normals_smem_batch(ope_ctx* ctx, const float4* pts, const int* d_counts, int stride, int clouds, int max_n, int k, const float vp[3],
                       float4* out);
int fpfh_smem_batch(ope_ctx* ctx, const float4* pts, const float4* nrm, const int* d_counts, int stride, int clouds, int max_n, float radius,
                    float* spfh, float* fpfh);
int feature_knn_batch(ope_ctx* ctx, const float* ftgt, const int* d_counts, int stride, int frames, int max_nt, const float* fqry, int nq,
                      int qstride, const int* d_qcounts, int dim, int k, int* out_idx);
// scores hypotheses [h_begin, h_end) of every frame and writes each frame's winner to d_results: from shared memory (grid null,
// every target <= max_nt <= 8 192 points) or, for one frame, through the target's grid index
int sacia_batch_device(ope_ctx* ctx, const SaciaBatch& a, int frames, int max_nt, const GridView* grid, ope_reg_result* d_results);
int fitness_batch_device(ope_ctx* ctx, const float4* tgt, const int* tgt_counts, const float4* src, const int* src_counts, int stride, int frames,
                         int max_nt, const ope_reg_result* d_icp, const int* d_active, double* d_out);
bool icp_small_batch_applicable(const ope_icp_params& prm, size_t n_src, size_t n_tgt);
int icp_small_batch_device(ope_ctx* ctx, const ope_icp_params& prm, const IcpBatchFrame* frames, int n_frames, ope_reg_result* d_results);

// one tracker's state commit (track_commit_kernel): the new alignedSource and the copy that replaces the source, and the dense
// Umeyama of the model onto the source
struct TrackCommit {
  const float4* in; int n_in; int pre;          // points to move: through coarse first (pre = 1), then through fine
  float coarse[16], fine[16];
  float4* out_aligned; float4* out_source;      // n_in points each
  const float4* model; const float4* src; int n_model;   // moments of model[i] -> src[i], i < n_model (0: no Umeyama)
  int nb;                                       // blocks: umeyama_blocks(n_model), or of n_in when there is no Umeyama
};
// the block count of umeyama_device for n pairs
int umeyama_blocks(ope_ctx* ctx, size_t n);
// n commits (device and host copies of the same array); d_rigid: n x 16 floats, written where n_model > 0
int track_commit_device(ope_ctx* ctx, const TrackCommit* d_commits, const TrackCommit* h_commits, int n, float* d_rigid);

// ---- batch.cu: the stages of a chunk of frames ----
static constexpr int kBCap = 4096;        // capacity of a sampled cloud (normals / ICP shared-memory paths)
static constexpr int kBFeatCap = 2048;    // capacity of a 1 cm sample (FPFH shared-memory path)
struct BSampleArgs {
  const float4* const* src;         // frame f's cloud (a shared source is the same pointer in every frame)
  const int* counts;                // its points
  const ope_reg_result* xforms;     // null: points as they are; else frame f's points go through xforms[f] (an identity matrix is not
                                    // the same thing: it turns -0 into +0)
  const int* xform_on;              // with xforms: the frames whose points are transformed (null: all)
  const int* active;                // frames to process (null: all)
  float inv_leaf[2];
  int cap[2];                       // output capacity per leaf
  float4* out[2];                   // leaf l, frame f: out[l] + f * kBCap
  int* out_counts[2];               // leaf l: counts[f]
  int* flags;                       // per frame: |= 1 when a sample overflowed its capacity / the voxel frame is too large
};
// ---- batch.cu: one chunk of frames through the frame-spanning stages (ope_pose_batch, ope_pose_tracker_step_batch) ----
// Per frame i < B: what the caller fills in, what the table hook sees and sets, and what the chunk leaves for the active frames.
struct PoseChunk {
  const ope_frame_input* targets = nullptr;
  size_t first = 0;                          // the chunk's first frame in the call (messages)
  std::vector<int> active;                   // in: frames that try the fast path; out: frames finished here
  std::vector<int> coarse;                   // frames that run SAC-IA (empty: every frame)
  // SAC-IA's source: one cloud with its FPFH for every frame (src_pts, src_fpfh, src_n), or per frame a cloud (src_clouds,
  // src_cloud_n) that the chunk samples at the coarse leaf and describes itself
  const float4* src_pts = nullptr; const float* src_fpfh = nullptr; int src_n = 0;
  std::vector<const float4*> src_clouds; std::vector<int> src_cloud_n;
  std::vector<const float4*> fine_src; std::vector<int> fine_n;   // the fine stage's source (moved by the coarse pose after SAC-IA)
  // the table hook runs once per chunk, before SAC-IA: `active` and `n_src_coarse` are final (it may clear `active` to finish
  // nothing), a per-frame source sample is at src_samples + i * kBCap (device); it points tables[i] at each SAC-IA frame's table
  const float4* src_samples = nullptr;
  std::vector<const ope_rng_table*> tables;
  std::vector<ope_reg_result> coarse_res, fine;
  std::vector<double> fitness;
  std::vector<int> n_src_coarse, n_tgt_coarse, n_src_fine, n_tgt_fine;
  bool ran_coarse(int i) const { return coarse.empty() || coarse[(size_t)i]; }
};
int pose_chunk(ope_ctx* ctx, const ope_pose_params& P, int B, PoseChunk& c, const std::function<int(PoseChunk&)>& tables_hook);
// estimateFinalPose's result for finished frame i: finalPose = rigid * (coarse * fine)
ope_pose_result chunk_pose_result(const PoseChunk& c, int i, const Mat4& rigid);

// ---- pipeline.cu: the lanes of the frame-spanning batches (see there) ----
int run_chunks_on_lanes(ope_ctx* ctx, size_t n, const std::atomic<int>* stop,
                        const std::function<int(ope_ctx*, size_t, size_t, size_t)>& run_chunk, size_t chunk_items = 0);

// ---- track.cu: ope_pose_tracker_step_batch's argument checks (targets may be null: not checked) and its body ----
int step_batch_check(ope_ctx* ctx, ope_pose_tracker* const* trackers, ope_cloud* const* sources, const ope_frame_input* targets, size_t n);
int tracker_step_batch(ope_ctx* ctx, ope_pose_tracker* const* trackers, ope_cloud** sources, const ope_frame_input* targets, size_t n,
                       const ope_rng_table* tables, ope_pose_result* results, int32_t* status);

// ---- segment.cu: one block per cut copies the points of pts[0 .. n) whose label is `want` (INT_MIN: every point; labels may then
// be null) in index order to out + out_off ----
struct SceneCut { const float4* pts; const int* labels; int n; int want; long long out_off; };
int scene_cut_device(ope_ctx* ctx, const SceneCut* d_cuts, int n_cuts, float4* out);

// ---- p2plane.cu: TransformationEstimationPointToPlaneLLS / ...PointToPlane (Levenberg-Marquardt) ----
int point_to_plane_device(ope_ctx* ctx, const float4* src, const float4* tgt, const float4* tgt_n, const int* d_is, const int* d_it,
                          const float* d_d2, size_t n, int kind, Mat4* T, int* n_pairs, double* sum_d2, int32_t* lm_info);

}  // namespace ope
