/* ope_cuda.h — C ABI of libope_cuda.so: the B200 (sm_100a) implementation of the registration hot path of
 * gopi-erabati/Object-Pose-Estimation.
 *
 * The reference has no FFI for this path: it instantiates header-only PCL templates in its own translation
 * units (SURVEY 8b). The entry points below are what the PCL-style shim classes in include/ope_pcl/ bind;
 * each cites the reference interface it replaces (paths relative to /root/reference; VP =
 * DetectAndLocalize/include/pcl/registration; [UPSTREAM] = un-vendored PCL, restated in SURVEY Appendix A).
 *
 * Conventions
 *   - every function returns OPE_OK (0) or a negative OPE_ERR_* (include/ope_types.h); nothing throws or
 *     aborts across the ABI; ope_last_error() returns a description of the last failure of that context;
 *   - host buffers are caller-owned and only read/written during the call; device memory is library-owned
 *     behind opaque handles; points are float triples `stride` BYTES apart starting at byte `offset`
 *     (so PCL's 32-byte PointXYZRGB / 48-byte PointXYZRGBNormal structs can be passed as they are, A.9);
 *     normals are float triples (+ curvature where stated); matrices are 4x4 column-major (Eigen::Matrix4f);
 *   - calls are synchronous from the caller's view (like align()/compute()), one ope_ctx per host thread;
 *   - there is NO CPU fallback: without a usable CUDA device every call fails with OPE_ERR_NO_DEVICE.
 */
#ifndef OPE_CUDA_H_
#define OPE_CUDA_H_

#include "ope_types.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ope_ctx ope_ctx;
typedef struct ope_cloud ope_cloud;
typedef struct ope_pose_tracker ope_pose_tracker;
typedef struct ope_comm ope_comm;

/* ---- context -------------------------------------------------------------------------------------- */
/* `stream` is a cudaStream_t to run on (e.g. torch.cuda.current_stream().cuda_stream) or NULL to create one. */
int ope_ctx_create(int device, void* stream, ope_ctx** out);
void ope_ctx_destroy(ope_ctx* ctx);
const char* ope_last_error(const ope_ctx* ctx);
int ope_ctx_synchronize(ope_ctx* ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
int64_t ope_ctx_launch_count(const ope_ctx* ctx);
/* device time (ms, CUDA events on the context's stream) of the last launch of the named dominant kernel:
 * which = 0: icp_kernel (the fused ICP loop), 1: the SAC-IA scorer (sacia_score_batch_kernel or sacia_kernel), 2: featgemm_kernel
 * (tcgen05 feature-distance GEMM). Negative if it never ran. */
double ope_ctx_last_kernel_ms(ope_ctx* ctx, int which);
/* feature-space k-NN bookkeeping: queries answered through the tcgen05 distance GEMM so far, and how many of them the exact
 * float32 kernel re-answered because the candidate set could not be proven complete */
int ope_ctx_feature_knn_stats(const ope_ctx* ctx, int64_t* gemm_queries, int64_t* fallbacks);
/* model-side cache of the pose trackers of this context (SURVEY 8f-3): the reference recomputes the 1 cm sample, normals and FPFH
 * of the source cloud every time the coarse stage runs (D&L/src/poseestimator.cpp:34,116); here a source cloud with the same size
 * and content hash as one seen before (and the same leaf / k / radius) reuses them. Results are bit-identical with and without
 * the cache (OPE_MODEL_CACHE=0 disables it). hits/misses: coarse stages served from / added to the cache. */
int ope_ctx_model_cache_stats(const ope_ctx* ctx, int64_t* hits, int64_t* misses);
/* library / build identification: "ope_cuda <version> sm_100a" */
const char* ope_version(void);

/* ---- clouds (device-resident float4 copies of PCL clouds; SURVEY A.9) -------------------------------- */
/* pcl::PointCloud<PointT> -> device. normals may be NULL. Replaces PCLBase::setInputCloud /
 * Registration::setInputSource / setInputTarget (VP/registration_mod.h:150-200) as the point where data is handed over. */
int ope_cloud_upload(ope_ctx* ctx, const void* pts, size_t n, size_t stride, size_t offset,
                     const void* normals, size_t nstride, size_t noffset, ope_cloud** out);
int ope_cloud_free(ope_ctx* ctx, ope_cloud* cloud);
size_t ope_cloud_size(const ope_cloud* cloud);
int ope_cloud_has_normals(const ope_cloud* cloud);
/* device -> host: xyz as float triples (3*n floats), normals as nx,ny,nz,curvature (4*n floats); either may be NULL */
int ope_cloud_download(ope_ctx* ctx, const ope_cloud* cloud, float* xyz, float* normals4);
/* pcl::copyPointCloud(cloud, indices, out) on the device (D&L/src/poseestimator.cpp:145) */
int ope_cloud_select(ope_ctx* ctx, const ope_cloud* cloud, const int32_t* idx, size_t n, ope_cloud** out);
/* pcl::transformPointCloud[WithNormals] -> new cloud (D&L/src/poseestimator.cpp:68,358; VP/impl/icp_mod.hpp:48-115) */
int ope_cloud_transform(ope_ctx* ctx, const ope_cloud* cloud, const float T[16], ope_cloud** out);
/* drop the cached search grids of a cloud, so the next call rebuilds its index (what setInputTarget's
 * target_cloud_updated_ = true does to the kd-tree, VP/impl/registration_mod.hpp:57-67,80-84) */
int ope_cloud_invalidate(ope_ctx* ctx, ope_cloud* cloud);
/* `*dst += *src` (pcl::PointCloud::operator+=, BM/src/regmeshpcd.cpp:254): src's points are appended to dst on the device;
 * normals are kept only if both clouds carry them; dst's cached search index is dropped. */
int ope_cloud_append(ope_ctx* ctx, ope_cloud* dst, const ope_cloud* src);
/* attach normals computed by ope_normals_knn to the cloud (pcl::copyPointCloud(normals, pointnormal), :201) */
int ope_cloud_set_normals(ope_ctx* ctx, ope_cloud* cloud, const float* normals4);

/* ---- depth image -> cloud (SURVEY 8f-1: the stage before the path) ------------------------------------------ */
/* DataGrabber::rgbd2Pcl + depthToMeter (D&L/src/datagrabber.cpp:9-62,121-174): host uint16 depth (rows x cols, row-major) ->
 * device cloud, compacted in the reference's column-outer / row-inner order, with its row/column swap quirk; Kinect
 * intrinsics are fx = fy = 525, cx = 319.5, cy = 239.5, scale 1000, z_max 2.0 (:34,146-150). */
int ope_depth_to_cloud(ope_ctx* ctx, const uint16_t* depth, int rows, int cols, float fx, float fy, float cx, float cy, float scale,
                       float z_max, ope_cloud** out);
/* the same for a batch of frames already resident on the device, one launch (layout: see csrc/depth.cu) */
int ope_depth_to_cloud_batch(ope_ctx* ctx, const uint16_t* d_depth, int frames, int rows, int cols, float fx, float fy, float cx, float cy,
                             float scale, float z_max, void* d_out, int32_t* d_col_start);

/* ---- scene preparation in front of the path (SURVEY 8f-2) ----------------------------------------------------------------------- */
/* ProcessingPcd::getPassThrough (D&L/src/processingpcd.cpp:8-41): pcl::PassThrough on z, then y, then x; a point survives iff it
 * is finite and inside all three closed intervals. limits = x_min, x_max, y_min, y_max, z_min, z_max (the reference's argument
 * order). *out: the surviving points in input order (device); out_idx (room for ope_cloud_size entries) / out_n may be NULL. */
int ope_pass_through(ope_ctx* ctx, const ope_cloud* cloud, const float limits[6], ope_cloud** out, int32_t* out_idx, size_t* out_n);
/* pcl::EuclideanClusterExtraction as ObjectSegmentationPlane::getClusters configures it (D&L/src/objectsegmentationplane.cpp:74-90:
 * setClusterTolerance(0.05), sizes 300 .. 1e5): connected components of the graph "squared distance < tolerance^2". labels: one
 * per point — cluster number (0 = largest, as extract() orders them; equal sizes by the smaller first index) or -1. */
int ope_euclidean_clusters(ope_ctx* ctx, const ope_cloud* cloud, float tolerance, int min_size, int max_size, int32_t* labels,
                           int* n_clusters);

/* pcl::SACSegmentation as ObjectSegmentationPlane::getPlaneIndicesAndCoeffSAC configures it (D&L/src/objectsegmentationplane.cpp:
 * 36-55: SACMODEL_PLANE, SAC_RANSAC, threshold 0.01, optimised coefficients; 50 iterations, probability 0.99, the fixed sampling
 * seed of PCL) on a device cloud without NaN points: refined plane (a, b, c, d), ascending inlier indices (out_idx: room for
 * ope_cloud_size entries, may be NULL), RANSAC iterations. *found = 0 when no plane exists. prm == NULL: the reference's values. */
int ope_plane_ransac(ope_ctx* ctx, const ope_cloud* cloud, const ope_segment_params* prm, float coeff[4], int32_t* out_idx, size_t* out_n,
                     int32_t* iterations, int32_t* found);
/* ObjectSegmentationPlane::getSegmentedObjectsOnPlane (D&L/src/objectsegmentationplane.cpp:122-282) on a pass-through-filtered
 * device cloud: table plane, polygonal prism over the padded bounding rectangle of the plane's hull, second plane on the prism's
 * points, Euclidean clusters of the rest. labels (ope_cloud_size entries): OPE_SEG_OUTSIDE_PRISM / OPE_SEG_PLANE /
 * OPE_SEG_NO_CLUSTER / cluster number (0 = largest = cloudClusterVector order). plane1 / plane2 / iters may be NULL.
 * *n_clusters = -1 when a plane fit failed (the reference then hands the whole cloud on, :149-152). */
int ope_segment_objects_on_plane(ope_ctx* ctx, const ope_cloud* cloud, const ope_segment_params* prm, int32_t* labels, float plane1[4],
                                 float plane2[4], int32_t iters[2], int32_t* n_clusters);
void ope_segment_params_default(ope_segment_params* p);

/* ---- depth images -> segmented scenes -> poses, many frames per call -------------------------------------------------------------- */
/* The reference's online loop for every Kinect frame (D&L/src/rosinterface.cpp:212-250): rgbd2Pcl -> getPassThrough ->
 * getSegmentedObjectsOnPlane -> estimateFinalPose on a cluster, here for a stack of frames at once. */
typedef struct ope_scene_batch ope_scene_batch;   /* opaque; holds its ope_ctx and must be destroyed before it */
void ope_scene_params_default(ope_scene_params* p);
/* depth: frames x rows x cols uint16, host OR device memory. For every frame: ope_depth_to_cloud -> ope_pass_through ->
 * ope_segment_objects_on_plane (DataGrabber::rgbd2Pcl, D&L/src/datagrabber.cpp:9-62; ProcessingPcd::getPassThrough,
 * D&L/src/processingpcd.cpp:8-41; ObjectSegmentationPlane::getSegmentedObjectsOnPlane, D&L/src/objectsegmentationplane.cpp:122-282),
 * each frame's result equal to those calls' bit for bit. The cropped clouds and their labels stay on the device in *out.
 * info / status: one entry per frame (status may be NULL); a degenerate RANSAC sample fails only its frame (OPE_ERR_UNSUPPORTED).
 * Returns OPE_OK when every frame succeeded, else the first failing frame's code (*out is then still valid). */
int ope_scene_batch_create(ope_ctx* ctx, const ope_scene_params* prm, const uint16_t* depth, int frames, int rows, int cols,
                           ope_scene_batch** out, ope_scene_frame* info, int32_t* status);
/* host copies of one frame: xyz (n_cropped x 3) and/or labels (n_cropped), either may be NULL; info may be NULL.
 * labels are exactly ope_segment_objects_on_plane's. */
int ope_scene_batch_frame(const ope_scene_batch* s, size_t frame, float* xyz, int32_t* labels, ope_scene_frame* info);
void ope_scene_batch_destroy(ope_scene_batch* s);
/* ope_pose_batch on the segmented frames. Frame f's target is cluster cluster[f] (NULL: 0 for every frame) = the points of the
 * cropped cloud labelled with that number, in ascending index order (what pcl::ExtractIndices returns for the cluster's sorted
 * indices). n_clusters == -1: the whole cropped cloud (the reference hands it on, D&L/src/objectsegmentationplane.cpp:149-152).
 * A rank >= n_clusters, or a frame whose scene status is an error: an empty target. Results, tables, status: as ope_pose_batch
 * (tables == NULL draws from libc rand() in frame order, empty targets included). workers: ignored; kept for ABI compatibility.
 * Concurrency comes from the lanes (OPE_BATCH_LANES). */
int ope_scene_pose_batch(const ope_scene_batch* s, const ope_pose_params* prm, const float* model_xyz, size_t n_model,
                         const int32_t* cluster, const ope_rng_table* tables, int workers, ope_pose_result* results, int32_t* status);

/* pcl::compute3DCentroid of a device cloud (include/ope_pcl/filters.h): serial float sums over the finite points in index order,
 * then each divided by (float) n; c = 0 when no point is finite. n_used (may be NULL): the number of finite points. */
int ope_cloud_centroid(ope_ctx* ctx, const ope_cloud* cloud, float c[3], int32_t* n_used);
/* the same for the clusters of frame f in rank order: xyz gets n_clusters x 3 floats (the whole cropped cloud, one centroid, when
 * n_clusters == -1; none when the frame's scene status is an error); *n_out: the number of centroids written. */
int ope_scene_batch_centroids(const ope_scene_batch* s, size_t frame, float* xyz, int32_t* n_out);
void ope_track_params_default(ope_track_params* p);
/* The node's cluster choice and the tracker step in one call (D&L/src/rosinterface.cpp:243-327, SURVEY 3.1 and A.0): camera i
 * is frame i of s (n == the number of frames) with trackers[i] and its device source *sources[i]. The call equals this serial
 * loop of public calls bit for bit, libc rand() consumption included:
 *   - branch: a frame whose scene status is an error -> NO_SCENE (tracker and source untouched, the frame's code in status[i]);
 *     a tracker that never completed a step (firstTimePose == 0) -> acquisition; any other -> tracking.
 *   - tracking: m = ope_cloud_centroid(*sources[i]) (the model as last placed in the scene), c_k = the centroid of cluster k
 *     (ope_scene_batch_centroids); the chosen cluster is the FIRST in rank order with sqrtf((dx*dx + dy*dy) + dz*dz) < gate
 *     (float, no FMA). The tracker steps on it as ope_pose_tracker_step_batch steps it -> TRACKED. No cluster inside the gate
 *     (n_clusters == 0 included): with reacquire the camera goes to acquisition (REACQUIRED on success), else LOST (tracker and
 *     source untouched). The reference keeps "the cluster whose centroid is less than 5 cm from the model's"; first-in-rank rather
 *     than nearest is this library's reading of that sentence (the reference file is not in this tree).
 *   - acquisition: try r (r = 0, 1, ... < n_clusters, at most max_tries; one try on the whole cloud when n_clusters == -1) is a
 *     fresh tracker with trackers[i]'s parameters on a device copy of the pristine model (trackers[i]'s cloudModel if it has one,
 *     else *sources[i]) against cluster r, as ope_scene_pose_batch cuts it. The first try with fitness < accept_fitness ||
 *     align_strength > accept_strength is committed: trackers[i] is then what a freshly created tracker is after
 *     ope_pose_estimate_final_device(copy of the model, that cluster), and *sources[i] is replaced by that call's source.
 *     No accepted try -> NOT_FOUND: tracker and source untouched, results[i] = the last try's (zero without a try).
 *   - order (the rand() stream): rounds r = 0, 1, ...; round 0 holds every tracking camera's step and every acquiring camera's
 *     rank-0 try (a reacquiring camera enters at round 0, after its failed gate), round r >= 1 the rank-r tries of the cameras
 *     still searching; in a round the cameras go in index order, and the round is ONE ope_pose_tracker_step_batch call (tables
 *     drawn from libc rand()).
 * results / choice / status: n entries each; status[i] is the code of the step whose result is results[i] (OPE_OK for a
 * camera that made no step, a failed try counts as not accepted). Returns OPE_OK or the first failing camera's code.
 * Argument checks are those of ope_pose_tracker_step_batch (distinct trackers and sources, all on s's context) and n; a violation
 * returns OPE_ERR_INVALID before anything changes. tp == NULL: ope_track_params_default. */
int ope_scene_track_step(const ope_scene_batch* s, const ope_track_params* tp, ope_pose_tracker* const* trackers, ope_cloud** sources,
                         size_t n, ope_pose_result* results, ope_track_choice* choice, int32_t* status);
/* host wall time (ms) of the phases of the context's last ope_scene_track_step: out[0] centroids + gate (one launch, one
 * read-back), out[1] commit of the accepted tries, out[2 + r] round r (cut + tracker step). *n_out: 2 + rounds; at most cap
 * entries are written. */
int ope_scene_track_phase_ms(const ope_ctx* ctx, double* out, int cap, int32_t* n_out);

/* ---- spatial search: replaces pcl::search::KdTree / KdTreeFLANN (SURVEY A.3) -------------------------- */
/* nearestKSearch for nq host queries; out_idx/out_d2 are nq*k, ascending (d2, index), padded with -1 / +inf. 1 <= k <=
 * OPE_KNN_MAX_K (256), OPE_ERR_INVALID otherwise. */
int ope_knn(ope_ctx* ctx, const ope_cloud* tgt, const void* qry, size_t nq, size_t stride, size_t offset, int k,
            int32_t* out_idx, float* out_d2);
/* same with the queries already on the device */
int ope_knn_cloud(ope_ctx* ctx, const ope_cloud* tgt, const ope_cloud* qry, int k, int32_t* out_idx, float* out_d2);
/* radiusSearch (d2 < r*r, ascending index). offsets: nq+1; out_idx/out_d2 up to `capacity` entries (may be NULL
 * to only count). Returns OPE_ERR_CAPACITY when total > capacity; *total is always set. */
int ope_radius_cloud(ope_ctx* ctx, const ope_cloud* tgt, const ope_cloud* qry, float radius, int64_t capacity,
                     int64_t* offsets, int32_t* out_idx, float* out_d2, int64_t* total);

/* ---- down-sampling ------------------------------------------------------------------------------------ */
/* pcl::UniformSampling::setRadiusSearch(leaf) + compute(indices) (D&L/src/poseestimator.cpp:141-144; SURVEY A.1).
 * out_idx must hold ope_cloud_size entries; ascending voxel-key order. OPE_ERR_GRID_TOO_LARGE when the voxel frame has more than
 * INT_MAX voxels (PCL's int voxel index would overflow); larger frames below that are processed in windows of voxels. */
int ope_uniform_sample(ope_ctx* ctx, const ope_cloud* cloud, float leaf, int32_t* out_idx, size_t* out_n);
/* the same, result kept on the device as a new cloud (fused copyPointCloud) */
int ope_uniform_sample_cloud(ope_ctx* ctx, const ope_cloud* cloud, float leaf, ope_cloud** out);
/* pcl::VoxelGrid::setLeafSize + filter (D&L/src/processingpcd.cpp:45-59; SURVEY A.2). rgb: packed float per
 * point or NULL. out_xyz holds 3*n floats, out_rgb n floats (or NULL). OPE_ERR_GRID_TOO_LARGE where PCL refuses ("Leaf size is
 * too small for the input dataset": more than INT_MAX voxels by its own count). */
int ope_voxel_grid(ope_ctx* ctx, const ope_cloud* cloud, const float* rgb, float lx, float ly, float lz,
                   float* out_xyz, float* out_rgb, size_t* out_n);

/* ---- features ------------------------------------------------------------------------------------------- */
/* pcl::NormalEstimation::setKSearch(k) + compute (D&L/src/poseestimator.cpp:151-156, BM/src/regmeshpcd.cpp:74-90;
 * SURVEY A.4). Writes the normals into the cloud (device) and, if out4 != NULL, to the host (n*4). 1 <= k <= OPE_KNN_MAX_K,
 * OPE_ERR_INVALID otherwise. The covariance is summed over the k nearest in ascending (d2, index) order. */
int ope_normals_knn(ope_ctx* ctx, ope_cloud* cloud, int k, const float viewpoint[3], float* out4);
/* pcl::NormalEstimation::setRadiusSearch(radius) + compute. Neighbours: the finite points with d2 < radius^2 (strict; the query
 * itself included), summed in ascending (d2, index) order. A non-finite point, or one with fewer than 3 neighbours, gets NaN normal
 * and curvature. The normal is flipped toward the viewpoint (NULL: the origin). Writes the normals into the cloud (device) and, if
 * out4 != NULL, to the host (n*4). Any neighbour count runs; lists longer than the shared-memory capacity take device scratch in
 * tiles bounded by OPE_RADIUS_NORMALS_SCRATCH_BYTES (INTEGRATION.md section 5). radius <= 0 or not finite: OPE_ERR_INVALID. */
int ope_normals_radius(ope_ctx* ctx, ope_cloud* cloud, float radius, const float viewpoint[3], float* out4);
/* pcl::FPFHEstimation::setRadiusSearch + compute (D&L/src/poseestimator.cpp:121-125; SURVEY A.5). The cloud must
 * carry normals. out: n*33 floats (host). out_spfh (n*33) may be NULL. */
int ope_fpfh(ope_ctx* ctx, const ope_cloud* cloud, float radius, float* out, float* out_spfh);
/* KdTreeFLANN<FPFHSignature33>::nearestKSearch over whole feature sets (SAC-IA findSimilarFeatures, SURVEY A.6/K6):
 * exact float32 L2_Simple ranking; host feature arrays (rows of `dim` floats). k <= 16. */
int ope_feature_knn(ope_ctx* ctx, const float* ftgt, size_t nt, const float* fqry, size_t nq, int dim, int k,
                    int32_t* out_idx, float* out_d2);

/* ---- rigid transform estimation ---------------------------------------------------------------------------- */
/* TransformationEstimationSVD::estimateRigidTransformation (D&L/src/poseestimator.cpp:306,435; SURVEY A.7).
 * isrc/itgt: n host indices each, or NULL for identity correspondences over the first n points. */
int ope_umeyama(ope_ctx* ctx, const ope_cloud* src, const ope_cloud* tgt, const int32_t* isrc, const int32_t* itgt,
                size_t n, float T[16]);

/* TransformationEstimationPointToPlaneLLS (kind = OPE_TE_POINT_TO_PLANE_LLS; the default of IterativeClosestPointWithNormals,
 * VP/icp_mod.h:352-357) and TransformationEstimationPointToPlane (kind = OPE_TE_POINT_TO_PLANE: Levenberg-Marquardt over the
 * 6-parameter rigid warp, what BuildModel sets, BM/src/regmeshpcd.cpp:162,193) ::estimateRigidTransformation [UPSTREAM].
 * tgt must carry normals. lm_info: 3 ints (Eigen LM status, function evaluations, iterations) or NULL. */
int ope_point_to_plane(ope_ctx* ctx, const ope_cloud* src, const ope_cloud* tgt, const int32_t* isrc, const int32_t* itgt, size_t n,
                       int kind, float T[16], int32_t* lm_info);

/* ---- registration --------------------------------------------------------------------------------------------- */
/* Registration::getFitnessScore(max_range), VP/impl/registration_mod.hpp:131-165. */
int ope_fitness(ope_ctx* ctx, const ope_cloud* src, const ope_cloud* tgt, const float T[16], double max_range,
                double* out);
/* determineCorrespondences + rejector chain on the clouds as given (VP/impl/correspondence_estimation_mod.hpp:127-213,
 * VP/impl/correspondence_estimation_normal_shooting_weighted.hpp:104-145, VP/impl/icp_mod.hpp:194-208). out: ns entries. */
int ope_correspondences(ope_ctx* ctx, const ope_cloud* src, const ope_cloud* tgt, const ope_icp_params* prm,
                        ope_correspondence* out, size_t* out_n);
/* IterativeClosestPoint[WithNormals]::align(output, guess): VP/impl/registration_mod.hpp:176-219 +
 * VP/impl/icp_mod.hpp:118-272 (variant VP/impl/icp_modCorr.hpp:118-230). guess may be NULL (identity).
 * out_corr (ns entries, last iteration's correspondences_) and out_aligned (device cloud = `output`) may be NULL. */
int ope_icp_align(ope_ctx* ctx, const ope_cloud* src, const ope_cloud* tgt, const ope_icp_params* prm,
                  const float guess[16], ope_reg_result* res, ope_correspondence* out_corr, ope_cloud** out_aligned);
/* The same with the reference's own extension of ICP, fixed correspondences (IterativeClosestPoint::setFixedCorrespondences,
 * VP/icp_mod.h:267-281; VP/impl/icp_mod.hpp:150-151,209-225; VP/impl/correspondence_estimation_mod.hpp:134-161): with the
 * nearest-neighbour estimator, pairs the caller pins enter every iteration's list in front with distance = squared distance * 1e10
 * (written back into `fixed`). Whatever the estimator, when rejectors exist they enter a second time at the end after rejector 0
 * alone, with the distances `fixed` holds. The reciprocal and the normal-shooting estimators omit the front entries but keep that
 * tail, with the caller's distances unchanged. The MODCORR variant ignores the list. `fixed` is in/out; out_corr must hold
 * ns + 2 * n_fixed entries. A pair whose source or target point is not finite is refused (OPE_ERR_INVALID).
 * prm->use_reciprocal (either entry point) selects determineReciprocalCorrespondences (VP/impl/correspondence_estimation_mod.hpp:
 * 216-303) for the nearest-neighbour estimator. */
int ope_icp_align_fixed(ope_ctx* ctx, const ope_cloud* src, const ope_cloud* tgt, const ope_icp_params* prm, const float guess[16],
                        ope_correspondence* fixed, size_t n_fixed, ope_reg_result* res, ope_correspondence* out_corr,
                        ope_cloud** out_aligned);
/* SampleConsensusInitialAlignment::align [UPSTREAM ia_ransac.hpp] (D&L/src/poseestimator.cpp:50-64; SURVEY A.6).
 * fsrc/ftgt: host FPFHSignature33 arrays (ns*33, nt*33). table == NULL: the decisions are drawn from libc rand()
 * exactly as PCL does (the host owns the RNG stream; the device evaluates the whole pool in one launch).
 * prm->hypothesis_begin/end restrict the evaluated shard (multi-GPU pools); out_errors: max_iterations floats or NULL. */
int ope_sacia_align(ope_ctx* ctx, const ope_cloud* src, const float* fsrc, const ope_cloud* tgt, const float* ftgt,
                    const ope_sacia_params* prm, const ope_rng_table* table, ope_reg_result* res, float* out_errors);
/* ---- the SAC-IA hypothesis pool sharded over the GPUs of one box (SURVEY 8e row 2) -------------------------------------------
 * One process per GPU, each with its own ope_ctx. NCCL (libnccl.so.2, bound at run time) carries 8 + 64 bytes per alignment over
 * NVLink: ncclAllReduce(MIN) of a packed (error bits, hypothesis index) key, then ncclBroadcast of the winner's 4x4, both on the
 * context's stream. ope_comm_unique_id: rank 0 calls it and hands the bytes (128) to the other ranks by any means (a file,
 * torch.distributed, MPI); ope_comm_create: every rank, same id, world, own rank (world == 1 needs no id and no NCCL).
 * ope_sacia_align_sharded: every rank passes the SAME clouds, features and pre-drawn table; rank r evaluates hypotheses
 * [H r / world, H (r + 1) / world); every rank returns the pool's winner — bit for bit what one GPU returns for the whole pool. */
int ope_comm_unique_id(void* out, size_t bytes);
int ope_comm_nccl_version(void);
int ope_comm_create(ope_ctx* ctx, const void* unique_id, size_t bytes, int world, int rank, ope_comm** out);
void ope_comm_destroy(ope_comm* comm);
int ope_comm_rank(const ope_comm* comm);
int ope_comm_world(const ope_comm* comm);
int ope_sacia_align_sharded(ope_ctx* ctx, ope_comm* comm, const ope_cloud* src, const float* fsrc, const ope_cloud* tgt, const float* ftgt,
                            const ope_sacia_params* prm, const ope_rng_table* table, ope_reg_result* res);
/* draw the SAC-IA decision table on the host from libc rand() (selectSamples + the pick of findSimilarFeatures) */
int ope_sacia_draw(const float* src_xyz, size_t ns, size_t stride_bytes, int iterations, int nr_samples,
                   int k_correspondences, float* min_sample_distance, int32_t* samples, int32_t* picks);

/* RegMeshPcd::registerPointClouds (BM/src/regmeshpcd.cpp:210-271) with the merged cloud resident on the device for the whole
 * chain: for every pair i, source = the merged cloud so far, target = view i+1; getIcpNormal (:62-208): normals k = normal_k (12)
 * of BOTH clouds recomputed from scratch (the reference recomputes all of them every pair), ICP-with-normals as configured by
 * `prm` (normal shooting k = 20, surface-normal rejector, TransformationEstimationPointToPlane, eps 1e-8), the source
 * transformed by the final transformation (:204), then `*aligned += *target` (:254). views: n_views host clouds (points/n/stride/
 * offset) or device clouds (.cloud); pair_results: n_views-1 records or NULL; *merged: the final cloud (device, caller frees).
 * The chain does not shard: pair i consumes the output of pair i-1. */
int ope_register_point_clouds(ope_ctx* ctx, const ope_frame_input* views, size_t n_views, const ope_icp_params* prm, int normal_k,
                              ope_reg_result* pair_results, ope_cloud** merged);

/* ---- PoseEstimator (D&L/src/poseestimator.cpp:16-448) ---------------------------------------------------------- */
int ope_pose_tracker_create(ope_ctx* ctx, const ope_pose_params* prm, ope_pose_tracker** out);
void ope_pose_tracker_destroy(ope_pose_tracker* t);
/* PoseEstimator::estimateFinalPose(p_sourceCloud, p_targetCloud, fitnessScore, alignStrength), :383-448.
 * source_xyz: ns*3 floats, in/out (overwritten with alignedSource, :441); target: nt points. */
int ope_pose_estimate_final(ope_pose_tracker* t, float* source_xyz, size_t ns, const void* target, size_t nt,
                            size_t tstride, size_t toffset, const ope_rng_table* table, ope_pose_result* res);
/* the same with both clouds resident on the device (bench.py `value`); *source is replaced by alignedSource. */
int ope_pose_estimate_final_device(ope_pose_tracker* t, ope_cloud** source, const ope_cloud* target,
                                   const ope_rng_table* table, ope_pose_result* res);
/* per-stage device time of the last call in milliseconds (CUDA events; same slots as the oracle's stage list:
 * [0] down-sample [1] normals [2] fpfh [3] sac-ia [4] icp [5] fitness [6] dense umeyama + transforms [7] total) */
int ope_pose_stage_ms(const ope_pose_tracker* t, double out[8]);

/* Batched localisation of independent frames against one model (BASELINE.json configs[4]; SURVEY 8e row 1 + 8f-3): every
 * frame runs the FIRST-frame path of estimateFinalPose (coarse SAC-IA + fine ICP, a fresh PoseEstimator per frame) with the
 * full-resolution model as the source. Chunks of frames run through one launch per stage on a few lanes at once (the calling
 * thread and helper threads, each with its own stream and scratch memory) so that one chunk's host work overlaps another's
 * kernels; the frames outside those launches' capacities then run on the same lanes, one frame at a time each, through the
 * single-frame path. The frame-invariant model side (1 cm sample, normals, FPFH — recomputed per frame by the reference,
 * D&L/src/poseestimator.cpp:34,116) is computed once. workers: ignored; kept for ABI compatibility. Concurrency comes from the
 * lanes (OPE_BATCH_LANES).
 * tables: n_frames pre-drawn SAC-IA decision tables, or NULL to draw them here, in frame order, from libc rand() (one
 * 400 x 5 draw per frame, exactly the stream a serial loop over fresh PoseEstimators would consume).
 * results: n_frames records; status: n_frames return codes (OPE_OK or the error of that frame) or NULL. A frame that fails on
 * the single-frame path (outside the frame-spanning launches) fails alone: the other frames still run, and the call returns the
 * lowest such frame's code. Any other failure (a decision table that does not fit a frame inside the launches, a device error)
 * stops the call with its code; results and status of frames not yet finished are then undefined. */
int ope_pose_batch(ope_ctx* ctx, const ope_pose_params* prm, const float* model_xyz, size_t n_model, const ope_frame_input* frames,
                   size_t n_frames, const ope_rng_table* tables, int workers, ope_pose_result* results, int32_t* status);

/* Advance n trackers of this context by one frame each. For every i the result is what
 *   ope_pose_estimate_final_device(trackers[i], &sources[i], target_i, tables ? &tables[i] : NULL, &results[i])
 * returns and leaves behind, the calls made in index order: the same results, the same tracker state
 * (alignedSource, cloudModel, fitnessScoreFine, alignedStrength, firstTimePose), the same *sources[i]
 * afterwards, and the same consumption of libc rand() when tables == NULL. A tracker draws a table, or
 * uses tables[i], only if it runs SAC-IA. targets: as ope_pose_batch's frames (host points or device
 * clouds; n == 0 means an empty target). Trackers and source handles must be distinct and belong to ctx.
 * Trackers may carry different models. Those whose parameters equal trackers[0]'s run through the frame-spanning launches of
 * ope_pose_batch with a per-tracker source; the others, and clouds outside those launches' capacities, through the single call.
 * status: n return codes or NULL; returns OPE_OK when every tracker succeeded, else the first failing tracker's code (a failing
 * tracker's state changes as the single call would change it). Duplicate or foreign trackers or sources, or a NULL source,
 * return OPE_ERR_INVALID before anything changes. */
int ope_pose_tracker_step_batch(ope_ctx* ctx, ope_pose_tracker* const* trackers, ope_cloud** sources,
                                const ope_frame_input* targets, size_t n, const ope_rng_table* tables,
                                ope_pose_result* results, int32_t* status);

/* Device time per stage of ope_pose_batch's frame-spanning launches (CUDA events on the context's stream), in milliseconds,
 * accumulated over the calls since the last reset: [0] staging + H2D of the clusters [1] target UniformSampling (1 cm + 8 mm)
 * [2] target normals [3] SPFH + FPFH [4] feature k-NN [5] SAC-IA pool [6] model under the coarse pose, 8 mm sampling [7] source
 * normals [8] NaN-normal compaction [9] ICP [10] fitness [11] unused. enable = 1 / 0: switch the laps on / off and reset the
 * sums; enable < 0: read only. out may be NULL. */
int ope_pose_batch_stage_ms(ope_ctx* ctx, int enable, double out[12]);

/* defaults of the reference classes (include/ope_types.h) */
void ope_icp_params_default(ope_icp_params* p);
void ope_sacia_params_default(ope_sacia_params* p);
void ope_pose_params_default(ope_pose_params* p);

#ifdef __cplusplus
}
#endif
#endif /* OPE_CUDA_H_ */
