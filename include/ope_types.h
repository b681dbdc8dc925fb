/* ope_types.h — plain-C parameter and result records shared by the CUDA library
 * (include/ope_cuda.h) and by the CPU checker used in tests (it includes this header; the product never includes it).
 *
 * Every default below is the default of the reference class it configures; the
 * citation is relative to /root/reference (D&L = DetectAndLocalize, BM = BuildModel,
 * VP = DetectAndLocalize/include/pcl/registration).
 */
#ifndef OPE_TYPES_H_
#define OPE_TYPES_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Error codes (all entry points return 0 on success, negative on failure; nothing
 * throws across the ABI — mirrors PCL_ERROR + silent return, VP/impl/registration_mod.hpp:73-77). */
enum {
  OPE_OK = 0,
  OPE_ERR_INVALID = -1,     /* bad argument (null pointer, k < 1, ...) */
  OPE_ERR_NO_DEVICE = -2,   /* CUDA device/runtime unavailable — there is NO CPU fallback */
  OPE_ERR_CUDA = -3,        /* a CUDA call failed; see ope_last_error() */
  OPE_ERR_EMPTY = -4,       /* empty cloud where the reference prints PCL_ERROR and returns */
  OPE_ERR_CAPACITY = -5,    /* caller-provided output buffer too small */
  OPE_ERR_GRID_TOO_LARGE = -6, /* voxel grid would overflow int32 (PCL: "Leaf size is too small") */
  OPE_ERR_UNSUPPORTED = -7
};

/* pcl::Correspondence, 12 bytes (SURVEY A.9): {index_query, index_match, distance} where
 * distance is the SQUARED euclidean distance (VP/impl/correspondence_estimation_mod.hpp:175). */
typedef struct ope_correspondence {
  int32_t index_query;
  int32_t index_match;
  float distance;
} ope_correspondence;

/* DefaultConvergenceCriteria::ConvergenceState, VP/default_convergence_criteria_mod.h:73-81 */
enum {
  OPE_CONV_NOT_CONVERGED = 0,
  OPE_CONV_ITERATIONS = 1,
  OPE_CONV_TRANSFORM = 2,
  OPE_CONV_ABS_MSE = 3,
  OPE_CONV_REL_MSE = 4,
  OPE_CONV_NO_CORRESPONDENCES = 5
};

/* correspondence estimators */
enum {
  OPE_EST_NEAREST = 0,         /* CorrespondenceEstimation, VP/impl/correspondence_estimation_mod.hpp:127-213 */
  OPE_EST_NORMAL_SHOOTING = 1  /* CorrespondenceEstimationNormalShooting; in-repo statement of the loop:
                                  VP/impl/correspondence_estimation_normal_shooting_weighted.hpp:104-145 */
};
/* correspondence rejectors */
enum {
  OPE_REJ_SURFACE_NORMAL = 1,       /* keep iff n_s.n_t > thr, VP/correspondence_rejection_mod.h:368-376 */
  OPE_REJ_SELF_OCCLUDED_NORMAL = 2  /* keep iff n_s.(-p_s/|p_s|) > thr, VP/correspondence_rejection_mod.h:382-391,
                                       VP/impl/correspondence_rejection_self_occluded_normal.cpp:43-64 */
};
/* transformation estimators */
enum {
  OPE_TE_SVD = 0,                /* TransformationEstimationSVD (Umeyama), ctor default VP/icp_mod.h:149 */
  OPE_TE_POINT_TO_PLANE_LLS = 1, /* IterativeClosestPointWithNormals default, VP/icp_mod.h:352-357 */
  OPE_TE_POINT_TO_PLANE = 2      /* TransformationEstimationPointToPlane (Levenberg-Marquardt on the 6-parameter rigid warp),
                                    what BuildModel sets: BM/src/regmeshpcd.cpp:162,193 */
};
/* which vendored ICP loop (SURVEY 3.2) */
enum {
  OPE_ICP_VARIANT_MOD = 0,     /* VP/impl/icp_mod.hpp:118-272: estimator/rejector normals refreshed every iteration */
  OPE_ICP_VARIANT_MODCORR = 1  /* VP/impl/icp_modCorr.hpp:118-230: normals stay as set once (stale) */
};

#define OPE_MAX_REJECTORS 4
/* largest k of ope_knn, ope_knn_cloud and ope_normals_knn (and of ope_pose_params.normal_k); k above it is OPE_ERR_INVALID */
#define OPE_KNN_MAX_K 256

/* IterativeClosestPoint[WithNormals] configuration. Defaults: VP/registration_mod.h:102-130,
 * VP/default_convergence_criteria_mod.h:94-110, VP/icp_mod.h:136-152. */
typedef struct ope_icp_params {
  int32_t max_iterations;              /* Registration::max_iterations_ = 10 */
  double transformation_epsilon;       /* 0 */
  double euclidean_fitness_epsilon;    /* -DBL_MAX */
  double max_correspondence_distance;  /* sqrt(DBL_MAX) */
  int32_t min_number_correspondences;  /* 3 */
  int32_t estimator;                   /* OPE_EST_* */
  int32_t k_search;                    /* normal shooting k (PCL default 10; apps use 20, D&L/src/poseestimator.cpp:246) */
  int32_t use_reciprocal;              /* use_reciprocal_correspondence_ = false, VP/icp_mod.h:143 */
  int32_t n_rejectors;
  int32_t rejector_kind[OPE_MAX_REJECTORS];
  double rejector_threshold[OPE_MAX_REJECTORS];
  int32_t transformation;              /* OPE_TE_* */
  int32_t variant;                     /* OPE_ICP_VARIANT_* */
  int32_t with_normals;                /* 1: IterativeClosestPointWithNormals::transformCloud rotates normals,
                                          VP/impl/icp_mod.hpp:311-318 */
  double mse_threshold_absolute;       /* 1e-12 */
  int32_t max_iterations_similar_transforms; /* 0 */
  int32_t failure_after_max_iterations;      /* false */
  int32_t force_all_iterations;        /* 0. Benchmark-only switch (SURVEY 8d, C2): evaluate the convergence
                                          tests but keep iterating until max_iterations. */
} ope_icp_params;

/* Result of an align() call: Registration::final_transformation_, converged_, nr_iterations_,
 * the convergence state and the size of the last correspondence set (for getAlignStrength,
 * VP/icp_mod.h:249-260). T is column-major like Eigen::Matrix4f. */
typedef struct ope_reg_result {
  float T[16];
  int32_t converged;
  int32_t state;
  int32_t iterations;
  int32_t n_correspondences;
  double last_mse;       /* ICP: correspondences_cur_mse_ of the last evaluated iteration; SAC-IA: min_sample_distance_ as the
                            run left it (selectSamples halves the member after 3*N failed draws and it STAYS halved) */
  double best_error;     /* SAC-IA: lowest_error; ICP: unused (0) */
  int32_t best_iteration;/* SAC-IA: index of the winning hypothesis; ICP: unused */
  int32_t reserved;
} ope_reg_result;

/* SampleConsensusInitialAlignment configuration [UPSTREAM ia_ransac.h]; values used by the app:
 * D&L/src/poseestimator.cpp:55-59 (400 / 5 / 5 / 0.05 / 0.01). */
typedef struct ope_sacia_params {
  int32_t max_iterations;        /* Registration default 10; app 400 */
  int32_t nr_samples;            /* 3; app 5 */
  int32_t k_correspondences;     /* 10; app 5 */
  float min_sample_distance;     /* 0; app 0.01 */
  double max_correspondence_distance; /* TruncatedError threshold, applied to SQUARED distances (SURVEY A.6) */
  int32_t hypothesis_begin;      /* shard [begin, end) of the hypothesis pool evaluated by this call; */
  int32_t hypothesis_end;        /* begin = end = 0 means the whole pool */
} ope_sacia_params;

/* Pre-drawn libc rand() decisions of one SAC-IA run (SURVEY hard part 3): for hypothesis h,
 * samples[h*nr_samples + s] is the source index and picks[h*nr_samples + s] in [0, k) selects among
 * the k nearest target features. */
typedef struct ope_rng_table {
  int32_t n_hypotheses;
  int32_t nr_samples;
  const int32_t* samples;
  const int32_t* picks;
} ope_rng_table;

/* PoseEstimator parameter sheet (SURVEY A.0), every literal of D&L/src/poseestimator.cpp. */
typedef struct ope_pose_params {
  float coarse_leaf;             /* 0.01  (:116) */
  float fine_leaf;               /* 0.008 (:199,206) */
  int32_t normal_k;              /* 30    (:153) */
  float fpfh_radius;             /* 0.03  (:122) */
  ope_sacia_params sacia;        /* 400/5/5/0.05/0.01 (:55-59) */
  int32_t min_target_features;   /* 10    (:40) */
  int32_t min_target_points;     /* 100   (:218) */
  ope_icp_params icp;            /* :310-341 */
  double coarse_refit_threshold; /* 1e-4: re-run SAC-IA iff last fine fitness > this (:399) */
} ope_pose_params;

/* Per-tracker state carried across frames: D&L/include/poseestimator.h:50-53. */
typedef struct ope_pose_result {
  float final_pose[16];    /* finalPose = rigidmodelPose * (coarse * fine), :421-439 */
  float coarse_pose[16];
  float fine_pose[16];
  float rigid_model_pose[16];
  double fitness;          /* fitnessScoreFine, :354 */
  double align_strength;   /* alignedStrength, :363 */
  int32_t ran_coarse;
  int32_t icp_iterations;
  int32_t icp_converged;
  int32_t icp_state;
  int32_t n_src_coarse, n_tgt_coarse, n_src_fine, n_tgt_fine;
  int32_t sacia_best_iteration;
  int32_t reserved;
  double sacia_best_error;
} ope_pose_result;

/* ObjectSegmentationPlane::getSegmentedObjectsOnPlane parameter sheet (D&L/src/objectsegmentationplane.cpp:36-90,174-203). */
typedef struct ope_segment_params {
  double distance_threshold;     /* 0.01  sacSeg.setDistanceThreshold (:43) */
  int32_t max_iterations;        /* 50    pcl::SACSegmentation default */
  int32_t min_cluster_size;      /* 300   (:84) */
  double probability;            /* 0.99  pcl::SACSegmentation default */
  double hull_margin;            /* 0.1   padding of the hull's bounding rectangle, a double literal in the reference (:180-183) */
  float cluster_tolerance;       /* 0.05  (:83) */
  int32_t max_cluster_size;      /* 1e5   (:85) */
} ope_segment_params;

/* per-point labels of ope_segment_objects_on_plane */
enum { OPE_SEG_OUTSIDE_PRISM = -3, OPE_SEG_PLANE = -2, OPE_SEG_NO_CLUSTER = -1 };

/* Camera, crop and segmentation of ope_scene_batch_create; ope_scene_params_default gives the values below. */
typedef struct ope_scene_params {
  float fx, fy, cx, cy, scale, z_max;  /* DataGrabber::rgbd2Pcl: 525, 525, 319.5, 239.5, 1000, 2.0 (D&L/src/datagrabber.cpp:34,146-150) */
  float limits[6];                     /* ProcessingPcd::getPassThrough x_min, x_max, y_min, y_max, z_min, z_max:
                                          -0.5, 0.5, -0.5, 0.3, 0.5, 1.6 (ObjectSegmentationPlane::getFiltered, D&L/src/objectsegmentationplane.cpp:17-18) */
  ope_segment_params seg;              /* ope_segment_params_default */
} ope_scene_params;

/* One frame of ope_scene_batch_create. */
typedef struct ope_scene_frame {
  int32_t n_points;                    /* after depth -> cloud */
  int32_t n_cropped;                   /* after the pass-through; the length of the frame's labels */
  float plane1[4], plane2[4];          /* table plane, second plane (zero when n_clusters == -1) */
  int32_t iterations[2];               /* RANSAC iterations of the two plane fits */
  int32_t n_clusters;                  /* as ope_segment_objects_on_plane: -1 = a plane fit failed */
  int32_t reserved;
} ope_scene_frame;

/* ope_scene_track_step: the cluster choice of the reference's online loop (D&L/src/rosinterface.cpp:243-327, SURVEY 3.1 and A.0);
 * ope_track_params_default gives the values below. */
typedef struct ope_track_params {
  double accept_fitness;    /* 1e-4: a pose is accepted iff fitness < accept_fitness || align_strength > accept_strength */
  double accept_strength;   /* 0.4 */
  float gate;               /* 0.05 m: centroid distance that keeps a tracked object on a cluster */
  int32_t max_tries;        /* acquisition tries per call; 0 = every cluster */
  int32_t reacquire;        /* 1: a tracker with no cluster inside the gate searches again in the same call */
} ope_track_params;

/* what one camera of ope_scene_track_step did */
enum {
  OPE_TRACK_TRACKED = 0,    /* stepped on the first cluster inside the gate */
  OPE_TRACK_ACQUIRED,       /* a fresh search accepted a cluster */
  OPE_TRACK_REACQUIRED,     /* lost by the gate, then a search in the same call accepted a cluster */
  OPE_TRACK_NOT_FOUND,      /* a search accepted no cluster */
  OPE_TRACK_LOST,           /* no cluster inside the gate and no search (reacquire = 0) */
  OPE_TRACK_NO_SCENE        /* the frame's scene status is an error */
};
typedef struct ope_track_choice {
  int32_t mode;             /* OPE_TRACK_* */
  int32_t cluster;          /* the rank stepped on (0 for a whole-cloud frame), -1 if none */
  int32_t tries;            /* acquisition tries made in this call */
  float gate_distance;      /* tracking: the distance of the chosen cluster (or of the nearest one when lost); NaN otherwise */
} ope_track_choice;

/* One frame of a batch (ope_pose_batch): the segmented scene cluster either as host points (stride/offset in BYTES as in
 * ope_cloud_upload) or, when points == NULL, as a device-resident cloud that no other call touches during the batch. */
typedef struct ope_frame_input {
  const void* points;
  size_t n;
  size_t stride;
  size_t offset;
  void* cloud;             /* ope_cloud* */
} ope_frame_input;

#ifdef __cplusplus
}
#endif
#endif /* OPE_TYPES_H_ */
