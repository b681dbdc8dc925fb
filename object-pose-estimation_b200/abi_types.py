"""ctypes mirrors of include/ope_types.h (the C-ABI records of libope_cuda.so).

Field order and widths must match the header exactly; tests/test_abi.py checks sizeof against the
values the C compiler reports.
"""
import ctypes as C

OPE_OK = 0
OPE_ERR_INVALID, OPE_ERR_NO_DEVICE, OPE_ERR_CUDA, OPE_ERR_EMPTY = -1, -2, -3, -4
OPE_ERR_CAPACITY, OPE_ERR_GRID_TOO_LARGE, OPE_ERR_UNSUPPORTED = -5, -6, -7

CONV_NOT_CONVERGED, CONV_ITERATIONS, CONV_TRANSFORM, CONV_ABS_MSE, CONV_REL_MSE, CONV_NO_CORRESPONDENCES = range(6)
EST_NEAREST, EST_NORMAL_SHOOTING = 0, 1
REJ_SURFACE_NORMAL, REJ_SELF_OCCLUDED_NORMAL = 1, 2
TE_SVD, TE_POINT_TO_PLANE_LLS, TE_POINT_TO_PLANE = 0, 1, 2
ICP_VARIANT_MOD, ICP_VARIANT_MODCORR = 0, 1
MAX_REJECTORS = 4


class Correspondence(C.Structure):
    _fields_ = [("index_query", C.c_int32), ("index_match", C.c_int32), ("distance", C.c_float)]


class IcpParams(C.Structure):
    _fields_ = [
        ("max_iterations", C.c_int32),
        ("transformation_epsilon", C.c_double),
        ("euclidean_fitness_epsilon", C.c_double),
        ("max_correspondence_distance", C.c_double),
        ("min_number_correspondences", C.c_int32),
        ("estimator", C.c_int32),
        ("k_search", C.c_int32),
        ("use_reciprocal", C.c_int32),
        ("n_rejectors", C.c_int32),
        ("rejector_kind", C.c_int32 * MAX_REJECTORS),
        ("rejector_threshold", C.c_double * MAX_REJECTORS),
        ("transformation", C.c_int32),
        ("variant", C.c_int32),
        ("with_normals", C.c_int32),
        ("mse_threshold_absolute", C.c_double),
        ("max_iterations_similar_transforms", C.c_int32),
        ("failure_after_max_iterations", C.c_int32),
        ("force_all_iterations", C.c_int32),
    ]


class RegResult(C.Structure):
    _fields_ = [
        ("T", C.c_float * 16),
        ("converged", C.c_int32),
        ("state", C.c_int32),
        ("iterations", C.c_int32),
        ("n_correspondences", C.c_int32),
        ("last_mse", C.c_double),
        ("best_error", C.c_double),
        ("best_iteration", C.c_int32),
        ("reserved", C.c_int32),
    ]


class SaciaParams(C.Structure):
    _fields_ = [
        ("max_iterations", C.c_int32),
        ("nr_samples", C.c_int32),
        ("k_correspondences", C.c_int32),
        ("min_sample_distance", C.c_float),
        ("max_correspondence_distance", C.c_double),
        ("hypothesis_begin", C.c_int32),
        ("hypothesis_end", C.c_int32),
    ]


class RngTable(C.Structure):
    _fields_ = [
        ("n_hypotheses", C.c_int32),
        ("nr_samples", C.c_int32),
        ("samples", C.POINTER(C.c_int32)),
        ("picks", C.POINTER(C.c_int32)),
    ]


class PoseParams(C.Structure):
    _fields_ = [
        ("coarse_leaf", C.c_float),
        ("fine_leaf", C.c_float),
        ("normal_k", C.c_int32),
        ("fpfh_radius", C.c_float),
        ("sacia", SaciaParams),
        ("min_target_features", C.c_int32),
        ("min_target_points", C.c_int32),
        ("icp", IcpParams),
        ("coarse_refit_threshold", C.c_double),
    ]


class PoseResult(C.Structure):
    _fields_ = [
        ("final_pose", C.c_float * 16),
        ("coarse_pose", C.c_float * 16),
        ("fine_pose", C.c_float * 16),
        ("rigid_model_pose", C.c_float * 16),
        ("fitness", C.c_double),
        ("align_strength", C.c_double),
        ("ran_coarse", C.c_int32),
        ("icp_iterations", C.c_int32),
        ("icp_converged", C.c_int32),
        ("icp_state", C.c_int32),
        ("n_src_coarse", C.c_int32),
        ("n_tgt_coarse", C.c_int32),
        ("n_src_fine", C.c_int32),
        ("n_tgt_fine", C.c_int32),
        ("sacia_best_iteration", C.c_int32),
        ("reserved", C.c_int32),
        ("sacia_best_error", C.c_double),
    ]


class SegmentParams(C.Structure):
    _fields_ = [("distance_threshold", C.c_double), ("max_iterations", C.c_int32), ("min_cluster_size", C.c_int32),
                ("probability", C.c_double), ("hull_margin", C.c_double), ("cluster_tolerance", C.c_float), ("max_cluster_size", C.c_int32)]


SEG_OUTSIDE_PRISM, SEG_PLANE, SEG_NO_CLUSTER = -3, -2, -1


class SceneParams(C.Structure):
    _fields_ = [("fx", C.c_float), ("fy", C.c_float), ("cx", C.c_float), ("cy", C.c_float), ("scale", C.c_float), ("z_max", C.c_float),
                ("limits", C.c_float * 6), ("seg", SegmentParams)]


class SceneFrame(C.Structure):
    _fields_ = [("n_points", C.c_int32), ("n_cropped", C.c_int32), ("plane1", C.c_float * 4), ("plane2", C.c_float * 4),
                ("iterations", C.c_int32 * 2), ("n_clusters", C.c_int32), ("reserved", C.c_int32)]


class TrackParams(C.Structure):
    _fields_ = [("accept_fitness", C.c_double), ("accept_strength", C.c_double), ("gate", C.c_float), ("max_tries", C.c_int32),
                ("reacquire", C.c_int32)]


TRACK_TRACKED, TRACK_ACQUIRED, TRACK_REACQUIRED, TRACK_NOT_FOUND, TRACK_LOST, TRACK_NO_SCENE = range(6)
TRACK_MODES = ("tracked", "acquired", "reacquired", "not_found", "lost", "no_scene")


class TrackChoice(C.Structure):
    _fields_ = [("mode", C.c_int32), ("cluster", C.c_int32), ("tries", C.c_int32), ("gate_distance", C.c_float)]


class FrameInput(C.Structure):
    _fields_ = [("points", C.c_void_p), ("n", C.c_size_t), ("stride", C.c_size_t), ("offset", C.c_size_t), ("cloud", C.c_void_p)]


def mat4(c_arr):
    """column-major float[16] -> numpy (4,4) row/col indexed like Eigen's M(r,c)."""
    import numpy as np
    return np.array(list(c_arr), dtype=np.float32).reshape(4, 4).T.copy()


def mat4_to_c(M):
    import numpy as np
    a = np.asarray(M, dtype=np.float32).T.reshape(16)
    return (C.c_float * 16)(*a.tolist())
