"""ctypes binding of libope_cuda.so (the C ABI in include/ope_cuda.h).

There is no CPU fallback anywhere in this module: if the shared library is missing or no CUDA device is usable,
every entry point raises.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from . import abi_types as T

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libope_cuda.so")
_LIB = None

f32p = C.POINTER(C.c_float)
i32p = C.POINTER(C.c_int32)
i64p = C.POINTER(C.c_int64)

EXPORTS = [
    "ope_ctx_create", "ope_ctx_destroy", "ope_last_error", "ope_ctx_synchronize", "ope_ctx_launch_count", "ope_version",
    "ope_ctx_last_kernel_ms", "ope_cloud_invalidate", "ope_ctx_feature_knn_stats", "ope_ctx_model_cache_stats",
    "ope_cloud_upload", "ope_cloud_free", "ope_cloud_size", "ope_cloud_has_normals", "ope_cloud_download",
    "ope_cloud_select", "ope_cloud_transform", "ope_cloud_set_normals", "ope_cloud_append", "ope_register_point_clouds",
    "ope_pass_through", "ope_euclidean_clusters", "ope_plane_ransac", "ope_segment_objects_on_plane", "ope_segment_params_default", "ope_knn", "ope_knn_cloud", "ope_radius_cloud", "ope_depth_to_cloud", "ope_depth_to_cloud_batch",
    "ope_uniform_sample", "ope_uniform_sample_cloud", "ope_voxel_grid",
    "ope_normals_knn", "ope_normals_radius", "ope_fpfh", "ope_feature_knn",
    "ope_umeyama", "ope_point_to_plane", "ope_fitness", "ope_correspondences", "ope_icp_align", "ope_icp_align_fixed", "ope_sacia_align", "ope_sacia_align_sharded",
    "ope_comm_unique_id", "ope_comm_nccl_version", "ope_comm_create", "ope_comm_destroy", "ope_comm_rank", "ope_comm_world", "ope_sacia_draw",
    "ope_pose_tracker_create", "ope_pose_tracker_destroy", "ope_pose_estimate_final", "ope_pose_estimate_final_device", "ope_pose_batch", "ope_pose_tracker_step_batch",
    "ope_pose_stage_ms", "ope_pose_batch_stage_ms", "ope_icp_params_default", "ope_sacia_params_default", "ope_pose_params_default",
    "ope_scene_params_default", "ope_scene_batch_create", "ope_scene_batch_frame", "ope_scene_batch_destroy", "ope_scene_pose_batch",
    "ope_cloud_centroid", "ope_scene_batch_centroids", "ope_track_params_default", "ope_scene_track_step", "ope_scene_track_phase_ms",
]


class OpeError(RuntimeError):
    def __init__(self, rc, msg):
        super().__init__("libope_cuda call failed: rc=%d (%s)" % (rc, msg))
        self.rc = rc


def build(verbose=False):
    """Compile csrc/ for sm_100a into libope_cuda.so (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", os.path.join(_HERE, "csrc"), "-j4"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or r.returncode != 0:
        print(r.stdout)
    if r.returncode != 0:
        raise RuntimeError("building libope_cuda.so failed")
    return LIB_PATH


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("libope_cuda.so is not built (run __graft_entry__.build()); there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        L.ope_last_error.restype = C.c_char_p
        L.ope_version.restype = C.c_char_p
        L.ope_ctx_launch_count.restype = C.c_int64
        L.ope_cloud_size.restype = C.c_size_t
        L.ope_ctx_last_kernel_ms.restype = C.c_double
        _LIB = L
    return _LIB


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def icp_params(**kw):
    p = T.IcpParams()
    lib().ope_icp_params_default(C.byref(p))
    _set(p, kw)
    return p


def sacia_params(**kw):
    p = T.SaciaParams()
    lib().ope_sacia_params_default(C.byref(p))
    _set(p, kw)
    return p


def pose_params(**kw):
    p = T.PoseParams()
    lib().ope_pose_params_default(C.byref(p))
    _set(p, kw)
    return p


def track_params(**kw):
    p = T.TrackParams()
    lib().ope_track_params_default(C.byref(p))
    _set(p, kw)
    return p


def _set(p, kw):
    for k, v in kw.items():
        if k == "rejectors":
            p.n_rejectors = len(v)
            for i, (kind, thr) in enumerate(v):
                p.rejector_kind[i] = kind
                p.rejector_threshold[i] = thr
        else:
            setattr(p, k, v)


def rng_table(samples, picks):
    samples = np.ascontiguousarray(samples, np.int32)
    picks = np.ascontiguousarray(picks, np.int32)
    t = T.RngTable(samples.shape[0], samples.shape[1], samples.ctypes.data_as(i32p), picks.ctypes.data_as(i32p))
    t._keep = (samples, picks)
    return t


class Cloud:
    def __init__(self, ctx, handle):
        self.ctx, self.h = ctx, handle

    def __len__(self):
        return int(lib().ope_cloud_size(self.h))

    @property
    def has_normals(self):
        return bool(lib().ope_cloud_has_normals(self.h))

    def free(self):
        # a cloud must never outlive its context: after Context.close() the device memory is gone with it
        if self.h and self.ctx.h:
            lib().ope_cloud_free(self.ctx.h, self.h)
        self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    def download(self, normals=False):
        n = len(self)
        xyz = np.empty((n, 3), np.float32)
        nr = np.empty((n, 4), np.float32) if normals else None
        self.ctx._chk(lib().ope_cloud_download(self.ctx.h, self.h, xyz.ctypes.data_as(f32p),
                                               nr.ctypes.data_as(f32p) if normals else None))
        return (xyz, nr) if normals else xyz


class Context:
    """One ope_ctx: a device, a stream, scratch memory. Not thread-safe (one per host thread)."""

    def __init__(self, device=0, stream=None):
        h = C.c_void_p()
        rc = lib().ope_ctx_create(int(device), C.c_void_p(stream) if stream else None, C.byref(h))
        if rc != 0:
            raise OpeError(rc, "ope_ctx_create: no usable CUDA device (there is no CPU fallback)" if rc == T.OPE_ERR_NO_DEVICE
                           else "ope_ctx_create")
        self.h = h

    def close(self):
        if self.h:
            lib().ope_ctx_synchronize(self.h)
            lib().ope_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc != 0:
            raise OpeError(rc, lib().ope_last_error(self.h).decode())

    def synchronize(self):
        self._chk(lib().ope_ctx_synchronize(self.h))

    @property
    def launches(self):
        return int(lib().ope_ctx_launch_count(self.h))

    def last_kernel_ms(self, which=0):
        """device time of the last icp_kernel (0) / SAC-IA scorer (1) launch, from CUDA events on the ctx stream"""
        return float(lib().ope_ctx_last_kernel_ms(self.h, int(which)))

    def feature_knn_stats(self):
        """(queries answered through the tcgen05 distance GEMM, queries the exact kernel re-answered)"""
        a, b = C.c_int64(0), C.c_int64(0)
        self._chk(lib().ope_ctx_feature_knn_stats(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def model_cache_stats(self):
        """(coarse stages served from the model-side cache, coarse stages that filled it)"""
        a, b = C.c_int64(0), C.c_int64(0)
        self._chk(lib().ope_ctx_model_cache_stats(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    BATCH_STAGES = ["h2d", "target_sampling", "target_normals", "fpfh", "feature_knn", "sacia", "model_sampling", "source_normals",
                    "nan_compaction", "icp", "fitness"]

    def batch_stage_ms(self, enable=-1):
        """per-stage device ms of ope_pose_batch's frame-spanning launches since the last reset; enable=1/0 switches + resets"""
        out = (C.c_double * 12)()
        self._chk(lib().ope_pose_batch_stage_ms(self.h, int(enable), out))
        return dict(zip(self.BATCH_STAGES, list(out)[:11]))

    def track_phase_ms(self):
        """host ms of the phases of the last SceneBatch.track: {"gate", "commit", "rounds": [round 0, 1, ...]}"""
        k = C.c_int32(0)
        self._chk(lib().ope_scene_track_phase_ms(self.h, None, 0, C.byref(k)))
        out = (C.c_double * max(k.value, 1))()
        self._chk(lib().ope_scene_track_phase_ms(self.h, out, k.value, C.byref(k)))
        v = list(out)[:k.value]
        return {"gate": v[0], "commit": v[1], "rounds": v[2:]} if v else {"gate": 0.0, "commit": 0.0, "rounds": []}

    def centroid(self, cloud):
        """pcl::compute3DCentroid of a device cloud: (xyz (3,) float32, number of finite points)"""
        c = (C.c_float * 3)()
        k = C.c_int32(0)
        self._chk(lib().ope_cloud_centroid(self.h, cloud.h, c, C.byref(k)))
        return np.array(list(c), np.float32), k.value

    def invalidate(self, cloud):
        self._chk(lib().ope_cloud_invalidate(self.h, cloud.h))

    # ---- clouds ----
    def upload(self, pts, normals=None):
        p = _f32(pts)
        assert p.ndim == 2 and p.shape[1] >= 3
        h = C.c_void_p()
        nr = None if normals is None else _f32(normals)
        self._chk(lib().ope_cloud_upload(self.h, p.ctypes.data_as(C.c_void_p), C.c_size_t(p.shape[0]),
                                         C.c_size_t(p.strides[0]), C.c_size_t(0),
                                         None if nr is None else nr.ctypes.data_as(C.c_void_p),
                                         C.c_size_t(0 if nr is None else nr.strides[0]), C.c_size_t(0), C.byref(h)))
        return Cloud(self, h)

    def depth_to_cloud(self, depth, fx=525.0, fy=525.0, cx=319.5, cy=239.5, scale=1000.0, z_max=2.0):
        """uint16 depth image (rows, cols) on the host -> device cloud (DataGrabber::rgbd2Pcl semantics)"""
        d = np.ascontiguousarray(depth, np.uint16)
        h = C.c_void_p()
        self._chk(lib().ope_depth_to_cloud(self.h, d.ctypes.data_as(C.POINTER(C.c_uint16)), d.shape[0], d.shape[1], C.c_float(fx),
                                           C.c_float(fy), C.c_float(cx), C.c_float(cy), C.c_float(scale), C.c_float(z_max), C.byref(h)))
        return Cloud(self, h)

    def depth_to_cloud_batch(self, d_depth_ptr, frames, rows, cols, d_out_ptr, d_col_start_ptr, fx=525.0, fy=525.0, cx=319.5, cy=239.5,
                             scale=1000.0, z_max=2.0):
        """device pointers (ints): uint16 depth [frames, rows, cols], float4 out [frames*rows*cols], int32 col_start [frames*cols+1]"""
        self._chk(lib().ope_depth_to_cloud_batch(self.h, C.c_void_p(d_depth_ptr), frames, rows, cols, C.c_float(fx), C.c_float(fy),
                                                 C.c_float(cx), C.c_float(cy), C.c_float(scale), C.c_float(z_max), C.c_void_p(d_out_ptr),
                                                 C.c_void_p(d_col_start_ptr)))

    def select(self, cloud, idx):
        idx = np.ascontiguousarray(idx, np.int32)
        h = C.c_void_p()
        self._chk(lib().ope_cloud_select(self.h, cloud.h, idx.ctypes.data_as(i32p), C.c_size_t(len(idx)), C.byref(h)))
        return Cloud(self, h)

    def transform(self, cloud, M):
        h = C.c_void_p()
        self._chk(lib().ope_cloud_transform(self.h, cloud.h, T.mat4_to_c(M), C.byref(h)))
        return Cloud(self, h)

    def append(self, dst, src):
        """*dst += *src on the device"""
        self._chk(lib().ope_cloud_append(self.h, dst.h, src.h))

    def _frame_inputs(self, frames):
        n = len(frames)
        arr = (T.FrameInput * max(n, 1))()
        keep = []
        for i, f in enumerate(frames):
            if isinstance(f, Cloud):
                arr[i] = T.FrameInput(None, 0, 0, 0, f.h)
            else:
                a = _f32(f) if len(f) else np.zeros((1, 3), np.float32)
                keep.append(a)
                arr[i] = T.FrameInput(a.ctypes.data, len(f), a.strides[0], 0, None)
        return arr, keep

    def register_point_clouds(self, views, prm, normal_k=12):
        """RegMeshPcd::registerPointClouds on the device: returns (merged Cloud, list of RegResult per pair)"""
        arr, keep = self._frame_inputs(views)
        res = (T.RegResult * max(len(views) - 1, 1))()
        h = C.c_void_p()
        self._chk(lib().ope_register_point_clouds(self.h, arr, C.c_size_t(len(views)), C.byref(prm), int(normal_k), res, C.byref(h)))
        return Cloud(self, h), [res[i] for i in range(len(views) - 1)]

    def set_normals(self, cloud, normals4):
        nr = _f32(normals4)
        self._chk(lib().ope_cloud_set_normals(self.h, cloud.h, nr.ctypes.data_as(f32p)))

    # ---- scene preparation (8f-2) ----
    def pass_through(self, cloud, limits, want_idx=False):
        """limits = (x_min, x_max, y_min, y_max, z_min, z_max); returns the filtered Cloud (and the kept indices)"""
        lim = (C.c_float * 6)(*[float(v) for v in limits])
        h = C.c_void_p()
        idx = np.empty(max(len(cloud), 1), np.int32) if want_idx else None
        m = C.c_size_t(0)
        self._chk(lib().ope_pass_through(self.h, cloud.h, lim, C.byref(h), None if idx is None else idx.ctypes.data_as(i32p), C.byref(m)))
        out = Cloud(self, h)
        return (out, idx[:m.value].copy()) if want_idx else out

    def euclidean_clusters(self, cloud, tolerance=0.05, min_size=300, max_size=100000):
        labels = np.empty(max(len(cloud), 1), np.int32)
        k = C.c_int(0)
        self._chk(lib().ope_euclidean_clusters(self.h, cloud.h, C.c_float(tolerance), int(min_size), int(max_size), labels.ctypes.data_as(i32p),
                                               C.byref(k)))
        return labels[:len(cloud)].copy(), k.value

    def plane_ransac(self, cloud, **kw):
        """pcl::SACSegmentation (plane): (found, coeff[4], inlier indices, iterations)"""
        prm = T.SegmentParams()
        lib().ope_segment_params_default(C.byref(prm))
        _set(prm, kw)
        coeff = (C.c_float * 4)()
        idx = np.empty(max(len(cloud), 1), np.int32)
        m, it, found = C.c_size_t(0), C.c_int32(0), C.c_int32(0)
        self._chk(lib().ope_plane_ransac(self.h, cloud.h, C.byref(prm), coeff, idx.ctypes.data_as(i32p), C.byref(m), C.byref(it), C.byref(found)))
        return bool(found.value), np.array(list(coeff), np.float32), idx[:m.value].copy(), it.value

    def segment_objects_on_plane(self, cloud, **kw):
        """getSegmentedObjectsOnPlane: (labels, n_clusters or -1, plane1, plane2, iterations)"""
        prm = T.SegmentParams()
        lib().ope_segment_params_default(C.byref(prm))
        _set(prm, kw)
        labels = np.empty(max(len(cloud), 1), np.int32)
        p1, p2 = (C.c_float * 4)(), (C.c_float * 4)()
        it = (C.c_int32 * 2)()
        k = C.c_int32(0)
        self._chk(lib().ope_segment_objects_on_plane(self.h, cloud.h, C.byref(prm), labels.ctypes.data_as(i32p), p1, p2, it, C.byref(k)))
        return labels[:len(cloud)].copy(), k.value, np.array(list(p1), np.float32), np.array(list(p2), np.float32), (it[0], it[1])

    def scene_batch(self, depth, **params):
        """Depth images -> cropped, segmented scenes, many frames per call (ope_scene_batch_create). depth: (frames, rows, cols)
        uint16 on the host (numpy) or a CUDA tensor of uint16 / int16 bits. params: fx, fy, cx, cy, scale, z_max, limits (x_min,
        x_max, y_min, y_max, z_min, z_max) and any ope_segment_params field. Returns a SceneBatch."""
        prm = T.SceneParams()
        lib().ope_scene_params_default(C.byref(prm))
        for k, v in params.items():
            if k == "limits":
                prm.limits = (C.c_float * 6)(*[float(x) for x in v])
            elif hasattr(prm, k) and k != "seg":
                setattr(prm, k, v)
            else:
                setattr(prm.seg, k, v)
        if hasattr(depth, "data_ptr"):
            import torch
            assert depth.is_cuda and depth.is_contiguous() and depth.element_size() == 2 and depth.dim() == 3
            torch.cuda.synchronize(depth.device)
            keep, ptr, shape = depth, C.c_void_p(depth.data_ptr()), tuple(depth.shape)
        else:
            keep = np.ascontiguousarray(depth, np.uint16)
            assert keep.ndim == 3
            ptr, shape = keep.ctypes.data_as(C.c_void_p), keep.shape
        n = shape[0]
        info = (T.SceneFrame * max(n, 1))()
        status = (C.c_int32 * max(n, 1))()
        h = C.c_void_p()
        rc = lib().ope_scene_batch_create(self.h, C.byref(prm), ptr, int(n), int(shape[1]), int(shape[2]), C.byref(h), info, status)
        del keep
        st = np.array(list(status)[:n], np.int32)
        if not h.value:
            self._chk(rc)
        return SceneBatch(self, h, [info[i] for i in range(n)], st)

    # ---- search ----
    def knn(self, tgt, qry, k):
        """tgt: Cloud; qry: Cloud or (N,>=3) array; 1 <= k <= 256 (OPE_KNN_MAX_K)."""
        nq = len(qry)
        idx = np.empty((nq, k), np.int32)
        d2 = np.empty((nq, k), np.float32)
        if isinstance(qry, Cloud):
            self._chk(lib().ope_knn_cloud(self.h, tgt.h, qry.h, k, idx.ctypes.data_as(i32p), d2.ctypes.data_as(f32p)))
        else:
            q = _f32(qry)
            self._chk(lib().ope_knn(self.h, tgt.h, q.ctypes.data_as(C.c_void_p), C.c_size_t(nq), C.c_size_t(q.strides[0]),
                                    C.c_size_t(0), k, idx.ctypes.data_as(i32p), d2.ctypes.data_as(f32p)))
        return idx, d2

    def radius(self, tgt, qry, r):
        nq = len(qry)
        off = np.empty(nq + 1, np.int64)
        total = C.c_int64(0)
        self._chk(lib().ope_radius_cloud(self.h, tgt.h, qry.h, C.c_float(r), C.c_int64(0), off.ctypes.data_as(i64p), None, None,
                                         C.byref(total)))
        idx = np.empty(max(total.value, 1), np.int32)
        d2 = np.empty(max(total.value, 1), np.float32)
        self._chk(lib().ope_radius_cloud(self.h, tgt.h, qry.h, C.c_float(r), C.c_int64(total.value), off.ctypes.data_as(i64p),
                                         idx.ctypes.data_as(i32p), d2.ctypes.data_as(f32p), C.byref(total)))
        return off, idx[:total.value], d2[:total.value]

    def feature_knn(self, ftgt, fqry, k):
        ft, fq = _f32(ftgt), _f32(fqry)
        idx = np.empty((fq.shape[0], k), np.int32)
        d2 = np.empty((fq.shape[0], k), np.float32)
        self._chk(lib().ope_feature_knn(self.h, ft.ctypes.data_as(f32p), C.c_size_t(ft.shape[0]), fq.ctypes.data_as(f32p),
                                        C.c_size_t(fq.shape[0]), ft.shape[1], k, idx.ctypes.data_as(i32p),
                                        d2.ctypes.data_as(f32p)))
        return idx, d2

    # ---- down-sampling ----
    def uniform_sample(self, cloud, leaf):
        out = np.empty(max(len(cloud), 1), np.int32)
        m = C.c_size_t(0)
        self._chk(lib().ope_uniform_sample(self.h, cloud.h, C.c_float(leaf), out.ctypes.data_as(i32p), C.byref(m)))
        return out[:m.value].copy()

    def uniform_sample_cloud(self, cloud, leaf):
        h = C.c_void_p()
        self._chk(lib().ope_uniform_sample_cloud(self.h, cloud.h, C.c_float(leaf), C.byref(h)))
        return Cloud(self, h)

    def voxel_grid(self, cloud, leaf, rgb=None):
        lx, ly, lz = (leaf, leaf, leaf) if np.isscalar(leaf) else leaf
        n = max(len(cloud), 1)
        oxyz = np.empty((n, 3), np.float32)
        orgb = np.empty(n, np.float32)
        m = C.c_size_t(0)
        rgbp = None
        if rgb is not None:
            rgb = _f32(rgb)
            rgbp = rgb.ctypes.data_as(f32p)
        self._chk(lib().ope_voxel_grid(self.h, cloud.h, rgbp, C.c_float(lx), C.c_float(ly), C.c_float(lz),
                                       oxyz.ctypes.data_as(f32p), orgb.ctypes.data_as(f32p), C.byref(m)))
        return oxyz[:m.value].copy(), (orgb[:m.value].copy() if rgb is not None else None)

    # ---- features ----
    def normals_knn(self, cloud, k, vp=(0, 0, 0)):
        out = np.empty((len(cloud), 4), np.float32)
        v = (C.c_float * 3)(*vp)
        self._chk(lib().ope_normals_knn(self.h, cloud.h, k, v, out.ctypes.data_as(f32p)))
        return out

    def normals_radius(self, cloud, r, vp=(0, 0, 0)):
        """NormalEstimation with setRadiusSearch(r): (n, 4) nx, ny, nz, curvature; also written into the cloud."""
        out = np.empty((len(cloud), 4), np.float32)
        v = (C.c_float * 3)(*vp)
        self._chk(lib().ope_normals_radius(self.h, cloud.h, C.c_float(r), v, out.ctypes.data_as(f32p)))
        return out

    def fpfh(self, cloud, r, want_spfh=False):
        n = len(cloud)
        out = np.empty((n, 33), np.float32)
        sp = np.empty((n, 33), np.float32) if want_spfh else None
        self._chk(lib().ope_fpfh(self.h, cloud.h, C.c_float(r), out.ctypes.data_as(f32p),
                                 sp.ctypes.data_as(f32p) if want_spfh else None))
        return (out, sp) if want_spfh else out

    def pose_batch(self, model, frames, prm=None, tables=None, workers=8):
        """Batched first-frame localisation (C5). frames: list of host arrays (M, >=3) float32 or device Clouds. Returns
        (list of PoseResult, status array)."""
        m = np.ascontiguousarray(model[:, :3], np.float32)
        n = len(frames)
        arr, keep = self._frame_inputs(frames)
        res = (T.PoseResult * max(n, 1))()
        status = (C.c_int32 * max(n, 1))()
        tb = None
        if tables is not None:
            tb = (T.RngTable * n)(*tables)
        rc = lib().ope_pose_batch(self.h, None if prm is None else C.byref(prm), m.ctypes.data_as(f32p), C.c_size_t(len(m)), arr,
                                  C.c_size_t(n), tb, int(workers), res, status)
        st = np.array(list(status)[:n], np.int32)
        self._chk(rc)
        return [res[i] for i in range(n)], st

    def pose_track_batch(self, trackers, sources, targets, tables=None):
        """Advance each PoseTracker by one frame (ope_pose_tracker_step_batch): trackers[i] with its device Cloud sources[i]
        (its handle is replaced in place, as estimate_final_device does) against targets[i] (host array or Cloud). Returns
        (list of PoseResult, status array); a tracker that failed has its code in status, a failure of the call itself raises."""
        n = len(trackers)
        assert len(sources) == n and len(targets) == n
        arr, keep = self._frame_inputs(targets)
        th = (C.c_void_p * max(n, 1))(*[t.h for t in trackers])
        sh = (C.c_void_p * max(n, 1))(*[s.h for s in sources])
        res = (T.PoseResult * max(n, 1))()
        status = (C.c_int32 * max(n, 1))()
        tb = None if tables is None else (T.RngTable * n)(*tables)
        rc = lib().ope_pose_tracker_step_batch(self.h, th, sh, arr, C.c_size_t(n), tb, res, status)
        for i, s in enumerate(sources):
            s.h = C.c_void_p(sh[i])
        st = np.array(list(status)[:n], np.int32)
        if rc != 0 and not (st == rc).any():
            self._chk(rc)
        return [res[i] for i in range(n)], st

    # ---- registration ----
    def umeyama(self, src, tgt, isrc=None, itgt=None, n=None):
        a = None if isrc is None else np.ascontiguousarray(isrc, np.int32)
        b = None if itgt is None else np.ascontiguousarray(itgt, np.int32)
        if n is None:
            n = len(a) if a is not None else (len(b) if b is not None else len(src))
        Tm = (C.c_float * 16)()
        self._chk(lib().ope_umeyama(self.h, src.h, tgt.h, None if a is None else a.ctypes.data_as(i32p),
                                    None if b is None else b.ctypes.data_as(i32p), C.c_size_t(n), Tm))
        return T.mat4(Tm)

    def point_to_plane(self, src, tgt, isrc=None, itgt=None, n=None, kind=T.TE_POINT_TO_PLANE, want_info=False):
        """TransformationEstimationPointToPlane (Levenberg-Marquardt) / ...LLS::estimateRigidTransformation; tgt carries normals"""
        a = None if isrc is None else np.ascontiguousarray(isrc, np.int32)
        b = None if itgt is None else np.ascontiguousarray(itgt, np.int32)
        if n is None:
            n = len(a) if a is not None else (len(b) if b is not None else min(len(src), len(tgt)))
        Tm = (C.c_float * 16)()
        info = (C.c_int32 * 3)()
        self._chk(lib().ope_point_to_plane(self.h, src.h, tgt.h, None if a is None else a.ctypes.data_as(i32p),
                                           None if b is None else b.ctypes.data_as(i32p), C.c_size_t(n), int(kind), Tm, info))
        return (T.mat4(Tm), tuple(info)) if want_info else T.mat4(Tm)

    def fitness(self, src, tgt, M, max_range=np.finfo(np.float64).max):
        out = C.c_double(0)
        self._chk(lib().ope_fitness(self.h, src.h, tgt.h, T.mat4_to_c(M), C.c_double(max_range), C.byref(out)))
        return out.value

    def correspondences(self, src, tgt, prm):
        buf = (T.Correspondence * max(len(src), 1))()
        m = C.c_size_t(0)
        self._chk(lib().ope_correspondences(self.h, src.h, tgt.h, C.byref(prm), buf, C.byref(m)))
        a = np.ctypeslib.as_array(buf)[:m.value]
        return a["index_query"].copy(), a["index_match"].copy(), a["distance"].copy()

    def icp(self, src, tgt, prm, guess=None, want_corr=False, want_aligned=False, fixed=None):
        """fixed: (query indices, match indices) pinned by the caller (setFixedCorrespondences); with want_corr their rewritten
        distances are appended to the correspondence tuple's container as a further output"""
        res = T.RegResult()
        nf = 0 if fixed is None else len(fixed[0])
        buf = (T.Correspondence * max(len(src) + 2 * nf, 1))() if want_corr else None
        g = None if guess is None else T.mat4_to_c(guess)
        h = C.c_void_p()
        if nf:
            fb = (T.Correspondence * nf)()
            for i in range(nf):
                fb[i] = T.Correspondence(int(fixed[0][i]), int(fixed[1][i]), float(fixed[2][i]) if len(fixed) > 2 else 0.0)
            rc = lib().ope_icp_align_fixed(self.h, src.h, tgt.h if tgt is not None else None, C.byref(prm), g, fb, C.c_size_t(nf),
                                           C.byref(res), buf, C.byref(h) if want_aligned else None)
        else:
            rc = lib().ope_icp_align(self.h, src.h, tgt.h if tgt is not None else None, C.byref(prm), g, C.byref(res), buf,
                                     C.byref(h) if want_aligned else None)
        self._chk(rc)
        out = [res]
        if want_corr:
            a = np.ctypeslib.as_array(buf)[:res.n_correspondences]
            out.append((a["index_query"].copy(), a["index_match"].copy(), a["distance"].copy()))
            if nf:
                out.append(np.ctypeslib.as_array(fb)["distance"].copy())
        if want_aligned:
            out.append(Cloud(self, h))
        return out[0] if len(out) == 1 else tuple(out)

    def sacia(self, src, fsrc, tgt, ftgt, prm, table=None, want_errors=False):
        fs, ft = _f32(fsrc), _f32(ftgt)
        res = T.RegResult()
        errs = np.full(prm.max_iterations, np.nan, np.float32) if want_errors else None
        self._chk(lib().ope_sacia_align(self.h, src.h, fs.ctypes.data_as(f32p), tgt.h, ft.ctypes.data_as(f32p), C.byref(prm),
                                        None if table is None else C.byref(table), C.byref(res),
                                        None if errs is None else errs.ctypes.data_as(f32p)))
        return (res, errs) if want_errors else res


class SceneBatch:
    """ope_scene_batch: the cropped clouds and labels of a stack of depth images, resident on the device. .info: one SceneFrame
    per frame; .status: per-frame return codes (OPE_ERR_UNSUPPORTED where a RANSAC sample was degenerate)."""

    def __init__(self, ctx, handle, info, status):
        self.ctx, self.h, self.info, self.status = ctx, handle, info, status

    def __len__(self):
        return len(self.info)

    def frame(self, f):
        """(xyz (n_cropped, 3) float32, labels (n_cropped,) int32) of frame f, as ope_pass_through + ope_segment_objects_on_plane"""
        n = self.info[f].n_cropped
        xyz = np.empty((max(n, 1), 3), np.float32)
        labels = np.empty(max(n, 1), np.int32)
        self.ctx._chk(lib().ope_scene_batch_frame(self.h, C.c_size_t(f), xyz.ctypes.data_as(f32p), labels.ctypes.data_as(i32p), None))
        return xyz[:n].copy(), labels[:n].copy()

    def pose(self, model, cluster=None, tables=None, workers=8, prm=None):
        """ope_scene_pose_batch: frame f localised on cluster rank cluster[f] (None: 0 everywhere). Returns (PoseResults, status)."""
        m = np.ascontiguousarray(model[:, :3], np.float32)
        n = len(self.info)
        cl = None if cluster is None else np.ascontiguousarray(cluster, np.int32)
        assert cl is None or len(cl) == n
        res = (T.PoseResult * max(n, 1))()
        status = (C.c_int32 * max(n, 1))()
        tb = None if tables is None else (T.RngTable * n)(*tables)
        rc = lib().ope_scene_pose_batch(self.h, None if prm is None else C.byref(prm), m.ctypes.data_as(f32p), C.c_size_t(len(m)),
                                        None if cl is None else cl.ctypes.data_as(i32p), tb, int(workers), res, status)
        st = np.array(list(status)[:n], np.int32)
        self.ctx._chk(rc)
        return [res[i] for i in range(n)], st

    def centroids(self, f):
        """compute3DCentroid of frame f's clusters in rank order: (k, 3) float32 (one row, the whole cloud, when n_clusters == -1)"""
        k = max(self.info[f].n_clusters, 1)
        xyz = np.empty((k, 3), np.float32)
        m = C.c_int32(0)
        self.ctx._chk(lib().ope_scene_batch_centroids(self.h, C.c_size_t(f), xyz.ctypes.data_as(f32p), C.byref(m)))
        return xyz[:m.value].copy()

    def track(self, trackers, sources, **track_params):
        """ope_scene_track_step: camera i = frame i with PoseTracker trackers[i] and its device Cloud sources[i] (the handle is
        replaced in place when the tracker steps or acquires). track_params: any ope_track_params field. Returns (list of
        PoseResult, list of TrackChoice, status array); a failing camera has its code in status, a failure of the call itself
        raises."""
        n = len(self.info)
        assert len(trackers) == n and len(sources) == n
        tp = globals()["track_params"](**track_params)
        th = (C.c_void_p * max(n, 1))(*[t.h for t in trackers])
        sh = (C.c_void_p * max(n, 1))(*[s.h for s in sources])
        res = (T.PoseResult * max(n, 1))()
        ch = (T.TrackChoice * max(n, 1))()
        status = (C.c_int32 * max(n, 1))()
        rc = lib().ope_scene_track_step(self.h, C.byref(tp), th, sh, C.c_size_t(n), res, ch, status)
        for i, s in enumerate(sources):
            s.h = C.c_void_p(sh[i])
        st = np.array(list(status)[:n], np.int32)
        if rc != 0 and not (st == rc).any():
            self.ctx._chk(rc)
        return [res[i] for i in range(n)], [ch[i] for i in range(n)], st

    def close(self):
        # the handle holds device memory of its context: destroyed before the context is
        if self.h and self.ctx.h:
            lib().ope_scene_batch_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def comm_unique_id():
    """rank 0: the 128-byte NCCL unique id to hand to the other ranks"""
    buf = C.create_string_buffer(128)
    rc = lib().ope_comm_unique_id(buf, C.c_size_t(128))
    if rc != 0:
        raise OpeError(rc, "ope_comm_unique_id (libnccl.so.2 not loadable?)")
    return buf.raw


class Comm:
    """ope_comm: the library's own NCCL communicator for the sharded SAC-IA pool (one process per GPU)"""

    def __init__(self, ctx, unique_id, world, rank):
        self.ctx = ctx
        h = C.c_void_p()
        uid = None if unique_id is None else C.create_string_buffer(unique_id, 128)
        ctx._chk(lib().ope_comm_create(ctx.h, uid, C.c_size_t(0 if uid is None else 128), int(world), int(rank), C.byref(h)))
        self.h = h

    def close(self):
        if self.h and self.ctx.h:
            lib().ope_comm_destroy(self.h)
        self.h = None

    def sacia(self, src, fsrc, tgt, ftgt, prm, table):
        fs, ft = _f32(fsrc), _f32(ftgt)
        res = T.RegResult()
        self.ctx._chk(lib().ope_sacia_align_sharded(self.ctx.h, self.h, src.h, fs.ctypes.data_as(f32p), tgt.h, ft.ctypes.data_as(f32p),
                                                    C.byref(prm), C.byref(table), C.byref(res)))
        return res


def sacia_draw(src_xyz, iterations, nr_samples, k_corr, min_sample_distance):
    s = _f32(src_xyz)
    samples = np.empty((iterations, nr_samples), np.int32)
    picks = np.empty((iterations, nr_samples), np.int32)
    msd = C.c_float(min_sample_distance)
    rc = lib().ope_sacia_draw(s.ctypes.data_as(f32p), C.c_size_t(s.shape[0]), C.c_size_t(s.strides[0]), iterations, nr_samples,
                              k_corr, C.byref(msd), samples.ctypes.data_as(i32p), picks.ctypes.data_as(i32p))
    if rc != 0:
        raise OpeError(rc, "ope_sacia_draw")
    return samples, picks


class PoseTracker:
    """PoseEstimator (D&L/src/poseestimator.cpp) on the device."""

    def __init__(self, ctx, prm=None):
        self.ctx = ctx
        h = C.c_void_p()
        ctx._chk(lib().ope_pose_tracker_create(ctx.h, None if prm is None else C.byref(prm), C.byref(h)))
        self.h = h

    def close(self):
        if self.h and self.ctx.h:
            lib().ope_pose_tracker_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def estimate_final(self, source, target, table=None):
        """Host buffers: source (N,3) float32 modified in place; target (M,>=3)."""
        assert source.dtype == np.float32 and source.flags.c_contiguous and source.shape[1] == 3
        t = _f32(target) if len(target) else np.zeros((0, 3), np.float32)
        res = T.PoseResult()
        self.ctx._chk(lib().ope_pose_estimate_final(self.h, source.ctypes.data_as(f32p), C.c_size_t(source.shape[0]),
                                                    t.ctypes.data_as(C.c_void_p), C.c_size_t(t.shape[0]),
                                                    C.c_size_t(t.strides[0] if len(t) else 12), C.c_size_t(0),
                                                    None if table is None else C.byref(table), C.byref(res)))
        return res

    def estimate_final_device(self, source_cloud, target_cloud, table=None):
        """Device-resident clouds; source_cloud's handle is replaced by alignedSource."""
        res = T.PoseResult()
        self.ctx._chk(lib().ope_pose_estimate_final_device(self.h, C.byref(source_cloud.h),
                                                           target_cloud.h if target_cloud is not None else None,
                                                           None if table is None else C.byref(table), C.byref(res)))
        return res

    def stage_ms(self):
        out = (C.c_double * 8)()
        lib().ope_pose_stage_ms(self.h, out)
        return list(out)
