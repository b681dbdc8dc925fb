"""k-NN with 32 < k <= 256, normals over k > 32 neighbours and over a search radius, against the CPU oracle; the pose entry points
with normal_k = 40; and NormalEstimation::setRadiusSearch through the PCL-style C++ shim.

Bars: k-NN indices and squared distances bit-equal (grid path; normals also on the shared-memory path below 4 096 points and with
the grid forced). Normals: the same finite mask as the oracle, bit-equal on the exact clouds of test_gpu_feature_paths.py (lattice,
plate, wire) and within 2e-6 elsewhere. Radius normals are unchanged when the scratch budget splits the queries into several
tiles. The pose paths equal their serial definitions as tests/test_gpu_pose_batch_frames.py and tests/test_gpu_track_batch.py
state them, and agree with the oracle's estimateFinalPose at the contract's bar."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import orc_radius
from test_gpu_feature_paths import feature_cases, size_cases
from test_gpu_track_batch import _compare, _play, _schedule

pytestmark = pytest.mark.gpu

libc = ctypes.CDLL(None)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KNN_KS = (33, 48, 64, 100, 255, 256)
NORMAL_KS = (33, 64, 256)
EXACT = ("lattice", "wire", "plate")
ATOL = 2e-6


def _same_normals(got, ref, exact, what):
    fg, fr = np.isfinite(got).all(1), np.isfinite(ref).all(1)
    assert np.array_equal(fg, fr), (what, np.nonzero(fg != fr)[0][:10])
    if exact:
        assert np.array_equal(got[fg].view(np.uint32), ref[fr].view(np.uint32)), what
    elif fg.any():
        assert np.abs(got[fg] - ref[fr]).max() <= ATOL, (what, np.abs(got[fg] - ref[fr]).max())


def _same_knn(ctx, orc, pts, qry, k, what):
    cl = ctx.upload(pts)
    try:
        idx, d2 = ctx.knn(cl, qry, k)
    finally:
        cl.free()
    ridx, rd2 = orc.knn(pts, qry, k)
    ok = np.isfinite(qry[:, :3]).all(1)
    assert np.array_equal(idx[ok], ridx[ok]), what
    assert np.array_equal(d2[ok].view(np.uint32), rd2[ok].view(np.uint32)), what
    assert (idx[~ok] == -1).all() and np.isinf(d2[~ok]).all(), what


@pytest.fixture(scope="module")
def scene(synth, model):
    """a 640 x 480 organised C3 frame (307 200 points)"""
    cloud = synth.make_frame(model, 940)[1]
    return np.ascontiguousarray(cloud.reshape(-1, cloud.shape[-1])[:, :3], np.float32)


# ------------------------------------------------------------------------------------------------------- k-NN ----
@pytest.mark.parametrize("k", KNN_KS)
def test_knn_above_32_on_the_adversarial_clouds(ctx, orc, k):
    for name, pts, *_ in feature_cases():
        _same_knn(ctx, orc, pts, pts, k, (name, k))
    for name, pts in size_cases():
        _same_knn(ctx, orc, pts, pts, k, (name, k))   # below and above 4 096 targets, fewer targets than k


@pytest.mark.parametrize("k", (33, 256))
def test_knn_above_32_on_the_model(ctx, orc, model, k):
    _same_knn(ctx, orc, model, model[::97].copy(), k, ("model", k))


def test_knn_k_above_the_cap_is_invalid(ctx, cuda_lib, small_model):
    cl = ctx.upload(small_model)
    L = cuda_lib.lib()
    k = 257
    idx = np.empty((4, k), np.int32)
    d2 = np.empty((4, k), np.float32)
    q = np.ascontiguousarray(small_model[:4, :3], np.float32)
    rc = L.ope_knn(ctx.h, cl.h, q.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(4), ctypes.c_size_t(12), ctypes.c_size_t(0), k,
                   idx.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), d2.ctypes.data_as(ctypes.POINTER(ctypes.c_float)))
    assert rc == cuda_lib.T.OPE_ERR_INVALID
    out = np.empty((len(small_model), 4), np.float32)
    rc = L.ope_normals_knn(ctx.h, cl.h, k, (ctypes.c_float * 3)(0, 0, 0), out.ctypes.data_as(ctypes.POINTER(ctypes.c_float)))
    assert rc == cuda_lib.T.OPE_ERR_INVALID
    cl.free()


# ---------------------------------------------------------------------------------------------- k-NN normals ----
def _normals_knn(ctx, pts, k, vp):
    cl = ctx.upload(pts)
    try:
        return ctx.normals_knn(cl, k, vp)
    finally:
        cl.free()


@pytest.mark.parametrize("force_grid", (False, True))
@pytest.mark.parametrize("k", NORMAL_KS)
def test_normals_above_32_on_the_adversarial_clouds(ctx, orc, monkeypatch, k, force_grid):
    if force_grid:
        monkeypatch.setenv("OPE_NORMALS_FORCE_GRID", "1")
    for name, pts, _, vps, _, exact in feature_cases():
        for vp in vps:
            _same_normals(_normals_knn(ctx, pts, k, vp), orc.normals_knn(pts, k, vp), exact, (name, k, vp))
    for name, pts in size_cases():
        if name in ("n4096", "n4097") or len(pts) <= k + 1:
            _same_normals(_normals_knn(ctx, pts, k, (0, 0, 0)), orc.normals_knn(pts, k), True, (name, k))


@pytest.mark.parametrize("k", (64, 256))
def test_normals_above_32_on_the_model(ctx, orc, model, k):
    _same_normals(_normals_knn(ctx, model, k, (0, 0, 0)), orc.normals_knn(model, k), False, ("model", k))


# -------------------------------------------------------------------------------------------- radius normals ----
def _normals_radius(ctx, pts, r, vp=(0, 0, 0)):
    cl = ctx.upload(pts)
    try:
        return ctx.normals_radius(cl, r, vp)
    finally:
        cl.free()


def test_radius_normals_on_the_adversarial_clouds(ctx, orc):
    for name, pts, _, vps, r, exact in feature_cases():
        for rr in (r, 2 * r):
            for vp in vps:
                _same_normals(_normals_radius(ctx, pts, rr, vp), orc_radius.normals_radius(pts, rr, vp), exact, (name, rr, vp))
    for name, pts in size_cases():
        _same_normals(_normals_radius(ctx, pts, 2 / 64), orc_radius.normals_radius(pts, 2 / 64), True, name)


def test_radius_normals_on_the_scene(ctx, orc, scene):
    got = _normals_radius(ctx, scene, 0.03)
    _same_normals(got, orc_radius.normals_radius(scene, 0.03), False, "scene 3 cm")


def test_radius_normals_on_the_model_in_several_tiles(ctx, orc, model, monkeypatch):
    """At 3 cm the model's neighbourhoods exceed the shared-memory lists (8 192 keys); a 32 MB budget cuts the queries into
    several tiles, and a budget smaller than one list runs each long list alone: the same bits every time."""
    from scipy.spatial import cKDTree
    counts = cKDTree(model[:, :3].astype(np.float64)).query_ball_point(model[:, :3], 0.03, return_length=True)
    assert counts.max() > 8192, counts.max()
    got = _normals_radius(ctx, model, 0.03)
    _same_normals(got, orc_radius.normals_radius(model, 0.03), False, "model 3 cm")
    for budget in (32 << 20, 4096):
        monkeypatch.setenv("OPE_RADIUS_NORMALS_SCRATCH_BYTES", str(budget))
        again = _normals_radius(ctx, model, 0.03)
        assert np.array_equal(again.view(np.uint32), got.view(np.uint32)), budget


def test_radius_argument_checks(ctx, cuda_lib, small_model):
    cl = ctx.upload(small_model)
    L = cuda_lib.lib()
    for r in (0.0, -0.01, float("inf"), float("nan")):
        assert L.ope_normals_radius(ctx.h, cl.h, ctypes.c_float(r), None, None) == cuda_lib.T.OPE_ERR_INVALID, r
    cl.free()


# ------------------------------------------------------------------------------------------ pose path, k = 40 ----
@pytest.fixture(scope="module")
def frames(synth, model):
    return [synth.make_frame(model, 950 + f)[0] for f in range(4)]


def test_pose_batch_with_normal_k_40_equals_fresh_trackers(ctx, synth, cuda_lib, model, frames, monkeypatch):
    T = cuda_lib.T
    prm = cuda_lib.pose_params(normal_k=40)
    runs = []
    for lanes, chunk in ((1, 64), (4, 3), (8, 1)):
        monkeypatch.setenv("OPE_BATCH_LANES", str(lanes))
        monkeypatch.setenv("OPE_BATCH_CHUNK", str(chunk))
        libc.srand(5)
        res, status = ctx.pose_batch(model, frames, prm=prm, tables=None)
        runs.append((res, list(status), libc.rand()))
    ref, ref_status, ref_after = runs[0]
    assert ref_status == [0] * len(frames)
    for res, status, after in runs[1:]:
        assert status == ref_status and after == ref_after
        assert all(bytes(g) == bytes(r) for g, r in zip(res, ref))
    libc.srand(5)
    for f, cl in enumerate(frames):
        tr = cuda_lib.PoseTracker(ctx, prm)
        s = tr.estimate_final(model.copy(), cl)
        tr.close()
        g = ref[f]
        for name in ("final_pose", "coarse_pose", "fine_pose", "rigid_model_pose"):
            rot, tr_ = synth.pose_error(T.mat4(getattr(g, name)), T.mat4(getattr(s, name)))
            assert rot < 1e-6 and tr_ < 1e-6, (f, name, rot, tr_)
        for name in ("ran_coarse", "icp_iterations", "icp_state", "icp_converged", "sacia_best_iteration", "n_src_coarse", "n_tgt_coarse",
                     "n_src_fine", "n_tgt_fine"):
            assert getattr(g, name) == getattr(s, name), (f, name)
        assert abs(g.fitness - s.fitness) < 1e-9, f
    assert libc.rand() == ref_after   # the serial loop consumed rand() as the batch did


@pytest.fixture(scope="module")
def sequences(synth, model):
    return [[f[0] for f in synth.make_sequence(model, 60 + s, 3)] for s in range(4)]


def test_tracker_step_batch_with_normal_k_40_equals_the_serial_loop(ctx, synth, cuda_lib, model, sequences, monkeypatch):
    specs = [(model, cuda_lib.pose_params(normal_k=40))] * len(sequences)
    sched = _schedule(sequences, 3)
    batch, rb = _play(ctx, cuda_lib, specs, sched, True)
    monkeypatch.setenv("OPE_ICP_SMALL", "1")
    serial, rs = _play(ctx, cuda_lib, specs, sched, False)
    exact, total = _compare(synth, cuda_lib.T, batch, serial)
    print("bit-identical results and sources: %d of %d" % (exact, total))
    assert rb == rs
    assert total > 0


def test_normal_k_40_against_the_oracle(ctx, orc, synth, cuda_lib, model, sequences):
    specs = [(model, cuda_lib.pose_params(normal_k=40))] * 2
    sched = _schedule(sequences[:2], 2)
    batch, _ = _play(ctx, cuda_lib, specs, sched, True, seed=3)
    orc.srand(3)
    ests = [orc.PoseEstimator(orc.pose_params(normal_k=40)) for _ in range(2)]
    srcs = [model.copy() for _ in range(2)]
    for k, step in enumerate(sched):
        for j, (i, t) in enumerate(step):
            o = ests[i].estimate_final(srcs[i], t)
            g = batch[k][j][0]
            rot, tr = synth.pose_error(cuda_lib.T.mat4(g.final_pose), np.array(o.final_pose, np.float64).reshape(4, 4).T)
            assert rot < 1e-4 and tr < 1e-5, (k, i, rot, tr)
            assert abs(g.fitness - o.fitness) < 1e-5
            assert (g.icp_iterations, g.icp_state) == (o.icp_iterations, o.icp_state)


# ---------------------------------------------------------------------------------------------- the C++ shim ----
@pytest.fixture(scope="module")
def normals_harness(cuda_lib, tmp_path_factory):
    cuda_lib.build()
    exe = str(tmp_path_factory.mktemp("shim") / "normals_harness")
    lib_dir = os.path.join(ROOT, "object-pose-estimation_b200")
    subprocess.run(["g++", "-O2", "-std=c++17", "-I" + os.path.join(ROOT, "include", "ope_pcl_compat"), "-o", exe,
                    os.path.join(ROOT, "tests", "cpp", "normals_harness.cpp"), "-L" + lib_dir, "-lope_cuda", "-Wl,-rpath," + lib_dir,
                    "-Wl,-rpath,/usr/local/cuda/lib64"], check=True)
    return exe


def _shim(exe, tmp_path, pts, k, r):
    src, dst = str(tmp_path / "in.f32"), str(tmp_path / "out.f32")
    np.ascontiguousarray(pts[:, :3], np.float32).tofile(src)
    p = subprocess.run([exe, src, str(k), repr(r), dst], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert p.returncode == 0, p.stderr
    n, untouched = map(int, p.stdout.split())
    return np.fromfile(dst, np.float32).reshape(-1, 4), n, untouched, p.stderr


def test_shim_radius_search(ctx, normals_harness, tmp_path, small_model):
    got, n, _, err = _shim(normals_harness, tmp_path, small_model, 0, 0.03)
    assert n == len(small_model), err
    assert np.array_equal(got.view(np.uint32), _normals_radius(ctx, small_model, 0.03).view(np.uint32))


def test_shim_both_or_neither_is_the_pcl_error(normals_harness, tmp_path, small_model):
    pts = small_model[:500]
    _, n, untouched, err = _shim(normals_harness, tmp_path, pts, 12, 0.03)
    assert "Both radius" in err and "and K (12) defined!" in err
    assert n == len(pts) and untouched == 1
    _, n, untouched, err = _shim(normals_harness, tmp_path, pts, 0, 0.0)
    assert "Neither radius nor K defined!" in err
    assert n == len(pts) and untouched == 1
