"""The single-frame scene preparation calls ope_pass_through -> ope_plane_ransac -> ope_segment_objects_on_plane against the oracle
on the frames and edge images that test_gpu_scene_batch.py only compares with the batch. The single-frame calls are one-frame runs of
the batch's stages, so that comparison cannot tell a wrong stage from a right one; the oracle can. Also a degenerate RANSAC sample,
which fails both calls."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

LIMITS = (-0.5, 0.5, -0.5, 0.3, 0.5, 1.6)      # ObjectSegmentationPlane::getFiltered, D&L/src/objectsegmentationplane.cpp:17-18
FRAMES = (23, 24, 25, 26, 27, 28)
SMALL_CAM = dict(fx=262.5, fy=262.5, cx=119.5, cy=159.5, scale=1000.0, z_max=2.0)


def _depth_mm(cloud):
    return np.rint(np.nan_to_num(cloud[..., 2], nan=0.0).astype(np.float64) * 1000.0).astype(np.uint16)


@pytest.fixture(scope="module")
def depths(synth, model):
    return {f: _depth_mm(synth.make_frame(model, f)[1]) for f in FRAMES}


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _check_against_oracle(ctx, orc, depth, **cam):
    """depth -> cloud -> pass-through -> plane RANSAC and segmentation, each equal to the oracle bit for bit; returns n_clusters"""
    pts = orc.depth_to_cloud(depth, **cam)
    keep = np.arange(len(pts), dtype=np.int32)
    for field, lo, hi in ((2, LIMITS[4], LIMITS[5]), (1, LIMITS[2], LIMITS[3]), (0, LIMITS[0], LIMITS[1])):   # z, y, x
        keep = keep[orc.pass_through(pts[keep], field, lo, hi)]
    sub = pts[keep]
    c = ctx.depth_to_cloud(depth, **cam)
    assert np.array_equal(_bits(c.download()), _bits(pts))
    filt, idx = ctx.pass_through(c, LIMITS, want_idx=True)
    assert np.array_equal(idx, keep) and np.array_equal(_bits(filt.download()), _bits(sub))
    ol, ok, op1, op2, oit = orc.segment_objects_on_plane(sub)
    gl, gk, gp1, gp2, git = ctx.segment_objects_on_plane(filt)
    assert gk == ok and git == tuple(oit)
    assert np.array_equal(_bits(gp1), _bits(op1)) and np.array_equal(_bits(gp2), _bits(op2))
    assert np.array_equal(gl, ol), int((gl != ol).sum())
    # the table plane alone: on these images it exists exactly when the oracle's segmentation succeeds
    found, coeff, inl, it = ctx.plane_ransac(filt)
    assert found == (ok >= 0) and it == oit[0] and np.array_equal(_bits(coeff), _bits(op1))
    if found:   # the inliers: |c . p| < 0.01 in the path's float order (c0 x + c1 y) + (c2 z + c3)
        d = (coeff[0] * sub[:, 0] + coeff[1] * sub[:, 1]) + (coeff[2] * sub[:, 2] + coeff[3] * np.float32(1.0))
        assert np.array_equal(inl, np.nonzero(np.abs(d).astype(np.float64) < 0.01)[0])
    else:
        assert len(inl) == 0
    return gk


@pytest.mark.parametrize("frame", FRAMES[1:])
def test_single_frame_calls_equal_the_oracle(ctx, orc, depths, frame):
    assert _check_against_oracle(ctx, orc, depths[frame]) >= 0


def _empty_table(synth, model):
    """a table with nothing on it: the object far outside the view, the wall beyond the crop, no noise"""
    pose = np.eye(4)
    pose[:3, 3] = (5.0, 0.1, 1.0)
    cloud, _ = synth.render_scene(model, pose, np.random.default_rng(0), wall_z=1.9, noise=False)
    return _depth_mm(cloud)


def test_edge_images_equal_the_oracle(ctx, orc, synth, model):
    zero = np.zeros((480, 640), np.uint16)
    two = np.zeros((480, 640), np.uint16)
    two[240, 320] = two[241, 320] = 1000                              # two points inside the crop: no plane
    assert _check_against_oracle(ctx, orc, zero) == -1
    assert _check_against_oracle(ctx, orc, two) == -1
    assert _check_against_oracle(ctx, orc, _empty_table(synth, model)) == 0


@pytest.mark.parametrize("frame", (23, 24, 25))
def test_other_intrinsics_equal_the_oracle(ctx, orc, depths, frame):
    """320 x 240 with other intrinsics"""
    assert _check_against_oracle(ctx, orc, depths[frame][::2, ::2].copy(), **SMALL_CAM) >= 0


def test_degenerate_sample_fails_both_calls(ctx, cuda_lib):
    """collinear points (i, 2i, 3i): PCL's ratio test is exact, so the first sample is degenerate. PCL would draw again; the path
    cannot replay that and fails with OPE_ERR_UNSUPPORTED"""
    T = cuda_lib.T
    i = np.arange(100, dtype=np.float32)
    cloud = ctx.upload(np.stack([i, 2 * i, 3 * i], 1))
    for call in (ctx.plane_ransac, ctx.segment_objects_on_plane):
        with pytest.raises(cuda_lib.OpeError) as e:
            call(cloud)
        assert e.value.rc == T.OPE_ERR_UNSUPPORTED and "degenerate" in str(e.value)
    # the raw outputs of the failed segmentation: every label outside the prism, no clusters, iterations and planes untouched
    labels = np.zeros(100, np.int32)
    p1, p2 = (C.c_float * 4)(7, 7, 7, 7), (C.c_float * 4)(7, 7, 7, 7)
    it = (C.c_int32 * 2)(-9, -9)
    k = C.c_int32(5)
    rc = cuda_lib.lib().ope_segment_objects_on_plane(ctx.h, cloud.h, None, labels.ctypes.data_as(C.POINTER(C.c_int32)), p1, p2, it,
                                                     C.byref(k))
    assert rc == T.OPE_ERR_UNSUPPORTED and k.value == -1 and (labels == T.SEG_OUTSIDE_PRISM).all()
    assert list(it) == [-9, -9] and list(p1) == [7] * 4 and list(p2) == [7] * 4
