"""ope_pose_batch finishes the frames outside its frame-spanning launches (tiny, empty or oversized clusters, or every frame when
the ICP parameters are outside them) on its chunk lanes, one frame per chunk. Whatever the lanes and chunks, every result is the same, and a
frame that fails there fails alone."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

libc = ctypes.CDLL(None)
H, S, K = 400, 5, 5
BIG, CLOUD = 4, 3     # the oversized frame (per-frame path), the frame given as a device cloud
CUTS = ((1, 64), (4, 3), (8, 1))   # (OPE_BATCH_LANES, OPE_BATCH_CHUNK)


@pytest.fixture(scope="module")
def frames(synth, model):
    fs = [synth.make_frame(model, 900 + f)[0] for f in range(4)]
    # four copies of a cluster side by side: more 1 cm and 8 mm voxels than the fast path's samples hold
    big = np.concatenate([fs[0] + np.array([dx, dy, 0], np.float32) for dx in (0, 0.4) for dy in (0, 0.4)])
    return fs + [big, fs[1][:60].copy(), fs[2][::40].copy(), np.zeros((0, 3), np.float32)]


@pytest.fixture(scope="module")
def inputs(ctx, frames):
    cloud = ctx.upload(frames[CLOUD])
    yield [cloud if f == CLOUD else x for f, x in enumerate(frames)]
    cloud.free()


def _run(ctx, model, inputs, monkeypatch, lanes, chunk, prm=None, seed=5):
    monkeypatch.setenv("OPE_BATCH_LANES", str(lanes))
    monkeypatch.setenv("OPE_BATCH_CHUNK", str(chunk))
    libc.srand(seed)
    res, status = ctx.pose_batch(model, inputs, prm=prm, tables=None)
    return res, list(status), libc.rand()


def _same_for_every_cut(ctx, model, inputs, monkeypatch, prm=None):
    runs = [_run(ctx, model, inputs, monkeypatch, lanes, chunk, prm) for lanes, chunk in CUTS]
    ref, ref_status, ref_after = runs[0]
    assert ref_status == [0] * len(inputs)
    for (lanes, chunk), (res, status, after) in zip(CUTS[1:], runs[1:]):
        assert status == ref_status, (lanes, chunk)
        assert after == ref_after, (lanes, chunk)   # rand() stands at the same place
        for f, (g, r) in enumerate(zip(res, ref)):
            assert bytes(g) == bytes(r), (lanes, chunk, f)
    return ref


def test_lanes_and_chunks_change_no_result(ctx, model, inputs, monkeypatch):
    res = _same_for_every_cut(ctx, model, inputs, monkeypatch)
    assert res[BIG].n_tgt_coarse > 2048   # beyond the fast path's 1 cm capacity: this frame ran on the per-frame path
    assert all(r.ran_coarse == 1 for r in res[:5])


def test_every_frame_on_the_per_frame_path(ctx, synth, cuda_lib, model, frames, inputs, monkeypatch):
    """The nearest-neighbour estimator is outside the frame-spanning ICP: every frame runs as a fresh tracker would, on the lanes."""
    T = cuda_lib.T
    prm = cuda_lib.pose_params()
    prm.icp.estimator = T.EST_NEAREST
    got = _same_for_every_cut(ctx, model, inputs, monkeypatch, prm)
    libc.srand(5)
    for f, cl in enumerate(frames):
        tr = cuda_lib.PoseTracker(ctx, prm)
        s = tr.estimate_final(model.copy(), cl)
        tr.close()
        g = got[f]
        for name in ("final_pose", "coarse_pose", "fine_pose", "rigid_model_pose"):
            rot, tr_ = synth.pose_error(T.mat4(getattr(g, name)), T.mat4(getattr(s, name)))
            assert rot < 1e-6 and tr_ < 1e-6, (f, name, rot, tr_)
        for name in ("ran_coarse", "icp_iterations", "icp_state", "icp_converged", "sacia_best_iteration", "n_src_coarse", "n_tgt_coarse",
                     "n_src_fine", "n_tgt_fine"):
            assert getattr(g, name) == getattr(s, name), (f, name, getattr(g, name), getattr(s, name))
        assert abs(g.fitness - s.fitness) < 1e-9, f


def test_failing_frames_fail_alone_and_the_lowest_is_reported(ctx, cuda_lib, model, inputs, frames, monkeypatch):
    """Two oversized frames in different chunks get a table with an out-of-range entry: each fails alone, and whatever the lanes
    and chunks, the call reports the lower one."""
    T = cuda_lib.T
    inputs = list(inputs) + [frames[BIG]]    # a second oversized frame, last
    bad_frames = (BIG, len(inputs) - 1)
    cl = ctx.upload(model)
    sp = ctx.uniform_sample_cloud(cl, 0.01)
    xyz = sp.download()
    sp.free(); cl.free()
    msd = cuda_lib.pose_params().sacia.min_sample_distance
    libc.srand(9)
    drawn = [cuda_lib.sacia_draw(xyz, H, S, K, msd) for _ in inputs]
    valid = [cuda_lib.rng_table(s, p) for s, p in drawn]
    ref, ref_status = ctx.pose_batch(model, inputs, tables=valid)
    assert (ref_status == 0).all()
    tables = list(valid)
    for f in bad_frames:
        bad_samples = drawn[f][0].copy()
        bad_samples[0, 0] = len(xyz) + 1000     # outside the model's 1 cm sample
        tables[f] = cuda_lib.rng_table(bad_samples, drawn[f][1])
    n = len(inputs)
    arr, keep = ctx._frame_inputs(inputs)
    m = np.ascontiguousarray(model[:, :3], np.float32)
    for lanes, chunk in CUTS:
        monkeypatch.setenv("OPE_BATCH_LANES", str(lanes))
        monkeypatch.setenv("OPE_BATCH_CHUNK", str(chunk))
        res = (T.PoseResult * n)()
        status = (ctypes.c_int32 * n)()
        rc = cuda_lib.lib().ope_pose_batch(ctx.h, None, m.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), ctypes.c_size_t(len(m)), arr,
                                           ctypes.c_size_t(n), (T.RngTable * n)(*tables), 16, res, status)
        assert rc == T.OPE_ERR_INVALID, (lanes, chunk)
        assert cuda_lib.lib().ope_last_error(ctx.h).decode().startswith("frame %d:" % BIG), (lanes, chunk)
        assert list(status) == [T.OPE_ERR_INVALID if f in bad_frames else T.OPE_OK for f in range(n)], (lanes, chunk)
        for f in range(n):
            if f not in bad_frames:
                assert bytes(res[f]) == bytes(ref[f]), (lanes, chunk, f)
