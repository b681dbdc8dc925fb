"""SAC-IA scoring paths against the oracle. The single-frame call is a one-frame run of the frame-spanning stages: targets that
fit (<= 8 192 points, with the source's terms in shared memory) go to the shared-memory scorer, everything else to the grid
index. Every path, every shard of the pool and every scorer setting must give the oracle's errors, winner and transform."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

KW = dict(max_iterations=400, nr_samples=5, k_correspondences=5, min_sample_distance=0.01, max_correspondence_distance=0.05)


@pytest.fixture(scope="module")
def pair(orc, synth, model):
    """the model's 1 cm sample with FPFH, a frame's 1 cm cluster sample with FPFH, and a 400-hypothesis table"""
    cl, _, _ = synth.make_frame(model, 2)
    sp = model[orc.uniform_sample(model, 0.01)]
    tp = cl[orc.uniform_sample(cl, 0.01)]
    sf = orc.fpfh(sp, orc.normals_knn(sp, 30), 0.03)
    tf = orc.fpfh(tp, orc.normals_knn(tp, 30), 0.03)
    orc.srand(1)
    samples, picks = orc.sacia_draw(sp, 400, 5, 5, 0.01)
    return sp, sf, tp, tf, samples, picks


def _oracle(orc, sp, sf, tp, tf, samples, picks, **kw):
    return orc.sacia(sp, sf, tp, tf, orc.sacia_params(**{**KW, **kw}), orc.rng_table(samples, picks), want_errors=True)


def _device(ctx, cuda_lib, sp, sf, tp, tf, samples, picks, want_errors=True, **kw):
    return ctx.sacia(ctx.upload(sp), sf, ctx.upload(tp), tf, cuda_lib.sacia_params(**{**KW, **kw}), cuda_lib.rng_table(samples, picks),
                     want_errors=want_errors)


def _same(g, o):
    assert g.best_iteration == o.best_iteration and g.best_error == o.best_error
    assert np.array_equal(np.array(list(g.T)), np.array(list(o.T)))


@pytest.mark.parametrize("nt", [8192, 8193])
def test_targets_either_side_of_the_scorer_choice(ctx, orc, cuda_lib, pair, nt):
    sp, sf, _, _, samples, picks = pair
    rng = np.random.default_rng(nt)
    base = pair[2]
    tp = np.concatenate([base + rng.normal(scale=0.004, size=base.shape).astype(np.float32) for _ in range(nt // len(base) + 1)])[:nt]
    tf = orc.fpfh(tp, orc.normals_knn(tp, 30), 0.03)
    o, oe = _oracle(orc, sp, sf, tp, tf, samples, picks)
    g, ge = _device(ctx, cuda_lib, sp, sf, tp, tf, samples, picks)
    assert np.array_equal(ge, oe), np.nanmax(np.abs(ge - oe))
    _same(g, o)
    _same(_device(ctx, cuda_lib, sp, sf, tp, tf, samples, picks, want_errors=False), o)


def test_source_too_large_for_shared_memory_terms(ctx, orc, cuda_lib, pair):
    """60 000 source points: 240 KB of terms alone exceed the shared memory of a block, so the grid scorer answers"""
    _, _, tp, tf, _, _ = pair
    rng = np.random.default_rng(11)
    sp = np.concatenate([pair[0] + rng.normal(scale=0.003, size=pair[0].shape).astype(np.float32) for _ in range(60000 // len(pair[0]) + 1)])[:60000]
    sf = np.concatenate([pair[1]] * (60000 // len(pair[1]) + 1))[:60000]
    H = 64
    orc.srand(3)
    samples, picks = orc.sacia_draw(sp, H, 5, 5, 0.01)
    o, oe = _oracle(orc, sp, sf, tp, tf, samples, picks, max_iterations=H)
    g, ge = _device(ctx, cuda_lib, sp, sf, tp, tf, samples, picks, max_iterations=H)
    assert np.array_equal(ge, oe), np.nanmax(np.abs(ge - oe))
    _same(g, o)


def test_duplicate_hypotheses_first_wins(ctx, orc, cuda_lib, pair):
    sp, sf, tp, tf, samples, picks = pair
    s = np.tile(samples.reshape(400, 5)[:100], (4, 1)).reshape(samples.shape)
    p = np.tile(picks.reshape(400, 5)[:100], (4, 1)).reshape(picks.shape)
    o, oe = _oracle(orc, sp, sf, tp, tf, s, p)
    assert o.best_iteration < 100 and (oe[:100] == oe[100:200]).all()
    for want_errors in (True, False):
        g = _device(ctx, cuda_lib, sp, sf, tp, tf, s, p, want_errors=want_errors)
        if want_errors:
            g, ge = g
            assert np.array_equal(ge, oe)
        _same(g, o)


def test_shards_of_the_pool(ctx, orc, cuda_lib, pair):
    sp, sf, tp, tf, samples, picks = pair
    full, fe = _device(ctx, cuda_lib, sp, sf, tp, tf, samples, picks)
    for b, e in ((0, 1), (399, 400), (137, 263), (400, 401)):
        g, ge = _device(ctx, cuda_lib, sp, sf, tp, tf, samples, picks, hypothesis_begin=b, hypothesis_end=e)
        e = min(e, 400)
        assert np.array_equal(ge[b:e], fe[b:e])
        assert np.isnan(ge[:b]).all() and np.isnan(ge[e:]).all()
        if b == e:
            assert (g.best_iteration, g.converged, g.best_error) == (-1, 0, 0.0)
            assert np.array_equal(np.array(list(g.T)), np.eye(4, dtype=np.float32).ravel())
        else:
            assert g.best_iteration == b + int(np.argmin(fe[b:e])) and g.best_error == fe[g.best_iteration]
            g_only = _device(ctx, cuda_lib, sp, sf, tp, tf, samples, picks, want_errors=False, hypothesis_begin=b, hypothesis_end=e)
            assert (g_only.best_iteration, g_only.best_error) == (g.best_iteration, g.best_error)


def test_every_scorer_setting_gives_the_same_bits(ctx, orc, cuda_lib, pair, monkeypatch):
    sp, sf, tp, tf, samples, picks = pair
    o, oe = _oracle(orc, sp, sf, tp, tf, samples, picks)
    for env in ({}, {"OPE_SACIA_PATH": "grid"}, {"OPE_SACIA_EARLY_EXIT": "0"}, {"OPE_SACIA_PATH": "smem"}):
        with monkeypatch.context() as m:
            for k, v in env.items():
                m.setenv(k, v)
            g, ge = _device(ctx, cuda_lib, sp, sf, tp, tf, samples, picks)
            assert np.array_equal(ge, oe), env
            _same(g, o)
            _same(_device(ctx, cuda_lib, sp, sf, tp, tf, samples, picks, want_errors=False), o)


def test_pose_batch_frames_equal_the_single_frame_sacia(ctx, synth, cuda_lib, model):
    """a batch of three frames (the scorer's blocks hold fewer hypotheses) gives every frame the single-frame SAC-IA winner"""
    libc = ctypes.CDLL(None)
    frames = [synth.make_frame(model, 910 + f)[0] for f in range(3)]
    libc.srand(5)
    serial = []
    for cl in frames:
        tr = cuda_lib.PoseTracker(ctx)
        serial.append(tr.estimate_final(model.copy(), cl))
        tr.close()
    libc.srand(5)
    got, status = ctx.pose_batch(model, frames, workers=1)
    assert (status == 0).all()
    for g, s in zip(got, serial):
        assert (g.sacia_best_iteration, g.sacia_best_error) == (s.sacia_best_iteration, s.sacia_best_error)
