"""ope_pose_tracker_step_batch: many trackers advanced by one frame per call must leave exactly what the serial loop of
ope_pose_estimate_final_device leaves — results, tracker state, the replaced source clouds and the libc rand() position."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

libc = ctypes.CDLL(None)
ROT_TOL = 1e-4    # rad (the contract bar against the oracle)
TRANS_TOL = 1e-5  # m
FIT_TOL = 1e-5


@pytest.fixture(scope="module")
def sequences(synth, model):
    return [[f[0] for f in synth.make_sequence(model, 40 + s, 4)] for s in range(10)]


def _play(ctx, cuda_lib, specs, schedule, batch, seed=11, tables=None):
    """specs: (model, params) per tracker; schedule: per step a list of (tracker, target). Returns per step the (result, status,
    downloaded source) of every entry, and libc rand() after the last step."""
    libc.srand(seed)
    trackers = [cuda_lib.PoseTracker(ctx, prm) for _, prm in specs]
    sources = [ctx.upload(m) for m, _ in specs]
    out = []
    for k, step in enumerate(schedule):
        if batch:
            res, st = ctx.pose_track_batch([trackers[i] for i, _ in step], [sources[i] for i, _ in step], [t for _, t in step],
                                           tables=None if tables is None else tables(k, [sources[i] for i, _ in step]))
        else:
            res, st = [], []
            for i, t in step:
                tg = ctx.upload(t) if len(t) else None
                try:
                    res.append(trackers[i].estimate_final_device(sources[i], tg))
                    st.append(0)
                except cuda_lib.OpeError as e:
                    res.append(None)
                    st.append(int(str(e).split("rc=")[1].split(" ")[0]))
                if tg is not None:
                    tg.free()
        out.append([(r, int(s), sources[i].download()) for r, s, (i, _) in zip(res, st, step)])
    after = libc.rand()
    for t in trackers:
        t.close()
    for s in sources:
        s.free()
    return out, after


def _compare(synth, T, got, ref):
    exact = total = 0
    for k, (gs, rs) in enumerate(zip(got, ref)):
        for j, ((g, gst, gsrc), (r, rst, rsrc)) in enumerate(zip(gs, rs)):
            assert gst == rst, (k, j, gst, rst)
            assert gsrc.shape == rsrc.shape, (k, j)
            if len(rsrc):
                assert np.nanmax(np.abs(gsrc.astype(np.float64) - rsrc)) <= 1e-6, (k, j)
            if rst != 0:
                continue
            for f in ("final_pose", "coarse_pose", "fine_pose", "rigid_model_pose"):
                rot, tr = synth.pose_error(T.mat4(getattr(g, f)), T.mat4(getattr(r, f)))
                assert rot < 1e-6 and tr < 1e-6, (k, j, f, rot, tr)
            for f in ("ran_coarse", "icp_iterations", "icp_state", "icp_converged", "sacia_best_iteration", "n_src_coarse", "n_tgt_coarse",
                      "n_src_fine", "n_tgt_fine"):
                assert getattr(g, f) == getattr(r, f), (k, j, f, getattr(g, f), getattr(r, f))
            assert abs(g.fitness - r.fitness) < 1e-9, (k, j)
            total += 1
            exact += int(bytes(g) == bytes(r) and np.array_equal(gsrc.view(np.uint32), rsrc.view(np.uint32)))
    return exact, total


def _schedule(seqs, n_steps):
    return [[(i, s[k]) for i, s in enumerate(seqs)] for k in range(n_steps)]


def test_step_batch_equals_the_serial_loop(ctx, synth, cuda_lib, model, sequences, monkeypatch):
    specs = [(model, None)] * len(sequences)
    sched = _schedule(sequences, 4)
    batch, rb = _play(ctx, cuda_lib, specs, sched, True)
    monkeypatch.setenv("OPE_ICP_SMALL", "1")
    serial, rs = _play(ctx, cuda_lib, specs, sched, False)
    exact, total = _compare(synth, cuda_lib.T, batch, serial)
    print("bit-identical results and sources: %d of %d" % (exact, total))
    assert rb == rs
    assert sum(r.ran_coarse for r, _, _ in batch[0]) == len(sequences)


def test_mixed_states_and_models_in_one_call(ctx, synth, cuda_lib, model, sequences, monkeypatch):
    """coarse_refit_threshold = 1: trackers track after their first frame; fresh trackers join at step 2, a second model for some."""
    other = synth.make_model(seed=1)
    prm = cuda_lib.pose_params(coarse_refit_threshold=1.0)
    specs = [(model if i % 3 else other, prm) for i in range(8)]
    tg_other = [[f[0] for f in synth.make_sequence(other, 70 + s, 4)] for s in range(3)]
    targets = [tg_other[i // 3] if i % 3 == 0 else sequences[i] for i in range(8)]
    sched = [[(i, targets[i][k]) for i in range(8) if i < 5 or k >= 2] for k in range(4)]
    batch, rb = _play(ctx, cuda_lib, specs, sched, True)
    monkeypatch.setenv("OPE_ICP_SMALL", "1")
    serial, rs = _play(ctx, cuda_lib, specs, sched, False)
    _compare(synth, cuda_lib.T, batch, serial)
    assert rb == rs
    kinds = {(r.ran_coarse, k) for k, step in enumerate(batch) for r, st, _ in step if st == 0}
    assert (0, 2) in kinds and (1, 2) in kinds      # tracking and first calls in the same call


def test_edge_frames_in_the_same_call(ctx, synth, cuda_lib, model, sequences, monkeypatch):
    s = sequences
    empty = np.zeros((0, 3), np.float32)
    specs = [(model, None)] * 5 + [(model, cuda_lib.pose_params(min_target_points=99))]
    sched = [[(0, s[0][0]), (1, s[1][0]), (2, s[2][0]), (3, empty), (4, s[4][0]), (5, s[5][0])],
             [(0, empty), (1, s[1][1][:60].copy()), (2, s[2][1][::40].copy()), (3, s[3][1]), (4, s[4][1]), (5, s[5][1])],
             [(0, s[0][2]), (1, s[1][2]), (2, s[2][2]), (3, s[3][2]), (4, s[4][2]), (5, s[5][2])]]
    batch, rb = _play(ctx, cuda_lib, specs, sched, True)
    monkeypatch.setenv("OPE_ICP_SMALL", "1")
    serial, rs = _play(ctx, cuda_lib, specs, sched, False)
    _compare(synth, cuda_lib.T, batch, serial)
    assert rb == rs


def test_explicit_tables_equal_drawn_ones(ctx, synth, cuda_lib, model, sequences):
    """Tables drawn with sacia_draw on every tracker's 1 cm source sample, in tracker order (every tracker re-runs SAC-IA here)."""
    T = cuda_lib.T
    seqs = sequences[:4]
    specs = [(model, None)] * len(seqs)
    sched = _schedule(seqs, 1)
    msd = cuda_lib.pose_params().sacia.min_sample_distance
    keep = []

    def tables(k, sources):
        out = []
        for src in sources:
            sp = ctx.uniform_sample_cloud(src, 0.01)
            s, p = cuda_lib.sacia_draw(sp.download(), 400, 5, 5, msd)
            sp.free()
            keep.append((s, p))
            out.append(cuda_lib.rng_table(s, p))
        return out

    drawn, _ = _play(ctx, cuda_lib, specs, sched, True, seed=5)
    given, _ = _play(ctx, cuda_lib, specs, sched, True, seed=5, tables=tables)
    _compare(synth, T, given, drawn)


def test_lanes_and_chunks_do_not_change_results(ctx, synth, cuda_lib, model, sequences, monkeypatch):
    specs = [(model, None)] * len(sequences)
    sched = _schedule(sequences, 2)
    runs = []
    for lanes, chunk in (("1", None), ("4", None), ("4", "3")):
        monkeypatch.setenv("OPE_BATCH_LANES", lanes)
        if chunk:
            monkeypatch.setenv("OPE_BATCH_CHUNK", chunk)
        runs.append(_play(ctx, cuda_lib, specs, sched, True))
    for out, after in runs[1:]:
        assert after == runs[0][1]
        exact, total = _compare(synth, cuda_lib.T, out, runs[0][0])
        assert exact == total


def test_two_sequences_against_the_oracle(ctx, orc, synth, cuda_lib, model, sequences):
    specs = [(model, None)] * 2
    sched = _schedule(sequences[:2], 3)
    batch, _ = _play(ctx, cuda_lib, specs, sched, True, seed=3)
    orc.srand(3)
    ests = [orc.PoseEstimator() for _ in range(2)]
    srcs = [model.copy() for _ in range(2)]
    for k, step in enumerate(sched):
        for j, (i, t) in enumerate(step):
            o = ests[i].estimate_final(srcs[i], t)
            g = batch[k][j][0]
            rot, tr = synth.pose_error(cuda_lib.T.mat4(g.final_pose), np.array(o.final_pose, np.float64).reshape(4, 4).T)
            assert rot < ROT_TOL and tr < TRANS_TOL, (k, i, rot, tr)
            assert abs(g.fitness - o.fitness) < FIT_TOL
            assert (g.icp_iterations, g.icp_state) == (o.icp_iterations, o.icp_state)


def test_argument_checks_change_nothing(ctx, cuda_lib, model, sequences):
    L = cuda_lib.lib()
    a, b = cuda_lib.PoseTracker(ctx), cuda_lib.PoseTracker(ctx)
    sa, sb = ctx.upload(model), ctx.upload(model)
    other = cuda_lib.Context()
    so = other.upload(model[:1000])
    arr, keep = ctx._frame_inputs([sequences[0][0], sequences[1][0]])
    res = (cuda_lib.T.PoseResult * 2)()
    st = (ctypes.c_int32 * 2)()

    def call(ts, ss):
        th = (ctypes.c_void_p * 2)(*[t.h for t in ts])
        sh = (ctypes.c_void_p * 2)(*[s.h for s in ss])
        rc = L.ope_pose_tracker_step_batch(ctx.h, th, sh, arr, ctypes.c_size_t(2), None, res, st)
        assert [sh[0], sh[1]] == [ss[0].h.value, ss[1].h.value]
        return rc

    assert call([a, a], [sa, sb]) == cuda_lib.T.OPE_ERR_INVALID
    assert call([a, b], [sa, sa]) == cuda_lib.T.OPE_ERR_INVALID
    assert call([a, b], [sa, so]) == cuda_lib.T.OPE_ERR_INVALID
    assert len(sa) == len(model) and len(sb) == len(model)
    assert L.ope_pose_tracker_step_batch(ctx.h, None, None, None, ctypes.c_size_t(0), None, None, None) == 0
    # nothing changed: both trackers still run their first call (cloudModel = the source, SAC-IA)
    r, st2 = ctx.pose_track_batch([a, b], [sa, sb], [sequences[0][0], sequences[1][0]])
    assert (st2 == 0).all() and all(x.ran_coarse == 1 for x in r)
    so.free(); other.close()
