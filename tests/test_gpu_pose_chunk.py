"""ope_pose_batch and ope_pose_tracker_step_batch run their fast-path frames through the same chunk of frame-spanning stages: a
fresh tracker's first step is ope_pose_batch's frame, and both read the decision tables by the single call's rule."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

H, S, K = 400, 5, 5


@pytest.fixture(scope="module")
def frames(synth, model):
    fs = [synth.make_frame(model, 900 + f)[0] for f in range(4)]
    # four copies of a cluster side by side: more 8 mm voxels than a fast-path sample holds, so the frame takes the per-frame path
    big = np.concatenate([fs[0] + np.array([dx, dy, 0], np.float32) for dx in (0, 0.4) for dy in (0, 0.4)])
    return fs + [big]


@pytest.fixture(scope="module")
def tables(ctx, cuda_lib, model, frames):
    """Explicit decision tables drawn on the model's 1 cm sample, one per frame."""
    cl = ctx.upload(model)
    sp = ctx.uniform_sample_cloud(cl, 0.01)
    xyz = sp.download()
    sp.free(); cl.free()
    msd = cuda_lib.pose_params().sacia.min_sample_distance
    return [cuda_lib.sacia_draw(xyz, H, S, K, msd) for _ in frames]


def _rows(cuda_lib, tables, n):
    """The tables cut or extended (by repeating their first row) to n hypotheses."""
    out = []
    for s, p in tables:
        reps = max(0, n - len(s))
        out.append(cuda_lib.rng_table(np.concatenate([s[:n], s[:1].repeat(reps, 0)]), np.concatenate([p[:n], p[:1].repeat(reps, 0)])))
    return out


def _first_steps(ctx, cuda_lib, model, frames, tables):
    trackers = [cuda_lib.PoseTracker(ctx) for _ in frames]
    sources = [ctx.upload(model) for _ in frames]
    try:
        return ctx.pose_track_batch(trackers, sources, frames, tables=tables)
    finally:
        for t in trackers:
            t.close()
        for s in sources:
            s.free()


def test_pose_batch_equals_the_first_tracker_step(ctx, synth, cuda_lib, model, frames, tables):
    T = cuda_lib.T
    tb = _rows(cuda_lib, tables, H)
    got, st = ctx.pose_batch(model, frames, tables=tb)
    ref, rst = _first_steps(ctx, cuda_lib, model, frames, tb)
    assert (st == 0).all() and (rst == 0).all()
    assert all(r.ran_coarse == 1 for r in got)
    for f in range(len(frames) - 1):   # the fast path: the same chunk, bit for bit
        assert bytes(got[f]) == bytes(ref[f]), f
    # the frame outside the envelope: ope_pose_batch's per-frame path and the tracker step's serial loop run different ICP kernels
    g, r = got[-1], ref[-1]
    assert g.n_tgt_coarse > 2048 and g.n_tgt_fine > 0
    for name in ("final_pose", "coarse_pose", "fine_pose", "rigid_model_pose"):
        rot, tr = synth.pose_error(T.mat4(getattr(g, name)), T.mat4(getattr(r, name)))
        assert rot < 1e-6 and tr < 1e-6, (name, rot, tr)
    for name in ("ran_coarse", "icp_iterations", "icp_state", "icp_converged", "sacia_best_iteration", "n_src_coarse", "n_tgt_coarse",
                 "n_src_fine", "n_tgt_fine"):
        assert getattr(g, name) == getattr(r, name), (name, getattr(g, name), getattr(r, name))
    assert abs(g.fitness - r.fitness) < 1e-9


def test_pose_batch_reads_the_first_h_hypotheses_of_a_longer_table(ctx, cuda_lib, model, frames, tables):
    picked = [frames[0], frames[-1]]   # one frame on the fast path, one on the per-frame path
    exact, st = ctx.pose_batch(model, picked, tables=_rows(cuda_lib, tables[:2], H))
    longer, st2 = ctx.pose_batch(model, picked, tables=_rows(cuda_lib, tables[:2], H + 1))
    assert (st == 0).all() and (st2 == 0).all()
    for f in range(2):
        assert bytes(exact[f]) == bytes(longer[f]), f


def test_a_short_table_is_invalid_in_both_apis(ctx, cuda_lib, model, frames, tables):
    short = _rows(cuda_lib, tables[:2], H - 1)
    with pytest.raises(cuda_lib.OpeError) as e:
        ctx.pose_batch(model, frames[:2], tables=short)
    assert e.value.rc == cuda_lib.T.OPE_ERR_INVALID
    with pytest.raises(cuda_lib.OpeError) as e:
        _first_steps(ctx, cuda_lib, model, frames[:2], short)
    assert e.value.rc == cuda_lib.T.OPE_ERR_INVALID
