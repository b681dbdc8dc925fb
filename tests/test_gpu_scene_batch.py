"""Depth images -> segmented scenes -> poses, many frames per call (ope_scene_batch_create / ope_scene_pose_batch): every frame's
result equals the single-frame chain ope_depth_to_cloud -> ope_pass_through -> ope_segment_objects_on_plane bit for bit, whatever
the frame's position in the batch or the chunking; the join equals ope_pose_batch on the host-cut clusters."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

LIMITS = (-0.5, 0.5, -0.5, 0.3, 0.5, 1.6)      # ObjectSegmentationPlane::getFiltered, D&L/src/objectsegmentationplane.cpp:17-18
FRAMES = (21, 22, 23, 24, 25, 26, 27, 28)


def _depth_mm(cloud):
    return np.rint(np.nan_to_num(cloud[..., 2], nan=0.0).astype(np.float64) * 1000.0).astype(np.uint16)


@pytest.fixture(scope="module")
def depths(synth, model):
    return {f: _depth_mm(synth.make_frame(model, f)[1]) for f in FRAMES}


def _single(ctx, d, **cam):
    """the single-frame chain: (n_points, xyz, labels, n_clusters, plane1, plane2, iterations)"""
    c = ctx.depth_to_cloud(d, **cam)
    filt = ctx.pass_through(c, LIMITS)
    xyz = filt.download()
    labels, k, p1, p2, it = ctx.segment_objects_on_plane(filt)
    return len(c), xyz, labels, k, p1, p2, tuple(it)


def _batch_frames(sb):
    out = []
    for f in range(len(sb)):
        xyz, labels = sb.frame(f)
        i = sb.info[f]
        out.append((i.n_points, xyz, labels, i.n_clusters, np.array(list(i.plane1), np.float32), np.array(list(i.plane2), np.float32),
                    (i.iterations[0], i.iterations[1])))
    return out


def _same(a, b):
    return (a[0] == b[0] and np.array_equal(a[1].view(np.uint32), b[1].view(np.uint32)) and np.array_equal(a[2], b[2]) and a[3] == b[3]
            and np.array_equal(a[4].view(np.uint32), b[4].view(np.uint32)) and np.array_equal(a[5].view(np.uint32), b[5].view(np.uint32))
            and a[6] == b[6])


def test_scene_batch_equals_the_single_frame_chain(ctx, depths):
    stack = np.stack([depths[f] for f in FRAMES])
    sb = ctx.scene_batch(stack)
    assert (sb.status == 0).all()
    got = _batch_frames(sb)
    for f, g in zip(FRAMES, got):
        s = _single(ctx, depths[f])
        assert sb.info[FRAMES.index(f)].n_cropped == len(s[1])
        assert _same(g, s), f
    assert all(g[3] >= 1 for g in got[:3])
    sb.close()


def test_scene_batch_equals_the_oracle(ctx, orc, depths):
    """the frames of test_plane_ransac_prism_and_object_clusters, from the depth image on: the oracle's rgbd2Pcl, PassThrough z, y, x
    and getSegmentedObjectsOnPlane"""
    frames = (21, 22, 23)
    sb = ctx.scene_batch(np.stack([depths[f] for f in frames]))
    for i, f in enumerate(frames):
        pts = orc.depth_to_cloud(depths[f])
        keep = np.arange(len(pts), dtype=np.int32)
        for field, lo, hi in ((2, LIMITS[4], LIMITS[5]), (1, LIMITS[2], LIMITS[3]), (0, LIMITS[0], LIMITS[1])):
            keep = keep[orc.pass_through(pts[keep], field, lo, hi)]
        sub = pts[keep]
        ol, ok, op1, op2, oit = orc.segment_objects_on_plane(sub)
        xyz, labels = sb.frame(i)
        info = sb.info[i]
        assert info.n_points == len(pts) and np.array_equal(xyz, sub)
        assert np.array_equal(labels, ol) and info.n_clusters == ok
        assert np.array_equal(np.array(list(info.plane1), np.float32), op1) and np.array_equal(np.array(list(info.plane2), np.float32), op2)
        assert (info.iterations[0], info.iterations[1]) == tuple(oit)
    sb.close()


def test_frame_index_does_not_leak(ctx, depths, monkeypatch):
    import torch
    stack = np.stack([depths[f] for f in FRAMES])
    one_call = ctx.scene_batch(stack)
    ref = _batch_frames(one_call)
    one_call.close()
    for i, f in enumerate(FRAMES):                                   # one frame per call
        sb = ctx.scene_batch(depths[f][None])
        assert _same(_batch_frames(sb)[0], ref[i]), f
        sb.close()
    sb = ctx.scene_batch(stack[::-1].copy())                          # reverse order
    for i, g in enumerate(_batch_frames(sb)[::-1]):
        assert _same(g, ref[i]), FRAMES[i]
    sb.close()
    monkeypatch.setenv("OPE_SCENE_CHUNK", "3")                        # 8 frames: chunks of 3, 3 and 2
    sb = ctx.scene_batch(stack)
    assert all(_same(g, r) for g, r in zip(_batch_frames(sb), ref))
    sb.close()
    monkeypatch.delenv("OPE_SCENE_CHUNK")
    dev = torch.from_numpy(stack.astype(np.int16)).cuda().contiguous()   # device-resident depth (uint16 bits)
    sb = ctx.scene_batch(dev)
    assert all(_same(g, r) for g, r in zip(_batch_frames(sb), ref))
    sb.close()


def _empty_table(synth, model):
    """a table with nothing on it: the object far outside the view, the wall beyond the crop, no noise"""
    pose = np.eye(4)
    pose[:3, 3] = (5.0, 0.1, 1.0)
    cloud, _ = synth.render_scene(model, pose, np.random.default_rng(0), wall_z=1.9, noise=False)
    return _depth_mm(cloud)


def test_edge_frames_in_a_mixed_batch(ctx, synth, cuda_lib, model, depths):
    zero = np.zeros((480, 640), np.uint16)
    two = np.zeros((480, 640), np.uint16)
    two[240, 320] = two[241, 320] = 1000                              # two points inside the crop: no plane
    table = _empty_table(synth, model)
    imgs = [zero, depths[21], two, table, depths[22]]
    sb = ctx.scene_batch(np.stack(imgs))
    assert (sb.status == 0).all()
    got = _batch_frames(sb)
    for img, g in zip(imgs, got):
        assert _same(g, _single(ctx, img))
    assert got[0][0] == 0 and got[0][3] == -1
    assert sb.info[2].n_cropped == 2 and got[2][3] == -1
    assert got[3][3] == 0 and sb.info[3].n_cropped > 1000
    res, st = sb.pose(model, workers=4)
    assert (st == 0).all()
    T = cuda_lib.T
    for f in (0, 3):                                                   # empty targets: identity, as ope_pose_batch
        r, t = synth.pose_error(T.mat4(res[f].final_pose), np.eye(4))
        assert r < 1e-5 and t < 1e-5, (f, r, t)
    sb.close()
    # 320 x 240 with other intrinsics: nothing assumes 640 x 480
    cam = dict(fx=262.5, fy=262.5, cx=119.5, cy=159.5, scale=1000.0, z_max=2.0)
    small = [depths[f][::2, ::2].copy() for f in (23, 24, 25)]
    sb = ctx.scene_batch(np.stack(small), **cam)
    assert (sb.status == 0).all()
    for img, g in zip(small, _batch_frames(sb)):
        assert _same(g, _single(ctx, img, **cam))
    sb.close()


def _cut(sb, f, rank):
    xyz, labels = sb.frame(f)
    i = sb.info[f]
    if sb.status[f] != 0:
        return np.zeros((0, 3), np.float32)
    if i.n_clusters < 0:
        return xyz
    return xyz[labels == rank] if rank < i.n_clusters else np.zeros((0, 3), np.float32)


def _check_pose_equal(synth, T, got, want):
    for f, (g, s) in enumerate(zip(got, want)):
        r, t = synth.pose_error(T.mat4(g.final_pose), T.mat4(s.final_pose))
        assert r < 1e-6 and t < 1e-6, (f, r, t)
        assert (g.icp_iterations, g.icp_state, g.icp_converged, g.sacia_best_iteration) == \
               (s.icp_iterations, s.icp_state, s.icp_converged, s.sacia_best_iteration), f
        assert abs(g.fitness - s.fitness) < 1e-9, f


def test_scene_pose_batch_equals_pose_batch_on_the_host_cut_clusters(ctx, orc, synth, cuda_lib, model, depths):
    T = cuda_lib.T
    libc = ctypes.CDLL(None)
    frames = [depths[f] for f in FRAMES[:6]] + [np.zeros((480, 640), np.uint16)]
    sb = ctx.scene_batch(np.stack(frames))
    n = len(frames)
    k = [sb.info[f].n_clusters for f in range(n)]
    multi = [f for f in range(n) if k[f] >= 2]
    assert multi, k
    ranks = np.zeros(n, np.int32)
    ranks[multi[0]] = 1                                                # the second-largest cluster
    ranks[2 if multi[0] != 2 else 3] = max(k) + 5                      # beyond the last cluster: an empty target
    for cluster in (None, ranks):
        cut = [_cut(sb, f, 0 if cluster is None else int(cluster[f])) for f in range(n)]
        libc.srand(7)
        got, st = sb.pose(model, cluster=cluster, workers=4)
        libc.srand(7)
        want, st2 = ctx.pose_batch(model, cut, workers=4)
        assert (st == 0).all() and (st2 == 0).all()
        _check_pose_equal(synth, T, got, want)
    # pre-drawn tables (ope_sacia_draw) instead of libc rand()
    sp = model[orc.uniform_sample(model, 0.01)]
    tables = []
    for f in range(n):
        orc.srand(100 + f)
        tables.append(cuda_lib.rng_table(*orc.sacia_draw(sp, 400, 5, 5, 0.01)))
    cut = [_cut(sb, f, 0) for f in range(n)]
    got, _ = sb.pose(model, tables=tables, workers=4)
    want, _ = ctx.pose_batch(model, cut, tables=tables, workers=4)
    _check_pose_equal(synth, T, got, want)
    # the oracle's estimateFinalPose on the first two frames' largest clusters, drawing from the same rand() stream
    libc.srand(7)
    got, _ = sb.pose(model, workers=4)
    orc.srand(7)
    for f in range(2):
        o = orc.PoseEstimator().estimate_final(model.copy(), cut[f])
        r, t = synth.pose_error(T.mat4(got[f].final_pose), np.array(o.final_pose, np.float64).reshape(4, 4).T)
        assert r < 1e-4 and t < 1e-5, (f, r, t)
    sb.close()


def localize(scene, model, fitness_max=1e-4, strength_min=0.4):
    """INTEGRATION.md's caller-side selection: every frame tries its clusters in size order and keeps the first one whose pose is
    accepted (rosinterface.cpp:243-327: fitness < 1e-4 or align strength > 0.4). Returns (rank per frame or -1, poses, tries)."""
    n = len(scene)
    done = 1 << 30                                                      # a rank past every frame's clusters: an empty target
    rank = np.zeros(n, np.int32)
    chosen = np.full(n, -1)
    poses = [None] * n
    tries = [[] for _ in range(n)]
    for f in range(n):
        if scene.status[f] != 0 or scene.info[f].n_clusters <= 0:
            rank[f] = done
    while (rank != done).any():
        res, _ = scene.pose(model, cluster=rank)
        for f in np.nonzero(rank != done)[0]:
            ok = res[f].fitness < fitness_max or res[f].align_strength > strength_min
            tries[f].append((int(rank[f]), bool(ok)))
            if ok:
                chosen[f], poses[f], rank[f] = rank[f], res[f], done
            elif rank[f] + 1 < scene.info[f].n_clusters:
                rank[f] += 1
            else:
                rank[f] = done
    return chosen, poses, tries


def test_caller_side_cluster_selection(ctx, model, depths):
    sb = ctx.scene_batch(np.stack([depths[f] for f in FRAMES]))
    chosen, poses, tries = localize(sb, model)
    for f in range(len(FRAMES)):
        ranks = [r for r, _ in tries[f]]
        assert ranks == list(range(len(ranks)))                         # size order, no cluster skipped
        accepted = [r for r, ok in tries[f] if ok]
        assert chosen[f] == (accepted[0] if accepted else -1)
        assert len(accepted) <= 1 and (not accepted or ranks[-1] == accepted[0])   # the search stops at the first accepted cluster
        if chosen[f] < 0:
            assert len(ranks) == max(sb.info[f].n_clusters, 0)
    sb.close()
