"""ope_scene_track_step: the node's cluster choice and the tracker step in one call must equal its definition, a serial loop of
public calls (SceneBatch.frame, the float32 gate, Context.pose_track_batch once per round, fresh PoseTrackers for the tries), bit for
bit and with the same libc rand() consumption; the centroids equal compute3DCentroid's serial float sums."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

libc = ctypes.CDLL(None)
GATE = np.float32(0.05)


def _centroid(pts):
    """compute3DCentroid: serial float32 sums over the finite points, then / n"""
    p = pts[np.isfinite(pts).all(1)]
    return np.array([np.cumsum(p[:, a], dtype=np.float32)[-1] / np.float32(len(p)) for a in range(3)], np.float32)


def _gate_distance(c, m):
    dx, dy, dz = (np.float32(c[a]) - np.float32(m[a]) for a in range(3))
    return np.float32(np.sqrt(np.float32((dx * dx + dy * dy) + dz * dz)))


def _two_points():
    d = np.zeros((480, 640), np.uint16)
    d[240, 320] = d[241, 320] = 1000              # two points inside the crop: no plane, the whole cloud is handed on
    return d


@pytest.fixture(scope="module")
def seqs(synth, model):
    """8 cameras x 4 frames: camera 0 sees the object alone (rank 0), the others next to a larger cylinder (rank 0) and a box;
    camera 2's object jumps 12 cm at frame 2; camera 3 sees an empty table (no cluster)"""
    out = []
    for c in range(8):
        if c == 3:
            pose = np.eye(4)
            pose[:3, 3] = (5.0, 0.1, 1.0)                                  # the object far outside the view, the wall beyond the crop
            cloud, _ = synth.render_scene(model, pose, np.random.default_rng(0), wall_z=1.9, noise=False)
            table = np.rint(np.nan_to_num(cloud[..., 2], nan=0.0).astype(np.float64) * 1000.0).astype(np.uint16)
            out.append(np.stack([table] * 4))
        else:
            d, _ = synth.make_scene_sequence(model, 100 + c, 4, distractors=0 if c == 0 else 2, jump_at=2 if c == 2 else None)
            out.append(d)
    return out


def _scenes(ctx, seqs, k):
    return ctx.scene_batch(np.stack([s[k] for s in seqs]))


# ---- 1. centroids ----------------------------------------------------------------------------------------------------------------
def test_centroids_equal_the_serial_float_sums(ctx, synth, model, seqs):
    others = [np.rint(np.nan_to_num(synth.make_frame(model, f)[1][..., 2], nan=0.0).astype(np.float64) * 1000.0).astype(np.uint16)
              for f in (21, 22, 23)]
    imgs = others + [s[0] for s in seqs[:3]] + [_two_points()]
    sb = ctx.scene_batch(np.stack(imgs))
    seen_whole = 0
    for f in range(len(imgs)):
        xyz, labels = sb.frame(f)
        k = sb.info[f].n_clusters
        got = sb.centroids(f)
        if k < 0:
            want = [_centroid(xyz)]
            seen_whole += 1
        else:
            want = [_centroid(xyz[labels == r]) for r in range(k)]
        assert len(got) == len(want), f
        for g, w in zip(got, want):
            assert np.array_equal(g.view(np.uint32), w.view(np.uint32)), (f, g, w)
    assert seen_whole == 1
    sb.close()
    src = ctx.upload(model)
    c, n = ctx.centroid(src)
    assert n == len(model) and np.array_equal(c.view(np.uint32), _centroid(model).view(np.uint32))
    with_nan = model[:5000].copy()
    with_nan[::7, 1] = np.nan
    c, n = ctx.centroid(ctx.upload(with_nan))
    assert n == len(with_nan) - len(with_nan[::7]) and np.array_equal(c.view(np.uint32), _centroid(with_nan).view(np.uint32))


# ---- the definition: a serial loop of public calls -----------------------------------------------------------------------------
class Camera:
    def __init__(self, ctx, cuda_lib, model, prm=None):
        self.tracker = cuda_lib.PoseTracker(ctx, prm)
        self.source = ctx.upload(model)
        self.found = False                    # the tracker completed a step (firstTimePose != 0)
        self.prm = prm


def reference_track(ctx, cuda_lib, sb, cams, model, accept_fitness, accept_strength, max_tries=0, reacquire=1, log=None):
    """what ope_scene_track_step is defined to do, with public calls only. Returns (results, choices as tuples, status)."""
    T = cuda_lib.T
    n = len(sb)
    frames = [sb.frame(f) for f in range(n)]

    def cut(f, r):
        xyz, labels = frames[f]
        return xyz if sb.info[f].n_clusters < 0 else np.ascontiguousarray(xyz[labels == r])

    res = [bytes(ctypes.sizeof(T.PoseResult))] * n
    choice = [[T.TRACK_NOT_FOUND, -1, 0, np.float32(np.nan)] for _ in range(n)]
    status = [0] * n
    chosen, search = {}, {}
    for i in range(n):
        if sb.status[i] != 0:
            choice[i][0], status[i] = T.TRACK_NO_SCENE, int(sb.status[i])
            continue
        K = 1 if sb.info[i].n_clusters < 0 else sb.info[i].n_clusters
        reacq = False
        if cams[i].found:
            m = _centroid(cams[i].source.download())
            ds = [_gate_distance(_centroid(cut(i, k)), m) for k in range(K)]
            if log is not None:
                log.extend(ds)
            inside = [k for k in range(K) if ds[k] < GATE]
            if inside:
                chosen[i] = inside[0]
                choice[i] = [T.TRACK_TRACKED, inside[0], 0, ds[inside[0]]]
                continue
            choice[i][3] = min(ds) if ds else np.float32(np.nan)
            if not reacquire:
                choice[i][0] = T.TRACK_LOST
                continue
            reacq = True
        limit = min(K, max_tries) if max_tries > 0 else K
        if limit > 0:
            search[i] = (limit, reacq)
    r = 0
    while True:
        entries = []
        for i in range(n):
            if r == 0 and i in chosen:
                entries.append((i, None, cams[i].tracker, cams[i].source, cut(i, chosen[i])))
            elif i in search:
                entries.append((i, r, cuda_lib.PoseTracker(ctx, cams[i].prm), ctx.upload(model), cut(i, r)))
        if not entries:
            break
        out, st = ctx.pose_track_batch([e[2] for e in entries], [e[3] for e in entries], [e[4] for e in entries])
        for (i, rank, t, s, _), o, c in zip(entries, out, st):
            res[i], status[i] = bytes(o), int(c)
            if rank is None:
                cams[i].source = s
                continue
            choice[i][2] += 1
            limit, reacq = search[i]
            if c == 0 and (o.fitness < accept_fitness or o.align_strength > accept_strength):
                cams[i].tracker.close()
                cams[i].source.free()
                cams[i].tracker, cams[i].source, cams[i].found = t, s, True
                choice[i][0], choice[i][1] = (T.TRACK_REACQUIRED if reacq else T.TRACK_ACQUIRED), rank
                del search[i]
                continue
            t.close()
            s.free()
            if rank + 1 >= limit:
                del search[i]
        r += 1
    for i in chosen:
        cams[i].found = True
    return res, [tuple(c) for c in choice], status


def _choice_tuple(c):
    return (c.mode, c.cluster, c.tries, np.float32(c.gate_distance))


def _same_choice(a, b):
    return a[:3] == b[:3] and np.array_equal(np.float32(a[3]).view(np.uint32), np.float32(b[3]).view(np.uint32))


def _play_library(ctx, cuda_lib, model, seqs, steps, seed, **tp):
    libc.srand(seed)
    trackers = [cuda_lib.PoseTracker(ctx) for _ in seqs]
    sources = [ctx.upload(model) for _ in seqs]
    out = []
    for k in steps:
        sb = _scenes(ctx, seqs, k)
        res, ch, st = sb.track(trackers, sources, **tp)
        out.append(([bytes(r) for r in res], [_choice_tuple(c) for c in ch], [int(x) for x in st], [s.download() for s in sources]))
        sb.close()
    after = libc.rand()
    for t in trackers:
        t.close()
    for s in sources:
        s.free()
    return out, after


def _play_reference(ctx, cuda_lib, model, seqs, steps, seed, log=None, **tp):
    libc.srand(seed)
    cams = [Camera(ctx, cuda_lib, model) for _ in seqs]
    out = []
    for k in steps:
        sb = _scenes(ctx, seqs, k)
        res, ch, st = reference_track(ctx, cuda_lib, sb, cams, model, log=log, **tp)
        out.append((res, ch, st, [c.source.download() for c in cams]))
        sb.close()
    after = libc.rand()
    for c in cams:
        c.tracker.close()
        c.source.free()
    return out, after


def _assert_same(got, want):
    for k, (g, w) in enumerate(zip(got, want)):
        assert g[2] == w[2], (k, g[2], w[2])
        for i in range(len(g[1])):
            assert _same_choice(g[1][i], w[1][i]), (k, i, g[1][i], w[1][i])
            assert g[0][i] == w[0][i], (k, i)
            assert g[3][i].shape == w[3][i].shape and np.array_equal(g[3][i].view(np.uint32), w[3][i].view(np.uint32)), (k, i)


@pytest.fixture(scope="module")
def acceptance(ctx, cuda_lib, model, seqs):
    """accept_fitness / accept_strength derived from a pass with acceptance switched off: every try of frames 0 and 2 is run (round 0
    with the seed the tests use, so camera 0's rank-0 result is the one they see), and accept_fitness is the threshold, among the
    midpoints of the recorded fitnesses, that accepts camera 0 at rank 0, rejects some camera's rank 0 but accepts a later rank,
    and accepts a try of camera 2 at its jump frame, with the widest margin to every recorded value; strength is switched off"""
    fits = {}
    for k in (0, 2):
        libc.srand(5)
        sb = _scenes(ctx, seqs, k)
        for r in range(6):
            idx = [i for i in range(len(seqs)) if r < max(sb.info[i].n_clusters, 0)]
            if not idx:
                break
            xyz = [sb.frame(i) for i in idx]
            ts = [cuda_lib.PoseTracker(ctx) for _ in idx]
            ss = [ctx.upload(model) for _ in idx]
            out, st = ctx.pose_track_batch(ts, ss, [x[l == r] for x, l in xyz])
            for i, o, c in zip(idx, out, st):
                if c == 0:
                    fits[(k, i, r)] = o.fitness
            for t in ts:
                t.close()
        sb.close()
    values = sorted(set(fits.values()))
    best = None
    for a, b in zip(values, values[1:]):
        thr = float(np.sqrt(a * b))
        ok0 = fits.get((0, 0, 0), np.inf) < thr
        later = any(fits[(0, c, 0)] > thr and any(f < thr for (k, i, r), f in fits.items() if k == 0 and i == c and r >= 1)
                    for c in range(1, len(seqs)) if (0, c, 0) in fits)
        jump = any(f < thr for (k, i, r), f in fits.items() if k == 2 and i == 2)
        if ok0 and later and jump and (best is None or b / a > best[0]):
            best = (b / a, thr)
    assert best is not None, sorted(fits.items())
    print("accept_fitness %.3g (margin x%.2f) from %d tries" % (best[1], best[0], len(fits)))
    return best[1], 1e9


# ---- 2. equality with the composition --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("reacquire,max_tries", [(1, 0), (0, 0), (1, 1)])
def test_track_step_equals_the_serial_loop(ctx, cuda_lib, model, seqs, acceptance, reacquire, max_tries):
    T = cuda_lib.T
    fit, strength = acceptance
    tp = dict(accept_fitness=fit, accept_strength=strength, reacquire=reacquire, max_tries=max_tries)
    got, ga = _play_library(ctx, cuda_lib, model, seqs, range(4), 5, **tp)
    log = []
    want, wa = _play_reference(ctx, cuda_lib, model, seqs, range(4), 5, log=log, **tp)
    _assert_same(got, want)
    assert ga == wa
    assert all(abs(float(d) - float(GATE)) >= 1e-5 for d in log)
    modes = [(k, i, c) for k, step in enumerate(got) for i, c in enumerate(step[1])]
    kinds = {c[0] for _, _, c in modes}
    assert T.TRACK_TRACKED in kinds and T.TRACK_NOT_FOUND in kinds
    assert got[0][1][0][:2] == (T.TRACK_ACQUIRED, 0)                              # the object alone: accepted at rank 0
    if max_tries == 0:
        assert any(c[0] == T.TRACK_ACQUIRED and c[1] >= 1 for c in got[0][1])     # the distractor first, then the object
        assert got[0][1][3][:3] == (T.TRACK_NOT_FOUND, -1, 0)                     # no cluster: no try
    if max_tries == 0 and reacquire:
        assert got[2][1][2][0] == T.TRACK_REACQUIRED                              # the jump
    if not reacquire:
        assert got[2][1][2][0] == T.TRACK_LOST and got[2][1][2][3] > GATE
    if max_tries == 1:                                                            # max_tries stopped searches with clusters left
        assert any(c[0] == T.TRACK_NOT_FOUND and c[2] == 1 for c in got[0][1][1:])


# ---- 3. lanes and chunks ---------------------------------------------------------------------------------------------------------
def test_lanes_and_chunks_do_not_change_results(ctx, cuda_lib, model, seqs, acceptance, monkeypatch):
    fit, strength = acceptance
    runs = []
    for lanes, chunk in (("1", None), ("4", None), ("4", "3")):
        monkeypatch.setenv("OPE_BATCH_LANES", lanes)
        if chunk:
            monkeypatch.setenv("OPE_BATCH_CHUNK", chunk)
        runs.append(_play_library(ctx, cuda_lib, model, seqs, range(3), 9, accept_fitness=fit, accept_strength=strength))
    for out, after in runs[1:]:
        assert after == runs[0][1]
        _assert_same(out, runs[0][0])


# ---- 4. oracle -------------------------------------------------------------------------------------------------------------------
def test_two_cameras_against_the_oracle(ctx, orc, synth, cuda_lib, model, seqs, acceptance):
    LIMITS = (-0.5, 0.5, -0.5, 0.3, 0.5, 1.6)
    T = cuda_lib.T
    fit, strength = acceptance
    cam_seqs = [seqs[1], seqs[2]]
    got, _ = _play_library(ctx, cuda_lib, model, cam_seqs, range(3), 3, accept_fitness=fit, accept_strength=strength)
    orc.srand(3)
    est = [None, None]
    src = [model.copy(), model.copy()]
    for k in range(3):
        clusters = []
        for c in range(2):
            pts = orc.depth_to_cloud(cam_seqs[c][k])
            keep = np.arange(len(pts), dtype=np.int32)
            for field, lo, hi in ((2, LIMITS[4], LIMITS[5]), (1, LIMITS[2], LIMITS[3]), (0, LIMITS[0], LIMITS[1])):
                keep = keep[orc.pass_through(pts[keep], field, lo, hi)]
            sub = pts[keep]
            labels, K, _, _, _ = orc.segment_objects_on_plane(sub)
            clusters.append([sub] if K < 0 else [np.ascontiguousarray(sub[labels == r]) for r in range(K)])
        # round 0: tracking steps and rank-0 tries in camera order, then the rank-r tries
        plan = {}
        for c in range(2):
            if est[c] is not None:
                m = _centroid(src[c])
                inside = [r for r, cl in enumerate(clusters[c]) if _gate_distance(_centroid(cl), m) < GATE]
                plan[c] = ("track", inside[0]) if inside else ("search", None)
            else:
                plan[c] = ("search", None)
        outcome = {}
        r = 0
        while True:
            todo = [c for c in range(2) if (r == 0 and plan[c][0] == "track") or (plan[c][0] == "search" and c not in outcome
                                                                                and r < len(clusters[c]))]
            if not todo:
                break
            for c in todo:
                if plan[c][0] == "track":
                    o = est[c].estimate_final(src[c], clusters[c][plan[c][1]])
                    outcome[c] = (plan[c][1], o)
                    continue
                e, s = orc.PoseEstimator(), model.copy()
                o = e.estimate_final(s, clusters[c][r])
                if o.fitness < fit or o.align_strength > strength:
                    est[c], src[c] = e, s
                    outcome[c] = (r, o)
            r += 1
        for c in range(2):
            g = cuda_lib.T.PoseResult.from_buffer_copy(got[k][0][c])
            ch = got[k][1][c]
            assert c in outcome, (k, c, ch)
            rank, o = outcome[c]
            assert ch[1] == rank and ch[0] in (T.TRACK_TRACKED, T.TRACK_ACQUIRED, T.TRACK_REACQUIRED), (k, c, ch, rank)
            rot, tr = synth.pose_error(T.mat4(g.final_pose), np.array(o.final_pose, np.float64).reshape(4, 4).T)
            assert rot < 1e-4 and tr < 1e-5, (k, c, rot, tr)
            assert abs(g.fitness - o.fitness) < 1e-5
            assert (g.icp_iterations, g.icp_state) == (o.icp_iterations, o.icp_state)


# ---- 5. argument checks ----------------------------------------------------------------------------------------------------------
def test_argument_checks_change_nothing(ctx, cuda_lib, model, seqs):
    L = cuda_lib.lib()
    T = cuda_lib.T
    two = [seqs[0], seqs[1]]
    sb = _scenes(ctx, two, 0)
    a, b = cuda_lib.PoseTracker(ctx), cuda_lib.PoseTracker(ctx)
    sa, sb_ = ctx.upload(model), ctx.upload(model)
    other = cuda_lib.Context()
    so = other.upload(model[:1000])
    res = (T.PoseResult * 3)()
    ch = (T.TrackChoice * 3)()
    st = (ctypes.c_int32 * 3)()

    def call(ts, ss, n=2):
        th = (ctypes.c_void_p * 3)(*[t.h for t in ts])
        sh = (ctypes.c_void_p * 3)(*[s.h for s in ss])
        rc = L.ope_scene_track_step(sb.h, None, th, sh, ctypes.c_size_t(n), res, ch, st)
        assert [sh[i] for i in range(len(ss))] == [s.h.value for s in ss]
        return rc

    assert call([a, a], [sa, sb_]) == T.OPE_ERR_INVALID
    assert call([a, b], [sa, sa]) == T.OPE_ERR_INVALID
    assert call([a, b], [sa, so]) == T.OPE_ERR_INVALID
    assert call([a, b, cuda_lib.PoseTracker(ctx)], [sa, sb_, ctx.upload(model)], n=3) == T.OPE_ERR_INVALID
    assert call([a], [sa], n=1) == T.OPE_ERR_INVALID
    assert len(sa) == len(model) and len(sb_) == len(model)
    libc.srand(21)
    r1, c1, s1 = sb.track([a, b], [sa, sb_])
    after = libc.rand()
    fresh = [cuda_lib.PoseTracker(ctx), cuda_lib.PoseTracker(ctx)]
    fs = [ctx.upload(model), ctx.upload(model)]
    libc.srand(21)
    r2, c2, s2 = sb.track(fresh, fs)
    assert libc.rand() == after
    assert [bytes(x) for x in r1] == [bytes(x) for x in r2] and list(s1) == list(s2)
    assert [_choice_tuple(x)[:3] for x in c1] == [_choice_tuple(x)[:3] for x in c2]
    assert np.array_equal(sa.download(), fs[0].download()) and np.array_equal(sb_.download(), fs[1].download())
    sb.close()
    so.free()
    other.close()
