"""UniformSampling, normal estimation, SPFH / FPFH and the batched first-frame path against the CPU oracle, on clouds built to hit
what smooth surfaces never do: exact k-NN ties and zero-distance duplicates, exactly degenerate covariances (a wire: rank 1, NaN
normals; a plate: rank 2, a viewpoint in its plane), pair features on the edges of their bins, neighbours at exactly the FPFH
radius, isolated and non-finite points, a large offset and a scale whose covariance falls below FLT_MIN, and clouds at the
capacity switches of the device paths (normals 4 096, FPFH 2 048, the batch envelope 2 048 / 4 096 samples and the 4 096-voxel
sampling hash). A cluster with one point metres away spans more than 2^28 voxels: the dense voxel tables process such frames in
windows and must still give PCL's result.

Bars: UniformSampling indices bit-exact; normals with the same finite mask, bit-equal on the exact clouds (lattice, plate, wire)
and within 2e-6 elsewhere; SPFH bit-exact; FPFH with the same NaN mask and within 1e-4 relative. Every path switch gives the same
bits. Batched frames equal one fresh ope_pose_estimate_final per frame as test_gpu_parity.py asks, and the oracle's counts,
SAC-IA winner and coarse pose.

test_cases_hit_what_they_are_built_for runs without a GPU: it checks on the oracle that every case reaches its edge."""
import ctypes

import numpy as np
import pytest

H = 1.0 / 64      # lattice spacing: a power of two, so squared distances between lattice points are exact in float
FPFH_RTOL = 1e-4
ROT_TOL = 1e-4    # rad
TRANS_TOL = 1e-5  # m
KS = (1, 2, 3, 12, 30, 32)
FAR = np.float32([7.0, 7.0, 7.0])   # the far outlier: with a cluster near the camera, > 2^28 voxels at 1 cm


# ------------------------------------------------------------------------------------------------- clouds ----
def _lattice(nx, ny, nz, h=H):
    g = np.stack(np.meshgrid(np.arange(nx), np.arange(ny), np.arange(nz), indexing="ij"), -1).reshape(-1, 3)
    return (g * h).astype(np.float32)


def lattice_ties():
    """A 12 x 12 x 6 lattice plus 64 duplicated points, shuffled: ties at the k-th neighbour, zero-distance pairs (SPFH bins a
    duplicate with f = 0, FPFH skips d^2 == 0), and with r = 2 h pairs at exactly d^2 == r^2."""
    rng = np.random.default_rng(201)
    lat = _lattice(12, 12, 6)
    dup = lat[rng.choice(len(lat), 64, replace=False)]
    pts = np.concatenate([lat, dup])
    return pts[rng.permutation(len(pts))]


def wire_blob():
    """60 exactly collinear points (y, z powers of two, spacing 1/512) 3 cm from a 400-point blob: with k = 12 every wire point's
    neighbours lie on the wire, its covariance has rank 1 and its normal is NaN; with r = 0.05 those NaN normals are FPFH
    neighbours of blob points."""
    rng = np.random.default_rng(202)
    wire = np.zeros((60, 3), np.float32)
    wire[:, 0] = np.arange(60, dtype=np.float32) / 512
    wire[:, 1] = 0.25
    wire[:, 2] = 0.5
    blob = rng.uniform([0.0, 0.28, 0.45], [0.12, 0.33, 0.55], (400, 3)).astype(np.float32)
    pts = np.concatenate([blob, wire])
    return pts[rng.permutation(len(pts))]


def plate():
    """600 exactly coplanar points (z = 0.5): normals exactly (0, 0, -1) with curvature 0 seen from the origin."""
    rng = np.random.default_rng(203)
    p = rng.uniform(0, 0.2, (600, 3)).astype(np.float32)
    p[:, 2] = 0.5
    return p


def slab():
    """Two parallel 16 x 16 lattice faces 3 h apart, seen from between them: with k = 12 every neighbourhood lies in one face
    (normals exactly +-z, pointing at each other), and with r = 3.5 h pairs across the faces have antiparallel normals, so pair
    features land on both edges of their ranges (f = +-1, +-pi / 2: the first bin and the last, clamped from 11 to 10)."""
    f = _lattice(16, 16, 1)
    return np.concatenate([f, f + np.float32([0, 0, 3 * H])])


SLAB_VP = (8 * H, 8 * H, 1.5 * H)


def isolated_nonfinite():
    """A lattice, an isolated point (no neighbour within r: all-zero SPFH and FPFH), and NaN / inf rows (NaN rows out)."""
    p = np.concatenate([_lattice(8, 8, 4), np.float32([[1, 1, 1], [np.nan, 0, 0], [0, np.inf, 0], [np.nan] * 3])])
    return p[np.random.default_rng(204).permutation(len(p))]


def offset():
    """lattice_ties() 100 m away (1/64 multiples stay exact at that magnitude)."""
    return lattice_ties() + np.float32([100, -100, 100])


def tiny():
    """A random blob scaled to 1e-21 m: the covariance (~1e-44) falls below FLT_MIN (eigen33's unit-scale branch)."""
    return (np.random.default_rng(205).normal(0, 1, (300, 3)) * 1e-21).astype(np.float32)


# (name, points, normal k values, viewpoints, fpfh radius, exact: normals must equal the oracle's bit for bit)
def feature_cases():
    return [
        ("lattice", lattice_ties(), KS, [(0, 0, 0), (0.3, -0.2, 1.0)], 2 * H, True),
        ("wire", wire_blob(), (3, 12), [(0, 0, 0)], 0.05, True),
        ("plate", plate(), (3, 12, 30), [(0, 0, 0), (0.1, 0.1, 0.5)], 0.03, True),
        ("slab", slab(), (12,), [SLAB_VP], 3.5 * H, False),
        ("isolated", isolated_nonfinite(), (3, 12, 30), [(0, 0, 0)], 2 * H, False),
        ("offset", offset(), (12, 30), [(100, -100, 99)], 2 * H, False),
        ("tiny", tiny(), (12, 30), [(0, 0, 0)], 3e-21, False),
    ]


def size_cases():
    """Prefixes of lattice_ties() at n = 1, 2, 3, k-1, k, k+1, and lattices at the normals (4 096) and FPFH (2 048) switches."""
    base = lattice_ties()
    out = [("n%d" % n, base[:n]) for n in sorted({1, 2, 3, 11, 12, 13, 29, 30, 31, 32, 33})]
    big = _lattice(16, 16, 16)
    out += [("n4096", big), ("n4097", np.concatenate([big, np.float32([[0.5 * H, 0.5 * H, 0.5 * H]])]))]
    half = _lattice(16, 16, 8)
    out += [("n2048", half), ("n2049", np.concatenate([half, np.float32([[0.5 * H, 0.5 * H, 0.5 * H]])]))]
    return out


# ----------------------------------------------------------------------------------------- batched clusters ----
def _voxels(orc, pts, leaf):
    return len(orc.uniform_sample(pts, leaf))


def _pad_to(orc, cl, leaf, want, z):
    """cl plus points at the centres of (want - samples of cl) voxels of a plane at depth z behind it."""
    need = want - _voxels(orc, cl, leaf)
    assert need > 0
    side = int(np.ceil(np.sqrt(need)))
    ij = np.stack(np.meshgrid(np.arange(side), np.arange(side), indexing="ij"), -1).reshape(-1, 2)[:need]
    base = np.floor(cl[:, :2].min(0) / leaf)
    pad = np.empty((need, 3), np.float32)
    pad[:, :2] = (base + ij + 0.5) * leaf
    pad[:, 2] = (np.floor(z / leaf) + 0.5) * leaf
    return np.concatenate([cl, pad]).astype(np.float32)


def batch_clusters(orc, synth, model):
    """(name, cluster) pairs for the pose entry points, from frames of the drill model."""
    fr = [synth.make_frame(model, 930 + i)[0] for i in range(8)]
    rng = np.random.default_rng(206)
    out = [("duplicated_shuffled", np.concatenate([fr[0], fr[0]])[rng.permutation(2 * len(fr[0]))])]
    out.append(("quantised_1mm", (np.round(fr[1].astype(np.float64) * 1000) / 1000).astype(np.float32)))
    w = fr[2][np.argmax(fr[2][:, 0])]
    wire = np.zeros((60, 3), np.float32)
    wire[:, 0] = np.float32(np.ceil(w[0] * 64) / 64) + np.arange(60, dtype=np.float32) / 64
    wire[:, 1] = np.float32(np.round(w[1] * 64) / 64)
    wire[:, 2] = np.float32(np.round(w[2] * 64) / 64)
    out.append(("wire", np.concatenate([fr[2], wire])))
    for name, leaf, want, f in (("s1cm_2048", 0.01, 2048, 3), ("s1cm_2049", 0.01, 2049, 3), ("s8mm_4096", 0.008, 4096, 4),
                                ("s8mm_4097", 0.008, 4097, 4)):
        out.append((name, _pad_to(orc, fr[f], leaf, want, fr[f][:, 2].max() + 0.05)))
    out.append(("hash_overflow", _pad_to(orc, fr[5], 0.01, 4300, fr[5][:, 2].max() + 0.05)))
    faces = (np.round(fr[6].astype(np.float64) * 100) / 100 - np.array([0.5, 0.5, 2.0])).astype(np.float32)
    out.append(("faces_negative", faces))
    nanrows = fr[7].copy()
    nanrows[::97] = np.nan
    nanrows[5, 1] = np.inf
    out.append(("nan_rows", nanrows))
    out.append(("far_outlier", np.concatenate([fr[0], FAR[None]])))
    return out


def _frame_cells(pts, leaf):
    """The PCL voxel frame's cell count, in float64 (UniformSampling's frame: floor(bbox * inv))."""
    p = pts[np.isfinite(pts).all(1)]
    inv = np.float32(1) / np.float32(leaf)
    lo, hi = np.floor(p.min(0) * inv), np.floor(p.max(0) * inv)
    return float(np.prod(hi - lo + 1))


def leaves_envelope(orc, cl):
    """Whether the batched fast path hands this frame to the per-frame path (batch.cu): a 1 cm sample above 2 048 points, an
    8 mm sample above 4 096, more than 4 096 occupied voxels in the sampling hash or a frame of more than 2^28 voxels."""
    n1, n2 = _voxels(orc, cl, 0.01), _voxels(orc, cl, 0.008)
    return n1 > 2048 or n2 > 4096 or max(_frame_cells(cl, 0.01), _frame_cells(cl, 0.008)) > 2 ** 28


# -------------------------------------------------------------------------------------------- CPU only ----
def test_cases_hit_what_they_are_built_for(orc, synth, model):
    lat = lattice_ties()
    idx, d2 = orc.knn(lat, lat, 13)
    assert (d2[:, 1] == 0).sum() == 128                     # every duplicate pair, both ways: zero-distance neighbours
    assert (d2[:, 11] == d2[:, 12]).mean() > 0.5            # a tie at the 12th neighbour for most points
    r2 = np.float32(2 * H) ** 2
    ri, rd = orc.knn(lat, lat, 64)
    assert (rd == r2).sum() > 1000                          # pairs at exactly the FPFH radius (left out by the strict <)
    wb = wire_blob()
    nw = orc.normals_knn(wb, 12)
    on_wire = (wb[:, 1] == 0.25) & (wb[:, 2] == 0.5)
    assert np.isnan(nw[on_wire, :3]).all() and np.isfinite(nw[~on_wire]).all()
    wi, wd = orc.knn(wb[on_wire], wb[~on_wire], 1)
    assert ((wd < 0.05 ** 2) & (wd > 0)).sum() > 20           # blob points with NaN-normal FPFH neighbours
    npl = orc.normals_knn(plate(), 12)
    assert (npl == np.float32([0, 0, -1, 0])).all()
    sl = slab()
    ns = orc.normals_knn(sl, 12, SLAB_VP)
    sp = orc.spfh(sl, ns, 3.5 * H)
    assert (sp[:, 10] > 0).sum() > 400 and (sp[:, 32] > 0).sum() > 400   # f1 and f3 in their last bin (clamped from 11)
    nl = orc.normals_knn(lat, 30, (0.3, -0.2, 1.0))
    assert ((orc.spfh(lat, nl, 2 * H)[:, [0, 11, 22]] > 0).sum(0) > 300).all()            # and in their first
    iso = isolated_nonfinite()
    ni = orc.normals_knn(iso, 12)
    fi = orc.fpfh(iso, ni, 2 * H)
    k = int(np.where((iso == 1).all(1))[0][0])
    assert (fi[k] == 0).all() and np.isnan(fi[~np.isfinite(iso).all(1)]).all()
    cov = np.cov(tiny().astype(np.float64).T)
    assert np.abs(cov).max() < np.finfo(np.float32).tiny
    # the batched clusters
    cl = dict(batch_clusters(orc, synth, model))
    assert _voxels(orc, cl["s1cm_2048"], 0.01) == 2048 and _voxels(orc, cl["s1cm_2049"], 0.01) == 2049
    assert _voxels(orc, cl["s8mm_4096"], 0.008) == 4096 and _voxels(orc, cl["s8mm_4097"], 0.008) == 4097
    assert _voxels(orc, cl["hash_overflow"], 0.01) > 4096
    tw = cl["wire"][orc.uniform_sample(cl["wire"], 0.008)]
    assert np.isnan(orc.normals_knn(tw, 30)).any(1).sum() > 0        # n_tgt_fine drops through removeNaNNormals
    assert _frame_cells(cl["far_outlier"], 0.01) > 2 ** 28 and _frame_cells(cl["far_outlier"], 0.008) > 2 ** 28
    assert _frame_cells(cl["far_outlier"], 0.008) < 2 ** 31 - 1
    assert np.isnan(cl["nan_rows"]).any() and (cl["faces_negative"] < 0).any()
    out = {n for n, c in cl.items() if leaves_envelope(orc, c)}
    # (the padding that takes the 8 mm sample to 4 096 also takes the 1 cm sample above 2 048)
    assert out == {"s1cm_2049", "s8mm_4096", "s8mm_4097", "hash_overflow", "far_outlier"}, out


# ----------------------------------------------------------------------------------------------- device ----
def _env(monkeypatch, **kv):
    for k, v in kv.items():
        if v is None:
            monkeypatch.delenv(k, raising=False)
        else:
            monkeypatch.setenv(k, v)


def _same_bits(a, b):
    return np.array_equal(np.asarray(a).view(np.uint32), np.asarray(b).view(np.uint32))


@pytest.mark.gpu
def test_uniform_sampling_on_adversarial_clouds(ctx, orc, monkeypatch):
    clouds = [c for c in feature_cases()] + [(n, p, (), (), 0, False) for n, p in size_cases()]
    for name, pts, *_ in clouds:
        c = ctx.upload(pts)
        for leaf in (0.01, 0.008, H, 2 * H):
            o = orc.uniform_sample(pts, leaf)
            for multi in (None, "1"):
                _env(monkeypatch, OPE_UNIFORM_MULTI_PASS=multi)
                g = ctx.uniform_sample(c, leaf)
                assert np.array_equal(g, o), (name, leaf, multi)
        c.free()


@pytest.mark.gpu
def test_normals_on_adversarial_clouds(ctx, orc, monkeypatch):
    for name, pts, ks, vps, _, exact in feature_cases():
        c = ctx.upload(pts)
        for k in ks:
            for vp in vps:
                o = orc.normals_knn(pts, k, vp)
                runs = []
                for grid in (None, "1"):
                    _env(monkeypatch, OPE_NORMALS_FORCE_GRID=grid)
                    runs.append(ctx.normals_knn(c, k, vp))
                g = runs[0]
                assert _same_bits(runs[1], g), (name, k, vp)
                assert np.array_equal(np.isfinite(g), np.isfinite(o)), (name, k, vp)
                fin = np.isfinite(o)
                if exact:
                    assert _same_bits(g[fin], o[fin]), (name, k, vp, np.abs(g[fin] - o[fin]).max())
                else:
                    assert np.allclose(g[fin], o[fin], rtol=0, atol=2e-6), (name, k, vp, np.abs(g[fin] - o[fin]).max())
        c.free()


@pytest.mark.gpu
@pytest.mark.parametrize("k", KS)
def test_normals_at_sizes_and_switches(ctx, orc, monkeypatch, k):
    for name, pts in size_cases():
        o = orc.normals_knn(pts, k, (0.1, -0.2, 0.7))
        c = ctx.upload(pts)
        runs = []
        for grid in (None, "1"):
            _env(monkeypatch, OPE_NORMALS_FORCE_GRID=grid)
            runs.append(ctx.normals_knn(c, k, (0.1, -0.2, 0.7)))
        c.free()
        assert _same_bits(runs[1], runs[0]), (name, k)
        assert np.array_equal(np.isfinite(runs[0]), np.isfinite(o)), (name, k)
        fin = np.isfinite(o)
        assert _same_bits(runs[0][fin], o[fin]), (name, k, np.abs(runs[0][fin] - o[fin]).max())


def _check_fpfh(ctx, orc, monkeypatch, name, pts, nr, r):
    o, os_ = orc.fpfh(pts, nr, r), orc.spfh(pts, nr, r)
    c = ctx.upload(pts, nr)
    runs = []
    for grid in (None, "1"):
        _env(monkeypatch, OPE_FPFH_FORCE_GRID=grid)
        runs.append(ctx.fpfh(c, r, want_spfh=True))
    c.free()
    fin = ~np.isnan(o).any(1)
    for g, gs in runs:
        assert np.array_equal(np.isnan(g), np.isnan(o)) and np.array_equal(np.isnan(gs), np.isnan(os_)), name
        assert _same_bits(gs[fin], os_[fin]), (name, np.argwhere(gs[fin] != os_[fin])[:8].tolist())   # integer counts + replayed adds
        scale = np.maximum(np.abs(o[fin]), 1.0)                                           # histograms are percentages
        assert (np.abs(g[fin] - o[fin]) / scale).max() < FPFH_RTOL if fin.any() else True, name


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c[0] for c in feature_cases()])
def test_fpfh_on_adversarial_clouds(ctx, orc, monkeypatch, case):
    name, pts, ks, vps, r, _ = next(c for c in feature_cases() if c[0] == case)
    nr = orc.normals_knn(pts, ks[-1] if name != "wire" else 12, vps[-1])
    _check_fpfh(ctx, orc, monkeypatch, name, pts, nr, r)


@pytest.mark.gpu
def test_fpfh_at_sizes_and_switches(ctx, orc, monkeypatch):
    for name, pts in size_cases():
        nr = orc.normals_knn(pts, 12, (0.1, -0.2, 0.7))
        _check_fpfh(ctx, orc, monkeypatch, name, pts, nr, 2 * H)


def _far_blob():
    """The 400-point blob with one point at (7, 7, 7) m: 701^3 voxels at 1 cm, 875^3 at 8 mm."""
    blob = np.random.default_rng(207).normal(0, 0.05, (400, 3)).astype(np.float32)
    return np.concatenate([blob, FAR[None]])


@pytest.mark.gpu
def test_uniform_sampling_beyond_2e28_voxels(ctx, orc, cuda_lib, monkeypatch):
    pts = _far_blob()
    c = ctx.upload(pts)
    for leaf in (0.01, 0.008):
        assert _frame_cells(pts, leaf) > 2 ** 28
        o = orc.uniform_sample(pts, leaf)
        for multi in (None, "1"):
            _env(monkeypatch, OPE_UNIFORM_MULTI_PASS=multi)
            assert np.array_equal(ctx.uniform_sample(c, leaf), o), leaf
            sc = ctx.uniform_sample_cloud(c, leaf)
            assert _same_bits(sc.download(), pts[o]), leaf
            sc.free()
    # beyond INT_MAX voxels PCL's int voxel index overflows: refused
    assert _frame_cells(pts, 0.004) > 2 ** 31
    with pytest.raises(cuda_lib.OpeError) as e:
        ctx.uniform_sample(c, 0.004)
    assert e.value.rc == cuda_lib.T.OPE_ERR_GRID_TOO_LARGE
    c.free()


@pytest.mark.gpu
def test_voxel_grid_beyond_2e28_voxels(ctx, orc, cuda_lib):
    pts = _far_blob()
    rgb = np.random.default_rng(208).integers(0, 1 << 24, len(pts)).astype(np.uint32).view(np.float32)
    c = ctx.upload(pts)
    for leaf in (0.01, 0.008):
        gx, gr = ctx.voxel_grid(c, leaf, rgb)
        ox, orr = orc.voxel_grid(pts, leaf, rgb)
        assert _same_bits(gx, ox) and _same_bits(gr, orr), leaf
    with pytest.raises(RuntimeError):
        orc.voxel_grid(pts, 0.004)
    with pytest.raises(cuda_lib.OpeError) as e:
        ctx.voxel_grid(c, 0.004)
    assert e.value.rc == cuda_lib.T.OPE_ERR_GRID_TOO_LARGE
    c.free()


def _counts(p):
    return (p.n_src_coarse, p.n_tgt_coarse, p.n_src_fine, p.n_tgt_fine, p.sacia_best_iteration)


def _batch_equals_single(synth, T, g, s, name):
    assert _counts(g) == _counts(s), (name, _counts(g), _counts(s))
    assert g.sacia_best_error == s.sacia_best_error, name
    assert _same_bits(np.array(g.coarse_pose), np.array(s.coarse_pose)), name
    r, t = synth.pose_error(T.mat4(g.final_pose), T.mat4(s.final_pose))
    assert r < 1e-6 and t < 1e-6, (name, r, t)
    assert (g.icp_iterations, g.icp_state, g.icp_converged) == (s.icp_iterations, s.icp_state, s.icp_converged), name
    assert abs(g.fitness - s.fitness) < 1e-9, name


def _against_oracle(synth, T, g, o, name):
    assert _counts(g) == (o.n_src_coarse, o.n_tgt_coarse, o.n_src_fine, o.n_tgt_fine, o.sacia_best_iteration), name
    r, t = synth.pose_error(T.mat4(g.coarse_pose), np.array(o.coarse_pose, np.float64).reshape(4, 4).T)
    assert r < ROT_TOL and t < TRANS_TOL, (name, r, t)


@pytest.fixture(scope="module")
def adversarial_frames(orc, synth, model):
    return batch_clusters(orc, synth, model)


@pytest.mark.gpu
def test_pose_batch_on_adversarial_clusters(ctx, orc, synth, cuda_lib, model, adversarial_frames, monkeypatch):
    T = cuda_lib.T
    libc = ctypes.CDLL(None)
    names = [n for n, _ in adversarial_frames]
    frames = [c for _, c in adversarial_frames]
    libc.srand(11)
    serial = []
    for cl in frames:
        tr = cuda_lib.PoseTracker(ctx)
        serial.append(tr.estimate_final(model.copy(), cl))
        tr.close()
    for env in ({}, {"OPE_BATCH_MORTON": "0"}, {"OPE_BATCH_CHUNK": "1"}):
        with monkeypatch.context() as m:
            for k, v in env.items():
                m.setenv(k, v)
            libc.srand(11)
            got, status = ctx.pose_batch(model, frames, workers=4)
        assert (status == 0).all(), (env, dict(zip(names, status)))
        for name, g, s in zip(names, got, serial):
            _batch_equals_single(synth, T, g, s, (name, env))
    orc.srand(11)
    for name, cl, s in zip(names, frames, serial):
        _against_oracle(synth, T, s, orc.PoseEstimator().estimate_final(model.copy(), cl), name)


@pytest.mark.gpu
def test_far_outlier_cluster_through_both_pose_entry_points(ctx, orc, synth, cuda_lib, model, adversarial_frames):
    """One point metres from the cluster: a frame of more than 2^28 voxels at 1 cm and 8 mm, which the device refused (-6)."""
    T = cuda_lib.T
    libc = ctypes.CDLL(None)
    cl = dict(adversarial_frames)["far_outlier"]
    orc.srand(3)
    o = orc.PoseEstimator().estimate_final(model.copy(), cl)
    libc.srand(3)
    tr = cuda_lib.PoseTracker(ctx)
    s = tr.estimate_final(model.copy(), cl)
    tr.close()
    _against_oracle(synth, T, s, o, "single")
    libc.srand(3)
    got, status = ctx.pose_batch(model, [cl], workers=1)
    assert (status == 0).all(), status
    _batch_equals_single(synth, T, got[0], s, "batch")


@pytest.mark.gpu
def test_tracker_step_batch_with_adversarial_sources(ctx, orc, synth, cuda_lib, model):
    """First calls of three trackers whose sources are the model duplicated and shuffled, quantised to 1 mm, and with the far
    outlier: ope_pose_tracker_step_batch equals one fresh ope_pose_estimate_final per tracker and the oracle."""
    T = cuda_lib.T
    libc = ctypes.CDLL(None)
    rng = np.random.default_rng(209)
    sources = [np.concatenate([model, model])[rng.permutation(2 * len(model))],
               (np.round(model.astype(np.float64) * 1000) / 1000).astype(np.float32),
               np.concatenate([model, FAR[None]])]
    targets = [synth.make_frame(model, 940 + i)[0] for i in range(3)]
    libc.srand(13)
    serial = []
    for src, tgt in zip(sources, targets):
        tr = cuda_lib.PoseTracker(ctx)
        serial.append(tr.estimate_final(src.copy(), tgt))     # the host source becomes alignedSource
        tr.close()
    trackers = [cuda_lib.PoseTracker(ctx) for _ in sources]
    dev = [ctx.upload(s) for s in sources]
    libc.srand(13)
    got, status = ctx.pose_track_batch(trackers, dev, targets)
    assert (status == 0).all(), status
    for i, (g, s) in enumerate(zip(got, serial)):
        _batch_equals_single(synth, T, g, s, i)
    orc.srand(13)
    for i, (src, tgt) in enumerate(zip(sources, targets)):
        _against_oracle(synth, T, serial[i], orc.PoseEstimator().estimate_final(src.copy(), tgt), i)
    for t, d in zip(trackers, dev):
        d.free()
        t.close()
