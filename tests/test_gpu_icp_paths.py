"""Every search path of the device ICP against the CPU oracle, on clouds built to hit what smooth surfaces never do: exact
ties, pairs at exactly the correspondence limit, queries crossing bisector planes between iterations (the certificates), queries
with thousands of near-equidistant candidates (the far-query queue and its split), NaN / inf rows, large offsets and small
scales, and degenerate sizes. The nearest-neighbour estimator must give one result, bit for bit, under every search tunable;
normal shooting must give the oracle's result through each of its device paths; fixed correspondences must follow the oracle in
every configuration of estimator, rejector chain, reciprocity, transformation estimator and variant.

Bars as in test_gpu_parity.py: correspondence lists (query, match, order) bit-exact, the same converged / state / iterations /
n_correspondences, poses within 1e-4 rad / 1e-5 m, fitness within 1e-5."""
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROT_TOL = 1e-4    # rad
TRANS_TOL = 1e-5  # m
FIT_TOL = 1e-5
H = 1.0 / 64      # lattice spacing: a power of two, so squared distances between (half-)lattice points are exact in float


# ------------------------------------------------------------------------------------------------- clouds ----
def _lattice(nx, ny, nz, h=H):
    g = np.stack(np.meshgrid(np.arange(nx), np.arange(ny), np.arange(nz), indexing="ij"), -1).reshape(-1, 3)
    return (g * h).astype(np.float32)


def _rot(axis, deg):
    a = np.asarray(axis, np.float64)
    a /= np.linalg.norm(a)
    t = np.deg2rad(deg)
    K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return np.eye(3) + np.sin(t) * K + (1 - np.cos(t)) * K @ K


def lattice_ties():
    """Target: a 16 x 16 x 12 lattice plus 64 duplicated points, shuffled so that a duplicate may come before or after its
    original. Source: midpoints of edges, faces and cells (2-, 4- and 8-way exact ties), the duplicated points themselves
    (zero-distance ties), and points one and two spacings outside the x = max face (squared distance exactly h^2 and 4 h^2)."""
    rng = np.random.default_rng(101)
    lat = _lattice(16, 16, 12)
    dup = lat[rng.choice(len(lat), 64, replace=False)]
    tgt = np.concatenate([lat, dup])[rng.permutation(len(lat) + 64)]
    inner = lat[(lat[:, 0] < 15 * H) & (lat[:, 1] < 15 * H) & (lat[:, 2] < 11 * H)]
    parts = [inner[rng.choice(len(inner), 300, replace=False)] + np.float32(H / 2) * np.array(off, np.float32)
             for off in ((1, 0, 0), (0, 1, 0), (1, 1, 0), (0, 1, 1), (1, 1, 1))]
    parts.append(dup[:40])
    face = lat[lat[:, 0] == 15 * H][rng.choice(16 * 12, 120, replace=False)]
    parts.append(face + np.array([H, 0, 0], np.float32))
    parts.append(face[:60] + np.array([2 * H, 0, 0], np.float32))
    src = np.concatenate(parts).astype(np.float32)
    return src[rng.permutation(len(src))], tgt


def crossing_bisectors():
    """Target: a 20 x 20 x 16 lattice. Source: 3 000 of its points, turned by 3 degrees about the lattice centre and moved by
    about 0.4 h, so that ICP drags many of them across the bisector planes between lattice points from one iteration to the
    next: the case a wrong cross-iteration certificate would get wrong."""
    rng = np.random.default_rng(102)
    tgt = _lattice(20, 20, 16)
    src = tgt[rng.choice(len(tgt), 3000, replace=False)].astype(np.float64)
    c = tgt.mean(0)
    src = (src - c) @ _rot((1, 2, 3), 3.0).T + c + np.array([0.4, -0.35, 0.3]) * H
    return src.astype(np.float32), tgt


def sphere_far():
    """Target: 8 000 points on a sphere (radius 0.1). Source: 150 points close to its centre (thousands of near-equidistant
    candidates each: far queries, split by start node), 40 points far outside the target's box, 400 points near the surface."""
    rng = np.random.default_rng(103)
    n = 8000
    i = np.arange(n) + 0.5
    phi, th = np.arccos(1 - 2 * i / n), np.pi * (1 + 5 ** 0.5) * i
    c = np.array([0.3, -0.2, 0.9])
    tgt = c + 0.1 * np.stack([np.cos(th) * np.sin(phi), np.sin(th) * np.sin(phi), np.cos(phi)], 1)
    centre = c + rng.normal(0, 0.002, (150, 3))
    d = rng.normal(size=(40, 3))
    outside = c + 0.8 * d / np.linalg.norm(d, axis=1, keepdims=True)
    surf = tgt[rng.choice(n, 400, replace=False)] * (1 + rng.normal(0, 0.003, (400, 1))) + np.array([0.004, -0.003, 0.002])
    src = np.concatenate([centre, outside, surf])
    return src[rng.permutation(len(src))].astype(np.float32), tgt.astype(np.float32)


def with_nonfinite(src):
    """NaN and +-inf rows spread through the source; returns the cloud and the positions of the finite rows"""
    out = src.copy()
    bad = np.arange(7, len(src), 97)
    vals = (np.nan, np.inf, -np.inf)
    for j, b in enumerate(bad):
        out[b, j % 3] = vals[j % 3]
    return out, np.setdiff1d(np.arange(len(src)), bad)


def _cases():
    src, tgt = lattice_ties()
    cs, ct = crossing_bisectors()
    ss, st = sphere_far()
    bad, _ = with_nonfinite(src)
    return {
        "lattice": (src, tgt, {}),
        "lattice-limit": (src, tgt, dict(max_correspondence_distance=H)),   # some pairs at exactly d2 == max^2
        "crossing": (cs, ct, dict(max_correspondence_distance=4 * H)),
        "sphere": (ss, st, {}),
        "sphere-limit": (ss, st, dict(max_correspondence_distance=0.0995)),   # the centre queries sit right at the limit
        "nonfinite": (bad, tgt, dict(max_correspondence_distance=H)),
        "offset-100m": (src + np.float32(100.0), tgt + np.float32(100.0), dict(max_correspondence_distance=H)),
        "scaled": (src * np.float32(2.0 ** -10), tgt * np.float32(2.0 ** -10), dict(max_correspondence_distance=H * 2.0 ** -10)),
        "tgt1": (src[:200], tgt[:1], {}),
        "tgt2": (src[:200], tgt[:2], {}),
        "tgt3": (src[:200], tgt[:3], {}),
    }


CASES = None


def case(name):
    global CASES
    if CASES is None:
        CASES = _cases()
    return CASES[name]


# -------------------------------------------------------------------------------------------------- checks ----
def _key(res):
    return res.converged, res.state, res.iterations, res.n_correspondences


def _same_as_oracle(synth, T, g, gc, o, oc, what):
    assert _key(g) == _key(o), (what, _key(g), _key(o))
    assert np.array_equal(gc[0], oc[0]) and np.array_equal(gc[1], oc[1]), (what, _first_diff(gc, oc))
    assert np.allclose(gc[2], oc[2], rtol=1e-5, atol=0), what
    r, t = synth.pose_error(T.mat4(g.T), T.mat4(o.T))
    assert r < ROT_TOL and t < TRANS_TOL, (what, r, t)


def _first_diff(a, b):
    n = min(len(a[0]), len(b[0]))
    d = np.nonzero((a[0][:n] != b[0][:n]) | (a[1][:n] != b[1][:n]))[0]
    j = int(d[0]) if len(d) else n
    return dict(len=(len(a[0]), len(b[0])), at=j, dev=[x[j:j + 3].tolist() for x in a], orc=[x[j:j + 3].tolist() for x in b])


def _same_bits(g, gc, h, hc, what):
    assert np.array_equal(np.array(list(g.T), np.float32).view(np.uint32), np.array(list(h.T), np.float32).view(np.uint32)), what
    assert _key(g) == _key(h), (what, _key(g), _key(h))
    assert all(np.array_equal(a.view(np.uint32), b.view(np.uint32)) for a, b in zip(gc, hc)), what


def _fitness_close(ctx, orc, T, cs, ct, src, tgt, g, o):
    gf, of = ctx.fitness(cs, ct, T.mat4(g.T)), orc.fitness(src, tgt, T.mat4(o.T))
    assert abs(gf - of) < FIT_TOL * max(1.0, abs(of)), (gf, of)


# ------------------------------------------------------------------------------------------ the clouds themselves ----
def test_the_cases_hit_what_they_are_built_for(orc):
    """CPU-side facts the GPU tests below rely on (checked against the oracle, so they hold wherever the oracle does)."""
    src, tgt = lattice_ties()
    i, d = orc.knn(tgt, src, 2, brute=True)
    assert (d[:, 0] == d[:, 1]).mean() > 0.5                    # most queries have an exactly tied second neighbour
    assert (d[:, 0] == np.float32(H * H)).sum() >= 100           # and many sit at exactly the 1-spacing limit
    cs, ct = crossing_bisectors()
    prm = dict(max_correspondence_distance=4 * H)
    _, c1 = orc.icp(cs, ct, orc.icp_params(max_iterations=1, **prm), want_corr=True)
    _, c30 = orc.icp(cs, ct, orc.icp_params(max_iterations=30, **prm), want_corr=True)
    assert np.array_equal(c1[0], c30[0])
    changed = (c1[1] != c30[1]).mean()
    print("crossing bisectors: %.1f %% of the matches change between iteration 1 and iteration 30" % (100 * changed))
    assert changed > 0.2


# ------------------------------------------------------------------------ nearest estimator, every tunable ----
TUNABLES = [{}, {"OPE_ICP_CERT_GAP": "0"}, {"OPE_ICP_CERT_GAP": "4"}, {"OPE_ICP_DFS_MAX": "1000000"}, {"OPE_ICP_SPLIT_MIN": "0"},
            {"OPE_ICP_SPLIT_MIN": "1000000000"}, {"OPE_ICP_FORCE_GRID": "1"}]
NEAREST_CASES = ["lattice", "lattice-limit", "crossing", "sphere", "sphere-limit", "nonfinite", "offset-100m", "scaled", "tgt1",
                 "tgt2", "tgt3"]


def _set_env(monkeypatch, env):
    for k in ("OPE_ICP_CERT_GAP", "OPE_ICP_DFS_MAX", "OPE_ICP_SPLIT_MIN", "OPE_ICP_FORCE_GRID", "OPE_ICP_SMALL"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


@pytest.mark.parametrize("name", NEAREST_CASES)
def test_nearest_one_result_for_every_tunable(ctx, orc, synth, cuda_lib, name, monkeypatch):
    """The fused kernel's search (seeded previous match, cross-iteration and range certificates, direct scan, per-thread DFS,
    grid-wide far-query queue with and without the split by start node, the no-room fallback) against the oracle, and every
    setting against every other bit for bit; iteration 1 also against ope_correspondences, a different kernel."""
    T = cuda_lib.T
    src, tgt, kw = case(name)
    cs, ct = ctx.upload(src), ctx.upload(tgt)
    for iters in (1, 3, 30):
        prm = dict(max_iterations=iters, transformation_epsilon=1e-10, euclidean_fitness_epsilon=1e-12, **kw)
        o, oc = orc.icp(src, tgt, orc.icp_params(**prm), want_corr=True)
        first = None
        for env in TUNABLES:
            _set_env(monkeypatch, env)
            g, gc = ctx.icp(cs, ct, cuda_lib.icp_params(**prm), want_corr=True)
            what = (name, iters, env)
            _same_as_oracle(synth, T, g, gc, o, oc, what)
            if first is None:
                first = (g, gc)
                _fitness_close(ctx, orc, T, cs, ct, src, tgt, g, o)
            else:
                _same_bits(g, gc, *first, what)
            if iters == 1:
                c = ctx.correspondences(cs, ct, cuda_lib.icp_params(**prm))
                assert all(np.array_equal(a, b) for a, b in zip(c, gc)), what
        _set_env(monkeypatch, {})


def test_nonfinite_rows_change_nothing_else(ctx, orc, synth, cuda_lib):
    """NaN / inf source rows get no correspondence, and every other row gets what it gets without them."""
    src, tgt = lattice_ties()
    bad, keep = with_nonfinite(src)
    clean = src[keep]
    ct = ctx.upload(tgt)
    for iters in (1, 3):
        prm = dict(max_iterations=iters, max_correspondence_distance=H)
        g, gc = ctx.icp(ctx.upload(bad), ct, cuda_lib.icp_params(**prm), want_corr=True)
        h, hc = ctx.icp(ctx.upload(clean), ct, cuda_lib.icp_params(**prm), want_corr=True)
        o, oc = orc.icp(clean, tgt, orc.icp_params(**prm), want_corr=True)
        assert np.isin(gc[0], keep).all()
        assert np.array_equal(gc[0], keep[hc[0]]) and np.array_equal(gc[1], hc[1]) and np.array_equal(gc[2], hc[2])
        assert np.array_equal(hc[0], oc[0]) and np.array_equal(hc[1], oc[1])
        assert _key(g) == _key(h) == _key(o)


def test_far_queries_really_happen(ctx, cuda_lib, monkeypatch, capfd):
    """The sphere's centre queries go through the grid-wide far-query queue under the default settings (OPE_PROFILE counts)."""
    src, tgt, kw = case("sphere")
    _set_env(monkeypatch, {})
    monkeypatch.setenv("OPE_PROFILE", "1")
    monkeypatch.setenv("OPE_PROFILE_ITER", "1")
    capfd.readouterr()
    ctx.icp(ctx.upload(src), ctx.upload(tgt), cuda_lib.icp_params(max_iterations=5, **kw))
    err = capfd.readouterr().err
    block0 = re.search(r"far queries of block 0: ([0-9.]+)", err)
    grid = [int(m.group(1)) for m in re.finditer(r"^\s+it\s+\d+:[^|]*\|\s*-?\d+\s*\|\s*(\d+)\s*\|", err, re.M)]
    print("sphere: far queries of block 0 per iteration %s; far queries of the grid per iteration %s"
          % (block0.group(1) if block0 else "?", grid))
    assert block0 is not None and len(grid) == 5, err[-2000:]
    assert grid[0] >= 100, grid                  # the centre queries (150 of them) cannot be answered by the fast path


# ----------------------------------------------------------------------------- normal shooting, every path ----
SHOOT_PATHS = [{}, {"OPE_ICP_FORCE_GRID": "1"}, {"OPE_ICP_SMALL": "1"}, {"OPE_ICP_SMALL": "0"}]
REJECTOR_CHAINS = [[], [(0, 0.7)], [(0, 0.2), (1, -0.5)]]    # kinds filled in from abi_types below


def _chain(T, i):
    kinds = (T.REJ_SURFACE_NORMAL, T.REJ_SELF_OCCLUDED_NORMAL)
    return [(kinds[k], thr) for k, thr in REJECTOR_CHAINS[i]]


def _shooting_cases():
    src, tgt = lattice_ties()
    cs, ct = crossing_bisectors()
    ss, st = sphere_far()
    return {
        "lattice": (src, tgt),
        "crossing": (cs, ct),
        "sphere": (ss, st),
        "offset-100m": (src + np.float32(100.0), tgt + np.float32(100.0)),
        "tgt3": (src[:200], tgt[:3]),                  # k_search above the number of targets
        "tgt4096": (cs[:1500], ct[:4096]),             # the largest target kept in shared memory
        "tgt4097": (cs[:1500], ct[:4097]),             # the smallest one that is not
        "src4096": (ct[:4096] + np.float32(0.3 * H), ct[:4000]),   # the largest source of the thread-per-query kernel
        "src4097": (ct[:4097] + np.float32(0.3 * H), ct[:4000]),
    }


@pytest.mark.parametrize("name", ["lattice", "crossing", "sphere", "offset-100m", "tgt3", "tgt4096", "tgt4097", "src4096", "src4097"])
def test_normal_shooting_every_path(ctx, orc, synth, cuda_lib, name, monkeypatch):
    T = cuda_lib.T
    src, tgt = _shooting_cases()[name]
    sn, tn = orc.normals_knn(src, 12), orc.normals_knn(tgt, 12)
    cs, ct = ctx.upload(src, sn), ctx.upload(tgt, tn)
    for k in (1, 20, 32):
        for chain in range(len(REJECTOR_CHAINS)):
            for variant in (T.ICP_VARIANT_MOD, T.ICP_VARIANT_MODCORR):
                prm = dict(max_iterations=8, transformation_epsilon=1e-10, euclidean_fitness_epsilon=1e-12, estimator=T.EST_NORMAL_SHOOTING,
                           k_search=k, rejectors=_chain(T, chain), with_normals=1, variant=variant)
                o, oc = orc.icp(src, tgt, orc.icp_params(**prm), src_normals=sn, tgt_normals=tn, want_corr=True)
                for env in SHOOT_PATHS:
                    _set_env(monkeypatch, env)
                    g, gc = ctx.icp(cs, ct, cuda_lib.icp_params(**prm), want_corr=True)
                    _same_as_oracle(synth, T, g, gc, o, oc, (name, k, chain, variant, env))
                _set_env(monkeypatch, {})


def test_min_number_correspondences_hit_exactly(ctx, orc, cuda_lib, monkeypatch):
    """n_correspondences == min_number_correspondences goes on; one more required stops with NO_CORRESPONDENCES."""
    T = cuda_lib.T
    src, tgt = lattice_ties()
    kw = dict(max_correspondence_distance=H)
    n1 = len(orc.correspondences(src, tgt, orc.icp_params(**kw))[0])
    cs, ct = ctx.upload(src), ctx.upload(tgt)
    for env in ({}, {"OPE_ICP_CERT_GAP": "0"}, {"OPE_ICP_FORCE_GRID": "1"}):
        _set_env(monkeypatch, env)
        for mn, state in ((n1, None), (n1 + 1, T.CONV_NO_CORRESPONDENCES)):
            prm = dict(max_iterations=1, min_number_correspondences=mn, **kw)
            g = ctx.icp(cs, ct, cuda_lib.icp_params(**prm))
            o = orc.icp(src, tgt, orc.icp_params(**prm))
            assert _key(g) == _key(o), (env, mn, _key(g), _key(o))
            if state is not None:
                assert g.state == state and g.iterations == 0
            else:
                assert g.iterations == 1 and g.n_correspondences == n1
    _set_env(monkeypatch, {})


# ---------------------------------------------------------------------- fixed correspondences x configuration ----
def _fixed_inputs(small_model):
    """2 000 points of the synthetic model, and 1 500 of them turned by 4 degrees and moved by a few millimetres (a surface
    without the symmetries that leave point-to-plane estimation singular); six source points to pin"""
    rng = np.random.default_rng(104)
    tgt = small_model[rng.choice(len(small_model), 2000, replace=False)].astype(np.float32)
    c = tgt.mean(0)
    src = (tgt[rng.choice(len(tgt), 1500, replace=False)].astype(np.float64) - c) @ _rot((0, 1, 1), 4.0).T + c
    src = (src + np.array([0.003, 0.002, -0.002])).astype(np.float32)
    return src, tgt, rng.choice(len(src), 6, replace=False)


@pytest.mark.parametrize("estimator", ["nearest", "nearest-reciprocal", "shooting"])
def test_fixed_correspondences_every_configuration(ctx, orc, synth, cuda_lib, small_model, estimator):
    """setFixedCorrespondences through the host-sequenced loop: the nearest estimator puts the pairs in front (whole chain,
    distance rewritten) and appends them after rejector 0; the reciprocal and shooting estimators only append them, with the
    caller's distances. Duplicate pairs included."""
    T = cuda_lib.T
    src, tgt, fq = _fixed_inputs(small_model)
    fm = orc.knn(tgt, src[fq], 3)[0][:, 2]
    fq = np.concatenate([fq, fq[:1], fq[1:2]]).astype(np.int32)            # an exact duplicate, and one query pinned twice
    fm = np.concatenate([fm, fm[:1], fm[2:3]]).astype(np.int32)
    fd = np.linspace(1e-4, 8e-4, len(fq)).astype(np.float32)                # what the loop keeps where it does not rewrite
    sn, tn = orc.normals_knn(src, 12), orc.normals_knn(tgt, 12)
    cs, ct = ctx.upload(src, sn), ctx.upload(tgt, tn)
    base = dict(max_iterations=6, max_correspondence_distance=0.02, transformation_epsilon=1e-10, euclidean_fitness_epsilon=1e-12)
    if estimator == "shooting":
        base.update(estimator=T.EST_NORMAL_SHOOTING, k_search=10, max_correspondence_distance=1.0)
    if estimator == "nearest-reciprocal":
        base.update(use_reciprocal=1)
    chains = [[], [(T.REJ_SURFACE_NORMAL, 0.5)], [(T.REJ_SURFACE_NORMAL, 0.2), (T.REJ_SELF_OCCLUDED_NORMAL, -0.5)]]
    n_checked = 0
    for chain in chains:
        for te in (T.TE_SVD, T.TE_POINT_TO_PLANE_LLS, T.TE_POINT_TO_PLANE):
            for variant in (T.ICP_VARIANT_MOD, T.ICP_VARIANT_MODCORR):
                prm = dict(base, rejectors=chain, transformation=te, variant=variant, with_normals=1)
                what = (estimator, len(chain), te, variant)
                g, gc, gd = ctx.icp(cs, ct, cuda_lib.icp_params(**prm), want_corr=True, fixed=(fq, fm, fd))
                o, oc, od = orc.icp(src, tgt, orc.icp_params(**prm), src_normals=sn, tgt_normals=tn, want_corr=True, fixed=(fq, fm, fd))
                _same_as_oracle(synth, T, g, gc, o, oc, what)
                assert np.allclose(gd, od, rtol=1e-5, atol=0), (what, gd, od)
                if estimator != "nearest":          # the caller's distances stay; the tail after rejector 0 carries them
                    assert np.array_equal(gd, fd), what
                    tail = np.isin(gc[2], fd).sum()
                    assert tail >= 1 if (variant == T.ICP_VARIANT_MOD and chain) else tail == 0, (what, tail)
                n_checked += 1
    assert n_checked == 18


def test_fixed_pair_on_a_nonfinite_point_is_refused(ctx, orc, cuda_lib, small_model):
    """A fixed pair whose query is a NaN row has no defined result (the oracle's transform turns NaN): the device refuses it,
    as it refuses indices out of range."""
    T = cuda_lib.T
    src, tgt, fq = _fixed_inputs(small_model)
    src = src.copy()
    src[fq[0]] = np.nan
    fm = np.arange(len(fq), dtype=np.int32)
    prm = dict(max_iterations=3, max_correspondence_distance=0.02)
    o = orc.icp(src, tgt, orc.icp_params(**prm), fixed=(fq, fm))
    assert not np.isfinite(np.array(list(o.T))).all()
    cs, ct = ctx.upload(src), ctx.upload(tgt)
    with pytest.raises(cuda_lib.OpeError):
        ctx.icp(cs, ct, cuda_lib.icp_params(**prm), fixed=(fq, fm))
    with pytest.raises(cuda_lib.OpeError):
        ctx.icp(cs, ct, cuda_lib.icp_params(**prm), fixed=(fq[1:], np.full(len(fq) - 1, len(tgt), np.int32)))
    g = ctx.icp(cs, ct, cuda_lib.icp_params(**prm), fixed=(fq[1:], fm[1:]))      # without it: accepted
    assert g.iterations >= 1 and T.CONV_NO_CORRESPONDENCES != g.state
