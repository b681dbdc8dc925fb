"""Pins the oracle to the reference's own code: oracle == oracle/_ref on the ICP configurations.

oracle/_ref holds the reference's VENDORED registration sources (VP = DetectAndLocalize/include/pcl/registration: the ICP loop,
Registration::align / getFitnessScore, CorrespondenceEstimation incl. reciprocal and fixed correspondences, the normal-shooting
loop, the rejector scores, the self-occluded-normal rejector, getAlignStrength, the convergence-criteria wiring), compiled
UNMODIFIED where they lie in the reference's source tree against the mock PCL of oracle/refstub (recipe: oracle/Makefile, target
`ref`; harness: oracle/ref_harness.cpp). The un-vendored PCL pieces ([UPSTREAM]: kd-tree, Umeyama/SVD, point-to-plane solvers,
transformPointCloud, hasConverged) are the oracle's own restatements on both sides and stay unpinned.

Both sides share the exact kd-tree and solvers, so every comparison is BIT-exact: transform, state, iteration count, the
last correspondence set, the fitness score, the align strength.

The reference's sources are not part of this repository: where oracle/_ref is not built, the same calls are answered from what
it returned, recorded in tests/golden/ref_registration.json (arrays as digests, so the comparisons stay bit-exact)."""
import numpy as np
import pytest

import ref_py


@pytest.fixture(scope="module")
def ref(orc):
    return ref_py if ref_py.available() else ref_py.Recorded()


@pytest.fixture(scope="module")
def drill(synth):
    return synth.bundled_model()


def _same(o, r, oc=None):
    assert np.array_equal(np.array(list(o.T)), np.array(list(r["res"].T))), np.abs(np.array(list(o.T)) - np.array(list(r["res"].T))).max()
    assert (o.converged, o.state, o.iterations, o.n_correspondences) == \
           (r["res"].converged, r["res"].state, r["res"].iterations, r["res"].n_correspondences)
    if oc is not None:
        assert all(ref_py.same_values(a, b) for a, b in zip(oc, r["corr"]))


def test_point_to_point_icp_c2(ref, orc, synth, drill):
    """BASELINE configs[1] shape (max-corr-distance 0.05, 50 iterations) at 8 000 points; getIcp's parameters
    (BM/src/regmeshpcd.cpp:16-41: transformation epsilon 1e-16, fitness epsilon left at its default)."""
    T = ref.T
    src, tgt, _ = synth.icp_pair(8000, seed=2, model=drill)
    for kw in (dict(max_iterations=50, max_correspondence_distance=0.05, transformation_epsilon=1e-8, euclidean_fitness_epsilon=1e-8),
               dict(max_iterations=80, max_correspondence_distance=0.05, transformation_epsilon=1e-16),
               dict(max_iterations=30, max_correspondence_distance=0.004, transformation_epsilon=1e-6, euclidean_fitness_epsilon=1e-3)):
        o, oc = orc.icp(src, tgt, orc.icp_params(**kw), want_corr=True)
        r = ref.icp(src, tgt, orc.icp_params(**kw))
        _same(o, r, oc)
        assert orc.fitness(src, tgt, T.mat4(o.T)) == r["fitness"]                       # Registration::getFitnessScore
        assert o.n_correspondences / (len(src) + len(tgt)) == r["align_strength"]       # getAlignStrength
        assert ref_py.same_values(orc.transform(src, T.mat4(o.T)), r["aligned"])        # `output`


def test_icp_with_guess_and_without_correspondences(ref, orc, synth, drill):
    src, tgt, _ = synth.icp_pair(3000, seed=4, model=drill)
    guess = synth.small_pose(np.random.default_rng(3), 2, 0.005).astype(np.float32)
    kw = dict(max_iterations=15, max_correspondence_distance=0.05)
    _same(orc.icp(src, tgt, orc.icp_params(**kw), guess=guess), ref.icp(src, tgt, orc.icp_params(**kw), guess=guess))
    far = (tgt + 100.0).astype(np.float32)
    kw = dict(max_iterations=5, max_correspondence_distance=0.01)
    o, r = orc.icp(src, far, orc.icp_params(**kw)), ref.icp(src, far, orc.icp_params(**kw))
    _same(o, r)
    assert o.state == ref.T.CONV_NO_CORRESPONDENCES and o.converged == 0


@pytest.mark.parametrize("variant", ["mod", "modcorr"])
def test_d_and_l_fine_stage(ref, orc, synth, drill, variant):
    """D&L/src/poseestimator.cpp:242-341: normal shooting k = 20, surface-normal 0.7 + self-occluded-normal 0.6, SVD,
    IterativeClosestPointWithNormals, 100 iterations, eps 1e-8 — through both vendored loops (icp_mod.hpp: estimator and
    rejectors re-fed from the transformed source every iteration; icp_modCorr.hpp: they keep what the application set once)."""
    T = ref.T
    cl, _, pose = synth.make_frame(drill, 1005)
    start = pose @ synth.small_pose(np.random.default_rng(8), 6, 0.01)
    sp_full = synth.apply(start, drill)
    sp = sp_full[orc.uniform_sample(sp_full, 0.008)]
    tp = cl[orc.uniform_sample(cl, 0.008)]
    sn, tn = orc.normals_knn(sp, 30), orc.normals_knn(tp, 30)
    keep_s, keep_t = np.isfinite(sn).all(1), np.isfinite(tn).all(1)
    sp, sn, tp, tn = sp[keep_s], sn[keep_s], tp[keep_t], tn[keep_t]
    kw = dict(max_iterations=100, transformation_epsilon=1e-8, euclidean_fitness_epsilon=1e-8, estimator=T.EST_NORMAL_SHOOTING,
              k_search=20, rejectors=[(T.REJ_SURFACE_NORMAL, 0.7), (T.REJ_SELF_OCCLUDED_NORMAL, 0.6)], with_normals=1,
              variant=T.ICP_VARIANT_MOD if variant == "mod" else T.ICP_VARIANT_MODCORR)
    o, oc = orc.icp(sp, tp, orc.icp_params(**kw), src_normals=sn, tgt_normals=tn, want_corr=True)
    r = ref.icp(sp, tp, orc.icp_params(**kw), src_normals=sn, tgt_normals=tn, variant=variant)
    _same(o, r, oc)
    assert o.iterations > 5
    assert orc.fitness(sp, tp, T.mat4(o.T)) == r["fitness"]
    assert o.n_correspondences / (len(sp) + len(tp)) == r["align_strength"]


@pytest.mark.parametrize("te", ["lm", "lls"])
def test_build_model_pair(ref, orc, synth, drill, te):
    """BM/src/regmeshpcd.cpp:62-208 (getIcpNormal): normal shooting k = 20, surface-normal rejector, point-to-plane
    Levenberg-Marquardt; and the constructor default of IterativeClosestPointWithNormals (LLS)."""
    T = ref.T
    (sp, _), (tp, _) = synth.turntable_views(drill[::4].copy(), n_views=36, first=2)
    sn, tn = orc.normals_knn(sp, 12), orc.normals_knn(tp, 12)
    kw = dict(max_iterations=40, transformation_epsilon=1e-8, euclidean_fitness_epsilon=1e-8, estimator=T.EST_NORMAL_SHOOTING,
              k_search=20, rejectors=[(T.REJ_SURFACE_NORMAL, 0.7)], with_normals=1,
              transformation=T.TE_POINT_TO_PLANE if te == "lm" else T.TE_POINT_TO_PLANE_LLS)
    o, oc = orc.icp(sp, tp, orc.icp_params(**kw), src_normals=sn, tgt_normals=tn, want_corr=True)
    r = ref.icp(sp, tp, orc.icp_params(**kw), src_normals=sn, tgt_normals=tn)
    _same(o, r, oc)


def test_reciprocal_correspondences(ref, orc, synth, drill):
    """determineReciprocalCorrespondences (VP/impl/correspondence_estimation_mod.hpp:216-303) alone and inside the loop
    (use_reciprocal_correspondence_, VP/impl/icp_mod.hpp:188-189)."""
    src, tgt, _ = synth.icp_pair(4000, seed=6, model=drill)
    tgt = tgt[:2500]                                  # unequal sizes: many source points share a target point
    for d in (0.05, 0.003):
        prm = orc.icp_params(max_correspondence_distance=d, use_reciprocal=1)
        oc = orc.correspondences_fixed(src, tgt, prm)
        rc = ref.correspondences(src, tgt, d, reciprocal=True)
        assert len(oc[0]) > 100 and all(ref_py.same_values(a, b) for a, b in zip(oc, rc))
        plain = orc.correspondences_fixed(src, tgt, orc.icp_params(max_correspondence_distance=d))
        assert len(oc[0]) < len(plain[0])
    kw = dict(max_iterations=25, max_correspondence_distance=0.05, transformation_epsilon=1e-8, euclidean_fitness_epsilon=1e-8,
              use_reciprocal=1)
    o, oc = orc.icp(src, tgt, orc.icp_params(**kw), want_corr=True)
    _same(o, ref.icp(src, tgt, orc.icp_params(**kw)), oc)


def test_fixed_correspondences(ref, orc, synth, drill):
    """The reference's own addition to ICP (VP/icp_mod.h:267-281, VP/impl/icp_mod.hpp:150-151,209-225,
    VP/impl/correspondence_estimation_mod.hpp:134-161): pinned pairs go in front with distance * 1e10 (rewritten in the
    caller's list every iteration) and, when rejectors exist, pass rejector 0 alone and are appended a second time."""
    T = ref.T
    rng = np.random.default_rng(11)
    src, tgt, _ = synth.icp_pair(3000, seed=7, model=drill)
    fq = rng.choice(len(src), 6, replace=False)
    fm = orc.knn(tgt, src[fq], 3)[0][:, 2]            # pin each to its THIRD nearest target point
    fixed = (fq, fm)
    prm = orc.icp_params(max_correspondence_distance=0.02)
    oc = orc.correspondences_fixed(src, tgt, prm, fixed)
    rc = ref.correspondences(src, tgt, 0.02, fixed=fixed)
    assert all(ref_py.same_values(a, b) for a, b in zip(oc, rc)) and np.array_equal(oc[0][:6], fq) and (oc[2][:6] > 1e3).all()
    kw = dict(max_iterations=20, max_correspondence_distance=0.05, transformation_epsilon=1e-10, euclidean_fitness_epsilon=1e-12)
    o, oc, od = orc.icp(src, tgt, orc.icp_params(**kw), want_corr=True, fixed=fixed)
    r = ref.icp(src, tgt, orc.icp_params(**kw), fixed=fixed)
    _same(o, r, oc)
    free = orc.icp(src, tgt, orc.icp_params(**kw))
    assert not np.array_equal(np.array(list(o.T)), np.array(list(free.T)))         # the pinned pairs do pull the estimate
    # with a rejector chain (nearest-neighbour estimator + surface-normal rejector): the fixed pairs appear twice
    sn, tn = orc.normals_knn(src, 12), orc.normals_knn(tgt, 12)
    ok_s, ok_t = np.isfinite(sn).all(1), np.isfinite(tn).all(1)
    assert ok_s.all() and ok_t.all()
    kw = dict(max_iterations=12, max_correspondence_distance=0.05, transformation_epsilon=1e-10, euclidean_fitness_epsilon=1e-12,
              rejectors=[(T.REJ_SURFACE_NORMAL, 0.2), (T.REJ_SELF_OCCLUDED_NORMAL, -2.0)])
    o, oc, od = orc.icp(src, tgt, orc.icp_params(**kw), src_normals=sn, tgt_normals=tn, want_corr=True, fixed=fixed)
    r = ref.icp(src, tgt, orc.icp_params(**kw), src_normals=sn, tgt_normals=tn, fixed=fixed)
    _same(o, r, oc)
