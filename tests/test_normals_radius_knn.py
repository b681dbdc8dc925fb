"""The CPU references for k-NN with k above 32 (the oracle's orc_knn) and for radius-based normal estimation (orc_radius.py),
against numpy restatements, on clouds built to
reach their edge cases: neighbours at exactly the radius (the strict d2 < r2), duplicates, 0 to 3 neighbours, NaN and inf points and
a 100 m offset. These are the references tests/test_gpu_normals_radius_knn.py holds the device to."""
import numpy as np
import pytest

import orc_radius

H = 0.25   # a power of two: squared distances between lattice points are exact in float, so d2 == r2 happens exactly


def _lattice(nx, ny, nz, h=H):
    g = np.stack(np.meshgrid(np.arange(nx), np.arange(ny), np.arange(nz), indexing="ij"), -1).reshape(-1, 3)
    return (g * h).astype(np.float32)


def exact_radius():
    """A lattice plus duplicates, shuffled: with r = h, every lattice neighbour sits at exactly d2 == r2 and is left out."""
    rng = np.random.default_rng(301)
    lat = _lattice(6, 6, 3)
    pts = np.concatenate([lat, lat[rng.choice(len(lat), 20, replace=False)]])
    return pts[rng.permutation(len(pts))]


def small_groups():
    """Groups 2 m apart of 1, 2, 3 and 4 points (0.1 m spread: within r = 0.5 of each other), and NaN / inf rows (no neighbour
    at all): every query has 0, 1, 2, 3 or 4 neighbours."""
    rng = np.random.default_rng(302)
    groups = [np.float32([2 * g, 0, 0]) + rng.uniform(0, 0.1, (g, 3)).astype(np.float32) for g in (1, 2, 3, 4)]
    bad = np.float32([[np.nan, 0, 0], [0, np.inf, 0], [-np.inf, np.nan, 1]])
    pts = np.concatenate(groups + [bad])
    return pts[rng.permutation(len(pts))]


def noisy_offset():
    """A noisy plate with duplicates, 100 m from the origin."""
    rng = np.random.default_rng(303)
    p = rng.uniform(0, 0.3, (700, 3)).astype(np.float32)
    p[:, 2] = rng.normal(0, 0.003, 700).astype(np.float32)
    p = np.concatenate([p, p[:40]])
    return p + np.float32([100, -100, 100])


def cases():
    # (name, points, radius, viewpoint)
    return [("exact_radius", exact_radius(), H, (0, 0, 0)), ("small_groups", small_groups(), 0.5, (0, 0, 5)),
            ("offset", noisy_offset(), 0.05, (100, -100, 101))]


def _d2(pts, q):
    """FLANN L2_Simple in float32: ((dx*dx + dy*dy) + dz*dz), left to right, no FMA."""
    d = (pts[:, :3] - q[None, :3]).astype(np.float32)
    return (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]


def _finite(pts):
    return np.isfinite(pts[:, :3]).all(1)


def _sorted_neighbours(pts, q, keep):
    """indices with `keep`, ascending (d2, index)"""
    d2 = _d2(pts, q)
    idx = np.nonzero(keep(d2) & _finite(pts))[0]
    order = np.lexsort((idx, d2[idx]))
    return idx[order], d2[idx][order]


def knn_restated(tgt, qry, k):
    idx = np.full((len(qry), k), -1, np.int32)
    d2 = np.full((len(qry), k), np.inf, np.float32)
    for i, q in enumerate(qry):
        ni, nd = _sorted_neighbours(tgt, q, lambda d: np.ones(len(d), bool))
        ni, nd = ni[:k], nd[:k]
        idx[i, :len(ni)] = ni
        d2[i, :len(nd)] = nd
    return idx, d2


def radius_sets(pts, r):
    r2 = np.float32(r) * np.float32(r)
    return [(_sorted_neighbours(pts, q, lambda d: d < r2) if np.isfinite(q).all() else (np.zeros(0, int), np.zeros(0, np.float32)))
            for q in pts[:, :3]]


def covariance_restated(pts, nbr):
    """computeMeanAndCovarianceMatrix: nine float32 sums, serial in the neighbour order, divided by the count"""
    acc = np.zeros(9, np.float32)
    for j in nbr:
        x, y, z = pts[j, :3]
        acc += np.float32([x * x, x * y, x * z, y * y, y * z, z * z, x, y, z])
    acc /= np.float32(len(nbr))
    m = acc[6:]
    c = np.empty((3, 3), np.float32)
    c[0, 0] = acc[0] - m[0] * m[0]; c[0, 1] = c[1, 0] = acc[1] - m[0] * m[1]; c[0, 2] = c[2, 0] = acc[2] - m[0] * m[2]
    c[1, 1] = acc[3] - m[1] * m[1]; c[1, 2] = c[2, 1] = acc[4] - m[1] * m[2]; c[2, 2] = acc[5] - m[2] * m[2]
    return c


# ------------------------------------------------------------------------------------------------------- k-NN ----
@pytest.mark.parametrize("k", [33, 64, 256])
@pytest.mark.parametrize("name", ["exact_radius", "small_groups", "offset"])
def test_orc_knn_above_32_equals_numpy(orc, name, k):
    pts = dict((c[0], c[1]) for c in cases())[name]
    for brute in (False, True):
        idx, d2 = orc.knn(pts, pts, k, brute=brute)
        ridx, rd2 = knn_restated(pts, pts, k)
        np.testing.assert_array_equal(idx, ridx)
        np.testing.assert_array_equal(d2, rd2)
    n_fin = int(_finite(pts).sum())
    assert (idx[0] >= 0).sum() == min(k, n_fin) if np.isfinite(pts[0]).all() else True


# ----------------------------------------------------------------------------------------------- radius normals ----
@pytest.mark.parametrize("name", ["exact_radius", "small_groups", "offset"])
def test_orc_normals_radius_equals_numpy(orc, name):
    _, pts, r, vp = [c for c in cases() if c[0] == name][0]
    got = orc_radius.normals_radius(pts, r, vp)
    sets = radius_sets(pts, r)
    off, oidx, _ = orc.radius(pts, pts, r)
    for i, (ni, _) in enumerate(sets):
        finite_q = np.isfinite(pts[i]).all()
        if finite_q:   # the tree's radius set is numpy's set
            assert sorted(oidx[off[i]:off[i + 1]].tolist()) == sorted(ni.tolist()), i
        if not finite_q or len(ni) < 3:
            assert np.isnan(got[i]).all(), i
            continue
        # the oracle's own k-NN normal with k = the set's size sums the same points in the same order: the same bits
        assert np.array_equal(orc.normals_knn(pts, len(ni), vp)[i].view(np.uint32), got[i].view(np.uint32)), i
        c = covariance_restated(pts, ni)
        w, v = np.linalg.eigh(c.astype(np.float64))
        n = v[:, 0]
        if np.dot(np.float64(vp) - pts[i].astype(np.float64), n) < 0:
            n = -n
        # the float32 sums hold the covariance to about ulp(max |p|^2): only where that is well below the eigenvalue gaps (not at
        # the 100 m offset, where it is all rounding, as in PCL) do the direction and curvature mean something to compare
        noise = 1e-6 * len(ni) * float(np.abs(pts[ni, :3]).max()) ** 2
        s = c[0, 0] + c[1, 1] + c[2, 2]
        if w[1] - w[0] > noise:
            assert np.abs(got[i, :3] - n).max() < 2e-3, (i, got[i], n)
        if s > 100 * noise:
            assert abs(got[i, 3] - abs(w[0] / s)) < 1e-3, i   # float32 rounding of a rank-2 covariance reaches ~4e-4 here


def test_cases_reach_their_edges(orc):
    pts = exact_radius()
    sets = radius_sets(pts, H)
    # neighbours at exactly d2 == r2 exist and are left out
    q = pts[0]
    assert (_d2(pts, q) == np.float32(H) * np.float32(H)).any()
    assert all(np.all(d < np.float32(H * H)) for _, d in sets)
    # duplicates: some sets hold a zero-distance pair other than the query itself
    assert any((d == 0).sum() >= 2 for _, d in sets)
    counts = {len(ni) for ni, _ in radius_sets(small_groups(), 0.5)}
    assert {0, 1, 2, 3, 4} <= counts
    off = noisy_offset()
    assert np.abs(off).min() > 99
    assert max(len(ni) for ni, _ in radius_sets(off, 0.05)) > 32
