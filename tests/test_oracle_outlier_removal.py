"""CPU checks of the outlier-removal reference (tests/outlier_reference.py) that the GPU filters are compared with:
a hand-computed case, agreement with an independent scipy cKDTree computation on seeded clouds, and the corner cases
of the contract (self-exclusion with duplicates, n <= k, non-finite rows, min_neighbors = 0, radius = 0).  Also the
argument checks of sycl_points_b200.OutlierRemoval, which run before anything touches the device."""
import math

import numpy as np
import pytest
from scipy.spatial import cKDTree

import outlier_reference as ref


def xyz1(a):
    a = np.asarray(a, np.float32).reshape(-1, 3)
    return np.c_[a, np.ones(len(a), np.float32)].astype(np.float32)


def square_and_far_point():
    return xyz1([[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0], [10, 0, 0]])


def test_hand_computed_square_and_far_point():
    # k = 2: a corner's two nearest others are its edge neighbours at 1 m -> d = 1.  The far point's are (1, 0) at 9 m
    # and (1, 1) at sqrt(82) m -> d = (9 + sqrt(82)) / 2 = 9.0276926.  mu = (4 + d) / 5, sigma from PCL's formula.
    keep, dbar, mu, sigma, thr = ref.statistical(square_and_far_point(), 2, 1.0)
    d_far = np.float32((np.float32(9.0) + np.sqrt(np.float32(82.0))) / np.float32(2.0))
    assert dbar.tolist() == [1.0, 1.0, 1.0, 1.0, float(d_far)]
    s1, s2 = 4.0 + float(d_far), 4.0 + float(d_far) ** 2
    assert mu == pytest.approx(s1 / 5, rel=1e-15) and mu == pytest.approx(2.6055385, rel=1e-7)
    assert sigma == pytest.approx(math.sqrt((s2 - s1 * s1 / 5) / 4), rel=1e-15) and sigma == pytest.approx(3.5900933, rel=1e-7)
    assert thr == pytest.approx(6.1956318, rel=1e-7)
    assert keep.tolist() == [True, True, True, True, False]
    # radius 1 m: each corner has its two edge neighbours at exactly 1 m (d^2 = 1 <= 1), the far point none
    assert ref.radius(square_and_far_point(), 1.0, 2).tolist() == [True, True, True, True, False]
    assert ref.radius(square_and_far_point(), 1.0, 3).tolist() == [False] * 5
    assert ref.radius(square_and_far_point(), 9.0, 1).tolist() == [True] * 5


def seeded_cloud(seed, n=3000):
    rs = np.random.RandomState(seed)
    blobs = np.concatenate([rs.normal(c, s, (n // 4, 3)) for c, s in (((0, 0, 0), 0.3), ((5, 1, 0), 0.6), ((-3, 4, 1), 1.0))])
    noise = rs.uniform(-10, 10, (n - len(blobs), 3))
    return xyz1(np.concatenate([blobs, noise]))


def independent_mean_distances(pts, k):
    """fp64 cKDTree version of step 1-2 (no duplicates in these clouds: the zero-distance entry is the point itself)"""
    t = cKDTree(pts[:, :3].astype(np.float64))
    d, i = t.query(pts[:, :3].astype(np.float64), k + 1)
    d, i = d.reshape(len(pts), -1), i.reshape(len(pts), -1)
    own = i == np.arange(len(pts))[:, None]
    drop = np.where(own.any(1), own.argmax(1), k)
    keep = np.ones_like(own)
    keep[np.arange(len(pts)), drop] = False
    return (d * keep).sum(1) / k


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("k", [1, 5, 20])
def test_statistical_matches_independent_kdtree(seed, k):
    pts = seeded_cloud(seed)
    indep = independent_mean_distances(pts, k)
    for alpha in (-0.5, 0.0, 1.0, 2.0):
        keep, dbar, mu, sigma, thr = ref.statistical(pts, k, alpha)
        np.testing.assert_allclose(dbar, indep, rtol=2e-6)
        mu_i, sd_i = indep.mean(), indep.std(ddof=1)
        thr_i = mu_i + alpha * sd_i
        assert thr == pytest.approx(thr_i, rel=1e-5)
        near = (np.abs(dbar - thr) <= 1e-9 * abs(thr)) | (np.abs(indep - thr_i) <= 1e-9 * abs(thr_i))
        assert near.sum() == 0
        assert np.array_equal(keep[~near], (indep <= thr_i)[~near])
        assert 0 < keep.sum() < len(pts)


@pytest.mark.parametrize("seed", [3, 4])
def test_radius_matches_independent_kdtree(seed):
    pts = seeded_cloud(seed)
    t = cKDTree(pts[:, :3].astype(np.float64))
    for r in (0.1, 0.5, 2.0):
        lo = t.query_ball_point(pts[:, :3].astype(np.float64), r * (1 - 5e-10), return_length=True) - 1
        hi = t.query_ball_point(pts[:, :3].astype(np.float64), r * (1 + 5e-10), return_length=True) - 1
        near = lo != hi  # a neighbour within 1e-9 relative of r^2
        for m in (0, 1, 5, 40):
            keep = ref.radius(pts, r, m)
            assert np.array_equal(keep[~near], (lo >= m)[~near]), (r, m)


def test_self_exclusion_with_duplicates():
    a = [0.5, -1.0, 2.0]
    pts = xyz1([a, [3, 3, 3], a, a, [3, 3, 4], a, a])  # five copies of a at rows 0, 2, 3, 5, 6
    # k = 2: every copy's two nearest others are copies at distance 0 (for rows 5 and 6 the k + 1 = 3 nearest are
    # rows 0, 2, 3: the point itself is not listed and the last entry is dropped)
    dbar = ref.mean_distances(pts, 2)
    assert dbar[[0, 2, 3, 5, 6]].tolist() == [0.0] * 5
    # rows 1 and 4: the other one at 1 m, then the lowest-index copy of a (d^2 = 23.25 and 26.25, exact in fp32)
    assert dbar[1] == (np.float32(1.0) + np.sqrt(np.float32(23.25))) / np.float32(2.0)
    assert dbar[4] == (np.float32(1.0) + np.sqrt(np.float32(26.25))) / np.float32(2.0)
    # duplicates count as others for the radius filter; at r = 0 they are the only ones
    assert ref.radius(pts, 0.0, 4).tolist() == [True, False, True, True, False, True, True]
    assert ref.radius(pts, 0.0, 5).tolist() == [False] * 7
    assert ref.radius(pts, 1.0, 1).tolist() == [True] * 7  # rows 1 and 4 are 1 m apart


def test_mean_distance_of_the_isolated_rows_by_hand():
    pts = xyz1([[0, 0, 0], [3, 0, 0], [3, 4, 0]])
    # n <= k: k = 5 leaves two others per point
    dbar = ref.mean_distances(pts, 5)
    assert dbar.tolist() == [np.float32((3 + 5) / 2), np.float32((3 + 4) / 2), np.float32((4 + 5) / 2)]
    keep, _, mu, sigma, thr = ref.statistical(pts, 5, 0.0)
    assert mu == pytest.approx(4.0) and keep.tolist() == [True, True, False]


def test_single_valid_point_keeps_it_and_empty_cloud():
    keep, dbar, mu, sigma, thr = ref.statistical(xyz1([[1, 2, 3]]), 3, -2.0)
    assert np.isnan(dbar[0]) and keep.tolist() == [False]  # no other point: invalid
    keep, dbar, mu, sigma, thr = ref.statistical(xyz1([[1, 2, 3], [1, 2, 4]]), 3, -2.0)
    assert sigma == 0.0 and thr == mu and keep.tolist() == [True, True]  # equal means: the variance is 0
    keep, dbar, *_ = ref.statistical(np.zeros((0, 4), np.float32), 3, 1.0)
    assert len(keep) == 0 and len(dbar) == 0
    assert len(ref.radius(np.zeros((0, 4), np.float32), 1.0, 1)) == 0


def test_non_finite_rows_are_removed_and_ignored():
    pts = seeded_cloud(5, 600)
    bad = pts.copy()
    rows = [3, 50, 51, 200, 599]
    for r, v in zip(rows, [np.nan, np.inf, -np.inf, np.nan, np.inf]):
        bad[r, r % 3] = v
    good = np.setdiff1d(np.arange(len(pts)), rows)
    for k in (1, 8):
        keep, dbar, mu, sigma, thr = ref.statistical(bad, k, 1.0)
        keep2, dbar2, mu2, sigma2, thr2 = ref.statistical(pts[good], k, 1.0)
        assert np.isnan(dbar[rows]).all() and not keep[rows].any()
        assert np.array_equal(dbar[good], dbar2) and (mu, sigma) == (mu2, sigma2)
        assert np.array_equal(keep[good], keep2)
    for r, m in ((0.5, 1), (2.0, 6), (1.0, 0)):
        keep = ref.radius(bad, r, m)
        assert not keep[rows].any()
        assert np.array_equal(keep[good], ref.radius(pts[good], r, m))
    assert ref.radius(bad, 1.0, 0).sum() == len(good)  # m = 0 keeps every finite point


def test_radius_zero_counts_exact_duplicates_only():
    pts = xyz1([[0, 0, 0], [0, 0, 1e-30], [0, 0, 0], [1, 1, 1]])
    assert ref.radius(pts, 0.0, 1).tolist() == [True, True, True, False]  # 1e-30^2 underflows to 0 in fp32
    pts = xyz1([[0, 0, 0], [0, 0, 1e-3], [0, 0, 0], [1, 1, 1]])
    assert ref.radius(pts, 0.0, 1).tolist() == [True, False, True, False]


class _Cloud:
    def size(self):
        return 3


@pytest.mark.parametrize("kw", [dict(mean_k=0, stddev_mul=1.0), dict(mean_k=128, stddev_mul=1.0),
                                dict(mean_k=2.0, stddev_mul=1.0), dict(mean_k=4, stddev_mul=float("nan")),
                                dict(mean_k=4, stddev_mul=float("inf"))])
def test_statistical_argument_checks(kw):
    from sycl_points_b200 import OutlierRemoval
    with pytest.raises(ValueError):
        OutlierRemoval(None).statistical(_Cloud(), **kw)


@pytest.mark.parametrize("kw", [dict(radius=-1.0, min_neighbors=1), dict(radius=float("inf"), min_neighbors=1),
                                dict(radius=float("nan"), min_neighbors=1), dict(radius=1.0, min_neighbors=-1),
                                dict(radius=1.0, min_neighbors=2 ** 32), dict(radius=1.0, min_neighbors=1.5)])
def test_radius_argument_checks(kw):
    from sycl_points_b200 import OutlierRemoval
    with pytest.raises(ValueError):
        OutlierRemoval(None).radius(_Cloud(), **kw)
