"""CPU checks of the Euclidean clustering reference (tests/cluster_reference.py) that the GPU clusters are compared with:
hand-computed cases (a chain at its spacing and one fp32 step below, a comb joined through one bridge point, size ties,
the size filter), agreement with an independent fp64 scipy computation on seeded clouds, and the corner cases of the
contract.  Also the argument checks of sycl_points_b200.EuclideanClustering, which run before anything touches the
device."""
import numpy as np
import pytest
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components
from scipy.spatial import cKDTree

import cluster_reference as ref


def xyz1(a):
    a = np.asarray(a, np.float32).reshape(-1, 3)
    return np.c_[a, np.ones(len(a), np.float32)].astype(np.float32)


def below(x):
    return float(np.nextafter(np.float32(x), np.float32(0.0)))


def test_chain_at_its_spacing_and_one_step_below():
    n = 40
    pts = xyz1(np.c_[0.25 * np.arange(n), np.zeros(n), np.zeros(n)])  # (exact in fp32: d^2 = 0.0625 = t * t)
    labels, indices, offsets = ref.clusters(pts, 0.25)
    assert labels.tolist() == [0] * n and indices.tolist() == list(range(n)) and offsets.tolist() == [0, n]
    # one step below: n singletons, equal sizes ordered by index
    labels, indices, offsets = ref.clusters(pts, below(0.25))
    assert labels.tolist() == list(range(n)) and indices.tolist() == list(range(n)) and offsets.tolist() == list(range(n + 1))


def comb():
    """three teeth of 4 points (x = 0, 1, 2; z = 0 ... 0.75) and one bridge point at (0.5, 0, 0), rows interleaved"""
    tooth = [[x, 0.0, 0.25 * k] for x in (0.0, 1.0, 2.0) for k in range(4)]  # rows 0-3, 4-7, 8-11 before the shuffle
    rows = tooth + [[0.5, 0.0, 0.0]]                                        # row 12: the bridge
    order = [8, 0, 4, 12, 9, 1, 5, 10, 2, 6, 11, 3, 7]
    return xyz1(np.asarray(rows)[order])


def test_comb_joined_through_one_bridge_point():
    pts = comb()
    # teeth 0 and 1 (rows 1, 5, 8, 11 and 2, 6, 9, 12) reach each other only through the bridge (row 3) at 0.5 m
    labels, indices, offsets = ref.clusters(pts, 0.5)
    big = [1, 2, 3, 5, 6, 8, 9, 11, 12]
    assert indices.tolist() == big + [0, 4, 7, 10] and offsets.tolist() == [0, 9, 13]
    assert [int(labels[i]) for i in range(13)] == [1 if i in (0, 4, 7, 10) else 0 for i in range(13)]
    # without the bridge: three teeth of 4, ordered by their smallest member (rows 0, 1, 2)
    pts[3, 0] = np.nan
    labels, indices, offsets = ref.clusters(pts, 0.5)
    assert labels[3] == -1 and offsets.tolist() == [0, 4, 8, 12]
    assert indices.tolist() == [0, 4, 7, 10, 1, 5, 8, 11, 2, 6, 9, 12]


def test_size_ties_and_the_size_filter():
    # blobs of sizes 3, 5, 3, 1, 5 centred 10 m apart, rows interleaved
    sizes = [3, 5, 3, 1, 5]
    owner = np.concatenate([np.full(s, b) for b, s in enumerate(sizes)])
    perm = np.random.RandomState(0).permutation(len(owner))
    owner = owner[perm]
    pts = xyz1(np.c_[10.0 * owner + 0.1 * (np.arange(len(owner)) % 3), np.zeros(len(owner)), np.zeros(len(owner))])
    first = {b: int(np.flatnonzero(owner == b)[0]) for b in range(5)}
    want = sorted(range(5), key=lambda b: (-sizes[b], first[b]))
    labels, indices, offsets = ref.clusters(pts, 0.25)
    assert [int(labels[first[b]]) for b in want] == list(range(5))
    assert offsets.tolist() == [0] + np.cumsum([sizes[b] for b in want]).tolist()
    for c, b in enumerate(want):
        assert indices[offsets[c]:offsets[c + 1]].tolist() == np.flatnonzero(owner == b).tolist()
    # min 2 drops the singleton, max 4 the two largest; min 4 max 4 keeps nothing
    for lo, hi, keep in ((2, 2 ** 31 - 1, [b for b in want if sizes[b] >= 2]), (1, 4, [b for b in want if sizes[b] <= 4]),
                         (4, 4, [])):
        labels, indices, offsets = ref.clusters(pts, 0.25, lo, hi)
        assert len(offsets) == len(keep) + 1
        for c, b in enumerate(keep):
            assert set(np.flatnonzero(labels == c)) == set(np.flatnonzero(owner == b))
        dropped = np.isin(owner, [b for b in range(5) if b not in keep])
        assert np.all(labels[dropped] == -1)


def blobs(seed, n=6000):
    rs = np.random.RandomState(seed)
    centres = rs.uniform(-20, 20, (40, 3))
    sd = rs.uniform(0.05, 0.6, 40)
    which = rs.randint(0, 40, n)
    return xyz1(centres[which] + rs.normal(0, 1, (n, 3)) * sd[which, None])


def clear_of(pts, t):
    """pts without the points that have a neighbour whose fp64 distance lies within 1e-3 relative of t (removing
    points creates no new pair, so every remaining pair is clear of the band)"""
    tree = cKDTree(pts[:, :3].astype(np.float64))
    pr = tree.query_pairs(t * (1 + 1e-3), output_type="ndarray")
    d = np.linalg.norm(pts[pr[:, 0], :3].astype(np.float64) - pts[pr[:, 1], :3], axis=1)
    near = np.zeros(len(pts), bool)
    near[pr[d >= t * (1 - 1e-3)].ravel()] = True
    return pts[~near]


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("t", [0.1, 0.3, 1.0])
def test_matches_independent_fp64_components(seed, t):
    pts = clear_of(blobs(seed), t)
    assert len(pts) > 5000
    labels, indices, offsets = ref.clusters(pts, t)
    pr = cKDTree(pts[:, :3].astype(np.float64)).query_pairs(t, output_type="ndarray")
    n = len(pts)
    _, comp = connected_components(coo_matrix((np.ones(len(pr)), (pr[:, 0], pr[:, 1])), shape=(n, n)), directed=False)
    # same partition, and labels ordered by (size desc, smallest member asc)
    for c in range(len(offsets) - 1):
        members = np.flatnonzero(labels == c)
        assert members.tolist() == indices[offsets[c]:offsets[c + 1]].tolist()
        assert set(np.flatnonzero(comp == comp[members[0]])) == set(members)
    sizes = np.diff(offsets.astype(np.int64))
    firsts = indices[offsets[:-1]]
    assert all((sizes[c], -firsts[c]) > (sizes[c + 1], -firsts[c + 1]) for c in range(len(sizes) - 1))
    assert len(sizes) == len(np.unique(comp)) and labels.min() == 0


def test_kdtree_candidates_agree_with_brute_force():
    pts = blobs(3, 5000)
    pts[::97, 1] = np.inf
    for t in (0.0, 0.2, below(0.2), 0.7):
        a, b = ref.edges(pts, t), ref.brute_edges(pts, t)
        assert np.array_equal(a[np.lexsort((a[:, 1], a[:, 0]))], b)


def test_corner_cases():
    assert [x.tolist() for x in ref.clusters(np.zeros((0, 4), np.float32), 1.0)] == [[], [], [0]]
    assert [x.tolist() for x in ref.clusters(np.full((5, 4), np.nan, np.float32), 1.0)] == [[-1] * 5, [], [0]]
    assert [x.tolist() for x in ref.clusters(xyz1([[1, 2, 3]]), 0.0)] == [[0], [0], [0, 1]]
    # t = 0 joins exact duplicates only (1e-30^2 underflows to 0 in fp32, so that pair counts as a duplicate)
    pts = xyz1([[0, 0, 0], [5, 0, 0], [0, 0, 0], [0, 0, 1e-30], [5, 0, 1e-3]])
    labels, indices, offsets = ref.clusters(pts, 0.0)
    assert labels.tolist() == [0, 1, 0, 0, 2] and offsets.tolist() == [0, 3, 4, 5]
    # a non-finite row between two clusters bridges nothing
    pts = xyz1([[0, 0, 0], [np.inf, 0, 0], [1, 0, 0], [0.5, np.nan, 0]])
    assert ref.clusters(pts, 0.6)[0].tolist() == [0, -1, 1, -1]


class _Cloud:
    def size(self):
        return 3


@pytest.mark.parametrize("kw", [dict(tolerance=-1.0), dict(tolerance=float("inf")), dict(tolerance=float("nan")),
                                dict(tolerance=1.0, min_cluster_size=0), dict(tolerance=1.0, min_cluster_size=5,
                                                                              max_cluster_size=4),
                                dict(tolerance=1.0, max_cluster_size=2 ** 32), dict(tolerance=1.0, min_cluster_size=1.5),
                                dict(tolerance=1.0, min_cluster_size=True)])
def test_argument_checks(kw):
    from sycl_points_b200 import EuclideanClustering
    with pytest.raises(ValueError):
        EuclideanClustering(None).extract(_Cloud(), **kw)
