"""The CPU reference of RANSAC plane segmentation (tests/plane_reference.py, DESIGN.md §3.5) against hand-computed
SplitMix64 draws and planes, the strict threshold, the axis test on both sides of eps, the no-model cases and an
independent fp64 computation (numpy distances and numpy.linalg.eigh)."""
import math

import numpy as np

import plane_reference as ref

M64 = 2 ** 64 - 1
GOLDEN = 0x9E3779B97F4A7C15


def splitmix64(z: int) -> int:  # an independent restatement, in Python integers
    z &= M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def py_draws(seed: int, h: int, nf: int):
    return [((splitmix64(seed + (3 * h + s + 1) * GOLDEN) >> 32) * nf) >> 32 for s in range(3)]


def xyz1(a):
    a = np.asarray(a, np.float32).reshape(-1, 3)
    return np.c_[a, np.ones(len(a), np.float32)].astype(np.float32)


def test_splitmix_draws_by_hand():
    # SplitMix64 seeded with 0 starts 0xe220a8397b1dcdaf, 0x6e789e6aa1b965f4, 0x06c45d188009454f, 0xf88bb8a8724c81ec:
    # hypothesis 0 draws the first three, hypothesis 1 starts at the fourth.  With n_f = 2^32, j is the high word.
    j = ref.draws(2, 0, 2 ** 32)
    assert [int(x) for x in j[0]] == [0xE220A839, 0x6E789E6A, 0x06C45D18]
    assert int(j[1, 0]) == 0xF88BB8A8
    assert [int(x) for x in ref.draws(1, 0, 3)[0]] == [2, 1, 0]  # 0xe220a839 * 3 >> 32 = 2, ...
    for seed in (0, 1, 12345, 2 ** 64 - 1):  # (the last one wraps around)
        for nf in (3, 1000, 2 ** 31 - 1):
            got = ref.draws(50, seed, nf)
            for h in (0, 1, 49):
                assert [int(x) for x in got[h]] == py_draws(seed, h, nf), (seed, nf, h)


def test_plane_by_hand():
    # n_f = 3 and seed 0 draw j = (2, 1, 0): p0 = (0, 3, 1), u = p1 - p0 = (2, -3, 0), v = p2 - p0 = (0, -3, 0),
    # n = u x v = (0, 0, -6) -> (0, 0, -1), d = -(n . p0) = 1
    pts = xyz1([[0, 0, 1], [2, 0, 1], [0, 3, 1]])
    coef, s0, counts = ref.hypotheses(pts, 0.1, 1)
    assert coef[0].tolist() == [0.0, 0.0, -1.0, 1.0] and s0[0] == 2 and counts[0] == 3
    r = ref.segment(pts, 0.1, 1)
    assert r.hypothesis == 0 and r.inliers.tolist() == [0, 1, 2] and r.remainder.tolist() == []


def seed_drawing(nf: int) -> int:
    """the smallest seed whose hypothesis 0 draws positions 0, 1, 2 of F in some order"""
    for seed in range(1_000_000):
        if sorted(py_draws(seed, 0, nf)) == [0, 1, 2]:
            return seed
    raise AssertionError


def test_strict_threshold():
    t = np.float32(0.25)
    inside = np.nextafter(t, np.float32(0))
    pts = xyz1([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0.5, 0.5, t], [0.25, 0.75, inside], [0.5, 0.25, -t],
                [0.75, 0.5, -inside]])
    seed = seed_drawing(len(pts))
    coef, _, counts = ref.hypotheses(pts, float(t), 1, seed)
    assert np.abs(coef[0]).tolist() == [0.0, 0.0, 1.0, 0.0]
    assert counts[0] == 5  # the plane's three points and the two one fp32 step inside; the two at exactly t are out
    assert ref.inlier_flags(pts, coef[0], float(t)).tolist() == [True, True, True, False, True, False, True]


def test_axis_on_both_sides_of_eps():
    th = math.radians(10.0)
    # n_f = 3, seed 0: p0 = row 2, the plane's normal is (sin th, 0, cos th) up to sign
    pts = xyz1([[0, 0, 0], [0, 1, 0], [math.cos(th), 0, -math.sin(th)]])
    coef, _, _ = ref.hypotheses(pts, 0.1, 1)
    assert abs(abs(float(coef[0, 2])) - math.cos(th)) < 1e-6
    for axis in ([0, 0, 1], [0, 0, -3.5]):
        ok = ref.hypotheses(pts, 0.1, 1, axis=axis, eps_angle=th + 1e-6)[2]
        rejected = ref.hypotheses(pts, 0.1, 1, axis=axis, eps_angle=th - 1e-6)[2]
        assert ok[0] == 3 and rejected[0] == ref.INVALID
    assert ref.hypotheses(pts, 0.1, 1, axis=[0, 0, 1], eps_angle=math.pi / 2)[2][0] == 3
    assert ref.hypotheses(pts, 0.1, 1, axis=[0, 0, 1], eps_angle=0.0)[2][0] == ref.INVALID


def assert_no_model(pts, H=200, **kw):
    r = ref.segment(pts, 0.2, H, **kw)
    assert r.hypothesis == -1 and np.isnan(r.coefficients).all()
    assert len(r.inliers) == 0 and r.remainder.tolist() == list(range(len(pts)))
    assert (r.counts == ref.INVALID).all()


def test_no_model_cases():
    rs = np.random.RandomState(2)
    two = xyz1(rs.uniform(-1, 1, (5, 3)))
    two[[0, 2, 4], rs.randint(0, 3, 3)] = [np.nan, np.inf, -np.inf]
    assert len(ref.finite_indices(two)) == 2
    assert_no_model(two)
    assert_no_model(np.tile(xyz1([[1.25, -3.5, 0.75]]), (5000, 1)))
    s = rs.randint(-1000, 1000, 3000).astype(np.float64)
    assert_no_model(xyz1(np.c_[s, 2 * s + 1, -3 * s + 0.5]))  # exactly collinear (and duplicates among them)
    assert_no_model(xyz1(np.c_[rs.uniform(-5, 5, (2000, 2)), np.zeros(2000)]), axis=[1, 0, 0], eps_angle=0.1)
    assert_no_model(np.zeros((0, 4), np.float32))


def test_against_independent_fp64():
    """every hypothesis's sample, plane and count against numpy in fp64 on a plane with clutter: a count may differ from
    numpy's only by the points whose fp64 distance lies within 1e-3 relative of t, and those are rare"""
    rs = np.random.RandomState(5)
    g = np.c_[rs.uniform(-20, 20, (4000, 2)), rs.normal(0, 0.02, 4000)]
    clutter = rs.uniform([-20, -20, 0.5], [20, 20, 5], (1500, 3))
    pts = xyz1(np.r_[g, clutter][rs.permutation(5500)] + [3.0, -1.0, -1.7])
    t, H, seed = 0.05, 300, 77
    coef, s0, counts = ref.hypotheses(pts, t, H, seed)
    P = pts[:, :3].astype(np.float64)
    near = 0
    for h in range(H):
        j = py_draws(seed, h, len(pts))
        if len(set(j)) < 3:
            assert counts[h] == ref.INVALID
            continue
        p = P[j]
        n = np.cross(p[1] - p[0], p[2] - p[0])
        n /= np.linalg.norm(n)
        assert s0[h] == j[0]
        assert np.allclose(coef[h, :3].astype(np.float64), n, atol=1e-6)
        assert abs(float(coef[h, 3]) + n @ p[0]) < 1e-5
        dist = np.abs(P @ coef[h, :3].astype(np.float64) + float(coef[h, 3]))
        amb = np.abs(dist - t) < 1e-3 * t
        near += int(amb.sum())
        want = int((dist[~amb] < t).sum())
        assert want <= counts[h] <= want + int(amb.sum()), h
    assert near < 0.001 * H * len(pts)
    # selection and refinement: the best count wins, the refined normal is numpy's eigh of the inliers' covariance
    r = ref.segment(pts, t, H, seed)
    assert counts[r.hypothesis] == counts.max() and r.hypothesis == int(np.flatnonzero(counts == counts.max())[0])
    first = np.abs(P @ coef[r.hypothesis, :3].astype(np.float64) + float(coef[r.hypothesis, 3])) < t
    q = P[first]
    w, V = np.linalg.eigh(np.cov(q.T, bias=True))
    nrm = V[:, 0] * np.sign(V[:, 0] @ coef[r.hypothesis, :3])
    assert np.allclose(r.coefficients[:3], nrm, atol=1e-6)
    assert abs(float(r.coefficients[3]) + nrm @ q.mean(0)) < 1e-5
    assert abs(float(r.coefficients[2])) > 0.999 and abs(abs(float(r.coefficients[3])) - 1.7) < 0.01
    assert np.array_equal(r.inliers, np.flatnonzero(ref.inlier_flags(pts, r.coefficients, t)))
    assert len(r.inliers) + len(r.remainder) == len(pts)
