"""The CPU reference of FPFH, feature correspondences and correspondence RANSAC (tests/global_reference.py) against
hand-computed cases and independent fp64 numpy computations: pair features and bins (the swap branch, skipped parallel
pairs, the (0, 0) and X < 0, Y = +-0 corners, points on every boundary ray), sector bins against numpy's arctan2,
FPFH against an fp64 numpy FPFH, triad poses against SVD Kabsch, the edge check at its boundary, the sampler against
the plane RANSAC's, and the brute-force feature search.  No GPU."""
import numpy as np
import pytest
from scipy.spatial import cKDTree

import global_reference as ref
import plane_reference


# ------------------------------------------------------------------ pair features and bins
def test_pair_feature_by_hand():
    z = [0.0, 0.0, 1.0]
    # no swap: u = n_i, v = e x u = (0, -1, 0), w = (1, 0, 0); X = 1, Y = 0 (bin 5), f2 = 0, f3 = 0
    f, b = ref.pair_feature([0, 0, 0], z, [1, 0, 0], z)
    assert f.tolist() == [0.0, 0.0, 1.0, 0.0, 0.0] and b.tolist() == [5, 5, 5]
    # swap (|a_i| = 0.5 < |a_j| = 1): u = n_j, o = n_i, e = -dp; v = (0, -1, 0), w = (0, 0, -1): X = 0, Y = -1
    # (theta = -pi/2, bin 2); f3 = -1 / sqrt(1.25) (bin 0)
    f, b = ref.pair_feature([0, 0, 0], z, [1, 0, 0.5], [1, 0, 0])
    assert f[4] == 1.0 and f[0] == 0.0 and f[2] == 0.0 and f[3] == -1.0
    assert abs(f[1] + 1 / np.sqrt(1.25)) < 1e-7 and b.tolist() == [2, 5, 0]
    # parallel: dp along u = n_i = n_j gives v = 0, the pair is skipped
    assert ref.pair_feature([0, 0, 0], z, [0, 0, 2], z) is None


def test_angle_bin_corners_and_rays():
    assert ref.angle_bin(0.0, 0.0) == 5 and ref.angle_bin(-0.0, -0.0) == 5
    assert ref.angle_bin(-1.0, 0.0) == 10 and ref.angle_bin(-1.0, -0.0) == 10
    assert ref.angle_bin(1.0, -0.0) == 5 and ref.angle_bin(1.0, 0.0) == 5
    # a point exactly on boundary ray k (the fp32 constants) falls in bin k; one fp32 step clockwise in bin k - 1
    for k in range(1, 11):
        a = -np.pi + 2 * np.pi * k / 11
        c, s = np.float32(np.cos(a)), np.float32(np.sin(a))
        assert ref.angle_bin(c, s) == k, k
        for scale in (np.float32(4.0), np.float32(0.25)):  # (powers of two: still exactly on the ray)
            assert ref.angle_bin(c * scale, s * scale) == k, (k, scale)
        # rotate by -1e-6 rad: below the ray
        e = -1e-6
        X, Y = np.float32(c * np.cos(e) - s * np.sin(e)), np.float32(c * np.sin(e) + s * np.cos(e))
        assert ref.angle_bin(X, Y) == k - 1, k


def test_angle_bins_equal_numpy_arctan2_away_from_boundaries():
    rng = np.random.default_rng(1)
    XY = rng.normal(size=(200_000, 2)).astype(np.float32)
    XY[:1000] *= np.float32(1e-20)
    XY[1000:2000] *= np.float32(1e20)
    th = np.arctan2(XY[:, 1].astype(np.float64), XY[:, 0].astype(np.float64))
    want = np.clip(np.floor(11 * (th + np.pi) / (2 * np.pi)), 0, 10).astype(int)
    bounds = -np.pi + 2 * np.pi * np.arange(1, 11) / 11
    far = np.min(np.abs(th[:, None] - bounds[None, :]), axis=1) > 1e-5
    got = np.array([ref.angle_bin(x, y) for x, y in XY[far]])
    assert far.sum() > 199_000 and np.array_equal(got, want[far])


# ------------------------------------------------------------------ FPFH against fp64 numpy
def radius_lists(p, r, k):
    """(idx int32 (n, k), dist float32 (n, k)): the k nearest within r ascending by (d^2, idx), -1 / FLT_MAX padded"""
    P = p[:, :3].astype(np.float32)
    n = len(P)
    idx = np.full((n, k), -1, np.int32)
    dist = np.full((n, k), np.finfo(np.float32).max, np.float32)
    Q = np.where(np.isfinite(P).all(1, keepdims=True), P, np.float32(1e6)).astype(np.float64)  # (never listed)
    for i, nb in enumerate(cKDTree(Q).query_ball_point(Q, r * 1.001)):
        nb = np.asarray(nb, np.int64)
        d = P[nb] - P[i]
        d2 = (d[:, 2] * d[:, 2] + (d[:, 1] * d[:, 1] + d[:, 0] * d[:, 0])).astype(np.float32)
        keep = d2 <= np.float32(r) * np.float32(r)
        nb, d2 = nb[keep], d2[keep]
        o = np.lexsort((nb, d2))[:k]
        idx[i, :len(o)], dist[i, :len(o)] = nb[o], d2[o]
    return idx, dist


def fpfh64(p, nrm, idx, dist):
    """independent fp64 FPFH: (rows, unsafe) with unsafe[i] when a feature of a pair it depends on lies within 2e-5 (in bin units) of
    a bin boundary (where fp32 and fp64 may bin differently)"""
    P, N = p[:, :3].astype(np.float64), nrm[:, :3].astype(np.float64)
    n, k = idx.shape
    valid = np.isfinite(P).all(1) & np.isfinite(N).all(1)
    S = np.zeros((n, 33))
    near = np.zeros(n, bool)
    for i in range(n):
        if not valid[i]:
            continue
        cnt, m = np.zeros(33), 0
        for r in range(k):
            j = idx[i, r]
            if j < 0 or j == i or not dist[i, r] > 0 or not valid[j]:
                continue
            dp = P[j] - P[i]
            ai, aj = N[i] @ dp, N[j] @ dp
            if abs(ai) < abs(aj):
                u, o, e, f3 = N[j], N[i], -dp, -aj / np.linalg.norm(dp)
            else:
                u, o, e, f3 = N[i], N[j], dp, ai / np.linalg.norm(dp)
            v = np.cross(e, u)
            if np.linalg.norm(v) < 1e-6 * np.linalg.norm(e):
                near[i] = True
                continue
            v /= np.linalg.norm(v)
            w = np.cross(u, v)
            th = np.arctan2(w @ o, u @ o)
            f2 = v @ o
            x1, x2, x3 = 11 * (th + np.pi) / (2 * np.pi), (f2 + 1) * 5.5, (f3 + 1) * 5.5
            near[i] |= any(abs(x - np.round(x)) < 2e-5 for x in (x1, x2, x3)) or abs(ai) - abs(aj) == 0
            cnt[int(np.clip(np.floor(x1), 0, 10))] += 1
            cnt[11 + int(np.clip(np.floor(x2), 0, 10))] += 1
            cnt[22 + int(np.clip(np.floor(x3), 0, 10))] += 1
            m += 1
        S[i] = cnt * (100.0 / m) if m else 0.0
    F = np.full((n, 33), np.nan)
    unsafe = near.copy()
    for i in range(n):
        if not valid[i]:
            continue
        acc = np.zeros(33)
        for r in range(k):
            j = idx[i, r]
            if j < 0 or j == i or not dist[i, r] > 0 or not valid[j]:
                continue
            acc += S[j] / float(dist[i, r])
            unsafe[i] |= near[j]
        F[i] = S[i]
        for g in range(3):
            s = acc[11 * g:11 * g + 11].sum()
            if s > 0:
                F[i, 11 * g:11 * g + 11] += acc[11 * g:11 * g + 11] * (100.0 / s)
    return F, unsafe


def surface_cloud(n=600, seed=3):
    rng = np.random.default_rng(seed)
    xy = rng.uniform(-3, 3, (n, 2))
    z = 0.3 * np.sin(xy[:, 0]) * np.cos(0.7 * xy[:, 1])
    p = np.c_[xy, z, np.ones(n)].astype(np.float32)
    g = np.c_[-0.3 * np.cos(xy[:, 0]) * np.cos(0.7 * xy[:, 1]), 0.21 * np.sin(xy[:, 0]) * np.sin(0.7 * xy[:, 1]),
              np.ones(n)]
    g /= np.linalg.norm(g, axis=1, keepdims=True)
    g += rng.normal(0, 0.05, g.shape)
    g /= np.linalg.norm(g, axis=1, keepdims=True)
    nrm = np.c_[g, np.zeros(n)].astype(np.float32)
    return p, nrm


def test_fpfh_equals_fp64_numpy():
    p, nrm = surface_cloud()
    p[5, 0] = np.nan
    nrm[9, 1] = np.inf
    p[17] = p[16]  # an exact duplicate
    idx, dist = radius_lists(p, 0.7, 40)
    F = ref.fpfh(p, nrm, idx, dist)
    F64, unsafe = fpfh64(p, nrm, idx, dist)
    assert np.isnan(F[5]).all() and np.isnan(F[9]).all()
    ok = np.isfinite(F64).all(1) & ~unsafe
    assert ok.sum() > 0.5 * len(p), ok.sum()
    np.testing.assert_allclose(F[ok], F64[ok], rtol=1e-4, atol=1e-4)
    # a finite row is the point's three normalised histograms plus its neighbours' three: it sums to 600
    s = F[np.isfinite(F).all(1)].sum(1)
    assert np.all(np.abs(s - 600) < 1e-2)


def test_isolated_point_has_zero_row():
    p = np.array([[0, 0, 0, 1], [10, 0, 0, 1]], np.float32)
    nrm = np.array([[0, 0, 1, 0], [0, 0, 1, 0]], np.float32)
    idx, dist = radius_lists(p, 1.0, 4)
    assert not ref.fpfh(p, nrm, idx, dist).any()


# ------------------------------------------------------------------ feature search
def test_feature_nn_ties_nan_and_mutual():
    rng = np.random.default_rng(4)
    s = rng.normal(size=(50, 33)).astype(np.float32)
    t = rng.normal(size=(70, 33)).astype(np.float32)
    d = ((s[:, None].astype(np.float64) - t[None].astype(np.float64)) ** 2).sum(-1)
    assert np.array_equal(ref.feature_nn(s, t), d.argmin(1))
    t2 = np.repeat(t[:5], 3, axis=0)  # equal rows: the lowest index wins
    nn = ref.feature_nn(s, t2)
    assert np.all(nn % 3 == 0)
    t3 = t.copy()
    t3[::2] = np.nan  # NaN rows never win; a NaN source row has no candidate
    s3 = s.copy()
    s3[7] = np.nan
    nn = ref.feature_nn(s3, t3)
    assert nn[7] == -1 and np.all(nn[np.arange(50) != 7] % 2 == 1)
    i, j = ref.correspondences(s, t, mutual=True)
    back = d.argmin(0)
    assert np.array_equal(i, np.flatnonzero(back[d.argmin(1)] == np.arange(50))) and np.array_equal(j, d.argmin(1)[i])


# ------------------------------------------------------------------ RANSAC pieces
def rot(axis, deg):
    a = np.deg2rad(deg)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]], np.float64)
    K /= np.linalg.norm(axis)
    return np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K


def test_triad_equals_svd_kabsch_on_noise_free_triples():
    rng = np.random.default_rng(5)
    for _ in range(200):
        R = rot(rng.normal(size=3), rng.uniform(-180, 180))
        t = rng.uniform(-20, 20, 3)
        p = rng.uniform(-30, 30, (3, 3)).astype(np.float32)
        q = (p.astype(np.float64) @ R.T + t).astype(np.float32)
        P64 = ref.triad(p, q, fp64=True)
        Rk, tk = ref.kabsch(p, q)
        # q is rounded to fp32: the two fits agree to that rounding
        assert np.abs(P64[:, :3] - Rk).max() < 1e-9 * 1e3 and np.abs(P64[:, 3] - tk).max() < 1e-9 * 1e4
        assert np.array_equal(ref.triad(p, q), P64.astype(np.float32))
    # exactly representable: a 90 degree turn about z of an integer triangle, recovered to 1e-9
    p = np.array([[0, 0, 0], [2, 0, 0], [0, 3, 1]], np.float32)
    q = np.array([[5, 1, 0], [5, 3, 0], [2, 1, 1]], np.float32)
    Rz = np.array([[0, -1, 0], [1, 0, 0], [0, 0, 1]], np.float64)
    P64 = ref.triad(p, q, fp64=True)
    Rk, tk = ref.kabsch(p, q)
    assert np.abs(P64[:, :3] - Rz).max() < 1e-9 and np.abs(P64[:, 3] - [5, 1, 0]).max() < 1e-9
    assert np.abs(Rk - Rz).max() < 1e-9 and np.abs(tk - [5, 1, 0]).max() < 1e-9
    # collinear or repeated vertices are degenerate
    assert ref.triad(np.array([[0, 0, 0], [1, 1, 1], [2, 2, 2]], np.float32), q) is None
    assert ref.triad(p, np.array([[1, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32)) is None


def test_edge_check_at_its_boundary():
    p = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32)
    q = 2 * p
    assert ref.edges_ok(p, q, 0.5)  # ds^2 = tau^2 dt^2 exactly: kept
    assert ref.edges_ok(q, p, 0.5)
    up = np.nextafter(np.float32(2), np.float32(3))
    assert not ref.edges_ok(p, p * up, 0.5)
    assert ref.edges_ok(p, p, 1.0) and not ref.edges_ok(p, p * up, 1.0)


def test_draws_equal_the_plane_sampler():
    for seed, m in ((0, 1000), (12345, 7), (2 ** 64 - 1, 2 ** 31 - 1)):
        assert np.array_equal(ref.draws(5000, seed, m), plane_reference.draws(5000, seed, m))


def test_ransac_recovers_a_pose_among_outliers():
    rng = np.random.default_rng(6)
    R, t = rot([0.1, 0.2, 1.0], 130.0), np.array([6.0, -3.0, 0.5])
    src = np.c_[rng.uniform(-20, 20, (400, 3)), np.ones(400)].astype(np.float32)
    tgt = src.copy()
    tgt[:, :3] = (src[:, :3].astype(np.float64) @ R.T + t).astype(np.float32)
    si = np.arange(400, dtype=np.int32)
    ti = si.copy()
    bad = rng.random(400) < 0.7
    ti[bad] = rng.integers(0, 400, bad.sum())
    r = ref.ransac(src, tgt, si, ti, 0.1, 3000, seed=1, optimize=True)
    assert r.hypothesis >= 0 and np.abs(r.pose[:, :3] - R).max() < 1e-5 and np.abs(r.pose[:, 3] - t).max() < 1e-4
    assert set(np.flatnonzero(~bad)) <= set(r.inliers.tolist())
    # M < 3 and M = 0: no model
    assert ref.ransac(src, tgt, si[:2], ti[:2], 0.1, 50).hypothesis == -1
    assert ref.ransac(src, tgt, si[:0], ti[:0], 0.1, 50).hypothesis == -1
