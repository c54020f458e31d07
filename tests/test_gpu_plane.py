"""RANSAC plane segmentation on the GPU (sycl_points_b200.PlaneSegmentation, spx_plane_segment) against the CPU
reference of tests/plane_reference.py.  Without refinement every hypothesis's count, the chosen hypothesis, the
coefficients bit for bit, the inliers and the remainder are equal on a drive revolution with its ground (level and
tilted, with and without an axis), far clouds, non-finite rows, a lattice at t, tiny clouds and the ~2 M-point raw
cloud.  With refinement the coefficients agree to 1 fp32 ulp and the inliers up to points within the coefficients'
difference of t.  Ground removal before clustering, determinism, gathered attributes and the C-ABI's argument checks."""
import ctypes as C
import math

import numpy as np
import pytest

import cluster_reference as cref
import plane_reference as ref
import synthetic
from test_gpu_outlier_removal import far_cloud, full_cloud, host_attrs, lattice, non_finite_rows, xyz1

pytestmark = pytest.mark.gpu

Z10 = dict(axis=[0.0, 0.0, 1.0], eps_angle=math.radians(10.0))


@pytest.fixture(scope="module")
def q(spx):
    return spx.DeviceQueue(0)


def tilt(pts, deg=4.0):
    a = np.deg2rad(deg)
    R = np.array([[1, 0, 0], [0, np.cos(a), -np.sin(a)], [0, np.sin(a), np.cos(a)]])
    out = pts.copy()
    out[:, :3] = (pts[:, :3].astype(np.float64) @ R.T).astype(np.float32)
    return out


def ground_truth(scan, beams=64, az_steps=1024, noise_seed=900):
    """(ground, height): which points of synthetic.drive's first revolution are ground returns, and every point's
    noise-free height above the ground.  scan() adds N(0, 0.02) range noise per ray from RandomState(noise_seed); the
    ray of a point follows from its direction, so the noise-free range is |p| minus that ray's noise, and a ground
    return is one whose noise-free range is the ray's distance to the ground plane."""
    p = scan[:, :3].astype(np.float64)
    r = np.linalg.norm(p, axis=1)
    a = np.rint(np.mod(np.arctan2(p[:, 1], p[:, 0]), 2 * np.pi) / (2 * np.pi / az_steps)).astype(int) % az_steps
    b = np.rint((np.rad2deg(np.arcsin(p[:, 2] / r)) + 24.8) / (26.8 / (beams - 1))).astype(int)
    noise = np.random.RandomState(noise_seed).normal(0.0, 0.02, (az_steps, beams))
    sin_e = np.sin(np.deg2rad(np.linspace(-24.8, 2.0, beams)))[b]
    r0 = r - noise[a, b]
    with np.errstate(divide="ignore"):
        ground = np.abs(r0 - synthetic.GROUND_Z / sin_e) < 2e-3
    return ground, r0 * sin_e - synthetic.GROUND_Z


@pytest.fixture(scope="module")
def revolution():
    _, scans = synthetic.drive(1)
    return scans[0]


def gpu_segment(spx, q, pts, t, H, cloud=None, **kw):
    cloud = cloud if cloud is not None else spx.PointCloudShared(q, pts)
    counts = spx.DeviceArray(q, (H,), np.uint32)
    r = spx.PlaneSegmentation(q).segment(cloud, t, H, hypothesis_counts=counts, **kw)
    inl = r.inliers.download() if len(r.inliers) else np.zeros(0, np.int32)
    rem = r.remainder.download() if len(r.remainder) else np.zeros(0, np.int32)
    return r, inl, rem, (counts.download() if len(pts) else None)


def check_exact(spx, q, pts, t, H, label, seed=0, **kw):
    """optimize_coefficients off: everything bit-exact"""
    want = ref.segment(pts, t, H, seed, kw.get("axis"), kw.get("eps_angle", 0.0), optimize=False)
    r, inl, rem, counts = gpu_segment(spx, q, pts, t, H, seed=seed, optimize_coefficients=False, **kw)
    if len(pts):
        assert np.array_equal(counts, want.counts), \
            f"{label}: counts differ at {np.flatnonzero(counts != want.counts)[:8]}"
    assert r.hypothesis == want.hypothesis, label
    assert np.array_equal(r.coefficients.view(np.uint32), want.coefficients.view(np.uint32)), \
        (label, r.coefficients, want.coefficients)
    assert np.array_equal(inl, want.inliers), f"{label}: {len(inl)} inliers, reference {len(want.inliers)}"
    assert np.array_equal(rem, want.remainder), label
    return want


def ulp_diff(a, b):
    """the distance in fp32 steps between two float32 arrays"""
    def ordered(x):
        i = x.view(np.int32).astype(np.int64)
        return np.where(i < 0, -(i & 0x7FFFFFFF), i)
    return np.abs(ordered(np.asarray(a, np.float32)) - ordered(np.asarray(b, np.float32)))


def check_refined(spx, q, pts, t, H, label, **kw):
    want = ref.segment(pts, t, H, 0, kw.get("axis"), kw.get("eps_angle", 0.0), optimize=True)
    r, inl, rem, counts = gpu_segment(spx, q, pts, t, H, **kw)
    assert np.array_equal(counts, want.counts) and r.hypothesis == want.hypothesis, label
    assert ulp_diff(r.coefficients, want.coefficients).max() <= 1, (label, r.coefficients, want.coefficients)
    if np.array_equal(r.coefficients.view(np.uint32), want.coefficients.view(np.uint32)):
        assert np.array_equal(inl, want.inliers) and np.array_equal(rem, want.remainder), label
        return 0
    # the two planes differ by a few ulps: a point may fall on either side of t only if its distance lies within that
    # difference (plus the rounding of the fp32 chain) of t
    P = pts[:, :3].astype(np.float64)
    g, w = r.coefficients.astype(np.float64), want.coefficients.astype(np.float64)
    dist = np.abs(P @ w[:3] + w[3])
    bound = np.abs(P) @ np.abs(g[:3] - w[:3]) + abs(g[3] - w[3]) + 4 * np.finfo(np.float32).eps * (np.abs(P) @ np.abs(w[:3]) + abs(w[3]))
    fin = np.isfinite(P).all(1)
    near = fin & (np.abs(dist - t) <= bound)
    a, b = np.zeros(len(pts), bool), np.zeros(len(pts), bool)
    a[inl], b[want.inliers] = True, True
    assert not np.any((a != b) & ~near), label
    print(f"{label}: refined planes {ulp_diff(r.coefficients, want.coefficients).tolist()} ulps apart, "
          f"{int(near.sum())} points within the bound of t, {int((a != b).sum())} differ")
    assert near.sum() <= 1e-4 * len(pts), label
    return int(near.sum())


# ------------------------------------------------------------------ unrefined: bit-exact
@pytest.mark.parametrize("tilted", [False, True])
@pytest.mark.parametrize("constrained", [False, True])
def test_drive_revolution_exact(spx, q, revolution, tilted, constrained):
    pts = tilt(revolution) if tilted else revolution
    kw = Z10 if constrained else {}
    for t in (0.05, 0.2, 0.5):
        for H in (1, 50, 1000):
            check_exact(spx, q, pts, t, H, f"tilted={tilted} axis={constrained} t={t} H={H}", **kw)


def hostile(revolution, case):
    return {"1km": lambda: far_cloud(revolution, (1000.0, -400.0, 25.0)),
            "22km": lambda: far_cloud(revolution, (21000.0, 6500.0, 40.0)),
            "non_finite": lambda: non_finite_rows(revolution)}[case]()


@pytest.mark.parametrize("case", ["1km", "22km", "non_finite"])
def test_hostile_geometry_exact(spx, q, revolution, case):
    pts = hostile(revolution, case)
    for t in (0.05, 0.2):
        for kw in ({}, Z10):
            check_exact(spx, q, pts, t, 1000, f"{case} t={t} {kw}", **kw)


def test_non_finite_rows_are_remainder(spx, q, revolution):
    pts = non_finite_rows(revolution)
    bad = np.flatnonzero(~np.isfinite(pts[:, :3]).all(1))
    assert len(bad) > 100
    r, inl, rem, _ = gpu_segment(spx, q, pts, 0.2, 200)
    assert np.isin(bad, rem).all() and not np.isin(bad, inl).any()


def test_lattice_at_t(spx, q):
    """a 0.25 m lattice: planes through lattice points have lattice points at exactly t = 0.25 (out) and, one fp32 step
    below, those are still out while the plane's own points are in"""
    pts = lattice()
    for t in (0.25, float(np.nextafter(np.float32(0.25), np.float32(1))), float(np.nextafter(np.float32(0.25), np.float32(0)))):
        check_exact(spx, q, pts, t, 500, f"lattice t={t}")


@pytest.mark.parametrize("n", [0, 1, 2, 3])
def test_tiny_clouds(spx, q, n):
    pts = xyz1(np.random.RandomState(n).uniform(-1, 1, (n, 3)))
    for H in (1, 7):
        w = check_exact(spx, q, pts, 0.5, H, f"n={n} H={H}")
        assert (w.hypothesis >= 0) == (n == 3)


def test_full_size_raw_cloud_exact(spx, q):
    pts, _, _ = synthetic.kitti_pair()
    assert len(pts) > 1_500_000
    w = check_exact(spx, q, pts, 0.1, 256, "2M")
    print(f"2M cloud: best hypothesis {w.hypothesis} with {int(w.counts[w.hypothesis])} inliers")


# ------------------------------------------------------------------ refined
@pytest.mark.parametrize("case", ["level", "tilted", "tilted_axis", "1km", "22km", "non_finite"])
def test_refined_within_one_ulp(spx, q, revolution, case):
    pts = {"level": revolution, "tilted": tilt(revolution), "tilted_axis": tilt(revolution)}.get(case)
    pts = hostile(revolution, case) if pts is None else pts
    kw = Z10 if case == "tilted_axis" else {}
    for t in (0.05, 0.2):
        check_refined(spx, q, pts, t, 1000, f"{case} t={t}", **kw)


# ------------------------------------------------------------------ usefulness: ground removal before clustering
def test_ground_removal_before_clustering(spx, q, revolution):
    ground, height = ground_truth(revolution)
    assert ground.mean() > 0.5
    pts = tilt(revolution)
    t = 0.05
    c = spx.PointCloudShared(q, pts)
    r = spx.PlaneSegmentation(q).segment(c, t, 1000, **Z10)
    inl = np.zeros(len(pts), bool)
    inl[r.inliers.download()] = True
    # returns of objects within t of the ground are indistinguishable from it; every other object return is "other"
    other = ~ground & (height > t)
    print(f"ground {ground.sum()}: {inl[ground].mean():.5f} inliers; others {other.sum()}: {inl[other].mean():.5f}; "
          f"object returns within t of the ground {int((~ground & ~other).sum())}: {inl[~ground & ~other].mean():.3f}")
    assert inl[ground].mean() >= 0.99 and inl[other].mean() <= 0.005
    normal = r.coefficients[:3].astype(np.float64)
    assert abs(abs(normal @ [0, -np.sin(np.deg2rad(4.0)), np.cos(np.deg2rad(4.0))]) - 1) < 1e-4
    rem = r.remainder_cloud()
    rem_pts = rem.points_host()
    assert np.array_equal(rem_pts, pts[~inl])
    got = spx.EuclideanClustering(q).extract(rem, 0.5)
    want = cref.clusters(rem_pts, 0.5)
    assert np.array_equal(got.labels.download(), want[0]) and np.array_equal(got.offsets, want[2])
    assert np.array_equal(got.indices.download(), want[1])
    whole = spx.EuclideanClustering(q).extract(c, 0.5)
    largest, largest_whole = int(np.diff(got.offsets.astype(np.int64)).max()), int(np.diff(whole.offsets.astype(np.int64)).max())
    print(f"largest cluster: {largest} points after ground removal, {largest_whole} with the ground")
    assert 4 * largest <= largest_whole


# ------------------------------------------------------------------ determinism, attributes, arguments
def test_two_runs_are_bit_identical_and_seeds_differ(spx, q, revolution):
    c = spx.PointCloudShared(q, revolution)
    a = gpu_segment(spx, q, revolution, 0.1, 1000, cloud=c)
    b = gpu_segment(spx, q, revolution, 0.1, 1000, cloud=c)
    assert np.array_equal(a[0].coefficients.view(np.uint32), b[0].coefficients.view(np.uint32))
    assert a[0].hypothesis == b[0].hypothesis
    for x, y in zip(a[1:], b[1:]):
        assert np.array_equal(x, y)
    s = gpu_segment(spx, q, revolution, 0.1, 1000, cloud=c, seed=2 ** 64 - 5)
    assert not np.array_equal(s[3], a[3])
    assert np.array_equal(s[3], ref.hypotheses(revolution, 0.1, 1000, 2 ** 64 - 5)[2])


def test_gathered_clouds_carry_every_attribute(spx, q, revolution):
    pts = revolution[::2].copy()
    c, host = full_cloud(spx, q, pts)
    r = spx.PlaneSegmentation(q).segment(c, 0.1, 300, optimize_coefficients=False)
    want = ref.segment(pts, 0.1, 300, optimize=False)
    assert len(want.inliers) > 1000 and len(want.remainder) > 1000
    for cloud, idx in ((r.inlier_cloud(), want.inliers), (r.remainder_cloud(), want.remainder)):
        got = host_attrs(cloud)
        for name, a in host.items():
            assert np.array_equal(got[name], a[idx]), name
    out = spx.PointCloudShared(q)
    assert r.inlier_cloud(output=out) is out and out.size() == len(want.inliers)


def test_empty_cloud_launches_nothing(spx, q):
    before = spx.kernel_launch_count()
    r = spx.PlaneSegmentation(q).segment(spx.PointCloudShared(q, np.zeros((0, 4), np.float32)), 0.2)
    assert spx.kernel_launch_count() == before
    assert r.hypothesis == -1 and np.isnan(r.coefficients).all() and len(r.inliers) == 0 and len(r.remainder) == 0
    assert r.inlier_cloud().size() == 0 and r.remainder_cloud().size() == 0


def test_argument_checks(spx, q):
    pts = xyz1(np.random.RandomState(1).uniform(-1, 1, (100, 3)))
    c = spx.PointCloudShared(q, pts)
    f = spx.PlaneSegmentation(q)
    for kw in (dict(distance_threshold=0.0), dict(distance_threshold=-1.0), dict(distance_threshold=float("nan")),
               dict(distance_threshold=float("inf")), dict(distance_threshold=0.1, max_iterations=0),
               dict(distance_threshold=0.1, max_iterations=2 ** 20 + 1), dict(distance_threshold=0.1, axis=[0, 0, 0]),
               dict(distance_threshold=0.1, axis=[0, float("nan"), 1]), dict(distance_threshold=0.1, axis=[0, 0, 1],
                                                                             eps_angle=-0.1),
               dict(distance_threshold=0.1, eps_angle=math.pi / 2 + 1e-9)):
        with pytest.raises(ValueError):
            f.segment(c, **kw)
    # the C-ABI itself refuses what the wrapper would have caught
    L = spx.lib()
    inl = spx.DeviceArray(q, (100,), np.int32)
    coef = np.zeros(4, np.float32)
    hyp, m = C.c_int32(), C.c_size_t()

    def call(n=100, t=0.1, H=10, axis=None, eps=0.0, points=c.points.ptr):
        ax = None if axis is None else np.asarray(axis, np.float32)
        return L.spx_plane_segment(q.handle, points, n, t, H, 0, None if ax is None else ax.ctypes.data, eps, 1,
                                   coef.ctypes.data, C.byref(hyp), inl.ptr, C.byref(m), None, None)
    for bad in (dict(t=0.0), dict(t=-0.1), dict(t=float("nan")), dict(t=float("inf")), dict(H=0), dict(H=2 ** 20 + 1),
                dict(axis=[0, 0, 0]), dict(axis=[0, float("inf"), 1]), dict(axis=[0, 0, 1], eps=-1e-12),
                dict(eps=math.pi / 2 + 1e-12), dict(eps=float("nan")), dict(n=2 ** 31),
                dict(points=C.c_void_p(c.points.ptr.value + 4))):
        assert call(**bad) == -1, bad
    assert call(H=2 ** 20) == 0 and call(axis=[0, 0, 1], eps=math.pi / 2) == 0 and call(n=0, points=None) == 0
