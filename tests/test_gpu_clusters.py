"""Euclidean cluster extraction on the GPU (sycl_points_b200.EuclideanClustering, spx_euclidean_clusters) against the
CPU reference of tests/cluster_reference.py: labels, offsets and member indices exactly equal, on a drive revolution
with the ground removed and airborne points added, on hostile geometry, on a 200 k-point helix (one deep component,
and n singletons), on a ~2 M-point raw cloud; plus determinism, every attribute of a gathered cluster and the
argument checks of the C-ABI."""
import ctypes as C

import numpy as np
import pytest
from scipy.optimize import brentq

import cluster_reference as ref
import synthetic
from test_gpu_outlier_removal import (copies_of_one_point, far_cloud, full_cloud, host_attrs, lattice, non_finite_rows,
                                      with_airborne, xyz1)

pytestmark = pytest.mark.gpu

INF = 2 ** 31 - 1
SIZES = [(1, INF), (10, INF), (1, 50), (100, 5000)]


@pytest.fixture(scope="module")
def q(spx):
    return spx.DeviceQueue(0)


@pytest.fixture(scope="module")
def drive_objects():
    """one revolution without the ground (z > -1.5 m), with 0.5 % airborne points"""
    _, scans = synthetic.drive(1)
    s = scans[0]
    return with_airborne(s[s[:, 2] > -1.5])[0]


@pytest.fixture(scope="module")
def drive_cloud():
    _, scans = synthetic.drive(1)
    return with_airborne(scans[0])[0]


def gpu_clusters(spx, q, pts, t, lo=1, hi=INF, cloud=None, tree=None):
    cloud = cloud if cloud is not None else spx.PointCloudShared(q, pts)
    r = spx.EuclideanClustering(q).extract(cloud, t, lo, hi, tree=tree)
    labels = r.labels.download() if len(pts) else np.zeros(0, np.int32)
    indices = r.indices.download() if r.offsets[-1] else np.zeros(0, np.int32)
    assert len(r) == len(r.offsets) - 1
    return labels, indices, r.offsets


def check(got, want, label):
    for name, g, w in zip(("labels", "indices", "offsets"), got, want):
        assert g.dtype == w.dtype and np.array_equal(g, w), \
            f"{label}: {name} differ ({len(g)} vs {len(w)} entries; first at {np.flatnonzero(g[:len(w)] != w[:len(g)])[:5]})"


def check_cloud(spx, q, pts, ts, sizes=((1, INF),), label="", cloud=None):
    cloud = cloud if cloud is not None else spx.PointCloudShared(q, pts)
    tree = spx.KDTree.build(q, cloud)
    for t in ts:
        e = ref.edges(pts, t)
        fin = np.isfinite(pts[:, :3]).all(1)
        for lo, hi in sizes:
            want = ref.clusters_from_edges(len(pts), fin, e, lo, hi)
            check(gpu_clusters(spx, q, pts, t, lo, hi, cloud=cloud, tree=tree), want, f"{label} t={t} ({lo}, {hi})")


def test_drive_revolution_without_ground(spx, q, drive_objects):
    check_cloud(spx, q, drive_objects, (0.0, 0.1, 0.5, 1.0, 3.0), SIZES, "drive")


# ------------------------------------------------------------------ hostile geometry
def between_two_clusters():
    """two 0.1 m chains 0.3 m apart end to end, and 1 % of rows with a non-finite coordinate placed in the gap"""
    rs = np.random.RandomState(7)
    a = np.c_[0.1 * np.arange(300), np.zeros(300), np.zeros(300)]
    b = np.c_[30.2 + 0.1 * np.arange(300), np.zeros(300), np.zeros(300)]
    bad = np.c_[rs.uniform(29.95, 30.15, 6), np.zeros(6), np.zeros(6)]
    vals = np.array([np.nan, np.inf, -np.inf])
    bad[np.arange(6), rs.randint(1, 3, 6)] = vals[rs.randint(0, 3, 6)]
    pts = np.r_[a, b, bad]
    return xyz1(pts[rs.permutation(len(pts))])


def hostile(drive_cloud, case):
    return {"copies": copies_of_one_point, "lattice": lattice, "between": between_two_clusters,
            "1km": lambda: far_cloud(drive_cloud, (1000.0, -400.0, 25.0)),
            "22km": lambda: far_cloud(drive_cloud, (21000.0, 6500.0, 40.0)),
            "non_finite": lambda: non_finite_rows(drive_cloud)}[case]()


@pytest.mark.parametrize("case", ["copies", "lattice", "between", "1km", "22km", "non_finite"])
def test_hostile_geometry(spx, q, drive_cloud, case):
    pts = hostile(drive_cloud, case)
    ts = {"copies": (0.0, 0.3, 2.0), "lattice": (0.25, float(np.nextafter(np.float32(0.25), np.float32(0))), 0.4),
          "between": (0.15, 0.2, 0.35)}.get(case, (0.0, 0.2, 0.6))
    check_cloud(spx, q, pts, ts, [(1, INF), (2, 500)], case)


def test_non_finite_rows_do_not_bridge(spx, q):
    pts = between_two_clusters()
    labels, indices, offsets = gpu_clusters(spx, q, pts, 0.2)
    assert offsets.tolist() == [0, 300, 600] and np.sum(labels == -1) == 6


def test_lattice_by_hand(spx, q):
    pts = lattice()
    assert gpu_clusters(spx, q, pts, 0.25)[2].tolist() == [0, len(pts)]
    labels, indices, offsets = gpu_clusters(spx, q, pts, float(np.nextafter(np.float32(0.25), np.float32(0))))
    assert labels.tolist() == list(range(len(pts))) and offsets.tolist() == list(range(len(pts) + 1))


@pytest.mark.parametrize("n", [1, 2])
def test_tiny_clouds(spx, q, n):
    pts = xyz1(np.random.RandomState(n).uniform(-1, 1, (n, 3)))
    check_cloud(spx, q, pts, (0.0, 0.5, 5.0), [(1, INF), (2, INF), (1, 1)], f"n={n}")


def test_empty_cloud_launches_nothing(spx, q):
    before = spx.kernel_launch_count()
    r = spx.EuclideanClustering(q).extract(spx.PointCloudShared(q, np.zeros((0, 4), np.float32)), 0.5)
    assert len(r) == 0 and r.offsets.tolist() == [0]
    assert spx.kernel_launch_count() == before


def test_voxel_grid_output_with_points_outside_the_hint_box(spx, q, drive_cloud):
    ds = spx.VoxelGrid(q, 0.2).downsampling(spx.PointCloudShared(q, drive_cloud))
    assert ds.index_hint is not None
    pts = ds.points_host()
    rs = np.random.RandomState(5)
    rows = rs.choice(len(pts), 60, replace=False)
    pts[rows[:30], 0] += 40.0
    pts[rows[30:], 2] -= 15.0
    pts[rows[:4], :3] = pts[rows[4], :3]
    ds.points = spx.DeviceArray.from_host(q, pts)  # (the hint stays: the index is built from the now-wrong box)
    assert ds.index_hint is not None
    check_cloud(spx, q, pts, (0.0, 0.3, 0.5, 2.0), [(1, INF), (3, 1000)], "hinted", cloud=ds)


def helix(n=200_000, spacing=0.05, radius=2.0, pitch=0.5):
    """n points along a helix, consecutive points `spacing` apart, turns `pitch` apart"""
    dphi = brentq(lambda a: np.hypot(2 * radius * np.sin(a / 2), pitch * a / (2 * np.pi)) - spacing, 1e-6, 1.0)
    phi = dphi * np.arange(n)
    return xyz1(np.c_[radius * np.cos(phi), radius * np.sin(phi), pitch * phi / (2 * np.pi)])


def test_helix_one_deep_component_and_n_singletons(spx, q):
    pts = helix()
    n = len(pts)
    hi, lo = 0.05 * 1.02, 0.05 * 0.98
    got = gpu_clusters(spx, q, pts, hi)
    assert got[2].tolist() == [0, n]
    check(got, ref.clusters(pts, hi), "helix above the spacing")
    got = gpu_clusters(spx, q, pts, lo)  # C = n: both sorts run over n entries, well beyond one radix tile
    assert len(got[2]) == n + 1
    check(got, ref.clusters(pts, lo), "helix below the spacing")


# ------------------------------------------------------------------ determinism, attributes, arguments
def test_two_runs_are_bit_identical(spx, q, drive_cloud):
    c = spx.PointCloudShared(q, drive_cloud)
    tree = spx.KDTree.build(q, c)
    a = gpu_clusters(spx, q, drive_cloud, 0.5, cloud=c, tree=tree)
    b = gpu_clusters(spx, q, drive_cloud, 0.5, cloud=c, tree=tree)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


def test_cluster_gathers_every_attribute_in_ascending_order(spx, q, drive_objects):
    pts = drive_objects[::2].copy()
    c, host = full_cloud(spx, q, pts)
    r = spx.EuclideanClustering(q).extract(c, 0.5, min_cluster_size=5)
    _, indices, offsets = ref.clusters(pts, 0.5, 5)
    assert np.array_equal(r.offsets, offsets) and len(r) >= 3
    for k in (0, 1, len(r) - 1):
        members = indices[offsets[k]:offsets[k + 1]]
        assert np.all(np.diff(members) > 0)
        got = host_attrs(r.cluster(k))
        for name, a in host.items():
            assert np.array_equal(got[name], a[members]), (k, name)
    out = spx.PointCloudShared(q)
    assert r.cluster(1, output=out) is out and out.size() == offsets[2] - offsets[1]
    with pytest.raises(IndexError):
        r.cluster(len(r))


def test_argument_checks(spx, q):
    pts = xyz1(np.random.RandomState(1).uniform(-1, 1, (100, 3)))
    c = spx.PointCloudShared(q, pts)
    other = spx.KDTree.build(q, spx.PointCloudShared(q, pts[:50]))
    f = spx.EuclideanClustering(q)
    with pytest.raises(ValueError):
        f.extract(c, 0.5, tree=other)
    for kw in (dict(tolerance=-1.0), dict(tolerance=float("nan")), dict(tolerance=0.5, min_cluster_size=0),
               dict(tolerance=0.5, min_cluster_size=3, max_cluster_size=2)):
        with pytest.raises(ValueError):
            f.extract(c, **kw)
    # the C-ABI itself refuses what the wrapper would have caught
    L = spx.lib()
    tree = spx.KDTree.build(q, c)
    lab = spx.DeviceArray(q, (100,), np.int32)
    idx = spx.DeviceArray(q, (100,), np.int32)
    off = spx.DeviceArray(q, (101,), np.uint32)
    nc, nm = C.c_size_t(), C.c_size_t()

    def call(n=100, t=0.5, lo=1, hi=INF):
        return L.spx_euclidean_clusters(tree.handle, c.points.ptr, n, t, lo, hi, lab.ptr, idx.ptr, off.ptr, C.byref(nc),
                                        C.byref(nm))
    assert call(n=99) == -1 and call(n=101) == -1
    assert call(t=-0.5) == -1 and call(t=float("inf")) == -1 and call(t=float("nan")) == -1
    assert call(lo=0) == -1 and call(lo=5, hi=4) == -1
    assert L.spx_euclidean_clusters(tree.handle, c.points.ptr, 100, 0.5, 1, INF, None, idx.ptr, off.ptr, C.byref(nc),
                                    C.byref(nm)) == 0
    want = ref.clusters(pts, 0.5)
    assert nc.value == len(want[2]) - 1 and nm.value == 100
    assert np.array_equal(idx.download(), want[1]) and np.array_equal(off.download(nc.value + 1), want[2])
    assert call() == 0 and np.array_equal(lab.download(), want[0])


# ------------------------------------------------------------------ full size
def test_full_size_raw_cloud(spx, q):
    pts, _, _ = synthetic.kitti_pair()
    assert len(pts) > 1_500_000
    t = 0.1
    e = ref.edges(pts, t)
    print(f"2M cloud at t = {t}: {len(e)} reference pairs")
    want = ref.clusters(pts, t, e=e)
    check(gpu_clusters(spx, q, pts, t), want, "2M")
    print(f"{len(want[2]) - 1} clusters, largest {int(np.diff(want[2].astype(np.int64)).max())}")
