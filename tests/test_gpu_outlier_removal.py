"""Statistical and radius outlier removal on the GPU (sycl_points_b200.OutlierRemoval, spx_statistical_outlier_indices,
spx_radius_outlier_indices) against the CPU reference of tests/outlier_reference.py: mean distances bit for bit, kept
indices exactly, on a synthetic LiDAR revolution with injected airborne outliers, on hostile geometry, with every
attribute carried along, and on a ~2 M-point raw cloud."""
import ctypes as C

import numpy as np
import pytest

import outlier_reference as ref
import synthetic

pytestmark = pytest.mark.gpu

BAND = 1e-9  # relative distance to the threshold below which a decision is reported and not compared


def with_airborne(scan, frac=0.005, seed=11):
    """the scan with frac * n points scattered through the air above and around it (rain, dust, birds), inserted at
    seeded positions"""
    rs = np.random.RandomState(seed)
    lo, hi = scan[:, :3].min(0), scan[:, :3].max(0)
    m = int(round(frac * len(scan)))
    air = np.c_[rs.uniform(lo[0], hi[0], m), rs.uniform(lo[1], hi[1], m), rs.uniform(lo[2] + 1.0, hi[2] + 8.0, m),
                np.ones(m)].astype(np.float32)
    at = np.sort(rs.choice(len(scan) + m, m, replace=False))
    out = np.empty((len(scan) + m, 4), np.float32)
    mask = np.zeros(len(out), bool)
    mask[at] = True
    out[mask] = air
    out[~mask] = scan
    return out, mask


@pytest.fixture(scope="module")
def q(spx):
    return spx.DeviceQueue(0)


@pytest.fixture(scope="module")
def drive_and_air():
    _, scans = synthetic.drive(1)
    return with_airborne(scans[0])


@pytest.fixture(scope="module")
def drive_cloud(drive_and_air):
    return drive_and_air[0]


def cloud_with_ids(spx, q, pts):
    """a cloud whose intensities are the row numbers: the output's intensities are the kept indices"""
    c = spx.PointCloudShared(q, pts)
    c.set_intensities(np.arange(len(pts), dtype=np.float32))
    return c


def kept(out):
    return out.intensities.download(out.size()).astype(np.int64) if out.size() else np.zeros(0, np.int64)


def gpu_statistical(spx, q, pts, k, alpha, cloud=None, tree=None):
    cloud = cloud if cloud is not None else cloud_with_ids(spx, q, pts)
    md = spx.DeviceArray(q, (max(len(pts), 1),), np.float32)
    out = spx.OutlierRemoval(q).statistical(cloud, k, alpha, tree=tree, mean_distances=md)
    return kept(out), (md.download()[:len(pts)] if len(pts) else np.zeros(0, np.float32))


def gpu_radius(spx, q, pts, r, m, cloud=None, tree=None):
    cloud = cloud if cloud is not None else cloud_with_ids(spx, q, pts)
    return kept(spx.OutlierRemoval(q).radius(cloud, r, m, tree=tree))


def check_statistical(got_idx, got_d, pts, k, alpha, label=""):
    want_d = ref.mean_distances(pts, k)
    assert np.array_equal(got_d.view(np.uint32), want_d.view(np.uint32)) or np.array_equal(got_d, want_d, equal_nan=True), \
        f"{label}: mean distances differ at {np.flatnonzero(~((got_d == want_d) | (np.isnan(got_d) & np.isnan(want_d))))[:10]}"
    mu, sigma, thr = ref.statistics(want_d, alpha)
    near = np.abs(want_d.astype(np.float64) - thr) <= BAND * abs(thr) if np.isfinite(thr) else np.zeros(len(pts), bool)
    print(f"{label}: k={k} alpha={alpha}: {int(near.sum())} points within {BAND:g} relative of mu + alpha sigma")
    keep = ~np.isnan(want_d) & (want_d.astype(np.float64) <= thr)
    mask = np.zeros(len(pts), bool)
    mask[got_idx] = True
    assert np.all(np.diff(got_idx) > 0)
    assert np.array_equal(mask[~near], keep[~near]), f"{label}: kept sets differ"
    return int(near.sum())


def check_radius(got_idx, pts, r, m, label=""):
    want = np.flatnonzero(ref.radius(pts, r, m))
    assert np.array_equal(got_idx, want), f"{label}: r={r} m={m}: {len(got_idx)} kept, reference {len(want)}"


@pytest.mark.parametrize("k", [1, 8, 50, 127])
def test_statistical_on_a_drive_revolution_with_airborne_outliers(spx, q, drive_cloud, k, capsys):
    pts = drive_cloud
    cloud = cloud_with_ids(spx, q, pts)
    tree = spx.KDTree.build(q, cloud)
    for alpha in (-0.5, 0.0, 1.0, 2.0):
        idx, d = gpu_statistical(spx, q, pts, k, alpha, cloud=cloud, tree=tree)
        n_near = check_statistical(idx, d, pts, k, alpha, "drive")
        assert f"{n_near} points within" in capsys.readouterr().out
        assert len(idx) < len(pts)  # (at alpha < 0 the airborne points' spread can put mu + alpha sigma below every d)
        assert alpha < 0 or len(idx) > 0


def test_statistical_and_radius_remove_the_airborne_points(spx, q, drive_and_air):
    pts, air = drive_and_air
    for idx in (gpu_statistical(spx, q, pts, 8, 1.0)[0], gpu_radius(spx, q, pts, 0.5, 2)):
        removed = np.ones(len(pts), bool)
        removed[idx] = False
        print(f"removed: {removed[air].mean():.3f} of the airborne points, {removed[~air].mean():.3f} of the scan")
        assert removed[air].mean() > 0.5 and removed[air].mean() > 5 * removed[~air].mean()


@pytest.mark.parametrize("r", [0.0, 0.05, 0.3, 2.0, 50.0])
def test_radius_on_a_drive_revolution_with_airborne_outliers(spx, q, drive_cloud, r):
    pts = drive_cloud
    cloud = cloud_with_ids(spx, q, pts)
    tree = spx.KDTree.build(q, cloud)
    for m in (0, 1, 5, 200, 10 ** 6):
        check_radius(gpu_radius(spx, q, pts, r, m, cloud=cloud, tree=tree), pts, r, m, "drive")


# ------------------------------------------------------------------ hostile geometry
def xyz1(a):
    a = np.asarray(a, np.float32).reshape(-1, 3)
    return np.c_[a, np.ones(len(a), np.float32)].astype(np.float32)


def copies_of_one_point():
    rs = np.random.RandomState(3)
    p = np.tile(xyz1([[1.25, -3.5, 0.75]]), (5000, 1))
    others = xyz1(rs.uniform(-2, 2, (6, 3)) + [1.25, -3.5, 0.75])
    return np.insert(p, [0, 17, 2500, 2500, 4999, 5000], others, axis=0)


def lattice(step=0.25, n=(16, 12, 6), origin=(-2.0, 3.0, -1.0)):
    g = np.stack(np.meshgrid(*[np.arange(k) for k in n], indexing="ij"), -1).reshape(-1, 3)
    return xyz1(np.asarray(origin, np.float32) + np.float32(step) * g.astype(np.float32))


def far_cloud(drive_cloud, offset):
    p = drive_cloud[::3].copy()
    p[:, :3] += np.asarray(offset, np.float32)
    return p


def non_finite_rows(drive_cloud):
    rs = np.random.RandomState(9)
    p = drive_cloud[::2].copy()
    rows = rs.choice(len(p), len(p) // 100, replace=False)
    vals = np.array([np.nan, np.inf, -np.inf], np.float32)
    p[rows, rs.randint(0, 3, len(rows))] = vals[rs.randint(0, 3, len(rows))]
    return p


def hostile_cases(drive_cloud):
    return {
        "copies": copies_of_one_point(),
        "lattice": lattice(),
        "1km": far_cloud(drive_cloud, (1000.0, -400.0, 25.0)),
        "22km": far_cloud(drive_cloud, (21000.0, 6500.0, 40.0)),
        "non_finite": non_finite_rows(drive_cloud),
        "all_nan": np.full((40, 4), np.nan, np.float32),
    }


@pytest.mark.parametrize("case", ["copies", "lattice", "1km", "22km", "non_finite", "all_nan"])
def test_statistical_on_hostile_geometry(spx, q, drive_cloud, case):
    pts = hostile_cases(drive_cloud)[case]
    for k in (1, 6, 50, 127):
        for alpha in (-0.5, 1.0):
            idx, d = gpu_statistical(spx, q, pts, k, alpha)
            check_statistical(idx, d, pts, k, alpha, case)


@pytest.mark.parametrize("case", ["copies", "lattice", "1km", "22km", "non_finite", "all_nan"])
def test_radius_on_hostile_geometry(spx, q, drive_cloud, case):
    pts = hostile_cases(drive_cloud)[case]
    radii = [0.0, 0.3, 2.0]
    if case == "lattice":  # exactly one lattice step, and one fp32 step below it
        radii = [0.25, float(np.nextafter(np.float32(0.25), np.float32(0.0))), 0.5, 0.6]
    ms = (0, 1, 6, 7, 26, 4999, 5000, 5005) if case in ("copies", "all_nan") else (0, 1, 6, 7, 26)
    for r in radii:
        for m in ms:
            check_radius(gpu_radius(spx, q, pts, r, m), pts, r, m, case)


def test_lattice_boundary_counts_by_hand(spx, q):
    pts = lattice()
    n6 = int(((np.array([16, 12, 6]) - 2).prod()))  # interior points: 6 neighbours at exactly 0.25 m
    assert len(gpu_radius(spx, q, pts, 0.25, 6)) == n6
    assert len(gpu_radius(spx, q, pts, float(np.nextafter(np.float32(0.25), np.float32(0.0))), 1)) == 0


@pytest.mark.parametrize("n", [0, 1, 8, 9])
def test_tiny_clouds(spx, q, n):
    rs = np.random.RandomState(n)
    pts = xyz1(rs.uniform(-1, 1, (n, 3)))
    for k in (1, 8):
        idx, d = gpu_statistical(spx, q, pts, k, 0.5)
        if n:
            check_statistical(idx, d, pts, k, 0.5, f"n={n}")
        else:
            assert len(idx) == 0
    for r, m in ((0.5, 1), (3.0, 8), (3.0, 0)):
        check_radius(gpu_radius(spx, q, pts, r, m), pts, r, m, f"n={n}")


def test_empty_cloud_launches_nothing(spx, q):
    before = spx.kernel_launch_count()
    c = spx.PointCloudShared(q, np.zeros((0, 4), np.float32))
    f = spx.OutlierRemoval(q)
    assert f.statistical(c, 8, 1.0).size() == 0
    assert f.radius(c, 0.5, 2, output=c) is c and c.size() == 0
    assert spx.kernel_launch_count() == before


def test_voxel_grid_output_with_points_outside_the_hint_box(spx, q, drive_cloud):
    vg = spx.VoxelGrid(q, 0.2)
    ds = vg.downsampling(spx.PointCloudShared(q, drive_cloud))
    assert ds.index_hint is not None
    pts = ds.points_host()
    rs = np.random.RandomState(5)
    rows = rs.choice(len(pts), 60, replace=False)
    pts[rows[:30], 0] += 40.0   # beyond the box on +x
    pts[rows[30:], 2] -= 15.0   # and below it
    pts[rows[:4], :3] = pts[rows[4], :3]  # a few duplicates out there
    ds.points = spx.DeviceArray.from_host(q, pts)  # (the hint stays: the index is built from the now-wrong box)
    ds.set_intensities(np.arange(len(pts), dtype=np.float32))
    assert ds.index_hint is not None
    for k in (6, 30):
        idx, d = gpu_statistical(spx, q, pts, k, 1.0, cloud=ds)
        check_statistical(idx, d, pts, k, 1.0, "hinted")
    for r, m in ((0.3, 1), (0.5, 4), (2.0, 3), (0.0, 1)):
        check_radius(gpu_radius(spx, q, pts, r, m, cloud=ds), pts, r, m, "hinted")


# ------------------------------------------------------------------ attributes, aliasing, determinism
def full_cloud(spx, q, pts):
    rs = np.random.RandomState(4)
    n = len(pts)
    a = rs.normal(0, 1, (n, 3, 3)).astype(np.float32)
    covs = np.zeros((n, 4, 4), np.float32)
    covs[:, :3, :3] = a @ a.transpose(0, 2, 1)
    normals = np.c_[rs.normal(0, 1, (n, 3)), np.zeros(n)].astype(np.float32)
    rgb = rs.uniform(0, 1, (n, 4)).astype(np.float32)
    inten = np.arange(n, dtype=np.float32)
    ts = rs.uniform(0, 100, n).astype(np.float32)
    c = spx.PointCloudShared(q, pts, covs, normals)
    c.set_rgb(rgb)
    c.set_intensities(inten)
    c.set_timestamp_offsets(ts)
    return c, dict(points=pts, covs=covs, normals=normals, rgb=rgb, intensities=inten, timestamp_offsets=ts)


def host_attrs(c):
    n = c.size()
    return dict(points=c.points_host(), covs=c.covs_host(), normals=c.normals_host(), rgb=c.rgb.download(n),
                intensities=c.intensities.download(n), timestamp_offsets=c.timestamp_offsets.download(n))


@pytest.mark.parametrize("which", ["statistical", "radius"])
def test_every_attribute_is_compacted_in_source_order(spx, q, drive_cloud, which):
    pts = drive_cloud[::4].copy()
    f = spx.OutlierRemoval(q)
    run = (lambda c, out: f.statistical(c, 10, 0.5, output=out)) if which == "statistical" else \
        (lambda c, out: f.radius(c, 0.4, 3, output=out))
    want = np.flatnonzero(ref.statistical(pts, 10, 0.5)[0] if which == "statistical" else ref.radius(pts, 0.4, 3))
    c, host = full_cloud(spx, q, pts)
    out1 = run(c, None)
    assert out1 is not c and c.size() == len(pts)
    got1 = host_attrs(out1)
    for name, a in host.items():
        assert np.array_equal(got1[name], a[want]), name
    out2 = run(c, None)  # a second run gives identical output
    got2 = host_attrs(out2)
    for name in host:
        assert np.array_equal(got2[name].view(np.uint32), got1[name].view(np.uint32)), name
    res = run(c, c)  # in place
    assert res is c and c.size() == len(want)
    got3 = host_attrs(c)
    for name in host:
        assert np.array_equal(got3[name], got1[name]), name


def test_argument_checks(spx, q):
    pts = xyz1(np.random.RandomState(1).uniform(-1, 1, (100, 3)))
    c = spx.PointCloudShared(q, pts)
    other = spx.KDTree.build(q, spx.PointCloudShared(q, pts[:50]))
    f = spx.OutlierRemoval(q)
    with pytest.raises(ValueError):
        f.statistical(c, 4, 1.0, tree=other)
    with pytest.raises(ValueError):
        f.radius(c, 0.5, 1, tree=other)
    for k in (0, 128):
        with pytest.raises(ValueError):
            f.statistical(c, k, 1.0)
    # the C-ABI itself refuses what the wrapper would have caught
    L = spx.lib()
    tree = spx.KDTree.build(q, c)
    idx = spx.DeviceArray(q, (100,), np.int32)
    m = C.c_size_t()
    assert L.spx_statistical_outlier_indices(tree.handle, c.points.ptr, 99, 4, 1.0, None, idx.ptr, C.byref(m)) == -1
    assert L.spx_statistical_outlier_indices(tree.handle, c.points.ptr, 100, 128, 1.0, None, idx.ptr, C.byref(m)) == -1
    assert L.spx_statistical_outlier_indices(tree.handle, c.points.ptr, 100, 4, float("nan"), None, idx.ptr, C.byref(m)) == -1
    assert L.spx_radius_outlier_indices(tree.handle, c.points.ptr, 100, -0.5, 1, idx.ptr, C.byref(m)) == -1
    assert L.spx_radius_outlier_indices(tree.handle, c.points.ptr, 100, float("inf"), 1, idx.ptr, C.byref(m)) == -1
    assert L.spx_radius_outlier_indices(tree.handle, c.points.ptr, 101, 0.5, 1, idx.ptr, C.byref(m)) == -1
    assert L.spx_statistical_outlier_indices(tree.handle, c.points.ptr, 100, 4, 1.0, None, idx.ptr, C.byref(m)) == 0
    assert 0 < m.value <= 100


# ------------------------------------------------------------------ full size
@pytest.fixture(scope="module")
def raw_2m():
    tgt, _, _ = synthetic.kitti_pair()
    return tgt


def test_full_size_statistical_and_radius(spx, q, raw_2m):
    pts = raw_2m
    n = len(pts)
    assert n > 1_500_000
    rows = np.sort(np.random.RandomState(2024).choice(n, 2000, replace=False))
    cloud = cloud_with_ids(spx, q, pts)
    tree = spx.KDTree.build(q, cloud)
    idx, d = gpu_statistical(spx, q, pts, 50, 1.0, cloud=cloud, tree=tree)
    want_d = ref.mean_distances(pts, 50, rows)
    assert np.array_equal(d[rows], want_d, equal_nan=True)
    mu, sigma, thr = ref.statistics(d, 1.0)  # fp64 statistics of the GPU's own mean distances
    near = np.abs(d.astype(np.float64) - thr) <= BAND * thr
    print(f"2M statistical: {int(near.sum())} points within {BAND:g} relative of mu + alpha sigma; "
          f"kept {len(idx)} of {n}")
    keep = ~np.isnan(d) & (d.astype(np.float64) <= thr)
    mask = np.zeros(n, bool)
    mask[idx] = True
    assert np.array_equal(mask[~near], keep[~near])
    rk = ~np.isnan(want_d) & (want_d.astype(np.float64) <= thr)
    assert np.array_equal(mask[rows][~near[rows]], rk[~near[rows]])
    idx_r = gpu_radius(spx, q, pts, 0.5, 5, cloud=cloud, tree=tree)
    mask_r = np.zeros(n, bool)
    mask_r[idx_r] = True
    assert np.array_equal(mask_r[rows], ref.radius(pts, 0.5, 5, rows))
    assert 0 < len(idx_r) < n
