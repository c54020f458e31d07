"""FPFH descriptors, feature correspondences and correspondence RANSAC on the GPU (sycl_points_b200.FPFHEstimation,
match_features, RANSACRegistration; spx_fpfh, spx_feature_correspondences, spx_ransac_registration) against the CPU
reference of tests/global_reference.py, and global registration end to end: a pair far outside ICP's basin is placed by
RANSAC within 0.5 m / 1 degree (the two other poses within 1 m / 2 degrees) and GICP from that pose ends within
0.02 m / 0.05 degrees."""
import ctypes as C

import numpy as np
import pytest

import global_reference as ref
import synthetic
from test_gpu_outlier_removal import far_cloud, lattice, non_finite_rows, xyz1

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def q(spx):
    return spx.DeviceQueue(0)


def Rz(deg):
    a = np.deg2rad(deg)
    T = np.eye(4)
    T[:2, :2] = [[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]]
    return T


def trans(x, y, z):
    T = np.eye(4)
    T[:3, 3] = [x, y, z]
    return T


POSES = {"t4_-2_r60": trans(4, -2, 0.05) @ Rz(60), "t-6_3_r150": trans(-6, 3, 0) @ Rz(150),
         "t2_5_r-100": trans(2, 5, -0.05) @ Rz(-100)}


def rot_angle(D):
    """the angle (radians) of a rotation close to the identity, from its skew part (arccos of the trace is too
    ill-conditioned there to resolve fp32 rounding); arccos beyond 0.1 rad"""
    s = 0.5 * np.linalg.norm([D[2, 1] - D[1, 2], D[0, 2] - D[2, 0], D[1, 0] - D[0, 1]])
    return float(np.arcsin(min(s, 1.0))) if s < 0.1 else float(np.arccos(np.clip((np.trace(D) - 1) / 2, -1, 1)))


def pose_error(T, T_gt):
    """(metres, degrees) between two poses"""
    d = np.linalg.inv(np.asarray(T_gt, np.float64)) @ np.asarray(T, np.float64)
    return float(np.linalg.norm(d[:3, 3])), float(np.degrees(rot_angle(d[:3, :3])))


def with_normals(spx, q, pts, k=15):
    cloud = spx.PointCloudShared(q, pts)
    tree = spx.KDTree.build(q, cloud)
    spx.covariance.estimate_normals(tree.knn_search(cloud, k), cloud)
    return cloud, tree


def gpu_fpfh(spx, q, cloud, tree, radius, max_nn=100):
    """(features, idx, dist, normals) on the host; the radius lists are the ones the descriptor used"""
    nn = tree.radius_search(cloud, max_nn, radius)
    f = spx.FPFHEstimation(q).compute(cloud, radius, max_nn, tree=tree)
    return f.download(), nn.indices_host(), nn.distances_host(), cloud.normals_host()


def check_fpfh(spx, q, cloud, tree, radius, label, max_nn=100):
    F, idx, dist, nrm = gpu_fpfh(spx, q, cloud, tree, radius, max_nn)
    want = ref.fpfh(cloud.points_host(), nrm, idx, dist)
    assert np.array_equal(F.view(np.uint32), want.view(np.uint32)), \
        f"{label}: rows differ at {np.flatnonzero((F.view(np.uint32) != want.view(np.uint32)).any(1))[:8]}"
    return F


@pytest.fixture(scope="module")
def offset_pair(spx, q):
    tgt_raw, src_raw, T_gt = synthetic.kitti_pair(42, T_gt=POSES["t4_-2_r60"])
    vg = spx.VoxelGrid(q, 1.0)
    out = {}
    for name, raw in (("src", src_raw), ("tgt", tgt_raw)):
        pts = vg.downsampling(spx.PointCloudShared(q, raw)).points_host()
        cloud, tree = with_normals(spx, q, pts)
        F = check_fpfh(spx, q, cloud, tree, 5.0, name)
        out[name] = dict(pts=pts, cloud=cloud, tree=tree, F=F)
    out["T_gt"] = T_gt
    out["raw"] = (src_raw, tgt_raw)
    return out


# ------------------------------------------------------------------ FPFH: bit-exact
def test_fpfh_bit_equal_on_the_voxel_pair(offset_pair):
    for name in ("src", "tgt"):
        F = offset_pair[name]["F"]
        assert 10_000 < len(F) < 20_000 and np.isfinite(F).all(), name


def test_fpfh_bit_equal_on_hostile_clouds(spx, q, offset_pair):
    base = offset_pair["tgt"]["pts"]
    far = far_cloud(base, (1e4, -1e4, 30.0))
    cloud, tree = with_normals(spx, q, far)
    check_fpfh(spx, q, cloud, tree, 5.0, "far")
    dup = np.concatenate([base[:3000], base[:3000:3]])
    cloud, tree = with_normals(spx, q, dup)
    check_fpfh(spx, q, cloud, tree, 5.0, "duplicates")
    iso = xyz1(np.array([[0, 0, 0], [50, 0, 0], [0, 50, 0], [0.5, 0, 0]], np.float32))
    cloud = spx.PointCloudShared(q, iso, normals=np.tile(np.float32([0, 0, 1, 0]), (4, 1)))
    F = check_fpfh(spx, q, cloud, spx.KDTree.build(q, cloud), 1.0, "isolated")
    assert not F[1:3].any()
    nf = non_finite_rows(base)
    rs = np.random.RandomState(2)
    cloud, tree = with_normals(spx, q, nf)
    nrm = cloud.normals_host()
    bad = rs.choice(len(nrm), 50, replace=False)
    nrm[bad, rs.randint(0, 3, 50)] = np.float32(np.nan)
    nrm[bad[:10], 0] = np.float32(np.inf)
    cloud.set_normals(nrm)
    F = check_fpfh(spx, q, cloud, tree, 5.0, "non-finite")
    assert np.isnan(F[bad]).all()
    lat = lattice(0.25, (24, 24, 6))
    cloud = spx.PointCloudShared(q, lat, normals=np.tile(np.float32([0.0, 0.6, 0.8, 0.0]), (len(lat), 1)))
    tree = spx.KDTree.build(q, cloud)
    assert (tree.radius_search(cloud, 100, 1.0).indices_host()[:, -1] >= 0).mean() > 0.3  # more than max_nn in the radius
    check_fpfh(spx, q, cloud, tree, 1.0, "lattice")


def test_fpfh_of_nothing_launches_nothing(spx, q):
    cloud = spx.PointCloudShared(q, np.zeros((0, 4), np.float32), normals=np.zeros((0, 4), np.float32))
    before = spx.kernel_launch_count()
    F = spx.FPFHEstimation(q).compute(cloud, 1.0)
    assert F.shape == (0, 33) and spx.kernel_launch_count() == before
    with pytest.raises(ValueError):
        spx.FPFHEstimation(q).compute(spx.PointCloudShared(q, xyz1([[0, 0, 0]])), 1.0)


# ------------------------------------------------------------------ correspondences: bit-exact
def gpu_matches(spx, q, s, t, mutual):
    a, b = spx.match_features(q, s, t, mutual=mutual)
    return (a.download() if len(a) else np.zeros(0, np.int32)), (b.download() if len(b) else np.zeros(0, np.int32))


@pytest.mark.parametrize("mutual", [False, True])
def test_correspondences_bit_equal(spx, q, offset_pair, mutual):
    s, t = offset_pair["src"]["F"], offset_pair["tgt"]["F"]
    gi, gj = gpu_matches(spx, q, s, t, mutual)
    wi, wj = ref.correspondences(s, t, mutual)
    assert np.array_equal(gi, wi) and np.array_equal(gj, wj), (len(gi), len(wi))
    # equal rows: the lowest index wins; NaN rows never match and find nothing
    t2 = np.repeat(t[:300], 3, axis=0)
    s2 = s[:2000].copy()
    s2[::7] = np.nan
    t2[1::5] = np.nan
    gi, gj = gpu_matches(spx, q, s2, t2, mutual)
    wi, wj = ref.correspondences(s2, t2, mutual)
    assert np.array_equal(gi, wi) and np.array_equal(gj, wj)
    assert not np.isin(np.arange(0, 2000, 7), gi).any()


# ------------------------------------------------------------------ RANSAC
@pytest.fixture(scope="module")
def pair_corr(spx, q, offset_pair):
    s, t = offset_pair["src"]["F"], offset_pair["tgt"]["F"]
    return ref.correspondences(s, t, False)


def gpu_ransac(spx, q, sp, tp, si, ti, eps, H, **kw):
    counts = spx.DeviceArray(q, (H,), np.uint32)
    S, T = spx.PointCloudShared(q, sp), spx.PointCloudShared(q, tp)
    r = spx.RANSACRegistration(q).align(S, T, (np.asarray(si, np.int32), np.asarray(ti, np.int32)), eps, H,
                                        hypothesis_counts=counts, **kw)
    inl = r.inliers.download() if len(r.inliers) else np.zeros(0, np.int32)
    return r, inl, counts.download()


def check_ransac_exact(spx, q, sp, tp, si, ti, eps, H, label, seed=0, tau=0.9):
    want = ref.ransac(sp, tp, si, ti, eps, H, seed, tau, optimize=False)
    r, inl, counts = gpu_ransac(spx, q, sp, tp, si, ti, eps, H, seed=seed, edge_length_similarity=tau, optimize=False)
    # every hypothesis's count (M = 0 too: then every one is invalid)
    assert np.array_equal(counts, want.counts), f"{label}: counts differ at {np.flatnonzero(counts != want.counts)[:8]}"
    assert r.hypothesis == want.hypothesis, label
    assert np.array_equal(r.T[:3].view(np.uint32), want.pose.view(np.uint32)), (label, r.T, want.pose)
    assert np.array_equal(inl, want.inliers), label
    return r, want


def test_ransac_exact_on_the_pair(spx, q, offset_pair, pair_corr):
    si, ti = pair_corr
    r, _ = check_ransac_exact(spx, q, offset_pair["src"]["pts"], offset_pair["tgt"]["pts"], si, ti, 1.0, 20_000, "pair")
    assert r.valid() and len(r.inliers) >= 20


def test_ransac_exact_on_edge_cases(spx, q, offset_pair, pair_corr):
    sp, tp = offset_pair["src"]["pts"], offset_pair["tgt"]["pts"]
    si, ti = pair_corr
    for m in (0, 1, 2):
        r, _ = check_ransac_exact(spx, q, sp, tp, si[:m], ti[:m], 1.0, 100, f"M={m}")
        assert not r.valid() and np.isnan(r.T).all()
    # tau = 1 with every target edge longer than its source edge: every hypothesis invalid
    rs = np.random.RandomState(1)
    P = xyz1(rs.uniform(-10, 10, (200, 3)))
    Q = P.copy()
    Q[:, :3] *= np.float32(1.5)
    idx = np.arange(200, dtype=np.int32)
    r, want = check_ransac_exact(spx, q, P, Q, idx, idx, 0.5, 500, "tau=1", tau=1.0)
    assert not r.valid() and (want.counts == ref.INVALID).all()
    # coplanar correspondences (a rotated ground patch), and non-finite points and out-of-range indices
    G = xyz1(np.c_[rs.uniform(-20, 20, (300, 2)), np.zeros(300)])
    T = POSES["t-6_3_r150"]
    GT = G.copy()
    GT[:, :3] = (G[:, :3].astype(np.float64) @ T[:3, :3].T + T[:3, 3]).astype(np.float32)
    idx = np.arange(300, dtype=np.int32)
    check_ransac_exact(spx, q, G, GT, idx, idx, 0.1, 3000, "coplanar")
    nf = non_finite_rows(np.concatenate([sp, sp]))[: len(sp)]
    si2, ti2 = si.copy(), ti.copy()
    si2[::50] = len(sp) + 5
    ti2[3::70] = -1
    check_ransac_exact(spx, q, nf, tp, si2, ti2, 1.0, 5000, "non-finite", seed=7)


def test_ransac_refined_equals_kabsch(spx, q, offset_pair, pair_corr):
    sp, tp = offset_pair["src"]["pts"], offset_pair["tgt"]["pts"]
    si, ti = pair_corr
    cases = [(sp, tp, si, ti, 1.0, 20_000)]
    rs = np.random.RandomState(3)
    G = xyz1(np.c_[rs.uniform(-20, 20, (300, 2)), rs.normal(0, 0.02, 300)])
    T = POSES["t2_5_r-100"]
    GT = G.copy()
    GT[:, :3] = (G[:, :3].astype(np.float64) @ T[:3, :3].T + T[:3, 3] + rs.normal(0, 0.02, (300, 3))).astype(np.float32)
    idx = np.arange(300, dtype=np.int32)
    GT[:, 2] = np.float32(0.25)  # target coplanar: a rank-2 cross-covariance
    cases.append((G, GT, idx, idx, 0.3, 3000))
    for k, (a, b, i, j, eps, H) in enumerate(cases):
        want = ref.ransac(a, b, i, j, eps, H, optimize=True)
        r, inl, counts = gpu_ransac(spx, q, a, b, i, j, eps, H)
        assert r.hypothesis == want.hypothesis and np.array_equal(counts, want.counts), k
        ps, qs = ref.gather_pairs(a, b, i, j)
        R, t = ref.kabsch(ps[want.hyp_inliers], qs[want.hyp_inliers])
        D = r.T[:3, :3].astype(np.float64) @ R.T
        dt, dang = np.abs(r.T[:3, 3] - t).max(), rot_angle(D)
        assert dt < 1e-6 * max(1.0, np.abs(t).max()) and dang < 1e-6, (k, dt, dang)
        # the inliers agree except for correspondences within the pose difference of eps
        d = np.linalg.norm(ps @ r.T[:3, :3].T.astype(np.float64) + r.T[:3, 3] - qs, axis=1)
        a_, b_ = np.zeros(len(ps), bool), np.zeros(len(ps), bool)
        a_[inl], b_[want.inliers] = True, True
        assert not np.any((a_ != b_) & (np.abs(d - eps) > 1e-4)), k
        assert r.fitness == len(inl) / len(i)


def test_determinism(spx, q, offset_pair):
    s, t = offset_pair["src"], offset_pair["tgt"]
    F1 = spx.FPFHEstimation(q).compute(s["cloud"], 5.0, tree=s["tree"]).download()
    F2 = spx.FPFHEstimation(q).compute(s["cloud"], 5.0, tree=s["tree"]).download()
    assert np.array_equal(F1.view(np.uint32), F2.view(np.uint32))
    m1 = gpu_matches(spx, q, F1, t["F"], True)
    m2 = gpu_matches(spx, q, F2, t["F"], True)
    assert all(np.array_equal(a, b) for a, b in zip(m1, m2))
    r1 = spx.RANSACRegistration(q).align(s["cloud"], t["cloud"], m1, 1.0, 20_000)
    r2 = spx.RANSACRegistration(q).align(s["cloud"], t["cloud"], m2, 1.0, 20_000)
    assert np.array_equal(r1.T.view(np.uint32), r2.T.view(np.uint32))
    assert np.array_equal(r1.inliers.download(), r2.inliers.download())


def test_c_abi_argument_checks(spx, q):
    L = spx.lib()
    d = spx.DeviceArray(q, (64, 33), np.float32)
    i = spx.DeviceArray(q, (64,), np.int32)
    Th = (C.c_float * 16)()
    h, m = C.c_int32(), C.c_size_t()
    assert L.spx_fpfh(q.handle, d.ptr, d.ptr, 4, i.ptr, d.ptr, 0, d.ptr) == -1  # k
    assert L.spx_fpfh(q.handle, d.ptr, d.ptr, 4, i.ptr, d.ptr, 129, d.ptr) == -1
    assert L.spx_fpfh(q.handle, None, d.ptr, 4, i.ptr, d.ptr, 8, d.ptr) == -1  # null
    assert L.spx_feature_correspondences(q.handle, d.ptr, 4, None, 4, 0, i.ptr, i.ptr, C.byref(m)) == -1
    assert L.spx_feature_correspondences(q.handle, d.ptr, 4, d.ptr, 4, 0, i.ptr, i.ptr, None) == -1

    def rr(eps=1.0, H=10, tau=0.9, pts=d.ptr, T=Th):
        return L.spx_ransac_registration(q.handle, pts, 4, d.ptr, 4, i.ptr, i.ptr, 4, eps, H, 0, tau, 1, T,
                                         C.byref(h), i.ptr, C.byref(m), None)
    assert rr() == 0
    for bad in (dict(eps=0.0), dict(eps=float("inf")), dict(eps=float("nan")), dict(H=0), dict(H=2 ** 20 + 1),
                dict(tau=0.0), dict(tau=1.5), dict(tau=float("nan")), dict(pts=None), dict(T=None)):
        assert rr(**bad) == -1, bad
    S = spx.PointCloudShared(q, xyz1(np.zeros((4, 3))))
    for kw in (dict(max_correspondence_distance=-1.0), dict(max_iterations=0), dict(edge_length_similarity=1.1),
               dict(seed=-1)):
        args = dict(max_correspondence_distance=1.0, **{k: v for k, v in kw.items() if k != "max_correspondence_distance"})
        if "max_correspondence_distance" in kw:
            args["max_correspondence_distance"] = kw["max_correspondence_distance"]
        with pytest.raises(ValueError):
            spx.RANSACRegistration(q).align(S, S, (np.arange(4), np.arange(4)), **args)
    with pytest.raises(ValueError):
        spx.FPFHEstimation(q).compute(spx.PointCloudShared(q, xyz1(np.zeros((2, 3))),
                                                           normals=np.zeros((2, 4), np.float32)), 0.0)


# ------------------------------------------------------------------ end to end
def gicp(spx, q, src_raw, tgt_raw, T0):
    vg = spx.VoxelGrid(q, 0.25)
    src = vg.downsampling(spx.PointCloudShared(q, src_raw))
    tgt = vg.downsampling(spx.PointCloudShared(q, tgt_raw))
    ts, tt = spx.KDTree.build(q, src), spx.KDTree.build(q, tgt)
    spx.covariance.estimate(ts.knn_search(src, 10), src)
    spx.covariance.estimate(tt.knn_search(tgt, 10), tgt)
    params = spx.RegistrationParams()
    params.robust.type = spx.RobustLossType.HUBER
    return spx.Registration(q, params).align(src, tgt, tt, np.asarray(T0, np.float32)).T


def global_pipeline(spx, q, src_raw, tgt_raw):
    vg = spx.VoxelGrid(q, 1.0)
    feats, clouds = [], []
    for raw in (src_raw, tgt_raw):
        pts = vg.downsampling(spx.PointCloudShared(q, raw)).points_host()
        cloud, tree = with_normals(spx, q, pts)
        feats.append(spx.FPFHEstimation(q).compute(cloud, 5.0, 100, tree=tree))
        clouds.append(cloud)
    corr = spx.match_features(q, feats[0], feats[1])
    return spx.RANSACRegistration(q).align(clouds[0], clouds[1], corr, 1.0, 100_000, seed=0)


@pytest.mark.parametrize("pose", list(POSES))
def test_global_registration_end_to_end(spx, q, pose):
    tgt_raw, src_raw, T_gt = synthetic.kitti_pair(42, T_gt=POSES[pose])
    r = global_pipeline(spx, q, src_raw, tgt_raw)
    et, er = pose_error(r.T, T_gt)
    print(f"{pose}: RANSAC {et:.3f} m {er:.3f} deg, {len(r.inliers)} inliers, fitness {r.fitness:.3f}")
    if pose == "t4_-2_r60":
        assert et < 0.5 and er < 1.0, (et, er)
    else:  # (the other two poses: RANSAC has to put GICP into its basin, about a metre and a few degrees)
        assert et < 1.0 and er < 2.0, (et, er)
    gt, gr = pose_error(gicp(spx, q, src_raw, tgt_raw, r.T), T_gt)
    print(f"{pose}: GICP from RANSAC {gt:.4f} m {gr:.4f} deg")
    assert gt < 0.02 and gr < 0.05, (gt, gr)
    if pose == "t4_-2_r60":
        it, ir = pose_error(gicp(spx, q, src_raw, tgt_raw, np.eye(4)), T_gt)
        print(f"{pose}: GICP from identity {it:.3f} m {ir:.3f} deg")
        assert it > 1.0
