"""The k = 1 correspondence search of every ICP align path against a brute-force reference on hostile geometry.

The search is not one piece of code: the cooperative align kernel (A, P = 1), the split loop with its keep test (B)
and without it (C), the host-decided LM / dog-leg loop (D), the batched align (E, P > 1) and the sharded one-launch
align (F) each carry their own copy of the non-finite guard and of the hand-off of runner-up bounds and allowances.
All of them claim "the brute-force answer, ties by index, bit for bit".  The scenarios below give them what the
bundled pair near the origin never does: a target kilometres from the origin, exact distance ties, targets at exactly
max_correspondence_distance, non-finite points, no overlap, empty and all-NaN targets, tiny and lopsided clouds, and
a sparse target that sends queries through the work list and onto the coarser grid levels.

Checks (convergence criteria off wherever iterations are compared):
  * search replay (A, B, C): after m iterations the cached neighbours equal the oracle's nearest neighbour at the
    pose the last search ran at — index and distance bit for bit within max_corr, beyond it otherwise;
  * one-step pose replay (GN): every step equals the oracle's single step from the same pose;
  * cross-path equality: A, B, C, E and F agree bit for bit;
  * LM / dog-leg (D) against the oracle's trajectory;
  * the keep test really keeps, and the sparse scenario really escalates.
The construction tests at the bottom run without a GPU and check that each scenario is what it claims to be.
"""
import contextlib
import ctypes as C
import functools
import os

import numpy as np
import pytest

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
F32 = np.float32

# ------------------------------------------------------------------------------------------------ scenario builders
# Each builder is seeded and returns host arrays near the origin: source / target points (n, 4), their covariances
# (n, 4, 4) and the target normals, both estimated from 10 neighbours BEFORE any corruption, thinning or move (the
# reference's un-centred fp32 sums would destroy covariances estimated kilometres away); `offset` moves the target
# on the device (transform_copy), `T0` is the initial guess, `iters` the iteration count of the pose checks.


@functools.lru_cache(maxsize=None)
def _bundled():
    d = np.load(os.path.join(GOLDEN, "bundled_pair.npz"))
    return d["source_ds"], d["target_ds"]


@functools.lru_cache(maxsize=None)
def _bundled_features():
    src, tgt = _bundled()
    return _features(src) + _features(tgt)


def _features(pts, k=10):
    idx, _ = oracle.KDTree(pts).knn(pts, k)
    return oracle.covariance(pts, idx), oracle.normals(pts, idx)


def _translation(t):
    T = np.eye(4, dtype=F32)
    T[:3, 3] = np.asarray(t, F32)
    return T


def _perturbation():
    return oracle.se3_exp(np.array([0.004, -0.003, 0.012, 0.3, -0.2, 0.05], F32))


def _scenario(name, src, cov_s, tgt, cov_t, nrm_t, T0, max_corr=2.0, iters=5, offset=None, exact_tree=False,
              **extra):
    return dict(name=name, src=np.ascontiguousarray(src, F32), cov_s=np.ascontiguousarray(cov_s, F32),
                tgt=np.ascontiguousarray(tgt, F32), cov_t=np.ascontiguousarray(cov_t, F32),
                nrm_t=np.ascontiguousarray(nrm_t, F32), T0=np.asarray(T0, F32), max_corr=float(max_corr), iters=iters,
                offset=offset, exact_tree=exact_tree, **extra)


def s1_world_frame(far=False):
    """Sensor-frame source, world-frame target ~1 km (S1) or ~22 km (S1b) from the origin."""
    src, tgt = _bundled()
    cs, _, ct, nt = _bundled_features()
    o = np.array([18000.0, -12500.0, 120.0] if far else [812.5, -640.25, 35.0], F32)
    T0 = (_translation(o).astype(np.float64) @ _perturbation().astype(np.float64)).astype(F32)
    return _scenario("S1b" if far else "S1", src, cs, tgt, ct, nt, T0, offset=o, iters=6)


def s2a_duplicate_targets(seed=21):
    """30 % of the target points appear twice; the permutation puts the lower index of a twin pair at random."""
    rs = np.random.RandomState(seed)
    src, tgt = _bundled()
    cs, _, ct, nt = _bundled_features()
    dup = np.sort(rs.choice(len(tgt), int(0.3 * len(tgt)), replace=False))
    rows = np.concatenate([np.arange(len(tgt)), dup])
    perm = rs.permutation(len(rows))
    rows = rows[perm]
    # rows: which bundled point each target row is; original: the row is the first copy of it (not the duplicate)
    return _scenario("S2a", src, cs, tgt[rows], ct[rows], nt[rows], _perturbation(), rows=rows,
                     original=perm < len(tgt))


def s2b_lattice_ties():
    """Both clouds snapped to a 0.25 m lattice, initial guess half a lattice step along x: many queries are exactly
    equidistant from two targets in the first search."""
    src, tgt = _bundled()
    snap = lambda p: np.unique(np.c_[np.round(p[:, :3] / 0.25) * 0.25, np.ones(len(p))].astype(F32), axis=0)
    s, t = snap(src), snap(tgt)
    cs, _ = _features(s)
    ct, nt = _features(t)
    return _scenario("S2b", s, cs, t, ct, nt, _translation([0.125, 0.0, 0.0]), iters=1)


def s3_radius_boundary(max_corr):
    """Sparse lattice of targets (spacing 8 max_corr, so nothing else lies within 3 max_corr of a query).  Source
    point i sits max_corr before its target along x (exact in fp32, distance exactly max_corr^2), one fp32 step
    farther, or at half the distance; T0 = I."""
    s = 8.0 * max_corr
    g = np.stack(np.meshgrid(np.arange(12), np.arange(10), np.arange(6), indexing="ij"), -1).reshape(-1, 3)
    tgt = np.c_[(g * s - np.array([40, 30, 20]) * max_corr).astype(F32), np.ones(len(g), F32)].astype(F32)
    kind = np.arange(len(tgt)) % 3  # 0 exactly at max_corr, 1 one step beyond, 2 well inside
    src = tgt.copy()
    x = tgt[:, 0] - F32(max_corr)
    src[:, 0] = np.where(kind == 0, x, np.where(kind == 1, np.nextafter(x, F32(-np.inf)), tgt[:, 0] - F32(0.5 * max_corr)))
    cs, _ = _features(src)
    ct, nt = _features(tgt)
    return _scenario(f"S3-{max_corr:g}", src, cs, tgt, ct, nt, np.eye(4, dtype=F32), max_corr=max_corr, iters=1,
                     kind=kind)


def _corrupt(pts, rs, frac=0.01):
    pts = pts.copy()
    rows = rs.choice(len(pts), max(3, int(frac * len(pts))), replace=False)
    bad = [np.nan, np.inf, -np.inf]
    for j, r in enumerate(rows):
        if j % 4 == 3:
            pts[r, :3] = bad[j % 3]
        else:
            pts[r, rs.randint(3)] = bad[j % 3]
    return pts, np.sort(rows)


def s4_non_finite(seed=4):
    """~1 % of the source rows and ~1 % of the target rows carry NaN or +-inf in one or all coordinates."""
    rs = np.random.RandomState(seed)
    src, tgt = _bundled()
    cs, _, ct, nt = _bundled_features()
    s, _ = _corrupt(src, rs)
    t, _ = _corrupt(tgt, rs)
    return _scenario("S4", s, cs, t, ct, nt, _perturbation())


def s5a_no_overlap():
    """The source starts 50 m beyond the far side of the target, max_corr 1: no correspondence, ever."""
    src, tgt = _bundled()
    cs, _, ct, nt = _bundled_features()
    shift = float(tgt[:, 0].max() - src[:, 0].min()) + 50.0
    return _scenario("S5a", src, cs, tgt, ct, nt, _translation([shift, 0.0, 0.0]), max_corr=1.0)


def s5b_half_overlap():
    """The half of the source with x above the median is moved 60 m along x (in the source frame)."""
    src, tgt = _bundled()
    cs, _, ct, nt = _bundled_features()
    s = src.copy()
    s[s[:, 0] > np.median(s[:, 0]), 0] += F32(60.0)
    return _scenario("S5b", s, cs, tgt, ct, nt, _perturbation())


def s6_empty_target(all_nan=False):
    """No target (nt = 0), or a target whose points are all NaN (an index over no finite point).  An empty cloud has
    no covariances (PointCloudShared::has_cov() needs a non-empty array), so the empty target is aligned with
    point-to-point, the factor the reference runs against it; GICP is refused (test_gicp_refuses_an_empty_target)."""
    src, _ = _bundled()
    cs, _, _, _ = _bundled_features()
    n = 200 if all_nan else 0
    t = np.full((n, 4), np.nan, F32)
    t[:, 3] = 1.0
    ct = np.tile(np.diag([1e-2, 1e-2, 1e-2, 0.0]).astype(F32), (n, 1, 1))
    nt = np.tile(np.array([0, 0, 1, 0], F32), (n, 1))
    return _scenario("S6-nan" if all_nan else "S6-empty", src, cs, t, ct, nt, _perturbation())


def s7_tiny(ns=None, nt=None, copies=None, seed=7):
    """ns source points against the whole target, the whole source against nt target points, or 5000 copies of one
    source point."""
    rs = np.random.RandomState(seed)
    src, tgt = _bundled()
    cs, _, ct, nrm = _bundled_features()
    if ns is not None:
        sel = np.sort(rs.choice(len(src), ns, replace=False))
        return _scenario(f"S7-ns{ns}", src[sel], cs[sel], tgt, ct, nrm, _perturbation())
    if nt is not None:
        sel = np.sort(rs.choice(len(tgt), nt, replace=False))
        return _scenario(f"S7-nt{nt}", src, cs, tgt[sel], ct[sel], nrm[sel], _perturbation())
    j = rs.randint(len(src))
    rows = np.full(copies, j)
    return _scenario(f"S7-copies{copies}", src[rows], cs[rows], tgt, ct, nrm, _perturbation())


@functools.lru_cache(maxsize=None)
def s8_sparse_escalation(seed=7):
    """A voxelised synthetic street pair, the target thinned to 3 % beyond x = 0, 1.5 m initial offset, max_corr 10,
    8 iterations: queries over the thinned half have their nearest target several cells away (work list, coarser
    grid levels), and the keep test runs from the third iteration on."""
    import synthetic
    rs = np.random.RandomState(seed)
    tgt_raw, src_raw, T_gt = synthetic.kitti_pair(seed, sweeps=4)
    src = oracle.voxel_downsample(src_raw, 0.2)
    tgt = oracle.voxel_downsample(tgt_raw, 0.2)
    cs, _ = _features(src)
    ct, nt = _features(tgt)
    keep = (tgt[:, 0] <= 0.0) | (rs.rand(len(tgt)) < 0.03)
    T0 = (T_gt.astype(np.float64) @ oracle.se3_exp(np.array([0.0, 0.0, 0.01, 1.2, -0.9, 0.0], F32))).astype(F32)
    return _scenario("S8", src, cs, tgt[keep], ct[keep], nt[keep], T0, max_corr=10.0, iters=8, exact_tree=True)


BUILDERS = {
    "S1": lambda: s1_world_frame(False),
    "S1b": lambda: s1_world_frame(True),
    "S2a": s2a_duplicate_targets,
    "S2b": s2b_lattice_ties,
    "S3-0.5": lambda: s3_radius_boundary(0.5),
    "S3-1": lambda: s3_radius_boundary(1.0),
    "S3-2": lambda: s3_radius_boundary(2.0),
    "S4": s4_non_finite,
    "S5a": s5a_no_overlap,
    "S5b": s5b_half_overlap,
    "S6-empty": lambda: s6_empty_target(False),
    "S6-nan": lambda: s6_empty_target(True),
    **{f"S7-ns{n}": functools.partial(s7_tiny, ns=n) for n in (1, 31, 32, 33, 257)},
    **{f"S7-nt{n}": functools.partial(s7_tiny, nt=n) for n in (1, 2, 7)},
    "S7-copies5000": functools.partial(s7_tiny, copies=5000),
    "S8": s8_sparse_escalation,
}
# factors each scenario runs with (the first one in the search replay and the LM / dog-leg checks); GICP elsewhere
SCENARIO_REGS = {"S1": ("GICP", "POINT_TO_PLANE"), "S1b": ("GICP", "POINT_TO_PLANE"), "S6-empty": ("POINT_TO_POINT",),
                 "S6-nan": ("GICP", "POINT_TO_POINT")}


def regs_of(name):
    return SCENARIO_REGS.get(name, ("GICP",))


# (scenario, factor) pairs of the Gauss-Newton checks
GN_CASES = [(s, r) for s in BUILDERS for r in regs_of(s)]
NEAR_ORIGIN = [s for s in BUILDERS if s not in ("S1", "S1b", "S8")]
KEEP_MUST_RUN = ("S1", "S2a", "S8")  # B's keep test must keep something here (S1b: only recorded, see below)


def oracle_nn(sc, src, tgt, T, tree=None):
    """(index, distance) of the nearest target of every source point at pose T: brute force, or the exact KD-tree
    for the large scenario (a KD-tree built over non-finite coordinates is no reference)."""
    if sc["exact_tree"]:
        i, d = tree.knn(src, 1, T, mode=0)
    else:
        i, d = oracle.knn_bruteforce(src, tgt, 1, T)
    return i.reshape(-1), d.reshape(-1)


# ------------------------------------------------------------------------------------------------ GPU side
OPT = {"GN": 0, "LM": 1, "DOGLEG": 2}
# environment of each Gauss-Newton path: A = cooperative one-launch loop (clouds below 400 k points), B = split
# loop with the keep test, C = split loop searching every query in every iteration
PATH_ENV = {"A": {"SPX_SPLIT_MIN": None, "SPX_KEEP_FRAC": None},
            "B": {"SPX_SPLIT_MIN": "0", "SPX_KEEP_FRAC": None},
            "C": {"SPX_SPLIT_MIN": "0", "SPX_KEEP_FRAC": "-1"}}


@contextlib.contextmanager
def _env(values):
    old = {k: os.environ.get(k) for k in values}
    try:
        for k, v in values.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def pose_delta(Ta, Tb):
    d = np.linalg.inv(Ta.astype(np.float64)) @ Tb.astype(np.float64)
    w = 0.5 * np.array([d[2, 1] - d[1, 2], d[0, 2] - d[2, 0], d[1, 0] - d[0, 1]])
    return np.linalg.norm(d[:3, 3]), float(np.arcsin(min(1.0, np.linalg.norm(w))))


def step_perturbation(Hg, bg, Ho, bo):
    """First-order bound on how far apart the solutions of H d = -b lie when H and b differ by (Hg - Ho, bg - bo):
    |dd| <= |Ho^-1| (|dH| |d| + |db|), with the differences the caller measured (H within 1e-5 relative is asserted
    before it is used).  It is the amplification of those differences by the conditioning of H: negligible for a
    well-posed problem, large when H is near singular — on the B200 only S7-nt1 (every source point paired with one
    and the same target) needs it.  Where it exceeds 1e-6 it is printed ("[sens]"), so that a pose bound it makes
    loose is visible; the H / b / inlier checks do not depend on it."""
    Ho, bo = Ho.astype(np.float64), bo.astype(np.float64)
    Hi = np.linalg.pinv(Ho)
    d = Hi @ bo
    return float(np.linalg.norm(Hi, 2) * (np.linalg.norm(Hg.astype(np.float64) - Ho, 2) * np.linalg.norm(d)
                                         + np.linalg.norm(bg.astype(np.float64) - bo)))


def rel(a, b):
    return np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)).max() / max(np.abs(b).max(), 1e-30)


class Case:
    """A scenario on the device.  The oracle reads back what the device holds (the target after its move)."""

    def __init__(self, spx, q, sc):
        self.sc, self.q = sc, q
        self.src = spx.PointCloudShared(q, sc["src"], sc["cov_s"])
        tgt = spx.PointCloudShared(q, sc["tgt"], sc["cov_t"], sc["nrm_t"])
        if sc["offset"] is not None:
            tgt = spx.transform.transform_copy(tgt, _translation(sc["offset"]))
        self.tgt = tgt
        self.tree = spx.KDTree.build(q, tgt)
        self.src_h, self.cov_s = sc["src"], sc["cov_s"]
        self.tgt_h = tgt.points_host()
        self.cov_t = tgt.covs_host() if tgt.size() else sc["cov_t"]
        self.nrm_t = tgt.normals_host() if tgt.size() else sc["nrm_t"]
        self.otree = oracle.KDTree(self.tgt_h) if sc["exact_tree"] else None
        self.T0 = sc["T0"]

    def nn(self, T):
        return oracle_nn(self.sc, self.src_h, self.tgt_h, T, self.otree)

    def oracle_align(self, reg, iters, opt="GN", T0=None, trace=False):
        P = oracle.default_params(reg_type=oracle.REG[reg], loss=0, opt_method=OPT[opt], max_iterations=iters,
                                  max_corr_dist=self.sc["max_corr"], crit_translation=0.0, crit_rotation=0.0,
                                  knn_mode=0 if self.sc["exact_tree"] else 2)
        return oracle.align(P, self.src_h, self.cov_s, self.tgt_h, self.cov_t, self.nrm_t, self.otree,
                            self.T0 if T0 is None else T0, trace=trace)


def gpu_params(spx, sc, reg, iters, opt="GN"):
    p = spx.RegistrationParams(reg_type=spx.RegType[reg], max_iterations=iters)
    p.max_correspondence_distance = sc["max_corr"]
    p.optimization_method = spx.OptimizationMethod(OPT[opt])
    p.criteria.translation = p.criteria.rotation = 0.0
    return p


def neighbours(spx, q, r):
    ip, dp, n = C.c_void_p(), C.c_void_p(), C.c_size_t()
    spx._lib.check(spx.lib().spx_registration_neighbors(r._h, C.byref(ip), C.byref(dp), C.byref(n)))
    idx, dist = np.empty(n.value, np.int32), np.empty(n.value, np.float32)
    if n.value:
        spx._lib.check(spx.lib().spx_memcpy_d2h(q.handle, idx.ctypes.data_as(C.c_void_p), ip, idx.nbytes))
        spx._lib.check(spx.lib().spx_memcpy_d2h(q.handle, dist.ctypes.data_as(C.c_void_p), dp, dist.nbytes))
    q.wait()
    return idx, dist


def run(spx, q, c, reg, iters, path="A", opt="GN"):
    """-> (result with trace, neighbour indices, distances, kept correspondences, launches)"""
    r = spx.Registration(q, gpu_params(spx, c.sc, reg, iters, opt))
    with _env(PATH_ENV[path]):
        res = r.align(c.src, c.tgt, c.tree, c.T0, trace=True)
    idx, dist = neighbours(spx, q, r)
    launches = r.last_timing()["launches"] if opt == "GN" else 0
    return res, idx, dist, r.kept_correspondences(), launches


def run_sharded(spx, q, comms, c, reg, iters):
    from sycl_points_b200.api import _ptr
    r = spx.Registration(q, gpu_params(spx, c.sc, reg, iters))
    spx._lib.check(spx.lib().spx_registration_set_params(r._h, r.params.to_c()))
    t16 = np.ascontiguousarray(c.T0.T).reshape(16)
    src, tgt = c.src, c.tgt
    with _env(PATH_ENV["A"]):
        spx._lib.check(spx.lib().spx_registration_align_sharded_launch(
            r._h, comms.handles[0], src.points.ptr, _ptr(src.covs), src.size(),
            tgt.points.ptr if tgt.size() else None, _ptr(tgt.covs) if tgt.size() else None,
            _ptr(tgt.normals) if tgt.size() else None, tgt.size(), c.tree.handle,
            t16.ctypes.data_as(C.POINTER(C.c_float)), -1.0))
        R = spx._lib.RegistrationResultC()
        spx._lib.check(spx.lib().spx_registration_align_sharded_finish(r._h, C.byref(R)))
    return spx.RegistrationResult.from_c(R), r.kept_correspondences()


def assert_same(a, b, what, trace=True):
    assert np.array_equal(a.T, b.T), f"{what}: T differs"
    assert np.array_equal(a.H, b.H) and np.array_equal(a.b, b.b), f"{what}: H / b differ"
    assert np.array_equal(np.float32(a.error), np.float32(b.error)), f"{what}: error {a.error} vs {b.error}"
    assert (a.inlier, a.iterations, a.converged) == (b.inlier, b.iterations, b.converged), \
        f"{what}: {(a.inlier, a.iterations, a.converged)} vs {(b.inlier, b.iterations, b.converged)}"
    if trace:
        assert np.array_equal(a.trace, b.trace), f"{what}: trace differs"


def assert_neighbours_exact(idx, dist, oi, od, max_corr, what):
    mc2 = F32(max_corr) * F32(max_corr)
    within = od <= mc2
    bad = np.flatnonzero(within & ((idx != oi) | (dist != od)))
    assert bad.size == 0, (f"{what}: {bad.size} of {within.sum()} correspondences differ from brute force, first "
                           f"query {bad[0]}: gpu ({idx[bad[0]]}, {dist[bad[0]]!r}) oracle ({oi[bad[0]]}, {od[bad[0]]!r})")
    out = np.flatnonzero(~within & ~(dist > mc2))
    assert out.size == 0, f"{what}: {out.size} entries beyond max_corr reported within, first query {out[0]}"


@pytest.fixture(scope="module")
def q(spx):
    return spx.DeviceQueue(0)


_CASES = {}


@pytest.fixture(scope="module")
def case(spx, q):
    def get(name):
        if name not in _CASES:
            _CASES[name] = Case(spx, q, BUILDERS[name]())
        return _CASES[name]
    yield get
    _CASES.clear()


@pytest.fixture(scope="module")
def plain(spx, q):
    src, tgt = _bundled()
    cs, _, ct, nt = _bundled_features()
    return Case(spx, q, _scenario("plain", src, cs, tgt, ct, nt, np.eye(4, dtype=F32)))


@pytest.fixture(scope="module")
def comms(spx, q):
    from sycl_points_b200.multi_gpu import LocalCommunicators
    cm = LocalCommunicators([q])
    yield cm
    cm.close()


def replay_iterations(c):
    return max(5, c.sc["iters"])


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["A", "B", "C"])
@pytest.mark.parametrize("name", list(BUILDERS))
def test_search_replay_equals_brute_force(spx, q, case, name, path):
    """After m = 1..M iterations the neighbours the loop used last equal the oracle's nearest neighbours at the pose
    that search ran at (T0 for m = 1, else trace[m - 2]); every run's trace is a prefix of the longest run's."""
    c = case(name)
    M = replay_iterations(c)
    reg = regs_of(name)[0]
    runs = [run(spx, q, c, reg, m, path) for m in range(1, M + 1)]
    longest = runs[-1][0].trace
    for m, (res, idx, dist, _, launches) in enumerate(runs, start=1):
        if path != "A":
            assert launches >= 3, "the split loop did not run"
        assert len(idx) == c.src.size()
        T_search = c.T0 if m == 1 else res.trace[m - 2]
        oi, od = c.nn(T_search)
        assert_neighbours_exact(idx, dist, oi, od, c.sc["max_corr"], f"{name} path {path} m={m}")
        assert np.array_equal(res.trace[:m], longest[:m]), f"{name} path {path}: run {m} left the longest run's trace"


@pytest.mark.gpu
@pytest.mark.parametrize("name,reg", GN_CASES)
def test_gauss_newton_steps_replay_on_the_oracle(spx, q, case, name, reg):
    """Every Gauss-Newton step of path A equals the oracle's single step from the same pose: rotation within 1e-5
    rad, translation within 1e-5 m + 4 ulp of the largest translation component (the pose is stored in fp32: one ulp
    is ~0.06 mm at 800 m, ~2 mm at 18 km), both widened by the first-order bound of the step's sensitivity to the
    H and b differences of that step (step_perturbation; negligible unless H is near singular).  The final H, b,
    error and inliers equal the oracle's step from trace[-2]."""
    c = case(name)
    M = c.sc["iters"]
    res, _, _, _, _ = run(spx, q, c, reg, M)
    for i in range(M):
        T_before = c.T0 if i == 0 else res.trace[i - 1]
        ores = c.oracle_align(reg, 1, T0=T_before)
        step = res if i == M - 1 else run(spx, q, c, reg, i + 1)[0]  # its H and b are those of step i
        assert np.array_equal(step.trace[i], res.trace[i])
        assert rel(step.H, ores["H"]) <= 1e-5, f"{name} {reg} step {i}: H differs by {rel(step.H, ores['H']):.2e}"
        sens = step_perturbation(step.H, step.b, ores["H"], ores["b"])
        dt, da = pose_delta(ores["T"], res.trace[i])
        if sens > 1e-6:
            print(f"[sens] {name} {reg} GN step {i}: widening {sens:.2e}, dt={dt:.2e} m, da={da:.2e} rad")
        tol_t = 1e-5 + 4 * float(np.spacing(np.abs(ores["T"][:3, 3]).max().astype(F32))) + sens
        assert dt <= tol_t and da <= 1e-5 + sens, \
            f"{name} {reg} step {i}: dt={dt:.3e} (tol {tol_t:.1e}) da={da:.3e} (sensitivity {sens:.1e})"
    assert res.inlier == ores["inlier"], (res.inlier, ores["inlier"])
    assert rel(res.H, ores["H"]) <= 1e-5
    assert np.abs(res.b - ores["b"]).max() <= 1e-5 * max(np.abs(ores["b"]).max(), 1e-2 * np.abs(ores["H"]).max())
    assert abs(res.error - ores["error"]) <= 1e-5 * abs(ores["error"])


@pytest.mark.gpu
@pytest.mark.parametrize("name,reg", GN_CASES)
def test_all_gauss_newton_paths_agree_bit_for_bit(spx, q, case, plain, comms, name, reg):
    """A (cooperative), B (split + keep), C (split, every query searched), E (batched, with a plain bundled pair and,
    for the S6 scenarios with point-to-point, a pair with an empty target in the same launch) and F (sharded
    one-launch, one rank): T, H, b, error, inliers, iterations, converged and, where returned, the trace are
    identical."""
    c = case(name)
    M = replay_iterations(c)
    A = run(spx, q, c, reg, M, "A")[0]
    B, _, _, kept_b, _ = run(spx, q, c, reg, M, "B")
    Cr, _, _, kept_c, _ = run(spx, q, c, reg, M, "C")
    assert kept_c == 0
    assert_same(B, A, f"{name}: B vs A")
    assert_same(Cr, A, f"{name}: C vs A")
    r = spx.Registration(q, gpu_params(spx, c.sc, reg, M))
    pairs = [(c.src, c.tgt, c.tree, c.T0), (plain.src, plain.tgt, plain.tree, None)]
    with_empty = name.startswith("S6") and reg == "POINT_TO_POINT"
    if with_empty:
        empty = Case(spx, q, s6_empty_target(False))
        pairs.append((c.src, empty.tgt, empty.tree, c.T0))
    with _env(PATH_ENV["A"]):
        E = r.align_batch(pairs)
        plain_one = spx.Registration(q, gpu_params(spx, c.sc, reg, M)).align(plain.src, plain.tgt, plain.tree)
        if with_empty:
            empty_one = spx.Registration(q, gpu_params(spx, c.sc, reg, M)).align(c.src, empty.tgt, empty.tree, c.T0)
            assert_same(E[2], empty_one, f"{name}: E (empty target) vs its single align", trace=False)
    assert_same(E[0], A, f"{name}: E vs A", trace=False)
    assert_same(E[1], plain_one, f"{name}: E (plain pair) vs its single align", trace=False)
    F, kept_f = run_sharded(spx, q, comms, c, reg, M)
    assert_same(F, A, f"{name}: F vs A", trace=False)
    print(f"[kept] {name} {reg}: B {kept_b}, F {kept_f} of {M * c.src.size()} correspondences")
    if name in KEEP_MUST_RUN:
        assert kept_b > 0, f"{name}: the keep test kept nothing"


@pytest.mark.gpu
@pytest.mark.parametrize("name,opt", [(s, "LM") for s in NEAR_ORIGIN] + [(s, "DOGLEG") for s in ("S4", "S5a", "S5b")])
def test_lm_and_dogleg_follow_the_oracle(spx, q, case, name, opt):
    """Path D (host-decided loop, nn_search_grid): pose after every iteration within 1e-5 of the oracle's
    trajectory (widened, as in the Gauss-Newton replay, by the step's first-order sensitivity to that iteration's H
    and b differences: the damped system is no worse conditioned than H), iterations / converged / inliers exact, and
    the last search's neighbours bit for bit."""
    c = case(name)
    M = c.sc["iters"]
    reg = regs_of(name)[0]
    res, idx, dist, _, _ = run(spx, q, c, reg, M, "A", opt)
    ores = c.oracle_align(reg, M, opt, trace=True)
    for it in range(M):
        g = res if it == M - 1 else run(spx, q, c, reg, it + 1, "A", opt)[0]
        o = ores if it == M - 1 else c.oracle_align(reg, it + 1, opt)
        sens = step_perturbation(g.H, g.b, o["H"], o["b"])
        dt, da = pose_delta(ores["trace"][it], res.trace[it])
        if sens > 1e-6:
            print(f"[sens] {name} {reg} {opt} iteration {it}: widening {sens:.2e}, dt={dt:.2e} m, da={da:.2e} rad")
        assert dt < 1e-5 + sens and da < 1e-5 + sens, \
            f"{name} {opt} iteration {it}: dt={dt:.2e} da={da:.2e} (sensitivity {sens:.1e})"
    assert (res.iterations, res.converged, res.inlier) == (ores["iterations"], ores["converged"], ores["inlier"])
    # the last search ran at the pose before the last iteration
    oi, od = c.nn(c.T0 if M == 1 else res.trace[M - 2])
    assert_neighbours_exact(idx, dist, oi, od, c.sc["max_corr"], f"{name} {opt}")


@pytest.mark.gpu
def test_sparse_scenario_escalates(spx, case):
    """S8 is only a test of the work list and the coarser levels if many queries have their nearest target more than
    two finest cells away: at T0 at least a quarter of them do, and the index has more than one level."""
    c = case("S8")
    info = c.tree.info()
    assert info["levels"] > 1
    oi, od = c.nn(c.T0)
    far = float(np.mean(od > (2.0 * info["cell_size"]) ** 2))
    print(f"[S8] {c.src.size()} / {c.tgt.size()} points, finest cell {info['cell_size']:.3f} m, "
          f"{info['levels']} levels, {100 * far:.1f} % of the queries > 2 cells from their nearest target")
    assert far >= 0.25, far


# ------------------------------------------------------------------------------------------------ CPU: construction
def test_s2_yields_exact_ties():
    for sc in (s2a_duplicate_targets(), s2b_lattice_ties()):
        i, d = oracle.knn_bruteforce(sc["src"], sc["tgt"], 2, sc["T0"])
        within = d[:, 0] <= F32(sc["max_corr"]) ** 2
        ties = within & (d[:, 0] == d[:, 1])
        assert ties.sum() >= 0.05 * len(d), (sc["name"], ties.sum())
        assert (i[ties, 0] < i[ties, 1]).all()  # the brute force resolves a tie to the lower index
    # in S2a the lower index of a twin pair is the first copy for some pairs and the duplicate for the others
    sc = s2a_duplicate_targets()
    rows, original = sc["rows"], sc["original"]
    order = np.lexsort((np.arange(len(rows)), rows))  # by bundled point, then by position
    r_sorted = rows[order]
    first_of_pair = np.flatnonzero(r_sorted[:-1] == r_sorted[1:])  # order[k] < order[k + 1]: the lower index
    assert len(first_of_pair) == int(0.3 * len(_bundled()[1]))
    share = float(original[order[first_of_pair]].mean())
    assert 0.4 < share < 0.6, share


@pytest.mark.parametrize("max_corr", [0.5, 1.0, 2.0])
def test_s3_distances_sit_on_the_radius(max_corr):
    sc = s3_radius_boundary(max_corr)
    i, d = oracle.knn_bruteforce(sc["src"], sc["tgt"], 2, sc["T0"])
    mc2 = F32(max_corr) * F32(max_corr)
    kind = sc["kind"]
    assert (i[:, 0] == np.arange(len(i))).all()
    assert (d[kind == 0, 0] == mc2).all()
    assert (d[kind == 1, 0] > mc2).all() and (d[kind == 1, 0] < mc2 * F32(1 + 1e-5)).all()  # one fp32 step beyond
    assert (d[kind == 2, 0] < mc2).all()
    assert (d[:, 1] > (3 * F32(max_corr)) ** 2).all()  # nothing else near


def test_s4_has_non_finite_rows_on_both_sides():
    sc = s4_non_finite()
    for pts in (sc["src"], sc["tgt"]):
        bad = ~np.isfinite(pts[:, :3]).all(1)
        assert 0.005 * len(pts) <= bad.sum() <= 0.02 * len(pts)
        assert np.isnan(pts).any() and np.isposinf(pts).any() and np.isneginf(pts).any()


def test_s5a_has_no_oracle_inliers():
    sc = s5a_no_overlap()
    P = oracle.default_params(reg_type=3, loss=0, max_iterations=5, max_corr_dist=sc["max_corr"], crit_translation=0.0,
                              crit_rotation=0.0, knn_mode=2)
    ores = oracle.align(P, sc["src"], sc["cov_s"], sc["tgt"], sc["cov_t"], None, None, sc["T0"], trace=True)
    assert ores["inlier"] == 0
    for T in [sc["T0"], *ores["trace"]]:
        _, d = oracle.knn_bruteforce(sc["src"], sc["tgt"], 1, T)
        assert (d > F32(sc["max_corr"]) ** 2).all()


@pytest.mark.gpu
def test_gicp_refuses_an_empty_target(spx, q, plain):
    """The reference's validate_params refuses GICP when the target has no covariances, and an empty cloud has none
    (PointCloudShared::has_cov() needs a non-empty array): the single and the batched align raise its error."""
    empty = spx.PointCloudShared(q, np.zeros((0, 4), F32), np.zeros((0, 4, 4), F32))
    tree = spx.KDTree.build(q, empty)
    params = spx.RegistrationParams(max_iterations=3)
    msg = "Covariance matrices of source and target must be pre-computed before performing GICP matching"
    with pytest.raises(RuntimeError, match=msg):
        spx.Registration(q, params).align(plain.src, empty, tree, plain.T0)
    with pytest.raises(RuntimeError, match=msg):
        spx.Registration(q, params).align_batch([(plain.src, plain.tgt, plain.tree), (plain.src, empty, tree, None)])
