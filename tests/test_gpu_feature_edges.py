"""Covariance, normal and preprocess-filter kernels against the oracle on hostile neighbourhoods and over their whole
k range.

Neighbour lists are written by hand and uploaded into a KNNResult, so every row is under the test's control:

- S1  the bundled target with lists from the index, plain k in {1, 2, 3, 4, 5, 7, 31, 64, 65, 128} and robust k in
      {1, 3, 4, 5, 7, 31, 63, 64} (robust k = 64 fills the local-memory weight arrays; k < 4 is the identity fallback)
- S2  -1 entries at the end, in the middle and at the front of rows, rows with exactly 3 and exactly 4 valid entries
      (either side of the cnt < 4 identity fallback), all -1 rows; odd and even k (the median is one element or the
      mean of two, and -1 entries enter it as 0)
- S3  every neighbour the same point (a zero covariance: its "inverse" is the zero matrix and the median is 0) and two
      distinct points repeated (rank 1)
- S4  collinear, exactly planar and cubic lattice neighbourhoods (repeated eigenvalues; exact in fp32 when the count
      is a power of two)
- S5  finite points whose lists hold a NaN or a +-inf row (NaN covariances and normals; NaN keys in the median sort)
- S6  the bundled target translated by [812.5, -640.25, 35] and [18000, -12500, 120] with lists from before the
      translation (the un-centred fp32 sums cancel: indefinite matrices)
- S7  S1-S5 under robust covariance with min_robust_scale in {0, 1e-3, 1}, mad_scale in {0, 1.5}, every loss and
      0, 1 and 3 iterations (a zero scale makes r / s infinite)

Covariances and robust covariances equal the oracle bit for bit (NaN in the same places), normals from the k-NN and
from stored covariances within 1e-5 per component, plane regularisation within 1e-6.  The box filter, the angle of
incidence filter and farthest point sampling (10^6-point lattice with exact ties across blocks, 10^6 random points:
the grid-stride loop; +-inf and NaN rows; a chosen first index through the C-ABI) select exactly the oracle's points.

The tests without the gpu mark check that each scenario is what it claims and check the oracle itself against
independent fp64 numpy restatements on inputs kept away from decision boundaries."""
import ctypes as C
import os
import shutil
import subprocess
from functools import lru_cache

import numpy as np
import pytest

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
F32 = np.float32
EPS32 = float(np.finfo(np.float32).eps)
LOSSES = ("NONE", "HUBER", "TUKEY", "CAUCHY", "GEMAN_MCCLURE")
PLAIN_K = (1, 2, 3, 4, 5, 7, 31, 64, 65, 128)
ROBUST_K = (1, 3, 4, 5, 7, 31, 63, 64)
FAR_OFFSETS = ((812.5, -640.25, 35.0), (18000.0, -12500.0, 120.0))
# Rows whose two smallest eigenvalues lie within this fraction of the largest |eigenvalue| (fp64, on the oracle's
# matrix) have no well-defined smallest eigenvector: any unit vector of the near-degenerate plane is a valid normal,
# and the fp32 Cardano solve picks one from rounding noise.  Such a row may exceed the 1e-5 bound and is then checked
# for what a normal must satisfy instead.
NEAR_REPEATED_GAP = 1e-2


# ------------------------------------------------------------------ shared helpers
def _bundled_target() -> np.ndarray:
    return np.load(os.path.join(GOLDEN, "bundled_pair.npz"))["target_ds"]


@lru_cache(maxsize=None)
def _bundled_lists(k: int) -> np.ndarray:
    """exact k-NN lists of the bundled target over itself (the oracle's brute force: what the index returns)"""
    tgt = _bundled_target()
    idx, _ = oracle.knn_bruteforce(tgt, tgt, k)
    idx.setflags(write=False)
    return idx


def _xyz1(xyz) -> np.ndarray:
    xyz = np.asarray(xyz, np.float64)
    return np.c_[xyz, np.ones(len(xyz))].astype(F32)


def assert_bits_equal(got, want, what=""):
    """equal bit for bit wherever neither side is NaN, NaN in exactly the same places (sign and payload free)"""
    got, want = np.asarray(got, F32), np.asarray(want, F32)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    gn, wn = np.isnan(got), np.isnan(want)
    assert np.array_equal(gn, wn), (what, "NaN positions differ", np.argwhere(gn != wn)[:5])
    ok = ~gn
    same = got[ok].view(np.uint32) == want[ok].view(np.uint32)
    if not same.all():
        bad = np.argwhere(ok)[~same][:5]
        pytest.fail(f"{what}: {int((~same).sum())} entries differ, first at {bad.tolist()}: "
                    f"{got[tuple(bad[0])]!r} vs {want[tuple(bad[0])]!r}")


def assert_close_nan_equal(got, want, tol, what=""):
    gn, wn = np.isnan(got), np.isnan(want)
    assert np.array_equal(gn, wn), (what, "NaN positions differ", np.argwhere(gn != wn)[:5])
    err = np.abs(np.where(gn, 0, got.astype(np.float64) - np.where(wn, 0, want)))
    assert err.max(initial=0.0) <= tol, (what, float(err.max()), np.unravel_index(err.argmax(), err.shape))


def check_normals(got, want, pts, covs, what):
    """<= 1e-5 per component against the oracle.  A row over the bound must have near-repeated smallest eigenvalues
    (fp64, on the oracle's covariance); it is then checked for unit length, a small eigen-residual and the sign rule
    dot(n, p) <= 1 on the GPU's own vector.  Returns how many rows took that path."""
    got, want = np.asarray(got, F32), np.asarray(want, F32)
    assert (got[:, 3] == 0).all(), what
    gn, wn = np.isnan(got), np.isnan(want)
    assert np.array_equal(gn, wn), (what, "NaN positions differ", np.argwhere(gn != wn)[:5])
    err = np.where(gn, 0, np.abs(got.astype(np.float64) - np.where(wn, 0, want))).max(axis=1)
    over = np.flatnonzero(err > 1e-5)
    if len(over):
        A = covs[over, :3, :3].astype(np.float64)
        assert np.isfinite(A).all(), (what, over[:5])
        lam = np.linalg.eigvalsh(A)
        scale = np.abs(lam).max(axis=1)
        gap = lam[:, 1] - lam[:, 0]
        far = gap > NEAR_REPEATED_GAP * scale
        assert not far.any(), (what, "normal off by more than 1e-5 on a well-separated row", over[far][:5],
                               err[over][far][:5], (gap / scale)[far][:5])
        n = got[over, :3].astype(np.float64)
        assert np.abs(np.linalg.norm(n, axis=1) - 1.0).max() <= 1e-5, what
        ray = np.einsum("ri,rij,rj->r", n, A, n)
        resid = np.linalg.norm(np.einsum("rij,rj->ri", A, n) - ray[:, None] * n, axis=1)
        assert (resid <= gap + 1e-4 * scale).all(), (what, resid, gap, scale)
        p = pts[over, :3].astype(np.float64)
        assert ((n * p).sum(1) <= 1.0 + 1e-5 * np.maximum(1.0, np.linalg.norm(p, axis=1))).all(), what
    print(f"{what}: {len(over)} normal rows took the near-repeated-eigenvalue path")
    return len(over)


def _unique_rows(covs) -> np.ndarray:
    flat = np.ascontiguousarray(covs.reshape(len(covs), 16)).view(np.uint32)
    _, first = np.unique(flat, axis=0, return_index=True)
    return covs[np.sort(first)]


# ------------------------------------------------------------------ scenario builders (seeded, host only)
def scenario_s2(k: int, seed: int = 2):
    """bundled target, exact lists with -1 written into the first 410 rows"""
    tgt = _bundled_target()
    idx = _bundled_lists(k).copy()
    rng = np.random.default_rng(seed)
    for r in range(0, 100):                       # at the end
        idx[r, k - rng.integers(1, k - 1):] = -1
    for r in range(100, 200):                     # in the middle, first and last entries kept
        s = int(rng.integers(1, k - 2))
        idx[r, s:s + int(rng.integers(1, k - s))] = -1
    for r in range(200, 300):                     # at the front
        idx[r, :rng.integers(1, k - 1)] = -1
    for r, valid in ((range(300, 350), 3), (range(350, 400), 4)):  # either side of cnt < 4
        for i in r:
            drop = np.setdiff1d(np.arange(k), rng.choice(k, valid, replace=False))
            idx[i, drop] = -1
    idx[400:410] = -1
    return tgt, idx


def scenario_s3(seed: int = 3):
    """duplicates: rows of 10 copies of one point (1/10 is inexact: near zero), 8 copies and two -1, two distinct
    points 5 + 5 and 4 + 4 with two -1 (rank 1); near the origin and ~100 m out.  The first 64 points have few
    significant bits, so every fp32 sum over them is exact and 8 copies give exactly the zero matrix; the last 64
    have full-precision coordinates."""
    rng = np.random.default_rng(seed)
    dyadic = np.r_[rng.integers(-320, 321, (32, 3)) / 16, rng.integers(320, 481, (32, 3)) / 4]
    pts = _xyz1(np.r_[dyadic, rng.uniform(-20, 20, (32, 3)), rng.uniform(80, 120, (32, 3))])
    n, k = len(pts), 10
    idx = np.empty((n, k), np.int32)
    for r in range(n):
        o = (r + 1 + int(rng.integers(0, n - 1))) % n
        kind = r % 4
        if kind == 0:
            row = [r] * 10
        elif kind == 1:
            row = [r] * 8 + [-1] * 2
        elif kind == 2:
            row = [r, o] * 5
        else:
            row = [r] * 4 + [o] * 4 + [-1] * 2
        idx[r] = rng.permutation(row) if kind != 2 else row
    return pts, idx


def _lattice_shapes():
    """(kind, axes, counts per axis): collinear, planar (orthogonal axes of equal length: the two in-plane
    eigenvalues repeat) and cubic (all three repeat)"""
    lines = [((1, 0, 0),), ((0, 0, 1),), ((1, 2, 2),), ((-2, 1, 2),)]
    planes = [((1, 0, 0), (0, 1, 0)), ((2, 1, 0), (-1, 2, 0)), ((1, 2, 2), (2, 1, -2))]
    cubes = [((1, 0, 0), (0, 1, 0), (0, 0, 1)), ((1, 2, 2), (2, 1, -2), (2, -2, 1))]
    out = []
    for ax in lines:
        for m in (8, 16, 5, 7):
            out.append(("line", ax, (m,)))
    for ax in planes:
        for m in (4, 2, 3):
            out.append(("plane", ax, (m, m)))
    for ax in cubes:
        out.append(("cube", ax, (2, 2, 2)))
    return out


def scenario_s4(seed: int = 4):
    """lattice neighbourhoods, k = 16 (shorter ones padded with -1 at random positions): every point of a
    neighbourhood lists exactly that neighbourhood.  Integer coordinates within +-40: every sum and product is exact
    in fp32, so with a power-of-two count the fp32 covariance is the exact one.  Returns pts, idx, kind per row and
    whether the row's count is a power of two."""
    rng = np.random.default_rng(seed)
    k = 16
    pts, rows, kinds, exact = [], [], [], []
    for kind, axes, counts in _lattice_shapes():
        for _ in range(3):
            p0 = rng.integers(-20, 21, 3)
            grid = np.stack(np.meshgrid(*[np.arange(m) for m in counts], indexing="ij"), -1).reshape(-1, len(counts))
            nb = p0 + grid @ np.asarray(axes)
            s, m = len(pts), len(nb)
            pts.extend(nb.tolist())
            for _ in range(m):
                rows.append(rng.permutation(np.r_[np.arange(s, s + m), np.full(k - m, -1)]))
                kinds.append(kind)
                exact.append(m & (m - 1) == 0)
    return _xyz1(pts), np.asarray(rows, np.int32), np.asarray(kinds), np.asarray(exact)


NONFINITE_ROWS = ((np.nan, 1.0, 2.0), (3.0, np.inf, 1.0), (-2.0, 4.0, -np.inf), (np.nan, np.nan, np.nan),
                  (np.inf, np.inf, np.inf))


def scenario_s5(seed: int = 5):
    """256 finite points and 5 non-finite rows; every third finite row lists one non-finite row among 10 finite
    neighbours, at a varying rank; the non-finite rows list finite neighbours"""
    rng = np.random.default_rng(seed)
    fin = rng.uniform(-30, 30, (256, 3))
    pts = _xyz1(np.r_[fin, np.asarray(NONFINITE_ROWS)])
    n, k = len(pts), 10
    idx = np.empty((n, k), np.int32)
    for r in range(n):
        idx[r] = rng.choice(256, k, replace=False)
        if r < 256 and r % 3 == 0:
            idx[r, (r // 3) % k] = 256 + (r // 3) % len(NONFINITE_ROWS)
    return pts, idx


def scenario_s6(offset):
    """the bundled target moved by offset (fp32 adds), lists from before the move"""
    tgt = _bundled_target()
    moved = tgt.copy()
    moved[:, :3] += np.asarray(offset, F32)
    return moved, _bundled_lists(10)


def robust_grid():
    """S7: every loss with min_robust_scale x mad_scale x iterations; NONE runs the plain estimate whatever the
    parameters, so once"""
    yield "NONE", 1.0, 1.0, 1
    for loss in LOSSES[1:]:
        for floor_ in (0.0, 1e-3, 1.0):
            for mad in (0.0, 1.5):
                for iters in (0, 1, 3):
                    yield loss, mad, floor_, iters


# ------------------------------------------------------------------ FPS reference with a chosen first point
_FPS_SRC = os.path.join(ROOT, "tests", "cpp", "fps_ref.cpp")
_FPS_SO = os.path.join(ROOT, "tests", "cpp", "_build", "libfps_ref.so")
_fps = None


def _fps_lib():
    global _fps
    if _fps is None:
        if not os.path.exists(_FPS_SO) or os.path.getmtime(_FPS_SO) < os.path.getmtime(_FPS_SRC):
            os.makedirs(os.path.dirname(_FPS_SO), exist_ok=True)
            tmp = _FPS_SO + f".{os.getpid()}.tmp"
            gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")
            env = {k: v for k, v in os.environ.items() if k not in ("CXX", "CC")}
            r = subprocess.run([gxx, "-std=c++20", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC",
                                "-march=x86-64-v3", "-shared", "-o", tmp, _FPS_SRC], capture_output=True, text=True,
                               env=env)
            assert r.returncode == 0, r.stderr[-4000:]
            os.replace(tmp, _FPS_SO)
        _fps = C.CDLL(_FPS_SO)
        _fps.ref_farthest_point_sampling.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_void_p]
        _fps.ref_farthest_point_sampling.restype = None
    return _fps


def fps_ref(points, num: int, first: int) -> np.ndarray:
    """selected indices, ascending, of farthest point sampling from `first` (the reference's loop)"""
    p = np.ascontiguousarray(points, F32)
    flags = np.zeros(len(p), np.uint8)
    _fps_lib().ref_farthest_point_sampling(p.ctypes.data, len(p), num, first, flags.ctypes.data)
    return np.flatnonzero(flags)


def oracle_first_index(points, seed: int = 1234) -> int:
    """the first point the operator draws from a fresh mt19937(seed) stream: the oracle's FPS stops after it at
    sampling_num = 1"""
    return int(np.flatnonzero(oracle.Rng(seed).farthest_point_sampling_flags(points, 1))[0])


def fps_lattice(side: int = 100) -> np.ndarray:
    """side^3 integer lattice in raster order: every distance is an exact integer, so ties are exact"""
    g = np.stack(np.meshgrid(*[np.arange(side)] * 3, indexing="ij"), -1).reshape(-1, 3)
    return _xyz1(g)


def fps_random(n: int = 1_000_000, seed: int = 7) -> np.ndarray:
    return _xyz1(np.random.default_rng(seed).uniform(-50, 50, (n, 3)))


def fps_nonfinite(seed: int = 8) -> np.ndarray:
    rng = np.random.default_rng(seed)
    pts = _xyz1(rng.uniform(-10, 10, (3000, 3)))
    pts[[700, 1500, 2900], 0] = [np.nan, np.inf, -np.inf]
    pts[2100, 3] = np.nan
    return pts


# ------------------------------------------------------------------ box / angle boundary points
BOX_MIN, BOX_MAX = F32(2.5), F32(40.0)


def box_cloud(seed: int = 9):
    """points whose L-inf range is exactly min / max and one fp32 step either side (on every axis, both signs),
    -0.0 coordinates, non-finite w, a point at FLT_MAX, and random points; returns (pts, which rows sit on a bound)"""
    rng = np.random.default_rng(seed)
    fmax = np.finfo(F32).max
    rows, on_bound = [], []
    for b in (BOX_MIN, BOX_MAX):
        for v in (b, np.nextafter(b, F32(np.inf)), np.nextafter(b, F32(-np.inf))):
            for axis in range(3):
                for sign in (1, -1):
                    p = rng.uniform(-0.9, 0.9, 3).astype(F32) * F32(BOX_MIN)
                    p[axis] = F32(sign) * v
                    rows.append([*p, 1.0])
                    on_bound.append(v == b)
    rows += [[-0.0, -0.0, -0.0, 1.0], [-0.0, 3.0, -0.0, 1.0], [0.0, -0.0, -BOX_MIN, 1.0], [-0.0, -0.0, -0.0, -0.0]]
    on_bound += [False, False, True, False]
    rows += [[3.0, 3.0, 3.0, w] for w in (np.nan, np.inf, -np.inf)]
    rows += [[fmax, 0.0, 0.0, 1.0], [0.0, -fmax, 1.0, 1.0], [np.inf, 0.0, 0.0, 1.0], [0.0, np.nan, 0.0, 1.0]]
    on_bound += [False] * 7
    rand = rng.uniform(-60, 60, (400, 3)).astype(F32)
    pts = np.r_[np.asarray(rows, F32), _xyz1(rand)]
    return pts, np.r_[np.asarray(on_bound), np.zeros(len(rand), bool)]


def box_runs():
    fmax = float(np.finfo(F32).max)
    return ((float(BOX_MIN), float(BOX_MAX)), (0.0, float(BOX_MAX)), (-0.0, fmax), (float(BOX_MAX), float(BOX_MIN)),
            (float(BOX_MIN), fmax), (float(BOX_MAX), float(BOX_MAX)))


def box_keep_numpy(pts, lo, hi):
    with np.errstate(invalid="ignore"):
        linf = np.abs(pts[:, :3]).max(axis=1)
        return np.isfinite(pts).all(axis=1) & ~((linf < F32(lo)) | (linf > F32(hi)))


_libm = None


def cosf(x: float) -> F32:
    """the C library's cosf, which the library and the oracle apply to the angle bounds on the host"""
    global _libm
    if _libm is None:
        _libm = C.CDLL("libm.so.6")
        _libm.cosf.restype, _libm.cosf.argtypes = C.c_float, [C.c_float]
    return F32(_libm.cosf(F32(x)))


TRIPLES = ((3, 4, 5), (5, 12, 13), (8, 15, 17), (7, 24, 25), (20, 21, 29), (9, 40, 41), (12, 35, 37), (11, 60, 61))


@lru_cache(maxsize=None)
def angle_bounds():
    """fp32 angles whose cosf is exactly a Pythagorean ratio a / c (fp32-rounded), by increasing angle:
    [(angle, cos, a, b, c)]"""
    out = []
    for a0, b0, c0 in TRIPLES:
        for a, b in ((a0, b0), (b0, a0)):
            target = F32(a) / F32(c0)
            up = dn = F32(np.arccos(np.float64(target)))
            for _ in range(64):  # outward from acos, the nearest fp32 angle first
                hit = next((x for x in (up, dn) if cosf(x) == target), None)
                if hit is not None:
                    out.append((hit, target, a, b, c0))
                    break
                up, dn = np.nextafter(up, F32(np.inf)), np.nextafter(dn, F32(-np.inf))
    return sorted(out, key=lambda t: t[0])


def angle_cloud():
    """points with stored normals: exactly at the cosine bounds (|cos| = a / c of a Pythagorean triple: every product,
    the norms and the denominator are exact integers), parallel (|cos| = 1 = cosf(0)), at the origin, normals with NaN
    or zero components, a zero normal, and random rows.  Returns pts, normals, the (min_angle, max_angle) runs and
    how many leading rows have exact integer products and norms."""
    rng = np.random.default_rng(10)
    bounds = angle_bounds()
    pts, nrm = [], []

    def add(p, n):
        pts.append([*p, 1.0])
        nrm.append([*n, 0.0])

    for _, _, a, b, c in bounds:
        for s, t in ((1, 1), (2, 3), (-1, 2)):
            add((s * a, s * b, 0), (t, 0, 0))              # |cos| = a / c
            add((0, s * b, s * a), (0, 0, -t))
    for s in (3, -5):
        add((s, 0, 0), (1, 0, 0))                          # |cos| = 1
        add((0, 0, s), (0, 0, 2))
    add((0, 0, 0), (1, 0, 0))                              # the origin
    add((-0.0, 0.0, -0.0), (0, 1, 0))
    for n in ((np.nan, 0, 1), (0, np.nan, 0), (np.nan, np.nan, np.nan), (0, 0, 0), (-0.0, 0, -0.0), (0, 1, 0), (1, 0, 0)):
        add(rng.uniform(-9, 9, 3), n)
    rp = rng.uniform(-30, 30, (300, 3))
    rn = rng.normal(size=(300, 3))
    rn /= np.linalg.norm(rn, axis=1, keepdims=True)
    for p, n in zip(rp, rn):
        add(p, n)
    pts, nrm = np.asarray(pts, F32), np.asarray(nrm, F32)
    half_pi = float(F32(np.pi / 2))
    runs = [(0.0, float(bounds[0][0])), (float(bounds[1][0]), float(bounds[2][0])), (0.0, half_pi),
            (float(bounds[-1][0]), half_pi)]
    return pts, nrm, runs, len(bounds) * 6 + 4


def exact_abs_cos(p, n):
    """|cos| of the angle filter for rows whose dot product, norms and denominator are exact small integers: then
    only the final division rounds"""
    d = (p[:, :3].astype(np.float64) * n[:, :3]).sum(1)
    den = np.sqrt((p[:, :3].astype(np.float64) ** 2).sum(1)) * np.sqrt((n[:, :3].astype(np.float64) ** 2).sum(1))
    assert np.array_equal(d, np.round(d)) and np.array_equal(den, np.round(den))
    return np.abs(d.astype(F32) / den.astype(F32))


# ================================================================== CPU: the scenarios are what they claim
def test_s4_lattices_have_repeated_eigenvalues():
    pts, idx, kinds, exact = scenario_s4()
    want_cov = oracle.covariance(pts, idx)
    for r in range(len(pts)):
        nb = pts[idx[r][idx[r] >= 0], :3].astype(np.float64)
        c = np.cov(nb.T, bias=True)
        lam = np.linalg.eigvalsh(c)
        tol = 1e-12 * lam[-1]
        if kinds[r] == "line":
            assert abs(lam[0]) <= tol and abs(lam[1]) <= tol and lam[2] > 0.1
        elif kinds[r] == "plane":
            assert abs(lam[0]) <= tol and abs(lam[2] - lam[1]) <= tol and lam[1] > 0.1
        else:
            assert abs(lam[2] - lam[0]) <= tol and lam[0] > 0.1
        if exact[r]:  # power-of-two count: the oracle's fp32 matrix IS the exact covariance
            assert np.array_equal(want_cov[r, :3, :3].astype(np.float64), c), r
    assert exact.sum() > 100 and (~exact).sum() > 100


def test_s6_covariances_are_indefinite():
    for off in FAR_OFFSETS:
        pts, idx = scenario_s6(off)
        lam = np.linalg.eigvalsh(oracle.covariance(pts, idx)[:, :3, :3].astype(np.float64))
        neg = lam[:, 0] < -1e-3 * np.abs(lam).max(axis=1)
        assert neg.sum() >= 10, (off, int(neg.sum()))


def test_s2_s3_s5_rows_are_as_built():
    for k in (9, 10):
        _, idx = scenario_s2(k)
        valid = (idx >= 0).sum(1)
        assert (idx[:100, -1] == -1).all() and (idx[100:200, [0, -1]] >= 0).all()
        assert (idx[100:200, 1:-1] == -1).any(axis=1).all() and (idx[200:300, 0] == -1).all()
        assert (valid[300:350] == 3).all() and (valid[350:400] == 4).all() and (valid[400:410] == 0).all()
    pts, idx = scenario_s3()
    cov = oracle.covariance(pts, idx)[:, :3, :3].astype(np.float64)
    size = (pts[idx.clip(0), :3].astype(np.float64) ** 2).sum(2).max(1)  # the largest |p|^2 a row lists
    assert (cov[1:64:4] == 0).all()                                  # 8 copies of a dyadic point: exactly zero
    assert (np.abs(cov[0::4]).max(axis=(1, 2)) <= 16 * EPS32 * size[0::4]).all()     # 10 copies: rounding only
    lam = np.linalg.eigvalsh(cov[2::4])                                # two points 5 + 5: rank 1 up to rounding
    assert (np.abs(lam[:, :2]).max(1) <= 16 * EPS32 * size[2::4]).all() and (lam[:, 2] > 1.0).all()
    pts, idx = scenario_s5()
    hit = (idx >= 256).any(1)
    assert hit[:256].sum() == 86 and not hit[256:].any()
    assert np.isnan(oracle.covariance(pts, idx)[hit]).any(axis=(1, 2)).all()


def test_box_boundary_points_sit_on_the_bounds():
    pts, on_bound = box_cloud()
    linf = np.abs(pts[:, :3]).max(1)
    assert np.isin(linf[on_bound], [BOX_MIN, BOX_MAX]).all() and on_bound.sum() == 13
    for b in (BOX_MIN, BOX_MAX):
        for v in (np.nextafter(b, F32(np.inf)), np.nextafter(b, F32(-np.inf))):
            assert (linf == v).sum() == 6
    assert (np.signbit(pts[:, :3]) & (pts[:, :3] == 0)).sum() >= 6


def test_angle_boundary_points_sit_on_the_cosines():
    bounds = angle_bounds()
    assert len(bounds) >= 6, bounds
    for ang, c, a, _, cc in bounds:
        assert cosf(ang) == c == F32(a) / F32(cc)
    pts, nrm, runs, n_exact = angle_cloud()
    ac = exact_abs_cos(pts[:n_exact], nrm[:n_exact])
    assert np.array_equal(ac, np.r_[np.repeat([b[1] for b in bounds], 6), np.ones(4, F32)])
    assert cosf(0.0) == 1.0
    for lo, hi in runs:  # every run has rows on at least one of its two bounds
        assert ((ac == cosf(lo)) | (ac == cosf(hi))).sum() >= 4, (lo, hi)
    assert (ac == cosf(runs[1][0])).sum() == 6 and (ac == cosf(runs[1][1])).sum() == 6


def test_fps_lattice_ties_resolve_to_the_lowest_index():
    """exact integer distances on the lattice: once the corners and edges are taken, most rounds have several equal
    maxima spread over different 256-point blocks (up to ~60 on the 10^6-point lattice), and the reference picks the
    lowest index among them"""
    pts = fps_lattice(40)
    g = pts[:, :3].astype(np.int64)
    first = 40 * 40 * 17 + 40 * 3 + 29
    rounds = 400
    sel = fps_ref(pts, rounds, first)
    order, dist, tied, most = [first], np.full(len(g), np.iinfo(np.int64).max), 0, 0
    for _ in range(rounds - 1):
        dist = np.minimum(dist, ((g - g[order[-1]]) ** 2).sum(1))
        ties = np.flatnonzero(dist == dist.max())
        tied += ties.max() // 256 != ties.min() // 256
        most = max(most, len(ties))
        order.append(int(ties[0]))
    assert np.array_equal(sel, np.unique(order)) and len(sel) == rounds
    assert tied >= rounds // 2 and most >= 20, (tied, most)


def test_fps_reference_matches_the_oracle():
    """the chosen-first reference, started where the oracle's stream starts, selects the oracle's points: random
    points, duplicates, non-finite rows, a lattice"""
    rng = np.random.default_rng(12)
    clouds = [_xyz1(rng.uniform(-5, 5, (4000, 3))), np.repeat(_xyz1(rng.uniform(-1, 1, (30, 3))), 7, axis=0),
              fps_nonfinite(), fps_lattice(16)]
    for pts in clouds:
        first = oracle_first_index(pts)
        for num in (n for n in (2, 37, 300) if n < len(pts)):  # (n <= num keeps every point: no selection runs)
            want = np.flatnonzero(oracle.Rng(1234).farthest_point_sampling_flags(pts, num))
            assert np.array_equal(fps_ref(pts, num, first), want), num
    # the quirk: a non-finite row keeps FLT_MAX and is selected again and again once it is the farthest
    pts = fps_nonfinite()
    got = fps_ref(pts, 50, 5)
    assert len(got) == 2 and 700 in got


# ================================================================== CPU: the oracle against fp64 numpy
def test_oracle_covariance_near_origin_vs_centred_fp64():
    """un-centred fp32 sums near the origin: within (k + 4) eps max|p|^2 of the centred fp64 covariance"""
    tgt = _bundled_target()
    for k in (5, 10, 31):
        idx = _bundled_lists(k)
        got = oracle.covariance(tgt, idx)[:, :3, :3].astype(np.float64)
        nb = tgt[idx, :3].astype(np.float64)
        d = nb - nb.mean(1, keepdims=True)
        want = np.einsum("rki,rkj->rij", d, d) / k
        bound = (k + 4) * EPS32 * (nb ** 2).sum(2).max(1)
        assert (np.abs(got - want).max(axis=(1, 2)) <= bound).all(), k


def _irls_fp64(pts, idx, loss, mad, floor_, iters):
    """covariance.hpp:97-250 in fp64: weighted covariance, squared Mahalanobis distances through the inverse (zero
    when |det| < 1e-6), median over all k entries (-1 ones count as 0), scale max(mad * median, floor).  Also returns
    the rows where a decision sits within 1e-3 relative of its threshold."""
    def weighted(P, w):
        tw = w.sum()
        mean = (P * w[:, None]).sum(0) / tw
        return (P.T * w) @ P / tw - np.outer(mean, mean), mean
    out, near = np.empty((len(idx), 3, 3)), np.zeros(len(idx), bool)
    for r, row in enumerate(idx):
        valid = row >= 0
        P = pts[row[valid], :3].astype(np.float64)
        Cm, mean = weighted(P, np.ones(len(P)))
        for _ in range(iters):
            det = np.linalg.det(Cm)
            Ci = np.linalg.inv(Cm) if abs(det) >= 1e-6 else np.zeros((3, 3))
            d = P - mean
            d2 = np.zeros(len(row))
            d2[valid] = np.einsum("ki,ij,kj->k", d, Ci, d)
            s = max(mad * np.median(d2), floor_)
            x = d2[valid] / s
            near[r] |= abs(abs(det) - 1e-6) < 1e-9 or abs(mad * np.median(d2) - floor_) < 1e-3 * floor_
            near[r] |= bool((np.abs(x - 1) < 1e-3).any() and loss == "TUKEY")
            with np.errstate(divide="ignore"):
                w = {"HUBER": np.minimum(1, 1 / x), "TUKEY": np.where(x >= 1, 0, (1 - x * x) ** 2),
                     "CAUCHY": 1 / (1 + x * x), "GEMAN_MCCLURE": 1 / (1 + x * x) ** 2}[loss]
            w = np.where(d2[valid] <= 1e-8, 1.0, w)
            Cm, mean = weighted(P, w)
        out[r] = Cm
    return out, near


def irls_blobs(seed: int = 17):
    """well-conditioned neighbourhoods near the origin: 10 points of an anisotropic Gaussian blob (sigma 0.3, 0.2,
    0.1 m) and 2 outliers ~1.5 m out, centres within 2 m of the origin; every point lists its own blob of 12.  The
    fp32 rounding of the un-centred sums (~eps |p|^2) stays five orders below the smallest variance."""
    rng = np.random.default_rng(seed)
    pts, rows = [], []
    for b in range(300):
        c = rng.uniform(-2, 2, 3)
        blob = c + rng.normal(size=(10, 3)) * [0.3, 0.2, 0.1]
        out_dir = rng.normal(size=(2, 3))
        out = c + 1.5 * out_dir / np.linalg.norm(out_dir, axis=1, keepdims=True)
        nb = np.r_[blob, out]
        rows += [rng.permutation(np.arange(12 * b, 12 * b + 12)) for _ in range(12)]
        pts.append(nb)
    return _xyz1(np.concatenate(pts)), np.asarray(rows, np.int32)


@pytest.mark.parametrize("loss", LOSSES[1:])
def test_oracle_robust_covariance_vs_fp64_irls(loss):
    """on well-conditioned neighbourhoods, rows with a decision near its threshold left out: within 1e-3 of the
    largest entry on every row and 2e-5 on the median row (three fp32 re-weightings through an inverse; a wrong weight
    function, median or scale rule is off by percents)"""
    pts, idx = irls_blobs()
    got = oracle.covariance_robust(pts, idx, oracle.LOSS[loss], 1.5, 1e-3, 3)[:, :3, :3].astype(np.float64)
    want, near = _irls_fp64(pts, idx, loss, 1.5, 1e-3, 3)
    rel = (np.abs(got - want).max(axis=(1, 2)) / np.abs(want).max(axis=(1, 2)))[~near]
    assert near.mean() < 0.05 and rel.max() <= 1e-3 and np.median(rel) <= 2e-5, (loss, near.mean(),
                                                                                   np.quantile(rel, [0.5, 1]))
    plain = oracle.covariance(pts, idx)[:, :3, :3]
    assert (np.abs(got - plain).max(axis=(1, 2)) > 1e-2 * np.abs(plain).max(axis=(1, 2))).mean() > 0.5  # weights act


def test_oracle_fps_vs_fp64_numpy():
    """random points, rounds compared only while the farthest point leads the next by more than fp32 can blur"""
    rng = np.random.default_rng(13)
    pts = _xyz1(rng.uniform(-10, 10, (2000, 3)))
    first = oracle_first_index(pts)
    p = pts[:, :3].astype(np.float64)
    sel, dist = [first], np.full(len(p), np.inf)
    while len(sel) < 40:
        dist = np.minimum(dist, ((p - p[sel[-1]]) ** 2).sum(1))
        top2 = np.sort(dist)[-2:]
        assert top2[1] - top2[0] > 1e-5 * top2[1], len(sel)  # no near-tie: fp32 and fp64 pick the same point
        sel.append(int(dist.argmax()))
    assert np.array_equal(np.flatnonzero(oracle.Rng(1234).farthest_point_sampling_flags(pts, 40)), np.unique(sel))


def test_oracle_box_and_angle_flags_vs_fp64_numpy():
    rng = np.random.default_rng(14)
    pts = _xyz1(rng.uniform(-50, 50, (5000, 3)))
    pts[::97, 1] = np.nan
    linf = np.abs(pts[:, :3].astype(np.float64)).max(1)
    lo, hi = 5.0, 35.0
    away = np.isnan(linf) | ((np.abs(linf - lo) > 1e-3) & (np.abs(linf - hi) > 1e-3))
    want = np.isfinite(linf) & (linf >= lo) & (linf <= hi)
    got = oracle.box_filter(pts, lo, hi)
    assert np.array_equal(got, pts[want]) and away.mean() > 0.99
    nrm = rng.normal(size=(5000, 4)).astype(F32)
    nrm[:, 3] = 0
    for amin, amax in ((0.0, 1.2), (0.3, 1.5)):
        p, n = pts[:, :3].astype(np.float64), nrm[:, :3].astype(np.float64)
        with np.errstate(invalid="ignore"):
            ac = np.abs((p * n).sum(1)) / (np.linalg.norm(p, axis=1) * np.linalg.norm(n, axis=1))
            want = ~np.isnan(ac) & (ac >= np.cos(amax)) & (ac <= np.cos(amin))
            near = (np.abs(ac - np.cos(amax)) < 1e-5) | (np.abs(ac - np.cos(amin)) < 1e-5)
        got = oracle.angle_incidence_flags(pts, amin, amax, normals=nrm).astype(bool)
        assert np.array_equal(got[~near], want[~near]) and near.sum() < 5


# ================================================================== GPU
@pytest.fixture(scope="module")
def q(spx):
    return spx.DeviceQueue(0)


def knn_from_host(spx, q, idx) -> "object":
    """a KNNResult holding the host int32 [n][k] lists as given (distances zero: no kernel here reads them)"""
    idx = np.ascontiguousarray(idx, np.int32)
    r = spx.KNNResult()
    r.allocate(q, idx.shape[0], idx.shape[1])
    r.indices.upload(idx)
    r.distances.upload(np.zeros(idx.shape, F32))
    return r


def check_plain(spx, q, pts, nn, idx, what):
    """covariance bit for bit, normals from the k-NN and from the stored covariances, plane regularisation; returns
    (covs, normals, near-repeated rows)"""
    cloud = spx.PointCloudShared(q, pts)
    spx.covariance.estimate(nn, cloud)
    covs = cloud.covs_host()
    want = oracle.covariance(pts, idx)
    assert_bits_equal(covs, want, f"{what} covariance")
    spx.covariance.estimate_normals(nn, cloud)
    nrm = cloud.normals_host()
    deg = check_normals(nrm, oracle.normals(pts, idx), pts, want, f"{what} normals")
    cloud.normals = None
    spx.covariance.extract_normals(cloud)
    deg += check_normals(cloud.normals_host(), oracle.normals_from_covs(pts, covs), pts, want,
                         f"{what} normals from covariances")
    check_plane(spx, q, covs, what)
    return covs, nrm, deg


def check_plane(spx, q, covs, what):
    u = _unique_rows(covs)
    pts = np.zeros((len(u), 4), F32)
    pts[:, 3] = 1
    c = spx.PointCloudShared(q, pts, u)
    spx.covariance.update_covariance_plane(c)
    assert_close_nan_equal(c.covs_host(), oracle.update_covariance_plane(u), 1e-6, f"{what} plane regularisation")


@pytest.mark.gpu
@pytest.mark.parametrize("k", PLAIN_K)
def test_covariance_and_normals_over_k(spx, q, k):
    """S1: lists from the index at every k up to its limit of 128"""
    tgt = _bundled_target()
    cloud = spx.PointCloudShared(q, tgt)
    nn = spx.KDTree.build(q, cloud).knn_search(cloud, k)
    idx = nn.indices_host()
    assert (idx >= 0).all()
    covs, _, _ = check_plain(spx, q, tgt, nn, idx, f"S1 k={k}")
    eye = (covs[:, :3, :3] == np.eye(3, dtype=F32)).all(axis=(1, 2))
    assert eye.all() == (k < 4)


PLAIN_SCENARIOS = {
    "S2-k9": lambda: scenario_s2(9), "S2-k10": lambda: scenario_s2(10), "S3": scenario_s3,
    "S4": lambda: scenario_s4()[:2], "S5": scenario_s5,
    "S6-near": lambda: scenario_s6(FAR_OFFSETS[0]), "S6-far": lambda: scenario_s6(FAR_OFFSETS[1]),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(PLAIN_SCENARIOS))
def test_covariance_and_normals_on_hostile_lists(spx, q, name):
    pts, idx = PLAIN_SCENARIOS[name]()
    covs, _, _ = check_plain(spx, q, pts, knn_from_host(spx, q, idx), idx, name)
    few = (idx >= 0).sum(1) < 4
    assert (covs[few, :3, :3] == np.eye(3, dtype=F32)).all()  # the identity fallback
    if name == "S5":
        assert np.isnan(covs).any(axis=(1, 2)).sum() == 86


def _robust_scenarios():
    out = {f"S1-k{k}": ("S1", k) for k in ROBUST_K}
    out.update({"S2-k9": lambda: scenario_s2(9), "S2-k10": lambda: scenario_s2(10), "S3": scenario_s3,
                "S4": lambda: scenario_s4()[:2], "S5": scenario_s5})
    return out


ROBUST_SCENARIOS = _robust_scenarios()


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(ROBUST_SCENARIOS))
def test_robust_covariance_scale_extremes(spx, q, name):
    """S7: every loss x min_robust_scale {0, 1e-3, 1} x mad_scale {0, 1.5} x iterations {0, 1, 3}, bit for bit"""
    sc = ROBUST_SCENARIOS[name]
    if isinstance(sc, tuple):
        pts = _bundled_target()
        c0 = spx.PointCloudShared(q, pts)
        nn = spx.KDTree.build(q, c0).knn_search(c0, sc[1])
        idx = nn.indices_host()
    else:
        pts, idx = sc()
        nn = knn_from_host(spx, q, idx)
    cloud = spx.PointCloudShared(q, pts)
    produced, differs = [], 0
    plain = oracle.covariance(pts, idx)
    for loss, mad, floor_, iters in robust_grid():
        spx.covariance.estimate_robust(nn, cloud, spx.RobustLossType[loss], mad, floor_, iters)
        got = cloud.covs_host()
        want = oracle.covariance_robust(pts, idx, oracle.LOSS[loss], mad, floor_, iters)
        assert_bits_equal(got, want, f"{name} {loss} mad={mad} floor={floor_} iters={iters}")
        produced.append(got)
        differs += not np.array_equal(got, plain, equal_nan=True)
    assert differs > 0 or idx.shape[1] < 4 or name == "S3"
    produced = _unique_rows(np.concatenate(produced))
    check_plane(spx, q, produced, f"{name} robust")
    # normals from the stored robust covariances (the sign rule needs a point: the origin, w = 1)
    origin = np.zeros((len(produced), 4), F32)
    origin[:, 3] = 1
    c = spx.PointCloudShared(q, origin, produced)
    spx.covariance.extract_normals(c)
    check_normals(c.normals_host(), oracle.normals_from_covs(origin, produced), origin, produced,
                  f"{name} robust normals from covariances")


def _kept(spx, out) -> np.ndarray:
    return out.intensities.download().astype(np.int64)


def _angle_runs(pf, spx, q, pts, normals, covs, runs, what):
    for lo, hi in runs:
        cloud = spx.PointCloudShared(q, pts, covs, normals)
        cloud.set_intensities(np.arange(len(pts), dtype=F32))
        out = pf.angle_incidence_filter(cloud, lo, hi, spx.PointCloudShared(q))
        want = np.flatnonzero(oracle.angle_incidence_flags(pts, lo, hi, normals=normals, covs=covs))
        got = _kept(spx, out)
        assert np.array_equal(got, want), (what, lo, hi, np.setxor1d(got, want)[:10])
        assert np.array_equal(out.points_host(), pts[want])
        if normals is not None:
            assert np.array_equal(out.normals_host(), normals[want], equal_nan=True)
        else:
            assert np.array_equal(out.covs_host(), covs[want], equal_nan=True)


ANGLE_RUNS = ((0.0, float(F32(80.0 * np.pi / 180.0))), (0.2, 1.2), (0.0, float(F32(np.pi / 2))))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(PLAIN_SCENARIOS))
def test_angle_filter_on_scenario_clouds(spx, q, name):
    """from the covariances and from the normals the scenario produces, including NaN ones (S5): a finite point with a
    NaN normal is kept, as the reference keeps it"""
    pts, idx = PLAIN_SCENARIOS[name]()
    nn = knn_from_host(spx, q, idx)
    cloud = spx.PointCloudShared(q, pts)
    spx.covariance.estimate(nn, cloud)
    spx.covariance.estimate_normals(nn, cloud)
    covs, nrm = cloud.covs_host(), cloud.normals_host()
    pf = spx.PreprocessFilter(q)
    _angle_runs(pf, spx, q, pts, None, covs, ANGLE_RUNS, f"{name} covariances")
    _angle_runs(pf, spx, q, pts, nrm, None, ANGLE_RUNS, f"{name} normals")
    if name == "S5":
        # a partly NaN covariance gives a NaN normal; an all-NaN one (a NaN or +inf row in every coordinate) looks
        # like the zero matrix to the eigen solver (fmax drops NaN) and gives the x axis
        nan_rows = np.flatnonzero(np.isnan(nrm).any(1) & np.isfinite(pts).all(1))
        assert len(nan_rows) == 52
        keep = oracle.angle_incidence_flags(pts, 0.0, 1.2, normals=nrm).astype(bool)
        assert keep[nan_rows].all()


@pytest.mark.gpu
def test_angle_filter_at_the_bounds_and_on_degenerate_normals(spx, q):
    pts, nrm, runs, _ = angle_cloud()
    pf = spx.PreprocessFilter(q)
    _angle_runs(pf, spx, q, pts, nrm, None, runs, "stored normals")
    # the same directions as covariances: diag with the smallest variance along the stored normal's axis
    axis_rows = np.flatnonzero(((np.abs(nrm[:, :3]) > 0).sum(1) == 1) & np.isfinite(nrm).all(1))
    covs = np.zeros((len(axis_rows), 4, 4), F32)
    for j, r in enumerate(axis_rows):
        a = int(np.argmax(np.abs(nrm[r, :3])))
        covs[j, :3, :3] = np.diag(np.where(np.arange(3) == a, F32(0.25), F32(4.0)))
    assert np.array_equal(np.abs(oracle.normals_from_covs(pts[axis_rows], covs)[:, :3]),
                          (np.abs(nrm[axis_rows, :3]) > 0).astype(F32))
    _angle_runs(pf, spx, q, pts[axis_rows], None, covs, runs, "covariances")
    # NaN covariances: a NaN normal, kept
    nanc = np.zeros((len(pts), 4, 4), F32)
    nanc[:, :3, :3] = np.eye(3, dtype=F32)
    nanc[::5, 1, 1] = np.nan
    _angle_runs(pf, spx, q, pts, None, nanc, runs[:2], "NaN covariances")


@pytest.mark.gpu
def test_box_filter_at_the_bounds(spx, q):
    pts, _ = box_cloud()
    n = len(pts)
    rng = np.random.default_rng(15)
    covs = rng.uniform(-1, 1, (n, 4, 4)).astype(F32)
    nrm, rgb = rng.uniform(-1, 1, (n, 4)).astype(F32), rng.uniform(0, 1, (n, 4)).astype(F32)
    ts = rng.uniform(0, 100, n).astype(F32)
    pf = spx.PreprocessFilter(q)
    for lo, hi in box_runs():
        keep = box_keep_numpy(pts, lo, hi)
        want = oracle.box_filter(pts, lo, hi)
        assert np.array_equal(want, pts[keep]), (lo, hi)
        cloud = spx.PointCloudShared(q, pts, covs, nrm)
        cloud.set_rgb(rgb)
        cloud.set_intensities(np.arange(n, dtype=F32))
        cloud.set_timestamp_offsets(ts)
        out = pf.box_filter(cloud, lo, hi, spx.PointCloudShared(q))
        assert np.array_equal(_kept(spx, out), np.flatnonzero(keep)), (lo, hi)
        assert np.array_equal(out.points_host().view(np.uint32), want.view(np.uint32))
        assert np.array_equal(out.covs_host(), covs[keep]) and np.array_equal(out.normals_host(), nrm[keep])
        assert np.array_equal(out.rgb.download(), rgb[keep]) and np.array_equal(out.timestamp_offsets.download(), ts[keep])
        # the points-only entry point
        dst = spx.DeviceArray(q, (n, 4), F32)
        m = C.c_size_t()
        spx.api.check(spx.lib().spx_box_filter(q.handle, cloud.points.ptr, n, lo, hi, dst.ptr, C.byref(m)))
        assert m.value == keep.sum() and np.array_equal(dst.download(m.value).view(np.uint32), want.view(np.uint32))
    assert box_keep_numpy(pts, *box_runs()[3]).sum() == 0 and box_keep_numpy(pts, *box_runs()[2]).sum() > 400


def fps_abi(spx, q, cloud, num: int, first: int) -> np.ndarray:
    """spx_farthest_point_sampling with a chosen first index: the call PreprocessFilter.farthest_point_sampling
    makes after drawing its first index"""
    idx = spx.DeviceArray(q, (max(num, 1),), np.int32)
    m = C.c_size_t()
    spx.api.check(spx.lib().spx_farthest_point_sampling(q.handle, cloud.points.ptr, cloud.size(), num, first, idx.ptr,
                                                       C.byref(m)))
    return idx.download(m.value).astype(np.int64)


def fps_wrapper(spx, q, cloud, num: int) -> np.ndarray:
    out = spx.PreprocessFilter(q).farthest_point_sampling(cloud, num)
    return _kept(spx, out)


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["lattice", "random"])
def test_fps_million_points(spx, q, which):
    """10^6 points: more than 2048 resident threads x SMs, so every thread strides over several points; on the
    lattice, massive exact ties across blocks resolve to the lowest index"""
    pts = fps_lattice(100) if which == "lattice" else fps_random()
    n = len(pts)
    assert n == 1_000_000 and n > 2048 * q.device_info()["sm_count"]
    cloud = spx.PointCloudShared(q, pts)
    cloud.set_intensities(np.arange(n, dtype=F32))
    first = oracle_first_index(pts)
    for num in (2, 64, 1000):
        got = fps_wrapper(spx, q, cloud, num)
        assert np.array_equal(got, fps_ref(pts, num, first)), (which, num)
        assert len(got) == num
    for first in (0, n - 1, n // 2 + 12345):
        assert np.array_equal(fps_abi(spx, q, cloud, 64, first), fps_ref(pts, 64, first)), (which, first)


@pytest.mark.gpu
def test_fps_small_and_nonfinite_clouds(spx, q):
    rng = np.random.default_rng(16)
    for n, num in ((100, 10), (100, 50), (255, 254), (65, 64), (1001, 1000), (3, 2)):
        pts = _xyz1(rng.uniform(-3, 3, (n, 3)))
        cloud = spx.PointCloudShared(q, pts)
        cloud.set_intensities(np.arange(n, dtype=F32))
        want = np.flatnonzero(oracle.Rng(1234).farthest_point_sampling_flags(pts, num))
        assert np.array_equal(fps_wrapper(spx, q, cloud, num), want), (n, num)
        for first in (0, n - 1, n // 2):
            assert np.array_equal(fps_abi(spx, q, cloud, num, first), fps_ref(pts, num, first)), (n, num, first)
    # +-inf and NaN rows keep FLT_MAX: the farthest one is selected again and again (the reference's behaviour)
    pts = fps_nonfinite()
    cloud = spx.PointCloudShared(q, pts)
    cloud.set_intensities(np.arange(len(pts), dtype=F32))
    for num in (2, 40):
        want = np.flatnonzero(oracle.Rng(1234).farthest_point_sampling_flags(pts, num))
        assert np.array_equal(fps_wrapper(spx, q, cloud, num), want), num
    for first in (0, 700, 1500, 2100, 2900, len(pts) - 1):
        got = fps_abi(spx, q, cloud, 40, first)
        assert np.array_equal(got, fps_ref(pts, 40, first)), first
        assert len(got) <= 3
