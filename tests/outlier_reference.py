"""CPU reference of the statistical and radius outlier filters (DESIGN.md §3.3), for the tests only.

Statistical: the k+1 nearest neighbours come from the oracle's exact brute force (orc_knn_bruteforce: the library's
fp32 distance chain, order (dist, index)); the mean distances are summed in fp32 in rank order, exactly as the
contract states, and mu / sigma are summed sequentially in fp64.  Radius: a brute-force count with the same fp32
chain (tests/cpp/outlier_count.cpp, compiled here with OpenMP and without floating-point contraction)."""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess

import numpy as np

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_SRC = os.path.join(ROOT, "tests", "cpp", "outlier_count.cpp")
_SO = os.path.join(ROOT, "tests", "cpp", "_build", "liboutlier_ref.so")
_GXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")
_lib = None


def _load():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(_SRC):
            os.makedirs(os.path.dirname(_SO), exist_ok=True)
            tmp = _SO + f".{os.getpid()}.tmp"
            env = {k: v for k, v in os.environ.items() if k not in ("CXX", "CC")}
            r = subprocess.run([_GXX, "-std=c++20", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC",
                                "-march=x86-64-v3", "-shared", "-o", tmp, _SRC], capture_output=True, text=True, env=env)
            assert r.returncode == 0, r.stderr[-4000:]
            os.replace(tmp, _SO)
        _lib = C.CDLL(_SO)
        _lib.ref_radius_outlier_keep.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_float, C.c_uint32,
                                                 C.c_void_p]
        _lib.ref_radius_outlier_keep.restype = None
    return _lib


def _pts(points) -> np.ndarray:
    p = np.ascontiguousarray(points, dtype=np.float32)
    assert p.ndim == 2 and p.shape[1] == 4
    return p


def mean_distances(points, k: int, rows=None) -> np.ndarray:
    """d_i of the listed rows (all when None) against the whole cloud: float32, NaN for invalid points."""
    p = _pts(points)
    rows = np.arange(len(p), dtype=np.int64) if rows is None else np.asarray(rows, np.int64)
    out = np.full(len(rows), np.nan, np.float32)
    if len(rows) == 0 or len(p) == 0:
        return out
    kk = k + 1
    idx, d2 = oracle.knn_bruteforce(p[rows], p, kk)
    is_self = idx == rows[:, None]
    drop = np.where(is_self.any(1), is_self.argmax(1), kk - 1)
    use = (idx >= 0) & np.isfinite(d2)
    use[np.arange(len(rows)), drop] = False
    s = np.zeros(len(rows), np.float32)
    c = np.zeros(len(rows), np.int64)
    with np.errstate(invalid="ignore"):
        for j in range(kk):  # rank order, fp32 adds
            v = use[:, j]
            s = np.where(v, s + np.sqrt(d2[:, j]), s).astype(np.float32)
            c += v
        finite = np.isfinite(p[rows, :3]).all(1)
        ok = finite & (c > 0)
        out[ok] = s[ok] / c[ok].astype(np.float32)
    return out


def statistics(dbar, alpha: float):
    """(mu, sigma, threshold) over the valid (non-NaN) mean distances: sequential fp64 sums, PCL's formula, the
    variance clamped at 0; threshold +inf when at most one point is valid."""
    x = np.asarray(dbar, np.float32)
    x = x[~np.isnan(x)].astype(np.float64)
    n = len(x)
    if n == 0:
        return 0.0, 0.0, np.inf
    s1 = float(np.cumsum(x)[-1])
    s2 = float(np.cumsum(x * x)[-1])
    mu = s1 / n
    if n <= 1:
        return mu, 0.0, np.inf
    sigma = float(np.sqrt(max((s2 - s1 * s1 / n) / (n - 1), 0.0)))
    return mu, sigma, mu + float(alpha) * sigma


def statistical(points, k: int, alpha: float):
    """(keep flags, d_i, mu, sigma, threshold) of the whole cloud."""
    dbar = mean_distances(points, k)
    mu, sigma, thr = statistics(dbar, alpha)
    keep = ~np.isnan(dbar) & (dbar.astype(np.float64) <= thr)
    return keep, dbar, mu, sigma, thr


def radius(points, r: float, min_neighbors: int, rows=None) -> np.ndarray:
    """Keep flags of the listed rows (all when None): at least min_neighbors others at fp32 d^2 <= r * r."""
    p = _pts(points)
    rows_a = None if rows is None else np.ascontiguousarray(rows, np.int64)
    m = len(p) if rows_a is None else len(rows_a)
    keep = np.zeros(m, np.uint8)
    if m:
        _load().ref_radius_outlier_keep(p.ctypes.data, len(p), None if rows_a is None else rows_a.ctypes.data, m,
                                        float(r), int(min_neighbors), keep.ctypes.data)
    return keep.astype(bool)
