"""CPU reference of RANSAC plane segmentation (DESIGN.md §3.5), for the tests only.

The sampler, the fp64 plane of every hypothesis, its validity, its fp32 coefficients and its strict fp32 inlier count
come from tests/cpp/plane_ref.cpp, compiled here with OpenMP and without floating-point contraction.  The selection,
the refinement (fp64 moments of the inliers shifted by p0, numpy.linalg.eigh) and the inlier / remainder lists are
built in numpy."""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
from dataclasses import dataclass

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_SRC = os.path.join(ROOT, "tests", "cpp", "plane_ref.cpp")
_SO = os.path.join(ROOT, "tests", "cpp", "_build", "libplane_ref.so")
_GXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")
INVALID = 0xFFFFFFFF
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
        _lib.ref_plane_draws.argtypes = [C.c_uint32, C.c_uint64, C.c_uint64, C.c_void_p]
        _lib.ref_plane_draws.restype = None
        _lib.ref_plane_hypotheses.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint64,
                                              C.c_void_p, C.c_double, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.ref_plane_hypotheses.restype = None
        _lib.ref_plane_inliers.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_float, C.c_void_p]
        _lib.ref_plane_inliers.restype = None
    return _lib


def _pts(points) -> np.ndarray:
    p = np.ascontiguousarray(points, dtype=np.float32)
    assert p.ndim == 2 and p.shape[1] == 4
    return p


def finite_indices(points) -> np.ndarray:
    return np.flatnonzero(np.isfinite(_pts(points)[:, :3]).all(1)).astype(np.int64)


def draws(H: int, seed: int, nf: int) -> np.ndarray:
    """uint32 [H, 3]: the positions in F that every hypothesis draws"""
    j = np.zeros((H, 3), np.uint32)
    _load().ref_plane_draws(H, seed % 2 ** 64, nf, j.ctypes.data)
    return j


def hypotheses(points, t: float, H: int, seed: int = 0, axis=None, eps_angle: float = 0.0):
    """(coef float32 [H, 4], sample0 int64 [H], counts uint32 [H]) of every hypothesis; NaN / -1 / INVALID when
    invalid"""
    p = _pts(points)
    F = finite_indices(p)
    coef = np.zeros((H, 4), np.float32)
    s0 = np.zeros(H, np.int64)
    counts = np.zeros(H, np.uint32)
    ax = None if axis is None else np.ascontiguousarray(axis, np.float32).reshape(3)
    _load().ref_plane_hypotheses(p.ctypes.data, len(p), F.ctypes.data, len(F), H, seed % 2 ** 64,
                                 None if ax is None else ax.ctypes.data, float(eps_angle), float(t), coef.ctypes.data,
                                 s0.ctypes.data, counts.ctypes.data)
    return coef, s0, counts


def inlier_flags(points, coef, t: float) -> np.ndarray:
    p = _pts(points)
    c = np.ascontiguousarray(coef, np.float32).reshape(4)
    f = np.zeros(len(p), np.uint8)
    if len(p):
        _load().ref_plane_inliers(p.ctypes.data, len(p), c.ctypes.data, float(t), f.ctypes.data)
    return f.astype(bool)


def select(counts) -> int:
    """the valid hypothesis with most inliers, ties to the lowest index; -1 when none is valid"""
    c = np.where(counts == INVALID, -1, counts.astype(np.int64))
    return int(np.argmax(c)) if len(c) and c.max() >= 0 else -1


def refine(points, coef, p0, inliers):
    """the least-squares plane of the inliers (fp64): smallest-eigenvalue direction of their covariance, oriented like
    coef's normal, through their centroid; coef itself when fewer than 3 inliers or not finite"""
    if len(inliers) < 3:
        return np.asarray(coef, np.float32)
    q = _pts(points)[inliers, :3].astype(np.float64) - np.asarray(p0[:3], np.float64)
    m = q.mean(0)
    cov = (q - m).T @ (q - m) / len(q)
    _, V = np.linalg.eigh(cov)
    nrm = V[:, 0]
    if nrm @ np.asarray(coef[:3], np.float64) < 0:
        nrm = -nrm
    c = np.asarray(p0[:3], np.float64) + m
    out = np.r_[nrm, -(nrm @ c)].astype(np.float32)
    return out if np.isfinite(out).all() else np.asarray(coef, np.float32)


@dataclass
class Result:
    coefficients: np.ndarray  # float32 [4]
    hypothesis: int
    inliers: np.ndarray       # int32, ascending
    remainder: np.ndarray     # int32, ascending
    counts: np.ndarray        # uint32 [H]


def segment(points, t: float, H: int, seed: int = 0, axis=None, eps_angle: float = 0.0, optimize: bool = True,
            hyp=None) -> Result:
    """what spx_plane_segment computes; hyp: the output of hypotheses() for the same arguments, if already at hand"""
    p = _pts(points)
    n = len(p)
    if n == 0:
        return Result(np.full(4, np.nan, np.float32), -1, np.zeros(0, np.int32), np.zeros(0, np.int32),
                      np.full(H, INVALID, np.uint32))
    coef, s0, counts = hypotheses(p, t, H, seed, axis, eps_angle) if hyp is None else hyp
    best = select(counts)
    if best < 0:
        return Result(np.full(4, np.nan, np.float32), -1, np.zeros(0, np.int32), np.arange(n, dtype=np.int32), counts)
    c = coef[best]
    if optimize:
        c = refine(p, c, p[s0[best]], np.flatnonzero(inlier_flags(p, c, t)))
    flags = inlier_flags(p, c, t)
    return Result(np.asarray(c, np.float32), best, np.flatnonzero(flags).astype(np.int32),
                  np.flatnonzero(~flags).astype(np.int32), counts)
