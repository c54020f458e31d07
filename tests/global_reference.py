"""CPU reference of FPFH descriptors, feature correspondences and correspondence RANSAC (DESIGN.md §3.6), for the
tests only.

The pair features, bins, SPFH / FPFH, the brute-force feature search, the sampler, the checks, the triad pose and the
strict fp32 count come from tests/cpp/fpfh_ref.cpp and tests/cpp/ransac_ref.cpp, compiled here with OpenMP and
without floating-point contraction.  The mutual filter, the selection, the least-squares refinement (numpy SVD
Kabsch) and the inlier lists are built in numpy."""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
from dataclasses import dataclass

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_GXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")
INVALID = 0xFFFFFFFF
DIM = 33
_libs: dict[str, C.CDLL] = {}


def _build(name: str) -> C.CDLL:
    if name not in _libs:
        src = os.path.join(ROOT, "tests", "cpp", f"{name}.cpp")
        so = os.path.join(ROOT, "tests", "cpp", "_build", f"lib{name}.so")
        if not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
            os.makedirs(os.path.dirname(so), exist_ok=True)
            tmp = so + f".{os.getpid()}.tmp"
            env = {k: v for k, v in os.environ.items() if k not in ("CXX", "CC")}
            r = subprocess.run([_GXX, "-std=c++20", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC",
                                "-march=x86-64-v3", "-shared", "-o", tmp, src], capture_output=True, text=True, env=env)
            assert r.returncode == 0, r.stderr[-4000:]
            os.replace(tmp, so)
        _libs[name] = C.CDLL(so)
    return _libs[name]


def _fpfh_lib() -> C.CDLL:
    L = _build("fpfh_ref")
    L.ref_angle_bin.argtypes = [C.c_float, C.c_float]
    L.ref_angle_bin.restype = C.c_int
    L.ref_pair_feature.argtypes = [C.c_void_p] * 6
    L.ref_pair_feature.restype = C.c_int
    L.ref_fpfh.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.ref_fpfh.restype = None
    L.ref_feature_nn.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]
    L.ref_feature_nn.restype = None
    return L


def _ransac_lib() -> C.CDLL:
    L = _build("ransac_ref")
    L.ref_ransac_draws.argtypes = [C.c_uint32, C.c_uint64, C.c_uint64, C.c_void_p]
    L.ref_ransac_draws.restype = None
    L.ref_triad.argtypes = [C.c_void_p] * 4
    L.ref_triad.restype = C.c_int
    L.ref_edges_ok.argtypes = [C.c_void_p, C.c_void_p, C.c_float]
    L.ref_edges_ok.restype = C.c_int
    L.ref_ransac_hypotheses.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_uint64, C.c_float,
                                        C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]
    L.ref_ransac_hypotheses.restype = None
    L.ref_ransac_inliers.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_float, C.c_void_p]
    L.ref_ransac_inliers.restype = None
    return L


def _f32(a, cols) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.float32)
    assert a.ndim == 2 and a.shape[1] == cols, a.shape
    return a


# ------------------------------------------------------------------ FPFH
def angle_bin(X: float, Y: float) -> int:
    return int(_fpfh_lib().ref_angle_bin(float(X), float(Y)))


def pair_feature(pi, ni, pj, nj):
    """(f2, f3, X, Y, swapped) and (b1, b2, b3) of the pair (i, j), or None when the pair is skipped"""
    a = [np.ascontiguousarray(v, np.float32).reshape(-1)[:3].copy() for v in (pi, ni, pj, nj)]
    out = np.zeros(5, np.float32)
    b = np.zeros(3, np.int32)
    ok = _fpfh_lib().ref_pair_feature(*(v.ctypes.data for v in a), out.ctypes.data, b.ctypes.data)
    return (out, b) if ok else None


def fpfh(points, normals, idx, dist, with_spfh: bool = False):
    """float32 (n, 33) FPFH rows (and the SPFH rows) from the radius neighbours idx / dist (n, k)"""
    p, nr = _f32(points, 4), _f32(normals, 4)
    idx = np.ascontiguousarray(idx, np.int32)
    dist = np.ascontiguousarray(dist, np.float32)
    n = len(p)
    k = idx.shape[1] if idx.ndim == 2 else 0
    F = np.zeros((n, DIM), np.float32)
    S = np.zeros((n, DIM), np.float32)
    if n:
        _fpfh_lib().ref_fpfh(p.ctypes.data, nr.ctypes.data, n, idx.ctypes.data, dist.ctypes.data, k, F.ctypes.data,
                             S.ctypes.data)
    return (F, S) if with_spfh else F


def feature_nn(src, tgt) -> np.ndarray:
    s, t = _f32(src, DIM), _f32(tgt, DIM)
    nn = np.full(len(s), -1, np.int32)
    if len(s) and len(t):
        _fpfh_lib().ref_feature_nn(s.ctypes.data, len(s), t.ctypes.data, len(t), nn.ctypes.data)
    return nn


def correspondences(src, tgt, mutual: bool = False):
    """(src_idx, tgt_idx) int32, ascending in the source row"""
    nn = feature_nn(src, tgt)
    keep = nn >= 0
    if mutual:
        back = feature_nn(tgt, src)
        keep &= back[np.where(keep, nn, 0)] == np.arange(len(nn))
    i = np.flatnonzero(keep).astype(np.int32)
    return i, nn[i].astype(np.int32)


# ------------------------------------------------------------------ RANSAC
def draws(H: int, seed: int, m: int) -> np.ndarray:
    c = np.zeros((H, 3), np.uint32)
    _ransac_lib().ref_ransac_draws(H, seed % 2 ** 64, m, c.ctypes.data)
    return c


def triad(p, q, fp64: bool = False):
    """float32 (3, 4) pose rows (R | t) of the triangle p (3, 3) -> q (3, 3) (with fp64: the fp64 pose before
    rounding), or None when degenerate"""
    p, q = np.ascontiguousarray(p, np.float32), np.ascontiguousarray(q, np.float32)
    P, P64 = np.zeros(12, np.float32), np.zeros(12, np.float64)
    if not _ransac_lib().ref_triad(p.ctypes.data, q.ctypes.data, P.ctypes.data, P64.ctypes.data):
        return None
    return P64.reshape(3, 4) if fp64 else P.reshape(3, 4)


def edges_ok(p, q, tau: float) -> bool:
    p, q = np.ascontiguousarray(p, np.float32), np.ascontiguousarray(q, np.float32)
    return bool(_ransac_lib().ref_edges_ok(p.ctypes.data, q.ctypes.data, float(tau)))


def gather_pairs(src_points, tgt_points, si, ti):
    """(ps, qs) float32 (M, 3); NaN rows where an index is out of range"""
    sp, tp = _f32(src_points, 4), _f32(tgt_points, 4)
    si, ti = np.asarray(si, np.int64), np.asarray(ti, np.int64)
    ok = (si >= 0) & (si < len(sp)) & (ti >= 0) & (ti < len(tp))
    ps = np.full((len(si), 3), np.nan, np.float32)
    qs = np.full((len(si), 3), np.nan, np.float32)
    ps[ok] = sp[si[ok], :3]
    qs[ok] = tp[ti[ok], :3]
    return np.ascontiguousarray(ps), np.ascontiguousarray(qs)


def hypotheses(ps, qs, H: int, seed: int, tau: float, eps: float):
    """(pose float32 (H, 3, 4), sample0 int64 (H,), counts uint32 (H,)); NaN / -1 / INVALID when invalid"""
    M = len(ps)
    pose = np.zeros((H, 12), np.float32)
    s0 = np.zeros(H, np.int64)
    counts = np.zeros(H, np.uint32)
    _ransac_lib().ref_ransac_hypotheses(ps.ctypes.data, qs.ctypes.data, M, H, seed % 2 ** 64, float(tau), float(eps),
                                        pose.ctypes.data, s0.ctypes.data, counts.ctypes.data)
    return pose.reshape(H, 3, 4), s0, counts


def inlier_flags(ps, qs, P, eps: float) -> np.ndarray:
    P = np.ascontiguousarray(P, np.float32).reshape(12)
    f = np.zeros(len(ps), np.uint8)
    if len(ps):
        _ransac_lib().ref_ransac_inliers(ps.ctypes.data, qs.ctypes.data, len(ps), P.ctypes.data, float(eps),
                                         f.ctypes.data)
    return f.astype(bool)


def select(counts) -> int:
    c = np.where(counts == INVALID, -1, counts.astype(np.int64))
    return int(np.argmax(c)) if len(c) and c.max() >= 0 else -1


def kabsch(P, Q):
    """fp64 least-squares (R, t) with R P + t ~ Q (SVD, reflection-corrected)"""
    P, Q = np.asarray(P, np.float64), np.asarray(Q, np.float64)
    pc, qc = P.mean(0), Q.mean(0)
    Hm = (P - pc).T @ (Q - qc)
    U, _, Vt = np.linalg.svd(Hm)
    D = np.diag([1.0, 1.0, np.sign(np.linalg.det(Vt.T @ U.T))])
    R = Vt.T @ D @ U.T
    return R, qc - R @ pc


@dataclass
class Result:
    pose: np.ndarray     # float32 (3, 4): rows (R | t); NaN without a model
    hypothesis: int
    inliers: np.ndarray  # int32 positions, ascending
    counts: np.ndarray   # uint32 [H]
    hyp_inliers: np.ndarray  # the winning hypothesis's inliers (what the refinement fits)


def ransac(src_points, tgt_points, si, ti, eps: float, H: int, seed: int = 0, tau: float = 0.9,
           optimize: bool = False) -> Result:
    """what spx_ransac_registration computes; with optimize the refined pose is numpy's SVD Kabsch (the device solver
    agrees with it to rounding, not bit for bit)"""
    ps, qs = gather_pairs(src_points, tgt_points, si, ti)
    M = len(ps)
    nanpose = np.full((3, 4), np.nan, np.float32)
    if M == 0:
        return Result(nanpose, -1, np.zeros(0, np.int32), np.full(H, INVALID, np.uint32), np.zeros(0, np.int32))
    pose, _, counts = hypotheses(ps, qs, H, seed, tau, eps)
    best = select(counts)
    if best < 0:
        return Result(nanpose, -1, np.zeros(0, np.int32), counts, np.zeros(0, np.int32))
    P = pose[best]
    hyp_in = np.flatnonzero(inlier_flags(ps, qs, P, eps)).astype(np.int32)
    if optimize and len(hyp_in) >= 3:
        R, t = kabsch(ps[hyp_in], qs[hyp_in])
        Pr = np.c_[R, t].astype(np.float32)
        if np.isfinite(Pr).all():
            P = Pr
    inl = np.flatnonzero(inlier_flags(ps, qs, P, eps)).astype(np.int32)
    return Result(np.asarray(P, np.float32), best, inl, counts, hyp_in)


def pose_to_T(P) -> np.ndarray:
    T = np.eye(4, dtype=np.float32)
    T[:3, :] = P
    return T
