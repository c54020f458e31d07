"""CPU reference of Euclidean cluster extraction (DESIGN.md §3.4), for the tests only.

Edges: every pair of finite points with the library's fp32 d^2 <= t * t (tests/cpp/cluster_edges.cpp, compiled here
with OpenMP and without floating-point contraction).  Small clouds are searched by brute force; larger ones take their
candidates from scipy's cKDTree.query_pairs at t (1 + 1e-4) in fp64, which covers the few-ulp gap between the fp32
chain and the exact distance, and keep the candidates that pass the fp32 test.  Components come from
scipy.sparse.csgraph.connected_components; the size filter, the order, the labels and the CSR are built in numpy."""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess

import numpy as np
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components
from scipy.spatial import cKDTree

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_SRC = os.path.join(ROOT, "tests", "cpp", "cluster_edges.cpp")
_SO = os.path.join(ROOT, "tests", "cpp", "_build", "libcluster_ref.so")
_GXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")
BRUTE_MAX = 4096  # finite points up to which the edges come from the O(n^2) brute force
MAX_SIZE = 2 ** 31 - 1
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
        _lib.ref_pairs_within.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_float, C.c_void_p]
        _lib.ref_pairs_within.restype = None
        _lib.ref_brute_pairs.argtypes = [C.c_void_p, C.c_size_t, C.c_float, C.c_void_p, C.c_size_t]
        _lib.ref_brute_pairs.restype = C.c_size_t
    return _lib


def _pts(points) -> np.ndarray:
    p = np.ascontiguousarray(points, dtype=np.float32)
    assert p.ndim == 2 and p.shape[1] == 4
    return p


def pairs_within(points, pairs, t: float) -> np.ndarray:
    """keep flags of the candidate pairs (int64 [m, 2]): fp32 d^2 <= t * t"""
    p = _pts(points)
    pr = np.ascontiguousarray(pairs, np.int64).reshape(-1, 2)
    keep = np.zeros(len(pr), np.uint8)
    if len(pr):
        _load().ref_pairs_within(p.ctypes.data, pr.ctypes.data, len(pr), float(t), keep.ctypes.data)
    return keep.astype(bool)


def brute_edges(points, t: float) -> np.ndarray:
    """every pair i < j of finite points at fp32 d^2 <= t * t, O(n^2)"""
    p = _pts(points)
    cap = 1 << 16
    while True:
        out = np.empty((cap, 2), np.int64)
        m = _load().ref_brute_pairs(p.ctypes.data, len(p), float(t), out.ctypes.data, cap)
        if m <= cap:
            return out[:m]
        cap = m


def edges(points, t: float) -> np.ndarray:
    """every pair i < j of finite points at fp32 d^2 <= t * t (int64 [m, 2])"""
    p = _pts(points)
    fin = np.flatnonzero(np.isfinite(p[:, :3]).all(1))
    if len(fin) <= BRUTE_MAX:
        return brute_edges(p, t)
    cand = cKDTree(p[fin, :3].astype(np.float64)).query_pairs(float(t) * (1 + 1e-4), output_type="ndarray")
    cand = fin[cand.astype(np.int64)] if len(cand) else np.zeros((0, 2), np.int64)
    return cand[pairs_within(p, cand, t)]


def clusters_from_edges(n: int, finite: np.ndarray, e: np.ndarray, min_size: int = 1, max_size: int = MAX_SIZE):
    """(labels int32[n], indices int32[M], offsets uint32[C + 1]) of the components of the graph on n nodes with edge
    list e; non-finite nodes belong to no cluster"""
    if n == 0:
        return np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(1, np.uint32)
    e = np.asarray(e, np.int64).reshape(-1, 2)
    g = coo_matrix((np.ones(len(e), np.int8), (e[:, 0], e[:, 1])), shape=(n, n))
    _, comp = connected_components(g, directed=False)
    comp = np.where(finite, comp, -1)
    ids = np.flatnonzero(finite)
    ucomp, first, size = np.unique(comp[ids], return_index=True, return_counts=True)
    smallest = ids[first]  # (ids ascending: the first occurrence is the smallest member)
    ok = (size >= min_size) & (size <= max_size)
    ucomp, smallest, size = ucomp[ok], smallest[ok], size[ok]
    order = np.lexsort((smallest, -size))
    rank = np.full(n + 1, -1, np.int64)  # (component ids are < n: rank[-1], for the non-finite nodes, stays -1)
    rank[ucomp[order]] = np.arange(len(order))
    labels = rank[comp].astype(np.int32)
    kept = np.flatnonzero(labels >= 0)
    indices = kept[np.argsort(labels[kept], kind="stable")].astype(np.int32)
    offsets = np.zeros(len(order) + 1, np.uint32)
    offsets[1:] = np.cumsum(size[order])
    return labels, indices, offsets


def clusters(points, t: float, min_size: int = 1, max_size: int = MAX_SIZE, e: np.ndarray | None = None):
    """(labels, indices, offsets) of the cloud, as spx_euclidean_clusters defines them"""
    p = _pts(points)
    e = edges(p, t) if e is None else e
    return clusters_from_edges(len(p), np.isfinite(p[:, :3]).all(1), e, min_size, max_size)
