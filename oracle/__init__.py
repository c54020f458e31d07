"""ORACLE — test infrastructure only.

ctypes binding of oracle/spx_oracle.cpp, the CPU restatement of the reference's hot path.
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this package; the product package (sycl_points_b200) never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "liborc.so")
_SRCS = [os.path.join(_HERE, f) for f in ("spx_oracle.cpp", "orc_math.hpp", "Makefile")]


def build(force: bool = False) -> str:
    """Compile the oracle with the committed Makefile (g++ only, no reference sources needed)."""
    stale = force or not os.path.exists(_SO) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in _SRCS)
    if stale:
        env = dict(os.environ)
        env.pop("CXX", None)
        subprocess.run(["make", "-C", _HERE] + (["-B"] if force else []), check=True, env=env,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    return _SO


def use_fast_build() -> str:
    """Switch this process to the timing build (-O3 -march=native, oracle/Makefile `fast`): bench.py's
    CPU-baseline legs only.  Must be called before the first oracle call.  The library is compiled for this
    host's CPU into a fresh private temporary directory (the source tree may be read-only), loaded, and the
    directory removed again: nothing is cached, so no other build and no other user's file is ever loaded."""
    global _SO, _lib
    import shutil
    import tempfile
    if _lib is not None:
        raise RuntimeError("oracle.use_fast_build() must be called before the oracle library is loaded")
    parity = _SO
    tmp = tempfile.mkdtemp(prefix="spx_oracle_")  # mode 0700, unpredictable name
    try:
        out = os.path.join(tmp, "liborc_fast_native.so")
        env = dict(os.environ)
        env.pop("CXX", None)
        subprocess.run(["make", "-C", _HERE, "fast", f"FAST_OUT={out}"], check=True, env=env, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT)
        _SO = out
        lib()  # mapped into the process: the file can go
    except BaseException:
        _SO = parity
        raise
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return out


class RegParams(C.Structure):
    """Field-for-field mirror of `struct orc_reg_params` (defaults: registration_params.hpp:46-114)."""
    _fields_ = [
        ("reg_type", C.c_int32), ("loss", C.c_int32), ("opt_method", C.c_int32), ("max_iterations", C.c_int32),
        ("max_corr_dist", C.c_float), ("robust_default_scale", C.c_float),
        ("crit_translation", C.c_float), ("crit_rotation", C.c_float), ("gn_lambda", C.c_float),
        ("lm_max_inner", C.c_int32), ("lm_lambda_factor", C.c_float), ("lm_init_lambda", C.c_float),
        ("lm_max_lambda", C.c_float), ("lm_min_lambda", C.c_float),
        ("dl_init_radius", C.c_float), ("dl_min_radius", C.c_float), ("dl_max_radius", C.c_float),
        ("dl_eta1", C.c_float), ("dl_eta2", C.c_float), ("dl_gamma_dec", C.c_float), ("dl_gamma_inc", C.c_float),
        ("sum_mode", C.c_int32), ("knn_mode", C.c_int32),
    ]


class RegResult(C.Structure):
    _fields_ = [
        ("T", C.c_float * 16), ("converged", C.c_int32), ("iterations", C.c_int32),
        ("H", C.c_float * 36), ("b", C.c_float * 6), ("error", C.c_float),
        ("H_raw", C.c_float * 36), ("b_raw", C.c_float * 6), ("error_raw", C.c_float), ("inlier", C.c_uint32),
    ]


REG = {"POINT_TO_POINT": 0, "POINT_TO_PLANE": 1, "POINT_TO_DISTRIBUTION": 2, "GICP": 3, "GENZ": 4}
LOSS = {"NONE": 0, "HUBER": 1, "TUKEY": 2, "CAUCHY": 3, "GEMAN_MCCLURE": 4}
OPT = {"GN": 0, "LM": 1, "DOGLEG": 2}

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if "liborc_fast_" not in _SO:
            build()
        _lib = C.CDLL(_SO)
        L = _lib
        L.orc_num_threads.restype = C.c_int
        L.orc_rng_create.restype = C.c_void_p
        L.orc_rng_create.argtypes = [C.c_uint32]
        L.orc_kdtree_build.restype = C.c_void_p
        L.orc_kdtree_size.restype = C.c_size_t
        L.orc_polar_downsample_attrs.restype = C.c_size_t
        L.orc_voxel_downsample.restype = C.c_size_t
        L.orc_voxel_downsample_unstable.restype = C.c_size_t
        L.orc_voxel_downsample_attrs.restype = C.c_size_t
        L.orc_box_filter.restype = C.c_size_t
        L.orc_voxel_key.restype = C.c_uint64
        L.orc_voxelmap_create.restype = C.c_void_p
        L.orc_voxelmap_create.argtypes = [C.c_float]
        L.orc_voxelmap_downsample.restype = C.c_size_t
        L.orc_voxelmap_overlap_ratio.restype = C.c_float
        L.orc_robust_weight.restype = C.c_float
        L.orc_robust_error.restype = C.c_float
        L.orc_robust_weight.argtypes = [C.c_int, C.c_float, C.c_float]
        L.orc_robust_error.argtypes = [C.c_int, C.c_float, C.c_float]
    return _lib


def _f(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_float))


def _i(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_int32))


def _pts(a) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.float32)
    assert a.ndim == 2 and a.shape[1] == 4
    return a


def _T(T) -> np.ndarray:
    """4x4 row-major numpy -> 16 floats column-major (Eigen::Matrix4f::data() order)."""
    T = np.asarray(T, dtype=np.float32).reshape(4, 4)
    return np.ascontiguousarray(T.T).reshape(16)


def _T_back(t16) -> np.ndarray:
    return np.array(t16, dtype=np.float32).reshape(4, 4).T.copy()


def num_threads() -> int:
    return int(lib().orc_num_threads())


def set_num_threads(n: int) -> None:
    lib().orc_set_num_threads(C.c_int(n))


class Rng:
    """std::mt19937 as the reference's test fixtures use it (test_kdtree.cpp:25-75)."""

    def __init__(self, seed: int):
        self._g = C.c_void_p(lib().orc_rng_create(seed))

    def __del__(self):
        if getattr(self, "_g", None):
            lib().orc_rng_destroy(self._g)
            self._g = None

    def uniform_points(self, n: int, rng: float) -> np.ndarray:
        out = np.empty((n, 4), np.float32)
        lib().orc_rng_uniform_points(self._g, C.c_size_t(n), C.c_float(rng), _f(out))
        return out

    def box_points(self, n: int, lo, hi) -> np.ndarray:
        out = np.empty((n, 4), np.float32)
        lo = np.asarray(lo, np.float32)
        hi = np.asarray(hi, np.float32)
        lib().orc_rng_box_points(self._g, C.c_size_t(n), _f(lo), _f(hi), _f(out))
        return out

    def weighted_random_sampling_flags(self, weights, num: int) -> np.ndarray:
        w = np.ascontiguousarray(weights, np.float32)
        flags = np.empty(len(w), np.uint8)
        lib().orc_weighted_random_sampling_flags(self._g, _f(w), C.c_size_t(len(w)), C.c_size_t(num),
                                                 flags.ctypes.data_as(C.POINTER(C.c_uint8)))
        return flags

    def farthest_point_sampling_flags(self, points, num: int) -> np.ndarray:
        p = _pts(points)
        flags = np.empty(len(p), np.uint8)
        lib().orc_farthest_point_sampling_flags(self._g, _f(p), C.c_size_t(len(p)), C.c_size_t(num),
                                                flags.ctypes.data_as(C.POINTER(C.c_uint8)))
        return flags

    def mixed_random_sampling_flags(self, weights, num: int, weighted_ratio: float) -> np.ndarray:
        w = np.ascontiguousarray(weights, np.float32)
        flags = np.empty(len(w), np.uint8)
        lib().orc_mixed_random_sampling_flags(self._g, _f(w), C.c_size_t(len(w)), C.c_size_t(num),
                                              C.c_float(weighted_ratio), flags.ctypes.data_as(C.POINTER(C.c_uint8)))
        return flags

    def random_sampling_flags(self, n: int, num: int) -> np.ndarray:
        flags = np.empty(n, np.uint8)
        lib().orc_random_sampling_flags(self._g, C.c_size_t(n), C.c_size_t(num),
                                        flags.ctypes.data_as(C.POINTER(C.c_uint8)))
        return flags


def angle_incidence_flags(points, min_angle: float, max_angle: float, normals=None, covs=None) -> np.ndarray:
    """angle_incidence_filter_operator.hpp:57-103; covs (n,16) column-major or (n,4,4) row-major"""
    p = _pts(points)
    nr = None if normals is None else _pts(normals)
    cv = None
    if covs is not None:
        cv = np.asarray(covs, np.float32)
        cv = np.ascontiguousarray(cv.transpose(0, 2, 1)).reshape(-1, 16) if cv.ndim == 3 else np.ascontiguousarray(cv)
    flags = np.empty(len(p), np.uint8)
    lib().orc_angle_incidence_flags(_f(p), _f(nr), _f(cv), C.c_size_t(len(p)), C.c_float(min_angle), C.c_float(max_angle),
                                    flags.ctypes.data_as(C.POINTER(C.c_uint8)))
    return flags


def transform_points(T, pts) -> np.ndarray:
    pts = _pts(pts)
    out = np.empty_like(pts)
    t = _T(T)
    lib().orc_transform_points(_f(t), _f(pts), C.c_size_t(len(pts)), _f(out))
    return out


def transform_cloud(T, pts, covs=None, normals=None):
    """transform::transform (transform.hpp:45-104): returns (points, covs | None, normals | None)."""
    pts = _pts(pts)
    n = len(pts)
    cv = None if covs is None else _covs_cm(covs)
    nr = None if normals is None else _pts(normals)
    o_p = np.empty_like(pts)
    o_c = None if cv is None else np.empty((n, 16), np.float32)
    o_n = None if nr is None else np.empty((n, 4), np.float32)
    t = _T(T)
    lib().orc_transform_cloud(_f(t), _f(pts), _f(cv), _f(nr), C.c_size_t(n), _f(o_p), _f(o_c), _f(o_n))
    if o_c is not None:
        o_c = np.ascontiguousarray(o_c.reshape(n, 4, 4).transpose(0, 2, 1))  # column-major -> row-major numpy
    return o_p, o_c, o_n


def knn_bruteforce(queries, targets, k: int, T=None):
    q, t = _pts(queries), _pts(targets)
    idx = np.empty((len(q), k), np.int32)
    dist = np.empty((len(q), k), np.float32)
    t16 = None if T is None else _T(T)
    lib().orc_knn_bruteforce(_f(q), C.c_size_t(len(q)), _f(t), C.c_size_t(len(t)), C.c_int(k), _f(t16), _i(idx),
                             _f(dist))
    return idx, dist


class KDTree:
    """Restatement of knn::KDTree (kdtree.hpp:292-553). mode 0 = exact oracle contract,
    mode 1 = the reference's traversal verbatim (16-entry stacks, first-visited ties)."""

    def __init__(self, points, leaf_threshold: int = 16):
        self.points = _pts(points)
        self._t = C.c_void_p(lib().orc_kdtree_build(_f(self.points), C.c_size_t(len(self.points)),
                                                    C.c_size_t(leaf_threshold)))

    def __del__(self):
        if getattr(self, "_t", None):
            lib().orc_kdtree_destroy(self._t)
            self._t = None

    @property
    def handle(self):
        return self._t

    def size(self) -> int:
        return int(lib().orc_kdtree_size(self._t))

    def knn(self, queries, k: int, T=None, mode: int = 0):
        q = _pts(queries)
        idx = np.empty((len(q), k), np.int32)
        dist = np.empty((len(q), k), np.float32)
        t16 = None if T is None else _T(T)
        lib().orc_kdtree_knn(self._t, _f(q), C.c_size_t(len(q)), C.c_int(k), _f(t16), C.c_int(mode), _i(idx),
                             _f(dist))
        return idx, dist


def eigen3(A):
    A = np.ascontiguousarray(A, np.float32).reshape(3, 3)
    vals = np.empty(3, np.float32)
    vecs = np.empty((3, 3), np.float32)
    lib().orc_eigen3(_f(A), _f(vals), _f(vecs))
    return vals, vecs


def inverse3(A):
    A = np.ascontiguousarray(A, np.float32).reshape(3, 3)
    out = np.empty((3, 3), np.float32)
    lib().orc_inverse3(_f(A), _f(out))
    return out


def covariance(points, idx) -> np.ndarray:
    """-> (n, 4, 4) row-major view of the reference's column-major Matrix4f (symmetric)."""
    p = _pts(points)
    idx = np.ascontiguousarray(idx, np.int32)
    covs = np.empty((len(p), 16), np.float32)
    lib().orc_covariance(_f(p), C.c_size_t(len(p)), _i(idx), C.c_int(idx.shape[1]), _f(covs))
    return covs.reshape(-1, 4, 4).transpose(0, 2, 1).copy()


def covariance_robust(points, idx, loss: int = 3, mad_scale: float = 1.0, min_robust_scale: float = 1.0,
                      robust_max_iterations: int = 1) -> np.ndarray:
    """covariance::estimate_robust (covariance.hpp:182-250, 323-373); default loss CAUCHY (3)"""
    p = _pts(points)
    idx = np.ascontiguousarray(idx, np.int32)
    covs = np.empty((len(p), 16), np.float32)
    lib().orc_covariance_robust(_f(p), C.c_size_t(len(p)), _i(idx), C.c_int(idx.shape[1]), C.c_int(loss),
                                C.c_float(mad_scale), C.c_float(min_robust_scale), C.c_int(robust_max_iterations), _f(covs))
    return covs.reshape(-1, 4, 4).transpose(0, 2, 1).copy()


def normals(points, idx) -> np.ndarray:
    p = _pts(points)
    idx = np.ascontiguousarray(idx, np.int32)
    out = np.empty((len(p), 4), np.float32)
    lib().orc_normals(_f(p), C.c_size_t(len(p)), _i(idx), C.c_int(idx.shape[1]), _f(out))
    return out


def _covs_cm(covs):
    if covs is None:
        return None
    c = np.asarray(covs, np.float32).reshape(-1, 4, 4)
    return np.ascontiguousarray(c.transpose(0, 2, 1)).reshape(-1, 16)


def normals_from_covs(points, covs) -> np.ndarray:
    p = _pts(points)
    c = _covs_cm(covs)
    out = np.empty((len(p), 4), np.float32)
    lib().orc_normals_from_covs(_f(p), _f(c), C.c_size_t(len(p)), _f(out))
    return out


def update_covariance_plane(covs) -> np.ndarray:
    c = _covs_cm(covs)
    out = np.empty_like(c)
    lib().orc_update_covariance_plane(_f(c), C.c_size_t(len(c)), _f(out))
    return out.reshape(-1, 4, 4).transpose(0, 2, 1).copy()


def set_genz_planarity_threshold(t: float) -> None:
    """RegistrationParams::genz.planarity_threshold (registration_params.hpp:51-53), default 0.2"""
    lib().orc_set_genz_planarity_threshold(C.c_float(t))


def set_rotation_constraint(enable: bool, weight: float = 1.0, robust_scale: float = 10.0) -> None:
    """RegistrationParams::rotation_constraint (registration_params.hpp:54-62); process-wide, default off"""
    lib().orc_set_rotation_constraint(C.c_int(1 if enable else 0), C.c_float(weight), C.c_float(robust_scale))


def genz_alpha(tgt_covs, idx, dist, max_corr_sq: float) -> float:
    """Registration::compute_genz_alpha (registration.hpp:464-511)"""
    idx = np.ascontiguousarray(idx, np.int32).reshape(-1)
    dist = np.ascontiguousarray(dist, np.float32).reshape(-1)
    lib().orc_genz_alpha.restype = C.c_float
    return float(lib().orc_genz_alpha(_f(_covs_cm(tgt_covs)), C.c_size_t(len(idx)), _i(idx), _f(dist), C.c_float(max_corr_sq)))


def robust_weight(loss: int, r: float, s: float) -> float:
    return float(lib().orc_robust_weight(loss, r, s))


def robust_error(loss: int, r: float, s: float) -> float:
    return float(lib().orc_robust_error(loss, r, s))


def linearize(reg: int, loss: int, src_pts, src_covs, tgt_pts, tgt_covs, tgt_normals, idx, dist, T, max_corr_sq,
              scale, mode: int = 1):
    sp, tp = _pts(src_pts), _pts(tgt_pts)
    sc, tc = _covs_cm(src_covs), _covs_cm(tgt_covs)
    tn = None if tgt_normals is None else _pts(tgt_normals)
    idx = np.ascontiguousarray(idx, np.int32).reshape(-1)
    dist = np.ascontiguousarray(dist, np.float32).reshape(-1)
    H = np.empty(36, np.float32)
    b = np.empty(6, np.float32)
    err = C.c_float()
    inl = C.c_uint32()
    t16 = _T(T)
    lib().orc_linearize(C.c_int(reg), C.c_int(loss), _f(sp), _f(sc), C.c_size_t(len(sp)), _f(tp), _f(tc), _f(tn),
                        _i(idx), _f(dist), _f(t16), C.c_float(max_corr_sq), C.c_float(scale), C.c_int(mode), _f(H),
                        _f(b), C.byref(err), C.byref(inl))
    return H.reshape(6, 6), b, float(err.value), int(inl.value)


def error(reg: int, loss: int, src_pts, src_covs, tgt_pts, tgt_covs, tgt_normals, idx, dist, T, max_corr_sq, scale,
          mode: int = 1):
    sp, tp = _pts(src_pts), _pts(tgt_pts)
    sc, tc = _covs_cm(src_covs), _covs_cm(tgt_covs)
    tn = None if tgt_normals is None else _pts(tgt_normals)
    idx = np.ascontiguousarray(idx, np.int32).reshape(-1)
    dist = np.ascontiguousarray(dist, np.float32).reshape(-1)
    err = C.c_float()
    inl = C.c_uint32()
    t16 = _T(T)
    lib().orc_error(C.c_int(reg), C.c_int(loss), _f(sp), _f(sc), C.c_size_t(len(sp)), _f(tp), _f(tc), _f(tn),
                    _i(idx), _f(dist), _f(t16), C.c_float(max_corr_sq), C.c_float(scale), C.c_int(mode),
                    C.byref(err), C.byref(inl))
    return float(err.value), int(inl.value)


def robust_weights(reg: int, loss: int, src_pts, src_covs, tgt_pts, tgt_covs, tgt_normals, idx, dist, T, max_corr_sq,
                   scale) -> np.ndarray:
    sp, tp = _pts(src_pts), _pts(tgt_pts)
    sc, tc = _covs_cm(src_covs), _covs_cm(tgt_covs)
    tn = None if tgt_normals is None else _pts(tgt_normals)
    idx = np.ascontiguousarray(idx, np.int32).reshape(-1)
    dist = np.ascontiguousarray(dist, np.float32).reshape(-1)
    w = np.empty(len(sp), np.float32)
    t16 = _T(T)
    lib().orc_robust_weights(C.c_int(reg), C.c_int(loss), _f(sp), _f(sc), C.c_size_t(len(sp)), _f(tp), _f(tc),
                             _f(tn), _i(idx), _f(dist), _f(t16), C.c_float(max_corr_sq), C.c_float(scale), _f(w))
    return w


def deskew_constant_velocity(pts, ts_ms, twist, duration, covs=None, normals=None):
    """deskew::deskew_point_cloud_constant_velocity (relative_pose_deskew.hpp:36-178) with twist =
    se3_log(prev^-1 * cur) given: returns (points, covs | None, normals | None)."""
    pts = _pts(pts)
    n = len(pts)
    ts = np.ascontiguousarray(ts_ms, np.float32)
    tw = np.ascontiguousarray(twist, np.float32)
    cv = None if covs is None else _covs_cm(covs)
    nr = None if normals is None else _pts(normals)
    o_p = np.empty_like(pts)
    o_c = None if cv is None else np.empty((n, 16), np.float32)
    o_n = None if nr is None else np.empty((n, 4), np.float32)
    lib().orc_deskew_constant_velocity(_f(pts), _f(nr), _f(cv), _f(ts), C.c_size_t(n), _f(tw), C.c_float(duration),
                                       _f(o_p), _f(o_n), _f(o_c))
    if o_c is not None:
        o_c = np.ascontiguousarray(o_c.reshape(n, 4, 4).transpose(0, 2, 1))
    return o_p, o_c, o_n


def se3_exp(twist) -> np.ndarray:
    tw = np.ascontiguousarray(twist, np.float32)
    out = np.empty(16, np.float32)
    lib().orc_se3_exp(_f(tw), _f(out))
    return _T_back(out)


def se3_log(T) -> np.ndarray:
    t16 = _T(T)
    out = np.empty(6, np.float32)
    lib().orc_se3_log(_f(t16), _f(out))
    return out


def so3_exp(om) -> np.ndarray:
    o = np.ascontiguousarray(om, np.float32)
    out = np.empty(4, np.float32)
    lib().orc_so3_exp(_f(o), _f(out))
    return out


def so3_log(q) -> np.ndarray:
    qq = np.ascontiguousarray(q, np.float32)
    out = np.empty(3, np.float32)
    lib().orc_so3_log(_f(qq), _f(out))
    return out


def solve6(H, b, lam: float):
    H = np.ascontiguousarray(H, np.float32).reshape(36)
    b = np.ascontiguousarray(b, np.float32)
    d = np.empty(6, np.float32)
    ok = lib().orc_solve6(_f(H), _f(b), C.c_float(lam), _f(d))
    return bool(ok), d


def dogleg_step(H, g, radius: float):
    H = np.ascontiguousarray(H, np.float32).reshape(36)
    g = np.ascontiguousarray(g, np.float32)
    p = np.empty(6, np.float32)
    sn = C.c_float()
    pr = C.c_float()
    lib().orc_dogleg_step(_f(H), _f(g), C.c_float(radius), _f(p), C.byref(sn), C.byref(pr))
    return p, float(sn.value), float(pr.value)


class Addons(C.Structure):
    """struct orc_addons: DegenerateRegularizationParams (degenerate_regularization.hpp:35-40) + MapPriorParams
    (map_prior.hpp:15-21)"""
    _fields_ = [("degenerate_type", C.c_int32), ("rot_thr", C.c_float), ("trans_thr", C.c_float),
                ("base_factor", C.c_float), ("map_prior_enabled", C.c_int32), ("rot_vel_sigma", C.c_float),
                ("trans_vel_sigma", C.c_float), ("rot_base_sigma", C.c_float), ("trans_base_sigma", C.c_float)]


def make_addons(nl_reg=False, rot_thr=10.0, trans_thr=1.0, base_factor=1.0, map_prior=False, rot_vel_sigma=1.0,
                trans_vel_sigma=1.0, rot_base_sigma=3.16e-2, trans_base_sigma=1e-2) -> Addons:
    return Addons(int(nl_reg), rot_thr, trans_thr, base_factor, int(map_prior), rot_vel_sigma, trans_vel_sigma,
                  rot_base_sigma, trans_base_sigma)


def set_addons(a: "Addons | None" = None):
    """process-wide add-on state of align() (also clears the stored prior)"""
    a = a if a is not None else make_addons()
    lib().orc_set_addons(C.byref(a))


def degenerate_regularize(a: Addons, H, b, inlier: int, T_cur, T_init):
    H = np.ascontiguousarray(H, np.float32).reshape(36).copy()
    b = np.ascontiguousarray(b, np.float32).reshape(6).copy()
    lib().orc_degenerate_regularize(C.byref(a), _f(H), _f(b), C.c_uint32(inlier), _f(_T(T_cur)), _f(_T(T_init)))
    return H.reshape(6, 6), b


def set_map_prior_state(prev: dict, T_pred):
    """MapPrior::update from an align() result dict -> (active, Omega 6x6)"""
    R = RegResult()
    R.T[:] = list(_T(prev["T"]))
    R.H_raw[:] = list(np.asarray(prev["H_raw"], np.float32).reshape(36))
    R.error_raw = float(prev["error_raw"])
    R.inlier = int(prev["inlier"])
    om = np.zeros(36, np.float32)
    lib().orc_set_map_prior_state.restype = C.c_int
    act = lib().orc_set_map_prior_state(C.byref(R), _f(_T(T_pred)), _f(om))
    return bool(act), om.reshape(6, 6)


def voxel_key(p, inv: float) -> int:
    pp = np.ascontiguousarray(p, np.float32)
    return int(lib().orc_voxel_key(_f(pp), C.c_float(inv)))


def voxel_downsample(points, voxel_size: float, min_voxel_count: int = 1, unstable: bool = False) -> np.ndarray:
    p = _pts(points)
    out = np.empty_like(p)
    fn = lib().orc_voxel_downsample_unstable if unstable else lib().orc_voxel_downsample
    m = fn(_f(p), C.c_size_t(len(p)), C.c_float(voxel_size), C.c_size_t(min_voxel_count), _f(out))
    return out[:m].copy()


class VoxelHashMap:
    """mapping::VoxelHashMap restated sequentially (voxel_hash_map.hpp:22-1066): points inserted in index order."""

    def __init__(self, voxel_size: float):
        if voxel_size <= 0:
            raise ValueError("voxel_size must be positive.")
        self.h = C.c_void_p(lib().orc_voxelmap_create(C.c_float(voxel_size)))
        self.voxel_size, self.max_staleness, self.remove_old_data_cycle = voxel_size, 100, 10
        self.rehash_threshold, self.min_num_point = 0.7, 1

    def __del__(self):
        if getattr(self, "h", None):
            lib().orc_voxelmap_destroy(self.h)
            self.h = None

    def set_params(self, **kw):
        for k, v in kw.items():
            assert hasattr(self, k), k
            setattr(self, k, v)
        lib().orc_voxelmap_set_params(self.h, C.c_float(self.voxel_size), C.c_uint32(self.max_staleness),
                                      C.c_uint32(self.remove_old_data_cycle), C.c_float(self.rehash_threshold),
                                      C.c_uint32(self.min_num_point))

    def add_point_cloud(self, points, sensor_pose=None, covs=None, rgb=None, intensities=None):
        p = _pts(points) if len(points) else np.zeros((0, 4), np.float32)
        T = _T(np.eye(4) if sensor_pose is None else sensor_pose)
        cv = None if covs is None else np.ascontiguousarray(covs, np.float32).reshape(len(p), 16)
        cl = None if rgb is None else _pts(rgb)
        it = None if intensities is None else np.ascontiguousarray(intensities, np.float32)
        lib().orc_voxelmap_add(self.h, _f(p), _f(cv), _f(cl), _f(it), C.c_size_t(len(p)), _f(T))

    def remove_old_data(self):
        lib().orc_voxelmap_remove_old(self.h)

    def info(self):
        cap, vn, st = C.c_uint64(), C.c_uint64(), C.c_uint32()
        fl = (C.c_int * 3)()
        lib().orc_voxelmap_info(self.h, C.byref(cap), C.byref(vn), C.byref(st), fl)
        return {"capacity": cap.value, "voxel_num": vn.value, "staleness_counter": st.value, "has_cov": bool(fl[0]),
                "has_rgb": bool(fl[1]), "has_intensity": bool(fl[2])}

    def downsampling(self, center=(0, 0, 0), distance=100.0):
        """-> dict(points, covs | None, rgb | None, intensities | None, keys), rows in slot order"""
        inf = self.info()
        n = inf["voxel_num"]
        pts = np.zeros((n, 4), np.float32)
        cv = np.zeros((n, 16), np.float32) if inf["has_cov"] else None
        cl = np.zeros((n, 4), np.float32) if inf["has_rgb"] else None
        it = np.zeros(n, np.float32) if inf["has_intensity"] else None
        keys = np.zeros(n, np.uint64)
        c = np.asarray(center, np.float32)
        m = lib().orc_voxelmap_downsample(self.h, _f(c), C.c_float(distance), _f(pts), _f(cv), _f(cl), _f(it),
                                          keys.ctypes.data_as(C.c_void_p)) if n else 0
        cut = lambda a: None if a is None else a[:m].copy()
        return {"points": pts[:m].copy(), "covs": cut(cv), "rgb": cut(cl), "intensities": cut(it), "keys": keys[:m].copy()}

    def compute_overlap_ratio(self, points, sensor_pose=None) -> float:
        p = _pts(points) if len(points) else np.zeros((0, 4), np.float32)
        T = _T(np.eye(4) if sensor_pose is None else sensor_pose)
        return float(lib().orc_voxelmap_overlap_ratio(self.h, _f(p), C.c_size_t(len(p)), _f(T)))


def spd_function(A, is_log: bool) -> np.ndarray:
    """log_spd_3x3 / exp_spd_3x3 (eigen_utils.hpp:646-677)"""
    a = np.ascontiguousarray(A, np.float32).reshape(9)
    out = np.empty(9, np.float32)
    lib().orc_spd_function(_f(a), C.c_int(int(is_log)), _f(out))
    return out.reshape(3, 3)


def voxel_downsample_attrs(points, voxel_size, min_voxel_count, rgb=None, intensity=None, timestamps=None):
    p = _pts(points)
    n = len(p)
    out = np.empty_like(p)
    rgb_a = None if rgb is None else _pts(rgb)
    it = None if intensity is None else np.ascontiguousarray(intensity, np.float32)
    ts = None if timestamps is None else np.ascontiguousarray(timestamps, np.float32)
    o_rgb = None if rgb is None else np.empty((n, 4), np.float32)
    o_it = None if intensity is None else np.empty(n, np.float32)
    o_ts = None if timestamps is None else np.empty(n, np.float32)
    m = lib().orc_voxel_downsample_attrs(_f(p), C.c_size_t(n), C.c_float(voxel_size), C.c_size_t(min_voxel_count),
                                         _f(rgb_a), _f(it), _f(ts), _f(out), _f(o_rgb), _f(o_it), _f(o_ts))
    cut = lambda a: None if a is None else a[:m].copy()
    return out[:m].copy(), cut(o_rgb), cut(o_it), cut(o_ts)


def polar_downsample_attrs(points, dist_size, elev_size, azim_size, coord_system=0, min_voxel_count=1, rgb=None,
                           intensity=None, timestamps=None):
    """filter::PolarGrid::downsampling (polar_downsampling.hpp); coord_system 0 LIDAR / 1 CAMERA."""
    p = _pts(points)
    n = len(p)
    out = np.empty_like(p)
    rgb_a = None if rgb is None else _pts(rgb)
    it = None if intensity is None else np.ascontiguousarray(intensity, np.float32)
    ts = None if timestamps is None else np.ascontiguousarray(timestamps, np.float32)
    o_rgb = None if rgb is None else np.empty((n, 4), np.float32)
    o_it = None if intensity is None else np.empty(n, np.float32)
    o_ts = None if timestamps is None else np.empty(n, np.float32)
    m = lib().orc_polar_downsample_attrs(_f(p), C.c_size_t(n), C.c_float(dist_size), C.c_float(elev_size),
                                         C.c_float(azim_size), C.c_int(coord_system), C.c_size_t(min_voxel_count),
                                         _f(rgb_a), _f(it), _f(ts), _f(out), _f(o_rgb), _f(o_it), _f(o_ts))
    cut = lambda a: None if a is None else a[:m].copy()
    return out[:m].copy(), cut(o_rgb), cut(o_it), cut(o_ts)


def box_filter(points, min_d: float, max_d: float) -> np.ndarray:
    p = _pts(points)
    out = np.empty_like(p)
    m = lib().orc_box_filter(_f(p), C.c_size_t(len(p)), C.c_float(min_d), C.c_float(max_d), _f(out))
    return out[:m].copy()


def default_params(**kw) -> RegParams:
    P = RegParams()
    lib().orc_default_params(C.byref(P))
    for k, v in kw.items():
        setattr(P, k, v)
    return P


def _result(R: RegResult) -> dict:
    return dict(T=_T_back(R.T), converged=bool(R.converged), iterations=int(R.iterations),
                H=np.array(R.H, np.float32).reshape(6, 6), b=np.array(R.b, np.float32), error=float(R.error),
                H_raw=np.array(R.H_raw, np.float32).reshape(6, 6), b_raw=np.array(R.b_raw, np.float32),
                error_raw=float(R.error_raw), inlier=int(R.inlier))


def align(P: RegParams, src_pts, src_covs, tgt_pts, tgt_covs, tgt_normals, tree: KDTree | None, T_init=None,
          robust_scale: float = -1.0, trace: bool = False):
    sp, tp = _pts(src_pts), _pts(tgt_pts)
    sc, tc = _covs_cm(src_covs), _covs_cm(tgt_covs)
    tn = None if tgt_normals is None else _pts(tgt_normals)
    t16 = _T(np.eye(4) if T_init is None else T_init)
    R = RegResult()
    tr = np.zeros((max(P.max_iterations, 1), 16), np.float32) if trace else None
    lib().orc_align(C.byref(P), _f(sp), _f(sc), C.c_size_t(len(sp)), _f(tp), _f(tc), _f(tn), C.c_size_t(len(tp)),
                    tree.handle if tree is not None else None, _f(t16), C.c_float(robust_scale), C.byref(R), _f(tr))
    out = _result(R)
    if trace:
        out["trace"] = np.stack([_T_back(t) for t in tr])
    return out


def robust_schedule(init_scale: float, min_scale: float, levels: int) -> np.ndarray:
    out = np.empty(levels, np.float32)
    lib().orc_robust_schedule(C.c_float(init_scale), C.c_float(min_scale), C.c_int(levels), _f(out))
    return out


def align_robust(P: RegParams, src_pts, src_covs, tgt_pts, tgt_covs, tgt_normals, tree: KDTree, T_init, init_scale,
                 min_scale, levels):
    sp, tp = _pts(src_pts), _pts(tgt_pts)
    sc, tc = _covs_cm(src_covs), _covs_cm(tgt_covs)
    tn = None if tgt_normals is None else _pts(tgt_normals)
    t16 = _T(np.eye(4) if T_init is None else T_init)
    R = RegResult()
    lib().orc_align_robust(C.byref(P), _f(sp), _f(sc), C.c_size_t(len(sp)), _f(tp), _f(tc), _f(tn),
                           C.c_size_t(len(tp)), tree.handle, _f(t16), C.c_float(init_scale), C.c_float(min_scale),
                           C.c_int(levels), C.byref(R))
    return _result(R)
