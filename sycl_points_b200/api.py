"""Host-side mirror of the reference's C++ interface for the hot path, on top of the C-ABI.

Names, argument meaning and error behaviour follow the reference (I/ = cpp/include/sycl_points/):
DeviceQueue (I/utils/sycl_utils.hpp:491), PointCloudShared (I/points/point_cloud.hpp:73),
knn.KNNResult / KNNBase / KDTree / knn_search_bruteforce (I/algorithms/knn/),
covariance.estimate / estimate_normals / extract_normals (I/algorithms/feature/covariance.hpp),
filter.VoxelGrid / PreprocessFilter.box_filter (I/algorithms/filter/),
registration.Registration / RegistrationParams / RegistrationResult / RegistrationPipeline
(I/algorithms/registration/).  numpy arrays are host data; every compute call runs on the GPU.
"""
from __future__ import annotations

import ctypes as C
import enum
import math
import os
from dataclasses import dataclass, field

import numpy as np

from . import _lib
from ._lib import (RegistrationAddonsC, RegistrationParamsC, RegistrationResultC, SpxError, SpxInvalidArgument,
                   check)

FLT_MAX = float(np.finfo(np.float32).max)


def _hostf(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_float))


def _T16(T) -> np.ndarray | None:
    """4x4 (row-major numpy) -> 16 floats column-major, the layout of Eigen::Matrix4f::data()."""
    if T is None:
        return None
    T = np.asarray(T, dtype=np.float32).reshape(4, 4)
    return np.ascontiguousarray(T.T).reshape(16)


def _T_from16(t16) -> np.ndarray:
    return np.array(t16, dtype=np.float32).reshape(4, 4).T.copy()


# ------------------------------------------------------------------ runtime
class DeviceQueue:
    """sycl_utils::DeviceQueue (sycl_utils.hpp:491-626): one in-order CUDA stream on one device."""

    def __init__(self, device: int = 0, cuda_stream: int | None = None, priority: int = 0):
        L = _lib.lib()
        h = C.c_void_p()
        if cuda_stream is None and priority != 0:
            check(L.spx_queue_create_with_priority(device, int(priority), C.byref(h)))
        elif cuda_stream is None:
            check(L.spx_queue_create(device, C.byref(h)))
        else:
            check(L.spx_queue_create_on_stream(device, C.c_void_p(cuda_stream), C.byref(h)))
        self._h = h
        self.device = device

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().spx_queue_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    def wait(self):
        """events.wait_and_throw()"""
        check(_lib.lib().spx_queue_sync(self._h))

    def set_blocking_sync(self, blocking: bool = True):
        """wait on an OS primitive instead of spinning (frees the core when many queues share a host)"""
        check(_lib.lib().spx_queue_set_blocking_sync(self._h, 1 if blocking else 0))

    def wait_event(self, event: "Event"):
        """later work on this queue starts only after `event` (recorded on any queue) has completed"""
        check(_lib.lib().spx_queue_wait_event(self._h, event._h))

    def is_cpu(self) -> bool:
        return False

    def is_gpu(self) -> bool:
        return True

    def is_nvidia(self) -> bool:
        return True

    def device_info(self) -> dict:
        name = C.create_string_buffer(256)
        sm, smc, l2 = C.c_int(), C.c_int(), C.c_int()
        mem = C.c_size_t()
        check(_lib.lib().spx_device_info(self.device, name, C.byref(sm), C.byref(smc), C.byref(mem), C.byref(l2)))
        return dict(name=name.value.decode(), sm=sm.value, sm_count=smc.value, global_mem=mem.value, l2=l2.value)


def device_count() -> int:
    n = C.c_int()
    check(_lib.lib().spx_device_count(C.byref(n)))
    return n.value


def kernel_launch_count() -> int:
    return int(_lib.lib().spx_kernel_launch_count())


class Event:
    def __init__(self):
        h = C.c_void_p()
        check(_lib.lib().spx_event_create(C.byref(h)))
        self._h = h

    def record(self, queue: DeviceQueue):
        check(_lib.lib().spx_event_record(queue.handle, self._h))
        return self

    def elapsed_ms(self, later: "Event") -> float:
        ms = C.c_float()
        check(_lib.lib().spx_event_elapsed_ms(self._h, later._h, C.byref(ms)))
        return ms.value

    def __del__(self):
        try:
            if self._h:
                _lib.lib().spx_event_destroy(self._h)
                self._h = None
        except Exception:
            pass


class PinnedArray:
    """Pinned host staging buffer (cudaMallocHost) viewed as a numpy array."""

    def __init__(self, shape, dtype=np.float32):
        self.shape = tuple(shape) if not isinstance(shape, int) else (shape,)
        self.dtype = np.dtype(dtype)
        nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        p = C.c_void_p()
        check(_lib.lib().spx_malloc_host(max(nbytes, 1), C.byref(p)))
        self._p = p
        buf = (C.c_char * max(nbytes, 1)).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(np.prod(self.shape))).reshape(self.shape)

    def __del__(self):
        try:
            if self._p:
                self.array = None
                _lib.lib().spx_free_host(self._p)
                self._p = None
        except Exception:
            pass


class DeviceArray:
    """shared_vector<T> (sycl_utils.hpp:630-635) as explicit device memory + host copies on demand."""

    def __init__(self, queue: DeviceQueue, shape, dtype=np.float32):
        self.queue = queue
        self.shape = tuple(shape) if not isinstance(shape, int) else (shape,)
        self.dtype = np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        p = C.c_void_p()
        check(_lib.lib().spx_malloc(queue.handle, self.nbytes, C.byref(p)))
        self._p = p

    @classmethod
    def from_host(cls, queue: DeviceQueue, a: np.ndarray) -> "DeviceArray":
        a = np.ascontiguousarray(a)
        d = cls(queue, a.shape, a.dtype)
        d.upload(a)
        return d

    @property
    def ptr(self):
        return self._p

    def __len__(self):
        return self.shape[0] if self.shape else 0

    def upload(self, a: np.ndarray, sync: bool = True):
        a = np.ascontiguousarray(a, dtype=self.dtype)
        assert a.nbytes == self.nbytes, (a.shape, self.shape)
        if self.nbytes:
            check(_lib.lib().spx_memcpy_h2d(self.queue.handle, self._p, a.ctypes.data_as(C.c_void_p), self.nbytes))
            if sync:
                self.queue.wait()  # pageable source: keep it alive until the copy has run

    def download(self, count: int | None = None) -> np.ndarray:
        shape = self.shape if count is None else (count,) + self.shape[1:]
        out = np.empty(shape, self.dtype)
        if out.nbytes:
            check(_lib.lib().spx_memcpy_d2h(self.queue.handle, out.ctypes.data_as(C.c_void_p), self._p, out.nbytes))
        self.queue.wait()
        return out

    def free(self):
        if getattr(self, "_p", None) and self._p:
            # (a queue already closed — members of a reference cycle are finalised in no particular order — passes
            # NULL: the library then frees synchronously)
            _lib.lib().spx_free(self.queue.handle, self._p)
            self._p = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def _ptr(a: DeviceArray | None):
    return None if a is None else a.ptr


def _addr(p):
    """c_void_p / int / None -> value assignable to a c_void_p structure field"""
    if p is None:
        return None
    return p.value if isinstance(p, C.c_void_p) else int(p)


# ------------------------------------------------------------------ containers
# A cloud that comes out of the voxel grid carries the box and cell edges KDTree.build needs (index_hint): with ~one
# point per occupied voxel on LiDAR surfaces, cells of 1.85 voxels hold ~3 points (the k = 1 optimum) and cells of
# 2.4 voxels ~5 (the k-NN first-pass grid) — what the adaptive build measures on such clouds.  SPX_INDEX_HINT=0 turns
# the hints off (every build measures its own occupancy curve).
INDEX_HINTS = os.environ.get("SPX_INDEX_HINT", "1") != "0"
INDEX_HINT_CELL = float(os.environ.get("SPX_INDEX_HINT_CELL", "1.85"))
INDEX_HINT_KNN_CELL = float(os.environ.get("SPX_INDEX_HINT_KNN_CELL", "2.4"))


class PointCloudShared:
    """PointCloudShared (point_cloud.hpp:73-476): per-attribute arrays on the device.
    points (n,4) xyz1; covs (n,4,4) symmetric, zero 4th row/col; normals (n,4) xyz0."""
    index_hint = None

    def __init__(self, queue: DeviceQueue, points: np.ndarray | None = None, covs: np.ndarray | None = None,
                 normals: np.ndarray | None = None):
        self.queue = queue
        self.points: DeviceArray | None = None
        self.covs: DeviceArray | None = None
        self.normals: DeviceArray | None = None
        self.rgb: DeviceArray | None = None          # (n, 4) RGBA in [0, 1]  (types.hpp:14-17)
        self.intensities: DeviceArray | None = None  # (n,)
        self.timestamp_offsets: DeviceArray | None = None  # (n,) ms relative to the first measurement
        self.start_time_ms = 0.0
        self.end_time_ms = 0.0
        self._n = 0
        if points is not None:
            self.set_points(points)
        if covs is not None:
            self.set_covs(covs)
        if normals is not None:
            self.set_normals(normals)

    def size(self) -> int:
        return self._n

    def __len__(self):
        return self._n

    def has_cov(self) -> bool:
        return self.covs is not None and len(self.covs) == self._n

    def has_normal(self) -> bool:
        return self.normals is not None and len(self.normals) == self._n

    def set_points(self, points: np.ndarray):
        p = np.ascontiguousarray(points, dtype=np.float32)
        if p.ndim != 2 or p.shape[1] != 4:
            raise ValueError("points must be (n, 4) float32 (xyz1)")
        self.points = DeviceArray.from_host(self.queue, p)
        self._n = len(p)
        self.index_hint = None

    def set_covs(self, covs: np.ndarray):
        c = np.asarray(covs, dtype=np.float32).reshape(-1, 4, 4)
        # host convention: row-major numpy; device/reference convention: column-major Matrix4f
        self.covs = DeviceArray.from_host(self.queue, np.ascontiguousarray(c.transpose(0, 2, 1)).reshape(-1, 16))

    def set_normals(self, normals: np.ndarray):
        self.normals = DeviceArray.from_host(self.queue, np.ascontiguousarray(normals, dtype=np.float32))

    def has_rgb(self) -> bool:
        return self.rgb is not None and len(self.rgb) == self._n and self._n > 0

    def has_intensity(self) -> bool:
        return self.intensities is not None and len(self.intensities) == self._n and self._n > 0

    def has_timestamps(self) -> bool:
        return self.timestamp_offsets is not None and len(self.timestamp_offsets) == self._n and self._n > 0

    def set_rgb(self, rgb: np.ndarray):
        self.rgb = DeviceArray.from_host(self.queue, np.ascontiguousarray(rgb, dtype=np.float32).reshape(-1, 4))

    def set_intensities(self, v: np.ndarray):
        self.intensities = DeviceArray.from_host(self.queue, np.ascontiguousarray(v, dtype=np.float32).reshape(-1))

    def set_timestamp_offsets(self, v: np.ndarray):
        self.timestamp_offsets = DeviceArray.from_host(self.queue,
                                                       np.ascontiguousarray(v, dtype=np.float32).reshape(-1))

    def set_points_xyz(self, xyz_dev: DeviceArray, n: int):
        """points <- packed xyz (device float[n][3]) expanded to xyz1 on the device (spx_points_from_xyz); the
        points array must already be allocated with room for n points.  Asynchronous."""
        check(_lib.lib().spx_points_from_xyz(self.queue.handle, xyz_dev.ptr, n, self.points.ptr))
        self._n = n

    def adopt_points(self, dev: DeviceArray, n: int):
        self.points = dev
        self._n = n
        self.index_hint = None

    def points_host(self) -> np.ndarray:
        return self.points.download(self._n) if self._n else np.zeros((0, 4), np.float32)

    def covs_host(self) -> np.ndarray:
        return self.covs.download(self._n).reshape(-1, 4, 4).transpose(0, 2, 1).copy()

    def normals_host(self) -> np.ndarray:
        return self.normals.download(self._n)


# ------------------------------------------------------------------ KNN
class KNNResult:
    """knn::KNNResult (result.hpp:12-34): indices int32 [q][k], squared distances float [q][k]."""

    def __init__(self):
        self.indices: DeviceArray | None = None
        self.distances: DeviceArray | None = None
        self.query_size = 0
        self.k = 0

    def allocate(self, queue: DeviceQueue, query_size: int = 0, k: int = 0):
        self.query_size, self.k = query_size, k
        self.indices = DeviceArray(queue, (query_size, k), np.int32)
        self.distances = DeviceArray(queue, (query_size, k), np.float32)

    def indices_host(self) -> np.ndarray:
        return self.indices.download() if self.query_size * self.k else np.zeros((self.query_size, self.k), np.int32)

    def distances_host(self) -> np.ndarray:
        return self.distances.download() if self.query_size * self.k else np.zeros((self.query_size, self.k),
                                                                                    np.float32)


class KNNBase:
    """knn::KNNBase (knn.hpp:14-61).  Subclass and implement knn_search_async to inject a KNN."""

    def knn_search_async(self, queries: PointCloudShared, k: int, result: KNNResult, depends=None, transT=None):
        raise NotImplementedError

    def knn_search(self, queries: PointCloudShared, k: int, depends=None, transT=None) -> KNNResult:
        result = KNNResult()
        self.knn_search_async(queries, k, result, depends, transT)
        queries.queue.wait()
        return result

    def nearest_neighbor_search_async(self, queries, result, depends=None, transT=None):
        return self.knn_search_async(queries, 1, result, depends, transT)

    def nearest_neighbor_search(self, queries, result, depends=None, transT=None):
        self.nearest_neighbor_search_async(queries, result, depends, transT)
        queries.queue.wait()


def knn_search_bruteforce(queue: DeviceQueue, queries: PointCloudShared, targets: PointCloudShared, k: int,
                          transT=None) -> KNNResult:
    """knn::knn_search_bruteforce (bruteforce.hpp:24-96); synchronous like the reference (:93)."""
    result = KNNResult()
    result.allocate(queue, queries.size(), k)
    t16 = _T16(transT)
    check(_lib.lib().spx_knn_bruteforce(queue.handle, _ptr(queries.points), queries.size(), _ptr(targets.points),
                                        targets.size(), k, _hostf(t16), result.indices.ptr, result.distances.ptr))
    queue.wait()
    return result


class KDTree(KNNBase):
    """knn::KDTree (kdtree.hpp:142-280) — same interface, GPU-resident exact cell-grid index inside."""

    def __init__(self, queue: DeviceQueue):
        self.queue = queue
        self._h = None
        self._n = 0

    @staticmethod
    def build(queue: DeviceQueue, cloud: PointCloudShared, leaf_threshold: int = 16, cell_size: float = 0.0):
        # leaf_threshold is the reference's KD-tree knob; it has no meaning for the grid (accepted, ignored)
        t = KDTree(queue)
        h = C.c_void_p()
        hint = getattr(cloud, "index_hint", None)
        if hint is not None and cell_size <= 0.0 and cloud.size() > 0:
            lo, hi, cell, cell_knn = hint
            check(_lib.lib().spx_index_build_hinted(queue.handle, _ptr(cloud.points), cloud.size(), _hostf(lo), _hostf(hi),
                                                    float(cell), float(cell_knn), C.byref(h)))
        else:
            check(_lib.lib().spx_index_build(queue.handle, _ptr(cloud.points), cloud.size(), float(cell_size),
                                             C.byref(h)))
        t._h = h
        t._n = cloud.size()
        return t

    @property
    def handle(self):
        return self._h

    def info(self) -> dict:
        cell = C.c_float()
        dims = (C.c_int32 * 3)()
        occ, npts = C.c_int64(), C.c_int64()
        check(_lib.lib().spx_index_info(self._h, C.byref(cell), dims, C.byref(occ), C.byref(npts)))
        lv = C.c_int32()
        check(_lib.lib().spx_index_levels(self._h, C.byref(lv)))
        return dict(cell_size=cell.value, dims=tuple(dims), occupied_cells=occ.value, n_points=npts.value,
                    levels=lv.value)

    def knn_search_async(self, queries: PointCloudShared, k: int, result: KNNResult, depends=None, transT=None):
        if k > 128:
            raise SpxInvalidArgument(-1, "[KDTree::knn_search_async] `k` is too large. not support.")
        nq = queries.size()
        if result.indices is None or result.query_size != nq or result.k != k:
            result.allocate(self.queue, nq, k if nq else 0)  # kdtree.hpp:429-450
        if nq == 0:
            return
        t16 = _T16(transT)
        check(_lib.lib().spx_index_knn(self._h, _ptr(queries.points), nq, k, _hostf(t16), result.indices.ptr,
                                       result.distances.ptr))

    def radius_search_async(self, queries: PointCloudShared, max_k: int, radius: float, result: KNNResult,
                            depends=None, transT=None):
        """kdtree.hpp:251-280: the max_k nearest targets within `radius` (dist² <= radius²), the remaining slots
        -1 / FLT_MAX."""
        if max_k > 100:
            raise SpxInvalidArgument(-1, "[KDTree::radius_search_async] `max_k` is too large. not support.")
        nq = queries.size()
        if nq == 0 or max_k == 0:
            result.allocate(self.queue, 0, 0)  # kdtree.hpp:580-587
            return
        if result.indices is None or result.query_size != nq or result.k != max_k:
            result.allocate(self.queue, nq, max_k)
        check(_lib.lib().spx_index_radius(self._h, _ptr(queries.points), nq, max_k, float(radius), _hostf(_T16(transT)),
                                          result.indices.ptr, result.distances.ptr))

    def radius_search(self, queries: PointCloudShared, max_k: int, radius: float, depends=None, transT=None):
        result = KNNResult()
        self.radius_search_async(queries, max_k, radius, result, depends, transT)
        queries.queue.wait()
        return result

    def remove_nodes_by_flags(self, flags: "DeviceArray", indices: "DeviceArray"):
        """kdtree.hpp:282-284: drop the points whose flag is 0 (REMOVE_FLAG) and renumber the kept ones by `indices`
        (old -> new, -1 where removed: FilterByFlags::calculate_indices)."""
        if len(flags) != len(indices):
            raise SpxInvalidArgument(-1, "[KDTree::remove_nodes_by_flags_impl] flags and indices must have the same size.")
        if self._h is None or len(flags) == 0:
            return
        host = indices.download()
        kept = int(host.max()) + 1 if host.size and host.max() >= 0 else 0
        check(_lib.lib().spx_index_remove_by_flags(self._h, flags.ptr, indices.ptr, len(flags), kept))
        self.queue.wait()
        self._n = kept

    def close(self):
        if self._h:
            _lib.lib().spx_index_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ------------------------------------------------------------------ features
class covariance:  # namespace sycl_points::algorithms::covariance
    @staticmethod
    def estimate(neighbors: KNNResult, points: PointCloudShared):
        """covariance::estimate_async(neighbors, points) (covariance.hpp:260-302)"""
        n = points.size()
        if points.covs is None or len(points.covs) != n:
            points.covs = DeviceArray(points.queue, (n, 16), np.float32)
        check(_lib.lib().spx_covariance(points.queue.handle, _ptr(points.points), n, _ptr(neighbors.indices),
                                        neighbors.k, points.covs.ptr))

    @staticmethod
    def estimate_robust(neighbors: KNNResult, points: PointCloudShared, robust_type=None, mad_scale: float = 1.0,
                        min_robust_scale: float = 1.0, robust_max_iterations: int = 1):
        """covariance::estimate_robust_async(neighbors, points, robust_type, mad_scale, min_robust_scale,
        robust_max_iterations) (covariance.hpp:323-390); default robust_type CAUCHY"""
        n = points.size()
        if neighbors.k > 64:
            raise RuntimeError("[covariance::estimate_robust_async] neighbor K is too large. MAX_K is 64")
        if points.covs is None or len(points.covs) != n:
            points.covs = DeviceArray(points.queue, (n, 16), np.float32)
        loss = int(RobustLossType.CAUCHY if robust_type is None else robust_type)
        check(_lib.lib().spx_covariance_robust(points.queue.handle, _ptr(points.points), n, _ptr(neighbors.indices),
                                               neighbors.k, loss, float(mad_scale), float(min_robust_scale),
                                               int(robust_max_iterations), points.covs.ptr))

    @staticmethod
    def estimate_knn(knn: KNNBase, points: PointCloudShared, k_correspondences: int):
        """covariance::estimate_async(knn, points, k) (covariance.hpp:304-311)"""
        neighbors = KNNResult()
        knn.knn_search_async(points, k_correspondences, neighbors)
        covariance.estimate(neighbors, points)

    @staticmethod
    def estimate_normals(neighbors: KNNResult, points: PointCloudShared):
        """covariance::estimate_normals_async (covariance.hpp:417-445)"""
        n = points.size()
        if points.normals is None or len(points.normals) != n:
            points.normals = DeviceArray(points.queue, (n, 4), np.float32)
        check(_lib.lib().spx_normals(points.queue.handle, _ptr(points.points), n, _ptr(neighbors.indices),
                                     neighbors.k, points.normals.ptr))

    @staticmethod
    def extract_normals(points: PointCloudShared):
        """covariance::extract_normals (covariance.hpp:467-503)"""
        if not points.has_cov():
            raise SpxInvalidArgument(-1, "[covariance::extract_normals_async] covariances not computed")
        n = points.size()
        if points.normals is None or len(points.normals) != n:
            points.normals = DeviceArray(points.queue, (n, 4), np.float32)
        check(_lib.lib().spx_normals_from_covs(points.queue.handle, _ptr(points.points), points.covs.ptr, n,
                                               points.normals.ptr))


    @staticmethod
    def update_covariance_plane(points: PointCloudShared):
        """kernel::update_covariance_plane over a cloud's covariances, in place (covariance.hpp:67-74)"""
        if not points.has_cov():
            raise SpxInvalidArgument(-1, "[covariance::update_covariance_plane] covariances not computed")
        check(_lib.lib().spx_covariance_update_plane(points.queue.handle, points.covs.ptr, points.size()))


def symmetric_eigen_decomposition_3x3(queue: "DeviceQueue", covs) -> tuple[np.ndarray, np.ndarray]:
    """eigen_utils::symmetric_eigen_decomposition_3x3 (eigen_utils.hpp:443-562) of n symmetric 3x3
    matrices given as (n, 3, 3) or the (n, 4, 4) covariance layout; returns (evals (n,3) ascending,
    evecs (n,3,3) with eigenvectors in columns)."""
    a = np.asarray(covs, np.float32)
    n = a.shape[0]
    c44 = np.zeros((n, 4, 4), np.float32)
    c44[:, :3, :3] = a[:, :3, :3]
    d = DeviceArray(queue, (n, 16), np.float32)
    d.upload(np.ascontiguousarray(c44.transpose(0, 2, 1)).reshape(n, 16))  # column-major 4x4
    ev, V = DeviceArray(queue, (n, 3), np.float32), DeviceArray(queue, (n, 9), np.float32)
    check(_lib.lib().spx_eigen3(queue.handle, d.ptr, n, ev.ptr, V.ptr))
    return ev.download(), V.download().reshape(n, 3, 3)


# ------------------------------------------------------------------ filters
class VoxelGrid:
    """filter::VoxelGrid (voxel_downsampling.hpp:14-79)."""

    def __init__(self, queue: DeviceQueue, voxel_size: float):
        if voxel_size <= 0.0:
            raise ValueError("voxel_size must be positive")  # std::invalid_argument, :23-25
        self.queue = queue
        self._voxel_size = float(voxel_size)
        self._min_voxel_count = 1

    def set_voxel_size(self, voxel_size: float):
        if voxel_size <= 0.0:
            raise ValueError("voxel_size must be positive")
        self._voxel_size = float(voxel_size)

    def get_voxel_size(self) -> float:
        return self._voxel_size

    def set_min_voxel_count(self, n: int):
        self._min_voxel_count = int(n)

    def downsampling(self, cloud: PointCloudShared, result: PointCloudShared | None = None) -> PointCloudShared:
        """voxel_downsampling.hpp:64-79 (+ :220-288 when the cloud carries RGB / intensity / timestamps)."""
        result = result if result is not None else PointCloudShared(self.queue)
        n = cloud.size()
        if n == 0:
            result.adopt_points(DeviceArray(self.queue, (0, 4), np.float32), 0)
            result.covs = result.normals = result.rgb = result.intensities = result.timestamp_offsets = None
            return result
        out = DeviceArray(self.queue, (n, 4), np.float32)
        m = C.c_size_t()
        rgb, inten, ts = cloud.has_rgb(), cloud.has_intensity(), cloud.has_timestamps()
        if not (rgb or inten or ts):
            check(_lib.lib().spx_voxel_downsample(self.queue.handle, cloud.points.ptr, n, self._voxel_size,
                                                  self._min_voxel_count, out.ptr, C.byref(m)))
            o_rgb = o_int = o_ts = None
        else:
            o_rgb = DeviceArray(self.queue, (n, 4), np.float32) if rgb else None
            o_int = DeviceArray(self.queue, (n,), np.float32) if inten else None
            o_ts = DeviceArray(self.queue, (n,), np.float32) if ts else None
            check(_lib.lib().spx_voxel_downsample_attrs(
                self.queue.handle, cloud.points.ptr, n, self._voxel_size, self._min_voxel_count,
                cloud.rgb.ptr if rgb else None, cloud.intensities.ptr if inten else None,
                cloud.timestamp_offsets.ptr if ts else None, out.ptr, _ptr(o_rgb), _ptr(o_int), _ptr(o_ts),
                C.byref(m)))
        mm = int(m.value)
        result.adopt_points(out, mm)
        # the voxel box of the output, known without touching the points: lets KDTree.build skip its bounding-box /
        # occupancy pass and the host round trip (spx_index_build_hinted).  Dropped by anything that moves the points.
        result.index_hint = None
        if mm > 0 and INDEX_HINTS:
            lo, hi = np.zeros(3, np.float32), np.zeros(3, np.float32)
            check(_lib.lib().spx_voxel_last_box(self.queue.handle, _hostf(lo), _hostf(hi), None))
            result.index_hint = (lo, hi, INDEX_HINT_CELL * self._voxel_size, INDEX_HINT_KNN_CELL * self._voxel_size)
        result.covs = None
        result.normals = None
        result.rgb = _trim(o_rgb, mm)
        result.intensities = _trim(o_int, mm)
        result.timestamp_offsets = _trim(o_ts, mm)
        return result


class VoxelHashMap:
    """mapping::VoxelHashMap (algorithms/mapping/voxel_hash_map.hpp:22-1066): the odometry submap — a device hash
    table of voxels accumulating centroid, log-Euclidean mean covariance, mean colour and mean intensity."""

    def __init__(self, queue: DeviceQueue, voxel_size: float):
        if voxel_size <= 0.0:
            raise ValueError("voxel_size must be positive.")  # std::invalid_argument, :41-43
        self.queue = queue
        self._voxel_size = float(voxel_size)
        self._max_staleness, self._remove_old_data_cycle = 100, 10
        self._rehash_threshold, self._min_num_point = 0.7, 1
        h = C.c_void_p()
        check(_lib.lib().spx_voxelmap_create(queue.handle, self._voxel_size, C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().spx_voxelmap_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _push(self):
        check(_lib.lib().spx_voxelmap_set_params(self._h, self._voxel_size, self._max_staleness,
                                                 self._remove_old_data_cycle, self._rehash_threshold,
                                                 self._min_num_point))

    def set_voxel_size(self, voxel_size: float):
        if voxel_size <= 0.0:
            raise ValueError("voxel_size must be positive.")
        self._voxel_size = float(voxel_size)
        self._push()

    def get_voxel_size(self) -> float:
        return self._voxel_size

    def set_max_staleness(self, v: int):
        self._max_staleness = int(v)
        self._push()

    def get_max_staleness(self) -> int:
        return self._max_staleness

    def set_remove_old_data_cycle(self, v: int):
        self._remove_old_data_cycle = int(v)
        self._push()

    def get_remove_old_data_cycle(self) -> int:
        return self._remove_old_data_cycle

    def set_rehash_threshold(self, v: float):
        self._rehash_threshold = float(v)
        self._push()

    def get_rehash_threshold(self) -> float:
        return self._rehash_threshold

    def set_min_num_point(self, v: int):
        self._min_num_point = int(v)
        self._push()

    def get_min_num_point(self) -> int:
        return self._min_num_point

    def clear(self):
        check(_lib.lib().spx_voxelmap_clear(self._h))

    def info(self) -> dict:
        cap, vn, st = C.c_uint64(), C.c_uint64(), C.c_uint32()
        hc, hr, hi = C.c_int(), C.c_int(), C.c_int()
        check(_lib.lib().spx_voxelmap_info(self._h, C.byref(cap), C.byref(vn), C.byref(st), C.byref(hc), C.byref(hr),
                                           C.byref(hi)))
        return {"capacity": cap.value, "voxel_num": vn.value, "staleness_counter": st.value, "has_cov": bool(hc.value),
                "has_rgb": bool(hr.value), "has_intensity": bool(hi.value)}

    def add_point_cloud(self, cloud: PointCloudShared, sensor_pose=None):
        """:117-140 — the cloud is in the sensor frame, sensor_pose (4x4) maps it into the map frame."""
        n = cloud.size()
        check(_lib.lib().spx_voxelmap_add(
            self._h, cloud.points.ptr if n else None, cloud.covs.ptr if n and cloud.has_cov() else None,
            cloud.rgb.ptr if n and cloud.has_rgb() else None,
            cloud.intensities.ptr if n and cloud.has_intensity() else None, n, _hostf(_T16(sensor_pose))))

    def remove_old_data(self):
        check(_lib.lib().spx_voxelmap_remove_old(self._h))

    def downsampling(self, result: PointCloudShared | None = None, center=(0.0, 0.0, 0.0), distance: float = 100.0,
                     return_keys: bool = False):
        """:146-188 — the voxels whose centroid lies within `distance` of `center` per axis, as a point cloud (with
        covariances / rgb / intensities when the map holds them)."""
        result = result if result is not None else PointCloudShared(self.queue)
        inf = self.info()
        n = inf["voxel_num"]
        result.covs = result.normals = result.rgb = result.intensities = result.timestamp_offsets = None
        if n == 0:
            result.adopt_points(DeviceArray(self.queue, (0, 4), np.float32), 0)
            return (result, np.zeros(0, np.uint64)) if return_keys else result
        pts = DeviceArray(self.queue, (n, 4), np.float32)
        covs = DeviceArray(self.queue, (n, 16), np.float32) if inf["has_cov"] else None
        rgb = DeviceArray(self.queue, (n, 4), np.float32) if inf["has_rgb"] else None
        inten = DeviceArray(self.queue, (n,), np.float32) if inf["has_intensity"] else None
        keys = DeviceArray(self.queue, (n,), np.uint64) if return_keys else None
        c = np.asarray(center, np.float32).reshape(3)
        m = C.c_size_t()
        check(_lib.lib().spx_voxelmap_downsample(self._h, _hostf(c), float(distance), pts.ptr, _ptr(covs), _ptr(rgb),
                                                 _ptr(inten), _ptr(keys), n, C.byref(m)))
        mm = int(m.value)
        result.adopt_points(pts, mm)
        result.covs = _trim(covs, mm)
        result.rgb = _trim(rgb, mm)
        result.intensities = _trim(inten, mm)
        if return_keys:
            return result, keys.download(mm)
        return result

    def compute_overlap_ratio(self, cloud: PointCloudShared, sensor_pose=None) -> float:
        """:194-246"""
        n = cloud.size()
        r = C.c_float()
        check(_lib.lib().spx_voxelmap_overlap_ratio(self._h, cloud.points.ptr if n else None, n,
                                                    _hostf(_T16(sensor_pose)), C.byref(r)))
        return float(r.value)


class CoordinateSystem(enum.IntEnum):  # common/coordinate_system.hpp:13
    LIDAR = 0
    CAMERA = 1


class PolarGrid:
    """filter::PolarGrid (polar_downsampling.hpp:111-452): the grid filter with cells in (range, elevation,
    azimuth); angles in radians."""

    def __init__(self, queue: DeviceQueue, distance_voxel_size: float, elevation_voxel_size: float,
                 azimuth_voxel_size: float, coord: CoordinateSystem = CoordinateSystem.LIDAR):
        if distance_voxel_size <= 0.0 or elevation_voxel_size <= 0.0 or azimuth_voxel_size <= 0.0:
            raise ValueError("voxel sizes must be positive")  # std::invalid_argument, :129-131
        self.queue = queue
        self.distance_voxel_size = float(distance_voxel_size)
        self.elevation_voxel_size = float(elevation_voxel_size)
        self.azimuth_voxel_size = float(azimuth_voxel_size)
        self.coord = CoordinateSystem(coord)
        self._min_voxel_count = 1

    def set_min_voxel_count(self, n: int):
        self._min_voxel_count = int(n)

    def set_coordinate_system(self, coord):
        self.coord = CoordinateSystem(coord)

    def downsampling(self, cloud: PointCloudShared, result: PointCloudShared | None = None) -> PointCloudShared:
        result = result if result is not None else PointCloudShared(self.queue)
        n = cloud.size()
        result.index_hint = None
        if n == 0:
            result.adopt_points(DeviceArray(self.queue, (0, 4), np.float32), 0)
            result.covs = result.normals = result.rgb = result.intensities = result.timestamp_offsets = None
            return result
        out = DeviceArray(self.queue, (n, 4), np.float32)
        m = C.c_size_t()
        rgb, inten, ts = cloud.has_rgb(), cloud.has_intensity(), cloud.has_timestamps()
        o_rgb = DeviceArray(self.queue, (n, 4), np.float32) if rgb else None
        o_int = DeviceArray(self.queue, (n,), np.float32) if inten else None
        o_ts = DeviceArray(self.queue, (n,), np.float32) if ts else None
        check(_lib.lib().spx_polar_downsample_attrs(
            self.queue.handle, cloud.points.ptr, n, self.distance_voxel_size, self.elevation_voxel_size,
            self.azimuth_voxel_size, int(self.coord), self._min_voxel_count, cloud.rgb.ptr if rgb else None,
            cloud.intensities.ptr if inten else None, cloud.timestamp_offsets.ptr if ts else None, out.ptr, _ptr(o_rgb),
            _ptr(o_int), _ptr(o_ts), C.byref(m)))
        mm = int(m.value)
        result.adopt_points(out, mm)
        result.index_hint = None
        result.covs = None
        result.normals = None
        result.rgb = _trim(o_rgb, mm)
        result.intensities = _trim(o_int, mm)
        result.timestamp_offsets = _trim(o_ts, mm)
        return result


def _trim(a: DeviceArray | None, m: int):
    """view the first m rows of an over-allocated output array (no copy)"""
    if a is None:
        return None
    a.shape = (m,) + a.shape[1:]
    a.nbytes = int(np.prod(a.shape)) * a.dtype.itemsize
    return a


_GATHER_ATTRS = ("points", "covs", "normals", "rgb", "intensities", "timestamp_offsets")


def _gather_attributes(queue: DeviceQueue, cloud: PointCloudShared, idx: DeviceArray | None, m: int,
                       output: PointCloudShared | None, first: int = 0) -> PointCloudShared:
    """filter_by_flags (common/filter_by_flags.hpp:29-57): every attribute the cloud carries is compacted to the m rows
    listed in idx[first:first + m] (device int32, ascending: source order is kept).  output may be the cloud itself;
    None makes a new cloud."""
    has = (True, cloud.has_cov(), cloud.has_normal(), cloud.has_rgb(), cloud.has_intensity(), cloud.has_timestamps())
    idx_ptr = C.c_void_p(idx.ptr.value + 4 * first) if m else None

    def take(a: DeviceArray | None, enable: bool):
        if not enable:
            return None
        row = int(np.prod(a.shape[1:])) if len(a.shape) > 1 else 1
        out = DeviceArray(queue, (m,) + a.shape[1:], a.dtype)
        if m:
            check(_lib.lib().spx_gather(queue.handle, a.ptr, row * a.dtype.itemsize, idx_ptr, m, out.ptr))
        return out

    res = [take(getattr(cloud, name), h) for name, h in zip(_GATHER_ATTRS, has)]
    output = output if output is not None else PointCloudShared(queue)
    for name, a in zip(_GATHER_ATTRS, res):
        setattr(output, name, a)
    output._n = m
    if output is not cloud:
        output.index_hint = getattr(cloud, "index_hint", None)  # a subset stays inside the box
    return output


class PreprocessFilter:
    """filter::PreprocessFilter (preprocess_filter.hpp + preprocess_operator/*.hpp): box filter, uniform / weighted /
    mixed random sampling, farthest point sampling, angle-of-incidence filter.  As in the reference every sampling
    operator owns its std::mt19937 (seed 1234); set_random_seed re-seeds all of them (preprocess_filter.hpp:46-51)."""

    _RNGS = ("_rng", "_rng_weighted", "_rng_mixed", "_rng_fps")

    def __init__(self, queue: DeviceQueue):
        self.queue = queue
        for name in self._RNGS:
            h = C.c_void_p()
            check(_lib.lib().spx_rng_create(1234, C.byref(h)))  # random_sampling_operator.hpp:20 and siblings
            setattr(self, name, h)

    def __del__(self):
        try:
            for name in self._RNGS:
                if getattr(self, name, None):
                    _lib.lib().spx_rng_destroy(getattr(self, name))
                    setattr(self, name, None)
        except Exception:
            pass

    def set_random_seed(self, seed: int):
        for name in self._RNGS:
            check(_lib.lib().spx_rng_seed(getattr(self, name), int(seed)))

    _ATTRS = _GATHER_ATTRS

    def _gather_all(self, cloud: PointCloudShared, idx: DeviceArray, m: int, output: PointCloudShared | None):
        """filter_by_flags (common/filter_by_flags.hpp:29-57): every attribute the cloud carries is compacted"""
        return _gather_attributes(self.queue, cloud, idx, m, output)

    def random_sampling(self, cloud: PointCloudShared, sampling_num: int,
                        output: PointCloudShared | None = None) -> PointCloudShared:
        """PreprocessFilter::random_sampling (random_sampling_operator.hpp:24-52): partial Fisher-Yates
        with the persistent mt19937, order-preserving compaction of every per-point attribute."""
        n = cloud.size()
        if n <= sampling_num:
            if output is None or output is cloud:
                return cloud
            # keep everything: the reference copies the source into the output (random_sampling_operator.hpp:26-30)
            for name in self._ATTRS:
                a = getattr(cloud, name)
                if a is None:
                    setattr(output, name, None)
                    continue
                b = DeviceArray(self.queue, a.shape, a.dtype)
                if a.nbytes:
                    check(_lib.lib().spx_memcpy_d2d(self.queue.handle, b.ptr, a.ptr, a.nbytes))
                setattr(output, name, b)
            output._n = n
            return output
        idx = DeviceArray(self.queue, (sampling_num,), np.int32)
        m = C.c_size_t()
        check(_lib.lib().spx_random_sampling(self.queue.handle, self._rng, n, sampling_num, idx.ptr, C.byref(m)))
        self._last_indices = idx
        return self._gather_all(cloud, idx, int(m.value), output)

    def mixed_random_sampling(self, cloud: PointCloudShared, weights, sampling_num: int, weighted_ratio: float,
                              output: PointCloudShared | None = None) -> PointCloudShared:
        """PreprocessFilter::mixed_random_sampling (mixed_random_sampling_operator.hpp:29-107): floor(num * ratio)
        points by weighted reservoir keys (weights: DeviceArray or host array of n floats), the rest uniformly."""
        n = cloud.size()
        if n <= sampling_num:
            return self.random_sampling(cloud, sampling_num, output)  # keep-all branch: copy, no draw
        w = weights if isinstance(weights, DeviceArray) else DeviceArray.from_host(self.queue,
                                                                                  np.ascontiguousarray(weights, np.float32))
        if len(w) != n:
            raise ValueError("[PreprocessFilter::mixed_random_sampling] weights size must match points")
        idx = DeviceArray(self.queue, (sampling_num,), np.int32)
        m = C.c_size_t()
        try:
            check(_lib.lib().spx_mixed_random_sampling(self.queue.handle, self._rng_mixed, w.ptr, n, sampling_num,
                                                       float(weighted_ratio), idx.ptr, C.byref(m)))
        except SpxInvalidArgument as e:
            raise ValueError(str(e)) from e
        self._last_indices = idx
        return self._gather_all(cloud, idx, int(m.value), output)

    def weighted_random_sampling(self, cloud: PointCloudShared, weights, sampling_num: int,
                                 output: PointCloudShared | None = None) -> PointCloudShared:
        """PreprocessFilter::weighted_random_sampling (weighted_sampling_operator.hpp:29-96)."""
        n = cloud.size()
        if n <= sampling_num:
            return self.random_sampling(cloud, sampling_num, output)  # keep-all branch: copy, no draw
        w = weights if isinstance(weights, DeviceArray) else DeviceArray.from_host(self.queue,
                                                                                  np.ascontiguousarray(weights, np.float32))
        if len(w) != n:
            raise ValueError("[PreprocessFilter::weighted_random_sampling] weights size must match points")
        idx = DeviceArray(self.queue, (sampling_num,), np.int32)
        m = C.c_size_t()
        try:
            check(_lib.lib().spx_weighted_random_sampling(self.queue.handle, self._rng_weighted, w.ptr, n, sampling_num,
                                                          idx.ptr, C.byref(m)))
        except SpxInvalidArgument as e:
            raise ValueError(str(e)) from e
        return self._gather_all(cloud, idx, int(m.value), output)

    def farthest_point_sampling(self, cloud: PointCloudShared, sampling_num: int,
                                output: PointCloudShared | None = None) -> PointCloudShared:
        """PreprocessFilter::farthest_point_sampling (farthest_point_sampling_operator.hpp:27-94): one cooperative
        launch for the whole selection."""
        n = cloud.size()
        if n <= sampling_num:
            return self.random_sampling(cloud, sampling_num, output)
        first = C.c_size_t()
        check(_lib.lib().spx_rng_uniform_index(self._rng_fps, n, C.byref(first)))
        idx = DeviceArray(self.queue, (sampling_num,), np.int32)
        m = C.c_size_t()
        check(_lib.lib().spx_farthest_point_sampling(self.queue.handle, cloud.points.ptr, n, sampling_num, first.value,
                                                     idx.ptr, C.byref(m)))
        return self._gather_all(cloud, idx, int(m.value), output)

    def angle_incidence_filter(self, cloud: PointCloudShared, min_angle: float, max_angle: float,
                               output: PointCloudShared | None = None) -> PointCloudShared:
        """PreprocessFilter::angle_incidence_filter (angle_incidence_filter_operator.hpp:23-111)."""
        output = output if output is not None else cloud
        n = cloud.size()
        if n == 0:
            return output
        if not cloud.has_normal() and not cloud.has_cov():
            raise RuntimeError("[PreprocessFilter::angle_incidence_filter] Normal vector or covariance matrices must be "
                               "pre-computed.")
        idx = DeviceArray(self.queue, (n,), np.int32)
        m = C.c_size_t()
        try:
            check(_lib.lib().spx_angle_incidence_indices(
                self.queue.handle, cloud.points.ptr, cloud.normals.ptr if cloud.has_normal() else None,
                None if cloud.has_normal() else cloud.covs.ptr, n, float(min_angle), float(max_angle), idx.ptr,
                C.byref(m)))
        except SpxInvalidArgument as e:
            raise ValueError(str(e)) from e
        return self._gather_all(cloud, idx, int(m.value), output)

    def box_filter(self, cloud: PointCloudShared, min_distance: float = 1.0, max_distance: float = FLT_MAX,
                   output: PointCloudShared | None = None) -> PointCloudShared:
        """PreprocessFilter::box_filter (box_filter_operator.hpp:19-54): keep points whose L-infinity range lies
        in [min, max]; every attribute the cloud carries is compacted with them, in source order."""
        output = output if output is not None else cloud
        n = cloud.size()
        if n == 0:
            return output
        idx = DeviceArray(self.queue, (n,), np.int32)
        m = C.c_size_t()
        check(_lib.lib().spx_box_filter_indices(self.queue.handle, cloud.points.ptr, n, min_distance, max_distance, idx.ptr,
                                                C.byref(m)))
        return self._gather_all(cloud, idx, int(m.value), output)


class OutlierRemoval:
    """filter::OutlierRemoval (outlier_removal_filter.hpp in the reference) with the semantics of PCL's
    StatisticalOutlierRemoval and RadiusOutlierRemoval, on the exact grid index (DESIGN.md §3.3).  Both filters keep
    the surviving points in source order and compact every attribute the cloud carries; `output` may be the cloud
    itself, None returns a new cloud.  Without a `tree`, a KDTree is built over the cloud (honouring its index_hint);
    a given tree must have been built over exactly this cloud."""

    def __init__(self, queue: DeviceQueue):
        self.queue = queue

    def _tree(self, cloud: PointCloudShared, tree: "KDTree | None"):
        if tree is None:
            return KDTree.build(self.queue, cloud), True
        if tree._n != cloud.size():
            raise ValueError("[OutlierRemoval] the tree was not built over this cloud")
        return tree, False

    def _run(self, cloud, output, tree, call):
        n = cloud.size()
        if n == 0:
            return _gather_attributes(self.queue, cloud, None, 0, output)
        t, owned = self._tree(cloud, tree)
        try:
            idx = DeviceArray(self.queue, (n,), np.int32)
            m = C.c_size_t()
            try:
                check(call(t.handle, idx, m))
            except SpxInvalidArgument as e:
                raise ValueError(str(e)) from e
            return _gather_attributes(self.queue, cloud, idx, int(m.value), output)
        finally:
            if owned:
                t.close()

    def statistical(self, cloud: PointCloudShared, mean_k: int, stddev_mul: float,
                    output: PointCloudShared | None = None, tree: "KDTree | None" = None,
                    mean_distances: DeviceArray | None = None) -> PointCloudShared:
        """Keep point i iff its mean distance to its mean_k nearest other points is at most mu + stddev_mul * sigma,
        mu and sigma taken over all points (PCL's StatisticalOutlierRemoval).  1 <= mean_k <= 127; stddev_mul finite,
        may be negative.  mean_distances (optional device float[n]) receives every point's mean distance, NaN for
        points that were removed as invalid (non-finite, or no neighbour at all)."""
        if isinstance(mean_k, bool) or not isinstance(mean_k, (int, np.integer)) or not 1 <= int(mean_k) <= 127:
            raise ValueError("[OutlierRemoval::statistical] `mean_k` must be an integer in [1, 127]")
        if not math.isfinite(float(stddev_mul)):
            raise ValueError("[OutlierRemoval::statistical] `stddev_mul` must be finite")
        n = cloud.size()
        if mean_distances is not None and (mean_distances.dtype != np.float32 or mean_distances.nbytes < 4 * n):
            raise ValueError("[OutlierRemoval::statistical] mean_distances must be a float32 device array of n values")
        return self._run(cloud, output, tree, lambda h, idx, m: _lib.lib().spx_statistical_outlier_indices(
            h, cloud.points.ptr, n, int(mean_k), float(stddev_mul), _ptr(mean_distances), idx.ptr, C.byref(m)))

    def radius(self, cloud: PointCloudShared, radius: float, min_neighbors: int,
               output: PointCloudShared | None = None, tree: "KDTree | None" = None) -> PointCloudShared:
        """Keep point i iff at least min_neighbors other points lie within `radius` (squared distances compared in fp32
        against radius * radius; PCL's RadiusOutlierRemoval).  radius finite and >= 0; min_neighbors = 0 keeps every
        finite point, radius = 0 counts exact duplicates only."""
        if not (math.isfinite(float(radius)) and float(radius) >= 0.0):
            raise ValueError("[OutlierRemoval::radius] `radius` must be finite and >= 0")
        if isinstance(min_neighbors, bool) or not isinstance(min_neighbors, (int, np.integer)) \
                or not 0 <= int(min_neighbors) < 2 ** 32:
            raise ValueError("[OutlierRemoval::radius] `min_neighbors` must be an integer in [0, 2^32)")
        n = cloud.size()
        return self._run(cloud, output, tree, lambda h, idx, m: _lib.lib().spx_radius_outlier_indices(
            h, cloud.points.ptr, n, float(radius), int(min_neighbors), idx.ptr, C.byref(m)))


class EuclideanClusters:
    """The result of EuclideanClustering.extract: C clusters, ordered by size descending (ties: smallest member
    ascending).  labels (device int32[n]): each point's cluster, -1 for non-finite points and dropped components;
    indices (device int32[offsets[C]]): the members of cluster 0, 1, ..., each ascending; offsets (host uint32[C + 1]):
    where each cluster's members start in indices."""

    def __init__(self, queue: DeviceQueue, cloud: PointCloudShared, labels: DeviceArray, indices: DeviceArray,
                 offsets: np.ndarray):
        self.queue = queue
        self.cloud = cloud
        self.labels = labels
        self.indices = indices
        self.offsets = offsets

    def __len__(self):
        return len(self.offsets) - 1

    def cluster(self, c: int, output: PointCloudShared | None = None) -> PointCloudShared:
        """Cluster c as a cloud: every attribute of the source cloud, members in ascending index order.  The source
        cloud must not have changed since extract."""
        if not 0 <= c < len(self):
            raise IndexError(f"[EuclideanClustering] cluster {c} of {len(self)}")
        first, end = int(self.offsets[c]), int(self.offsets[c + 1])
        return _gather_attributes(self.queue, self.cloud, self.indices, end - first, output, first)


class EuclideanClustering:
    """Euclidean cluster extraction (semantics of PCL's EuclideanClusterExtraction, DESIGN.md §3.4) on the exact grid
    index: the connected components of the graph joining two finite points whose fp32 squared distance is at most
    tolerance * tolerance.  Components with fewer than min_cluster_size or more than max_cluster_size points are
    dropped (not split).  Without a `tree`, a KDTree is built over the cloud (honouring its index_hint); a given tree
    must have been built over exactly this cloud.  libspx's own interface."""

    def __init__(self, queue: DeviceQueue):
        self.queue = queue

    def extract(self, cloud: PointCloudShared, tolerance: float, min_cluster_size: int = 1,
                max_cluster_size: int = 2 ** 31 - 1, tree: "KDTree | None" = None) -> EuclideanClusters:
        if not (math.isfinite(float(tolerance)) and float(tolerance) >= 0.0):
            raise ValueError("[EuclideanClustering] `tolerance` must be finite and >= 0")
        for v in (min_cluster_size, max_cluster_size):
            if isinstance(v, bool) or not isinstance(v, (int, np.integer)) or not 1 <= int(v) < 2 ** 32:
                raise ValueError("[EuclideanClustering] cluster sizes must be integers in [1, 2^32)")
        if int(min_cluster_size) > int(max_cluster_size):
            raise ValueError("[EuclideanClustering] need min_cluster_size <= max_cluster_size")
        n = cloud.size()
        if n >= 2 ** 31:
            raise ValueError("[EuclideanClustering] at most 2^31 - 1 points")
        labels = DeviceArray(self.queue, (n,), np.int32)
        indices = DeviceArray(self.queue, (n,), np.int32)
        if n == 0:
            return EuclideanClusters(self.queue, cloud, labels, indices, np.zeros(1, np.uint32))
        if tree is None:
            t, owned = KDTree.build(self.queue, cloud), True
        elif tree._n != n:
            raise ValueError("[EuclideanClustering] the tree was not built over this cloud")
        else:
            t, owned = tree, False
        try:
            offsets = DeviceArray(self.queue, (n + 1,), np.uint32)
            nc, nm = C.c_size_t(), C.c_size_t()
            try:
                check(_lib.lib().spx_euclidean_clusters(t.handle, cloud.points.ptr, n, float(tolerance),
                                                        int(min_cluster_size), int(max_cluster_size), labels.ptr,
                                                        indices.ptr, offsets.ptr, C.byref(nc), C.byref(nm)))
            except SpxInvalidArgument as e:
                raise ValueError(str(e)) from e
            return EuclideanClusters(self.queue, cloud, labels, _trim(indices, int(nm.value)),
                                     offsets.download(int(nc.value) + 1))
        finally:
            if owned:
                t.close()


class PlaneModel:
    """The result of PlaneSegmentation.segment.  coefficients (host float32[4]): the plane (a, b, c, d) with
    a x + b y + c z + d = 0 and (a, b, c) a unit normal, NaN without a model; hypothesis: the index of the winning
    hypothesis, -1 without a model; inliers (device int32[m]): the points within the threshold of the plane, ascending;
    remainder (device int32[n - m]): every other index ascending, non-finite rows included."""

    def __init__(self, queue: DeviceQueue, cloud: PointCloudShared, coefficients: np.ndarray, hypothesis: int,
                 inliers: DeviceArray, remainder: DeviceArray):
        self.queue = queue
        self.cloud = cloud
        self.coefficients = coefficients
        self.hypothesis = hypothesis
        self.inliers = inliers
        self.remainder = remainder

    def inlier_cloud(self, output: PointCloudShared | None = None) -> PointCloudShared:
        """The inliers as a cloud: every attribute of the source cloud, in ascending index order.  The source cloud
        must not have changed since segment."""
        return _gather_attributes(self.queue, self.cloud, self.inliers, self.inliers.shape[0], output)

    def remainder_cloud(self, output: PointCloudShared | None = None) -> PointCloudShared:
        """Every point but the inliers as a cloud (PCL's ExtractIndices with setNegative(true)): every attribute, in
        ascending index order."""
        return _gather_attributes(self.queue, self.cloud, self.remainder, self.remainder.shape[0], output)


class PlaneSegmentation:
    """RANSAC plane segmentation (semantics of PCL's SACSegmentation with SACMODEL_PLANE, or
    SACMODEL_PERPENDICULAR_PLANE when an axis is given, and SAC_RANSAC; DESIGN.md §3.5).  max_iterations hypotheses are
    drawn from a counter-based stream keyed by `seed` and scored over every finite point; the one with the most points
    at |a x + b y + c z + d| < distance_threshold wins (ties: the lowest index).  With an `axis`, a hypothesis whose
    normal lies more than eps_angle (radians) from it is rejected.  optimize_coefficients refits the plane to the
    inliers by least squares and selects them again.  libspx's own interface."""

    def __init__(self, queue: DeviceQueue):
        self.queue = queue

    def segment(self, cloud: PointCloudShared, distance_threshold: float, max_iterations: int = 1000, axis=None,
                eps_angle: float = 0.0, seed: int = 0, optimize_coefficients: bool = True,
                hypothesis_counts: DeviceArray | None = None) -> PlaneModel:
        """hypothesis_counts (optional device uint32[max_iterations]) receives every hypothesis's inlier count,
        0xFFFFFFFF for an invalid one."""
        t = float(distance_threshold)
        if not (math.isfinite(t) and t > 0.0):
            raise ValueError("[PlaneSegmentation] `distance_threshold` must be finite and > 0")
        if isinstance(max_iterations, bool) or not isinstance(max_iterations, (int, np.integer)) \
                or not 1 <= int(max_iterations) <= 2 ** 20:
            raise ValueError("[PlaneSegmentation] `max_iterations` must be an integer in [1, 2^20]")
        eps = float(eps_angle)
        if not 0.0 <= eps <= math.pi / 2:
            raise ValueError("[PlaneSegmentation] `eps_angle` must be in [0, pi/2]")
        if isinstance(seed, bool) or not isinstance(seed, (int, np.integer)) or not 0 <= int(seed) < 2 ** 64:
            raise ValueError("[PlaneSegmentation] `seed` must be an integer in [0, 2^64)")
        ax = None
        if axis is not None:
            ax = np.ascontiguousarray(axis, np.float32).reshape(-1)
            if ax.shape != (3,) or not np.isfinite(ax).all() or not ax.any():
                raise ValueError("[PlaneSegmentation] `axis` must be 3 finite values, not all zero")
        n = cloud.size()
        if n >= 2 ** 31:
            raise ValueError("[PlaneSegmentation] at most 2^31 - 1 points")
        H = int(max_iterations)
        if hypothesis_counts is not None and (hypothesis_counts.dtype != np.uint32 or hypothesis_counts.nbytes < 4 * H):
            raise ValueError("[PlaneSegmentation] hypothesis_counts must be a uint32 device array of max_iterations values")
        inliers = DeviceArray(self.queue, (n,), np.int32)
        remainder = DeviceArray(self.queue, (n,), np.int32)
        coef = np.empty(4, np.float32)
        hyp, m = C.c_int32(), C.c_size_t()
        try:
            check(_lib.lib().spx_plane_segment(self.queue.handle, cloud.points.ptr if n else None, n, t, H, int(seed),
                                               ax.ctypes.data if ax is not None else None, eps,
                                               int(bool(optimize_coefficients)), coef.ctypes.data, C.byref(hyp),
                                               inliers.ptr, C.byref(m), remainder.ptr, _ptr(hypothesis_counts)))
        except SpxInvalidArgument as e:
            raise ValueError(str(e)) from e
        m = int(m.value)
        return PlaneModel(self.queue, cloud, coef, int(hyp.value), _trim(inliers, m), _trim(remainder, n - m))


FPFH_DIM = 33


class FPFHEstimation:
    """FPFH descriptors (Rusu et al. 2009, with the point's own SPFH term; DESIGN.md §3.6) over the max_nn nearest
    neighbours within `radius` (Open3D's hybrid search).  The cloud must carry normals, oriented as
    covariance.estimate_normals writes them.  Without a `tree`, a KDTree is built over the cloud; a given tree must have
    been built over exactly this cloud.  libspx's own interface."""

    def __init__(self, queue: DeviceQueue):
        self.queue = queue

    def compute(self, cloud: PointCloudShared, radius: float, max_nn: int = 100,
                tree: "KDTree | None" = None) -> DeviceArray:
        """device float32 (n, 33): bins 0-10 f1, 11-21 f2, 22-32 f3; NaN rows for points with a non-finite coordinate
        or normal"""
        r = float(radius)
        if not (math.isfinite(r) and r > 0.0):
            raise ValueError("[FPFHEstimation] `radius` must be finite and > 0")
        if isinstance(max_nn, bool) or not isinstance(max_nn, (int, np.integer)) or not 1 <= int(max_nn) <= 100:
            raise ValueError("[FPFHEstimation] `max_nn` must be an integer in [1, 100]")
        n = cloud.size()
        if n >= 2 ** 31:
            raise ValueError("[FPFHEstimation] at most 2^31 - 1 points")
        if n and not cloud.has_normal():
            raise ValueError("[FPFHEstimation] the cloud has no normals (covariance.estimate_normals)")
        out = DeviceArray(self.queue, (n, FPFH_DIM), np.float32)
        if n == 0:
            return out
        if tree is None:
            t, owned = KDTree.build(self.queue, cloud), True
        elif tree._n != n:
            raise ValueError("[FPFHEstimation] the tree was not built over this cloud")
        else:
            t, owned = tree, False
        try:
            nn = KNNResult()
            t.radius_search_async(cloud, int(max_nn), r, nn)
            try:
                check(_lib.lib().spx_fpfh(self.queue.handle, cloud.points.ptr, cloud.normals.ptr, n, nn.indices.ptr,
                                          nn.distances.ptr, int(max_nn), out.ptr))
            except SpxInvalidArgument as e:
                raise ValueError(str(e)) from e
            self.queue.wait()
        finally:
            if owned:
                t.close()
        return out


def _feature_rows(queue: DeviceQueue, f) -> DeviceArray:
    if isinstance(f, DeviceArray):
        if f.dtype != np.float32 or len(f.shape) != 2 or f.shape[1] != FPFH_DIM:
            raise ValueError("features must be float32 (n, 33)")
        return f
    a = np.ascontiguousarray(f, np.float32)
    if a.ndim != 2 or a.shape[1] != FPFH_DIM:
        raise ValueError("features must be float32 (n, 33)")
    return DeviceArray.from_host(queue, a)


def match_features(queue: DeviceQueue, source_features, target_features, mutual: bool = False):
    """(src_idx, tgt_idx), device int32 arrays: for every source row i with a candidate, the target row with the
    smallest squared feature distance (ties: the lowest index; NaN rows never match), ascending in i.  mutual keeps a
    pair only if the reverse search picks i as well (DESIGN.md §3.6)."""
    s, t = _feature_rows(queue, source_features), _feature_rows(queue, target_features)
    ns, nt = s.shape[0], t.shape[0]
    if ns >= 2 ** 31 or nt >= 2 ** 31:
        raise ValueError("[match_features] at most 2^31 - 1 rows")
    si, ti = DeviceArray(queue, (ns,), np.int32), DeviceArray(queue, (ns,), np.int32)
    m = C.c_size_t()
    check(_lib.lib().spx_feature_correspondences(queue.handle, s.ptr if ns else None, ns, t.ptr if nt else None, nt,
                                                 int(bool(mutual)), si.ptr, ti.ptr, C.byref(m)))
    m = int(m.value)
    return _trim(si, m), _trim(ti, m)


class RANSACResult:
    """The result of RANSACRegistration.align.  T (host float32 4x4, row-major numpy): target <- source, NaN without a
    model; hypothesis: the winning hypothesis, -1 without a model; inliers (device int32[m]): positions into the
    correspondence list, ascending; fitness: m / number of correspondences (0 without any)."""

    def __init__(self, T: np.ndarray, hypothesis: int, inliers: DeviceArray, n_correspondences: int):
        self.T = T
        self.hypothesis = hypothesis
        self.inliers = inliers
        self.fitness = len(inliers) / n_correspondences if n_correspondences else 0.0

    def valid(self) -> bool:
        return self.hypothesis >= 0


class RANSACRegistration:
    """Global registration by RANSAC over feature correspondences with an edge-length check (the usual
    feature-matching RANSAC, as Open3D's registration_ransac_based_on_feature_matching; DESIGN.md §3.6).
    max_iterations three-correspondence hypotheses drawn from a counter-based stream keyed by `seed`, each posed in
    closed form (triad) and scored over every correspondence with |R p + t - q| < max_correspondence_distance; the most
    inliers win (ties: the lowest index).  optimize refits the pose to the inliers by least squares and selects them
    again.  Its pose is the initial guess to hand to Registration.align.  libspx's own interface."""

    def __init__(self, queue: DeviceQueue):
        self.queue = queue

    def align(self, source: PointCloudShared, target: PointCloudShared, correspondences,
              max_correspondence_distance: float, max_iterations: int = 100000, edge_length_similarity: float = 0.9,
              seed: int = 0, optimize: bool = True, hypothesis_counts: DeviceArray | None = None) -> RANSACResult:
        """correspondences: (src_idx, tgt_idx) as match_features returns them (device or host int32).
        hypothesis_counts (optional device uint32[max_iterations]) receives every hypothesis's inlier count,
        0xFFFFFFFF for an invalid one."""
        eps = float(max_correspondence_distance)
        if not (math.isfinite(eps) and eps > 0.0):
            raise ValueError("[RANSACRegistration] `max_correspondence_distance` must be finite and > 0")
        if isinstance(max_iterations, bool) or not isinstance(max_iterations, (int, np.integer)) \
                or not 1 <= int(max_iterations) <= 2 ** 20:
            raise ValueError("[RANSACRegistration] `max_iterations` must be an integer in [1, 2^20]")
        tau = float(edge_length_similarity)
        if not 0.0 < tau <= 1.0:
            raise ValueError("[RANSACRegistration] `edge_length_similarity` must be in (0, 1]")
        if isinstance(seed, bool) or not isinstance(seed, (int, np.integer)) or not 0 <= int(seed) < 2 ** 64:
            raise ValueError("[RANSACRegistration] `seed` must be an integer in [0, 2^64)")
        si, ti = correspondences
        si = si if isinstance(si, DeviceArray) else DeviceArray.from_host(self.queue, np.asarray(si, np.int32))
        ti = ti if isinstance(ti, DeviceArray) else DeviceArray.from_host(self.queue, np.asarray(ti, np.int32))
        if si.dtype != np.int32 or ti.dtype != np.int32 or si.shape != ti.shape or len(si.shape) != 1:
            raise ValueError("[RANSACRegistration] correspondences must be two int32 arrays of equal length")
        M = si.shape[0]
        H = int(max_iterations)
        if hypothesis_counts is not None and (hypothesis_counts.dtype != np.uint32 or hypothesis_counts.nbytes < 4 * H):
            raise ValueError("[RANSACRegistration] hypothesis_counts must be a uint32 device array of max_iterations values")
        inliers = DeviceArray(self.queue, (M,), np.int32)
        T = np.empty(16, np.float32)
        hyp, m = C.c_int32(), C.c_size_t()
        try:
            check(_lib.lib().spx_ransac_registration(
                self.queue.handle, _ptr(source.points), source.size(), _ptr(target.points), target.size(),
                si.ptr if M else None, ti.ptr if M else None, M, eps, H, int(seed), tau, int(bool(optimize)),
                T.ctypes.data, C.byref(hyp), inliers.ptr if M else None, C.byref(m), _ptr(hypothesis_counts)))
        except SpxInvalidArgument as e:
            raise ValueError(str(e)) from e
        return RANSACResult(T.reshape(4, 4).T.copy(), int(hyp.value), _trim(inliers, int(m.value)), M)


class transform:  # namespace sycl_points::algorithms::transform (common/transform.hpp:45-136)
    @staticmethod
    def transform(cloud: PointCloudShared, trans) -> None:
        """in place: points T p, covariances T C T^T, normals T n"""
        if cloud.size() == 0:
            return
        t16 = _T16(trans)
        check(_lib.lib().spx_transform(cloud.queue.handle, cloud.points.ptr,
                                       _ptr(cloud.covs) if cloud.has_cov() else None,
                                       _ptr(cloud.normals) if cloud.has_normal() else None, cloud.size(), _hostf(t16)))
        cloud.index_hint = None  # the points moved: the voxel box no longer describes them

    transform_async = transform

    @staticmethod
    def transform_copy(cloud: PointCloudShared, trans) -> PointCloudShared:
        out = PointCloudShared(cloud.queue)
        n = cloud.size()

        def dup(a: DeviceArray | None, enable: bool):
            if not enable:
                return None
            b = DeviceArray(cloud.queue, a.shape, a.dtype)
            check(_lib.lib().spx_memcpy_d2d(cloud.queue.handle, b.ptr, a.ptr, a.nbytes))
            return b

        out.points = dup(cloud.points, n > 0) if n else DeviceArray(cloud.queue, (0, 4), np.float32)
        out._n = n
        out.covs = dup(cloud.covs, cloud.has_cov())
        out.normals = dup(cloud.normals, cloud.has_normal())
        out.rgb = dup(cloud.rgb, cloud.has_rgb())
        out.intensities = dup(cloud.intensities, cloud.has_intensity())
        out.timestamp_offsets = dup(cloud.timestamp_offsets, cloud.has_timestamps())
        transform.transform(out, trans)
        return out


class deskew:  # namespace sycl_points::algorithms::deskew
    @staticmethod
    def deskew_point_cloud_constant_velocity(input_cloud: PointCloudShared, output_cloud: PointCloudShared,
                                             previous_relative_pose, current_relative_pose,
                                             inter_scan_duration_seconds: float = -1.0) -> bool:
        """relative_pose_deskew.hpp:36-178.  False (nothing done) for an empty cloud, a cloud without timestamps
        or a non-positive duration.  `output_cloud` may be `input_cloud`."""
        n = input_cloud.size()
        if n == 0 or not input_cloud.has_timestamps():
            return False
        dur = inter_scan_duration_seconds if inter_scan_duration_seconds > 0.0 else \
            float(np.float32((input_cloud.end_time_ms - input_cloud.start_time_ms) * 1e-3))
        if dur <= 0.0:
            return False
        q = input_cloud.queue
        if output_cloud is not input_cloud:
            def dup(a, enable):
                if not enable:
                    return None
                b = DeviceArray(q, a.shape, a.dtype)
                check(_lib.lib().spx_memcpy_d2d(q.handle, b.ptr, a.ptr, a.nbytes))
                return b
            output_cloud.start_time_ms, output_cloud.end_time_ms = input_cloud.start_time_ms, input_cloud.end_time_ms
            output_cloud.timestamp_offsets = dup(input_cloud.timestamp_offsets, True)
            output_cloud.points = DeviceArray(q, (n, 4), np.float32)
            output_cloud._n = n
            output_cloud.normals = DeviceArray(q, (n, 4), np.float32) if input_cloud.has_normal() else None
            output_cloud.covs = DeviceArray(q, (n, 4, 4), np.float32) if input_cloud.has_cov() else None
            output_cloud.rgb = dup(input_cloud.rgb, input_cloud.has_rgb())
            output_cloud.intensities = dup(input_cloud.intensities, input_cloud.has_intensity())
        output_cloud.index_hint = None
        prev = np.asarray(previous_relative_pose, np.float32).reshape(4, 4)
        cur = np.asarray(current_relative_pose, np.float32).reshape(4, 4)
        inv = np.eye(4, dtype=np.float32)  # Isometry3f::inverse(): R^T, -R^T t
        inv[:3, :3] = prev[:3, :3].T
        inv[:3, 3] = -(prev[:3, :3].T @ prev[:3, 3])
        delta = np.eye(4, dtype=np.float32)
        delta[:3, :3] = inv[:3, :3] @ cur[:3, :3]
        delta[:3, 3] = inv[:3, :3] @ cur[:3, 3] + inv[:3, 3]
        twist = se3_log(delta)
        nrm, cov = input_cloud.has_normal(), input_cloud.has_cov()
        check(_lib.lib().spx_deskew_constant_velocity(
            q.handle, input_cloud.points.ptr, _ptr(input_cloud.normals) if nrm else None,
            _ptr(input_cloud.covs) if cov else None, output_cloud.timestamp_offsets.ptr, n, _hostf(twist), float(dur),
            output_cloud.points.ptr, _ptr(output_cloud.normals) if nrm else None,
            _ptr(output_cloud.covs) if cov else None))
        q.wait()
        return True


# ------------------------------------------------------------------ registration
class RegType(enum.IntEnum):  # factor.hpp:18-32
    POINT_TO_POINT = 0
    POINT_TO_PLANE = 1
    POINT_TO_DISTRIBUTION = 2
    GICP = 3
    GENZ = 4


class RobustLossType(enum.IntEnum):  # robust.hpp:14-20
    NONE = 0
    HUBER = 1
    TUKEY = 2
    CAUCHY = 3
    GEMAN_MCCLURE = 4


class OptimizationMethod(enum.IntEnum):  # registration_params.hpp:17-21
    GAUSS_NEWTON = 0
    LEVENBERG_MARQUARDT = 1
    POWELL_DOGLEG = 2


def RegType_from_string(s: str) -> RegType:  # factor.hpp:43-61
    u = s.upper()
    if u == "P2D":
        return RegType.POINT_TO_DISTRIBUTION
    try:
        return RegType[u]
    except KeyError:
        raise RuntimeError(f"[RegType_from_string] Invalid RegType str '{s}'")


def RobustLossType_from_string(s: str) -> RobustLossType:  # robust.hpp:30-48
    try:
        return RobustLossType[s.upper()]
    except KeyError:
        raise RuntimeError(f"[RobustLossType_from_string] Invalid RobustLossType str '{s}'")


def OptimizationMethod_from_string(s: str) -> OptimizationMethod:  # registration_params.hpp:23-38
    u = s.upper()
    table = {"GN": 0, "GAUSS_NEWTON": 0, "LM": 1, "LEVENBERG_MARQUARDT": 1, "DOGLEG": 2, "POWELL_DOGLEG": 2}
    if u not in table:
        raise RuntimeError(f"[OptimizationMethod_from_string] Invalid OptimizationMethod str [{s}]")
    return OptimizationMethod(table[u])


@dataclass
class RobustParams:
    type: RobustLossType = RobustLossType.NONE
    default_scale: float = 10.0


@dataclass
class Criteria:
    translation: float = 1e-3
    rotation: float = 1e-3


@dataclass
class GaussNewtonParams:
    lambda_: float = 1.0


@dataclass
class LevenbergMarquardtParams:
    max_inner_iterations: int = 10
    lambda_factor: float = 2.0
    init_lambda: float = 1.0
    max_lambda: float = 1e3
    min_lambda: float = 1e-6


@dataclass
class DoglegParams:
    initial_trust_region_radius: float = 1.0
    min_trust_region_radius: float = 1e-4
    max_trust_region_radius: float = 10.0
    eta1: float = 0.25
    eta2: float = 0.75
    gamma_decrease: float = 0.25
    gamma_increase: float = 2.0


@dataclass
class GenZParams:
    planarity_threshold: float = 0.2  # registration_params.hpp:51-53


@dataclass
class RotationConstraintRobust:
    default_scale: float = 10.0


@dataclass
class RotationConstraintParams:
    """RegistrationFactorParams::RotationConstraint (registration_params.hpp:54-62)"""
    enable: bool = False
    weight: float = 1.0
    robust: RotationConstraintRobust = field(default_factory=RotationConstraintRobust)


class DegenerateRegularizationType(enum.IntEnum):  # degenerate_regularization.hpp:14-17
    none = 0
    nl_reg = 1


def DegenerateRegularizationType_from_string(s: str) -> DegenerateRegularizationType:  # :19-33
    u = s.upper()
    if u == "NONE":
        return DegenerateRegularizationType.none
    if u in ("NL-REG", "NL_REG"):
        return DegenerateRegularizationType.nl_reg
    raise RuntimeError(f"[DegenerateRegularizationType_from_string] Invalid DegenerateRegularizationType str [{s}]")


@dataclass
class DegenerateRegularizationParams:  # degenerate_regularization.hpp:35-40
    type: DegenerateRegularizationType = DegenerateRegularizationType.none
    rot_eigenvalue_threshold: float = 10.0
    trans_eigenvalue_threshold: float = 1.0
    base_factor: float = 1.0


@dataclass
class MapPriorParams:  # map_prior.hpp:15-21
    enabled: bool = False
    rot_vel_sigma: float = 1.0
    trans_vel_sigma: float = 1.0
    rot_base_sigma: float = 3.16e-2
    trans_base_sigma: float = 1e-2


@dataclass
class RegistrationParams:
    """RegistrationParams (registration_params.hpp:41-114), same defaults."""
    reg_type: RegType = RegType.GICP
    max_correspondence_distance: float = 2.0
    robust: RobustParams = field(default_factory=RobustParams)
    verbose: bool = False
    gn: GaussNewtonParams = field(default_factory=GaussNewtonParams)
    lm: LevenbergMarquardtParams = field(default_factory=LevenbergMarquardtParams)
    dogleg: DoglegParams = field(default_factory=DoglegParams)
    optimization_method: OptimizationMethod = OptimizationMethod.GAUSS_NEWTON
    max_iterations: int = 20
    criteria: Criteria = field(default_factory=Criteria)
    genz: GenZParams = field(default_factory=GenZParams)
    rotation_constraint: RotationConstraintParams = field(default_factory=RotationConstraintParams)
    degenerate_reg: DegenerateRegularizationParams = field(default_factory=DegenerateRegularizationParams)
    map_prior: MapPriorParams = field(default_factory=MapPriorParams)
    max_blocks: int = 0  # spx extension: cap on the align kernel's persistent grid (0 = one full wave)

    def addons_c(self) -> RegistrationAddonsC:
        d, m = self.degenerate_reg, self.map_prior
        return RegistrationAddonsC(int(d.type), d.rot_eigenvalue_threshold, d.trans_eigenvalue_threshold, d.base_factor,
                                   int(bool(m.enabled)), m.rot_vel_sigma, m.trans_vel_sigma, m.rot_base_sigma,
                                   m.trans_base_sigma)

    def to_c(self) -> RegistrationParamsC:
        P = RegistrationParamsC()
        _lib.lib().spx_default_registration_params(C.byref(P))
        P.reg_type = int(self.reg_type)
        P.robust_loss = int(self.robust.type)
        P.optimization_method = int(self.optimization_method)
        P.max_iterations = int(self.max_iterations)
        P.max_correspondence_distance = self.max_correspondence_distance
        P.robust_default_scale = self.robust.default_scale
        P.criteria_translation = self.criteria.translation
        P.criteria_rotation = self.criteria.rotation
        P.gn_lambda = self.gn.lambda_
        P.lm_max_inner_iterations = self.lm.max_inner_iterations
        P.lm_lambda_factor = self.lm.lambda_factor
        P.lm_init_lambda = self.lm.init_lambda
        P.lm_max_lambda = self.lm.max_lambda
        P.lm_min_lambda = self.lm.min_lambda
        P.dogleg_initial_trust_region_radius = self.dogleg.initial_trust_region_radius
        P.dogleg_min_trust_region_radius = self.dogleg.min_trust_region_radius
        P.dogleg_max_trust_region_radius = self.dogleg.max_trust_region_radius
        P.dogleg_eta1 = self.dogleg.eta1
        P.dogleg_eta2 = self.dogleg.eta2
        P.dogleg_gamma_decrease = self.dogleg.gamma_decrease
        P.dogleg_gamma_increase = self.dogleg.gamma_increase
        P.max_grid_blocks = int(self.max_blocks)
        P.genz_planarity_threshold = self.genz.planarity_threshold
        P.rotation_constraint_enable = 1 if self.rotation_constraint.enable else 0
        P.rotation_constraint_weight = self.rotation_constraint.weight
        P.rotation_constraint_robust_scale = self.rotation_constraint.robust.default_scale
        return P


@dataclass
class RegistrationResult:
    """RegistrationResult (result.hpp:13-28)."""
    T: np.ndarray = field(default_factory=lambda: np.eye(4, dtype=np.float32))
    converged: bool = False
    iterations: int = 0
    H: np.ndarray = field(default_factory=lambda: np.zeros((6, 6), np.float32))
    b: np.ndarray = field(default_factory=lambda: np.zeros(6, np.float32))
    error: float = FLT_MAX
    H_raw: np.ndarray = field(default_factory=lambda: np.zeros((6, 6), np.float32))
    b_raw: np.ndarray = field(default_factory=lambda: np.zeros(6, np.float32))
    error_raw: float = FLT_MAX
    inlier: int = 0
    trace: np.ndarray | None = None  # pose after every outer iteration (parity tests)

    @staticmethod
    def from_c(R: RegistrationResultC) -> "RegistrationResult":
        # one copy of the struct's 104 words, sliced by field offset (words): T 0, converged 16, iterations 17,
        # H 18, b 54, error 60, H_raw 61, b_raw 97, error_raw 103, inlier 104 — the call sits between the
        # align's last kernel and the caller, so it is kept short
        w = np.frombuffer(R, np.float32).copy()
        return RegistrationResult(T=w[0:16].reshape(4, 4).T.copy(), converged=bool(R.converged),
                                  iterations=int(R.iterations), H=w[18:54].reshape(6, 6), b=w[54:60],
                                  error=float(w[60]), H_raw=w[61:97].reshape(6, 6), b_raw=w[97:103],
                                  error_raw=float(w[103]), inlier=int(R.inlier))


@dataclass
class LinearizedResult:
    """LinearizedResult (linearized_result.hpp:12-23)."""
    H: np.ndarray
    b: np.ndarray
    error: float
    inlier: int


@dataclass
class ExecutionOptions:
    """Registration::ExecutionOptions (registration.hpp:92-100)."""
    robust_scale: float = -1.0
    rotation_robust_scale: float = -1.0
    dt: float = 0.1
    prev_pose: np.ndarray = field(default_factory=lambda: np.eye(4, dtype=np.float32))


def se3_exp(twist) -> np.ndarray:
    tw = np.ascontiguousarray(twist, np.float32)
    out = np.empty(16, np.float32)
    check(_lib.lib().spx_se3_exp(_hostf(tw), _hostf(out)))
    return _T_from16(out)


def se3_log(T) -> np.ndarray:
    """eigen_utils::lie::se3_log (eigen_utils.hpp:991-1034): [rx ry rz tx ty tz]."""
    out = np.empty(6, np.float32)
    check(_lib.lib().spx_se3_log(_hostf(_T16(T)), _hostf(out)))
    return out


def solve_6x6(H, b, lam: float):
    H = np.ascontiguousarray(H, np.float32).reshape(36)
    b = np.ascontiguousarray(b, np.float32)
    d = np.empty(6, np.float32)
    ok = C.c_int()
    check(_lib.lib().spx_solve_6x6(_hostf(H), _hostf(b), lam, _hostf(d), C.byref(ok)))
    return bool(ok.value), d


def dogleg_step(H, g, radius: float):
    H = np.ascontiguousarray(H, np.float32).reshape(36)
    g = np.ascontiguousarray(g, np.float32)
    p = np.empty(6, np.float32)
    sn, pr = C.c_float(), C.c_float()
    check(_lib.lib().spx_dogleg_step(_hostf(H), _hostf(g), radius, _hostf(p), C.byref(sn), C.byref(pr)))
    return p, sn.value, pr.value


class Registration:
    """registration::Registration (registration.hpp:88-965)."""

    def __init__(self, queue: DeviceQueue, params: RegistrationParams | None = None):
        self.queue = queue
        self.params = params if params is not None else RegistrationParams()
        h = C.c_void_p()
        Pc = self.params.to_c()
        check(_lib.lib().spx_registration_create(queue.handle, C.byref(Pc), C.byref(h)))
        self._h = h
        self._neighbors = KNNResult()  # registration.hpp:365 (used with injected KNNs)
        a = self.params.addons_c()
        check(_lib.lib().spx_registration_set_addons(self._h, C.byref(a)))  # registration.hpp:112-113
        self._addons_key = bytes(a)

    def set_map_prior_state(self, prev_result: "RegistrationResult", T_pred) -> bool:
        """Registration::set_map_prior_state (registration.hpp:124-126): arms the MAP prior of the next align from
        the previous result and the predicted pose; returns whether a prior is now in force."""
        self._sync_addons()
        R = RegistrationResultC()
        R.T[:] = list(_T16(prev_result.T))
        R.H_raw[:] = list(np.asarray(prev_result.H_raw, np.float32).reshape(36))
        R.error_raw = float(prev_result.error_raw)
        R.inlier = int(prev_result.inlier)
        act = C.c_int()
        self._prior_omega = np.zeros(36, np.float32)
        check(_lib.lib().spx_registration_set_map_prior_state(self._h, C.byref(R), _hostf(_T16(T_pred)), C.byref(act),
                                                              _hostf(self._prior_omega)))
        return bool(act.value)

    def _sync_addons(self):
        """params.degenerate_reg / params.map_prior edited after construction: pushed (and the prior dropped, as
        MapPrior::set_params does) only when they changed"""
        a = self.params.addons_c()
        if bytes(a) != self._addons_key:
            check(_lib.lib().spx_registration_set_addons(self._h, C.byref(a)))
            self._addons_key = bytes(a)

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().spx_registration_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _scale(self, options: ExecutionOptions | None) -> float:
        s = options.robust_scale if options is not None else -1.0
        return s if s > 0.0 else self.params.robust.default_scale  # registration.hpp:217-218

    def _genz(self):
        """the stateless C entry points take the GenZ planarity threshold from a thread-local setting"""
        if self.params.reg_type == RegType.GENZ:
            check(_lib.lib().spx_set_genz_planarity_threshold(float(self.params.genz.planarity_threshold)))
        rc = self.params.rotation_constraint
        check(_lib.lib().spx_set_rotation_constraint(1 if rc.enable else 0, float(rc.weight), float(rc.robust.default_scale)))

    def _loss(self) -> int:
        if self.params.robust.type != RobustLossType.NONE and self.params.robust.default_scale <= 0.0:
            print("[Caution] `robust.default_scale` must be greater than zero. Disable robust loss.")
            self.params.robust.type = RobustLossType.NONE  # registration.hpp:186-192
        return int(self.params.robust.type)

    def _validate(self, source: PointCloudShared, target: PointCloudShared):
        # registration.hpp:129-193
        if self.params.reg_type == RegType.POINT_TO_PLANE and not target.has_normal():
            if not target.has_cov():
                raise RuntimeError("[Registration::validate_params] Normal vector or covariance matrices of target "
                                   "must be pre-computed before performing Point-to-Plane ICP matching.")
            print("[Caution] Normal vectors for Point-to-Plane ICP are not provided. ")
            print("          Attempting to derive them from pre-computed covariance matrices.")
            covariance.extract_normals(target)
        if self.params.reg_type == RegType.GENZ:
            if not target.has_cov():
                raise RuntimeError("[Registration::validate_params] Covariance matrices of target must be pre-computed "
                                   "before performing GenZ-ICP matching.")
            if not target.has_normal():
                print("[Caution] Normal vectors for GenZ-ICP are not provided. ")
                print("          Attempting to derive them from pre-computed covariance matrices.")
                covariance.extract_normals(target)
        if self.params.rotation_constraint.enable:
            if not source.has_cov():
                raise RuntimeError("[Registration::validate_params] Covariance matrices of source are required for "
                                   "performing rotation constraint matching.")
            if not target.has_cov():
                raise RuntimeError("[Registration::validate_params] Covariance matrices of target are required for "
                                   "performing rotation constraint matching.")
        if self.params.reg_type == RegType.GICP and (not source.has_cov() or not target.has_cov()):
            raise RuntimeError("[Registration::validate_params] Covariance matrices of source and target must be "
                               "pre-computed before performing GICP matching.")
        if self.params.reg_type == RegType.POINT_TO_DISTRIBUTION and not target.has_cov():
            raise RuntimeError("[Registration::validate_params] Covariance matrices of target must be pre-computed "
                               "before performing Point-to-Distribution ICP matching.")

    def align(self, source: PointCloudShared, target: PointCloudShared, target_knn: KNNBase, initial_guess=None,
              options: ExecutionOptions | None = None, trace: bool = False) -> RegistrationResult:
        """Registration::align (registration.hpp:201-276)."""
        T0 = np.eye(4, dtype=np.float32) if initial_guess is None else np.asarray(initial_guess, np.float32)
        if source.size() == 0:
            return RegistrationResult(T=T0.copy())
        self._validate(source, target)
        self._loss()
        if not isinstance(target_knn, KDTree):
            return self._align_injected_knn(source, target, target_knn, T0, options, trace)
        Pc = self.params.to_c()
        if options is not None and options.rotation_robust_scale > 0.0:  # registration.hpp:219-221
            Pc.rotation_constraint_robust_scale = float(options.rotation_robust_scale)
        check(_lib.lib().spx_registration_set_params(self._h, C.byref(Pc)))
        self._sync_addons()
        R = RegistrationResultC()
        t16 = _T16(T0)
        tr = np.zeros((max(self.params.max_iterations, 1), 16), np.float32) if trace else None
        scale = options.robust_scale if options is not None else -1.0
        check(_lib.lib().spx_registration_align(
            self._h, source.points.ptr, _ptr(source.covs) if source.has_cov() else None, source.size(),
            target.points.ptr, _ptr(target.covs) if target.has_cov() else None,
            _ptr(target.normals) if target.has_normal() else None, target.size(), target_knn.handle, _hostf(t16),
            float(scale), C.byref(R), _hostf(tr)))
        out = RegistrationResult.from_c(R)
        if trace:
            out.trace = np.stack([_T_from16(t) for t in tr])
        return out

    def align_batch(self, pairs, options: ExecutionOptions | None = None) -> list:
        """P independent aligns in one set-up launch + one persistent cooperative launch
        (spx_registration_align_batch; BASELINE config 5).  pairs: sequence of
        (source, target, target_knn[, initial_guess]).  Each result equals what align() returns for that
        pair alone, bit for bit.  Reference semantics per pair: registration.hpp:201-276."""
        pairs = list(pairs)
        n = len(pairs)
        if n == 0:
            return []
        self._loss()
        Pc = self.params.to_c()
        check(_lib.lib().spx_registration_set_params(self._h, C.byref(Pc)))
        arr = (_lib.AlignPairC * n)()
        keep = []
        scale = options.robust_scale if options is not None else -1.0
        for j, pr in enumerate(pairs):
            source, target, knn = pr[0], pr[1], pr[2]
            T0 = np.eye(4, dtype=np.float32) if len(pr) < 4 or pr[3] is None else np.asarray(pr[3], np.float32)
            if source.size():
                self._validate(source, target)
                if not isinstance(knn, KDTree):
                    raise SpxInvalidArgument(-1, "[Registration::align_batch] target_knn must be a KDTree (spx_index)")
            t16 = _T16(T0)
            keep.append(t16)
            a = arr[j]
            a.src_points = _addr(source.points.ptr) if source.size() else None
            a.src_covs = _addr(_ptr(source.covs)) if source.has_cov() else None
            a.ns = source.size()
            a.tgt_points = _addr(target.points.ptr) if target.size() else None
            a.tgt_covs = _addr(_ptr(target.covs)) if target.has_cov() else None
            a.tgt_normals = _addr(_ptr(target.normals)) if target.has_normal() else None
            a.nt = target.size()
            a.target_index = _addr(knn.handle) if isinstance(knn, KDTree) else None
            a.T_init_host = _hostf(t16)
            a.robust_scale = float(scale)
        R = (RegistrationResultC * n)()
        check(_lib.lib().spx_registration_align_batch(self._h, n, arr, R))
        return [RegistrationResult.from_c(R[j]) for j in range(n)]

    def last_timing(self) -> dict:
        """CUDA-event time of the iteration kernels of the last Gauss-Newton align (bench.py)."""
        ms, launches, iters = C.c_float(), C.c_int32(), C.c_int32()
        check(_lib.lib().spx_registration_last_timing(self._h, C.byref(ms), C.byref(launches), C.byref(iters)))
        return dict(loop_ms=ms.value, launches=launches.value, iterations=iters.value)

    def kept_correspondences(self) -> int:
        """Correspondences the last align kept without a search, summed over its iterations (split-kernel loop)."""
        kept = C.c_uint64()
        check(_lib.lib().spx_registration_kept_correspondences(self._h, C.byref(kept)))
        return int(kept.value)

    # -- pieces usable with any KNNBase (the reference's tests inject host KNNs)
    def _linearize(self, source, target, nn: KNNResult, T, scale) -> LinearizedResult:
        H = np.empty(36, np.float32)
        b = np.empty(6, np.float32)
        err, inl = C.c_float(), C.c_uint32()
        mc = np.float32(self.params.max_correspondence_distance)
        t16 = _T16(T)
        self._genz()
        check(_lib.lib().spx_linearize(
            self.queue.handle, int(self.params.reg_type), self._loss(), source.points.ptr,
            _ptr(source.covs) if source.has_cov() else None, source.size(), target.points.ptr,
            _ptr(target.covs) if target.has_cov() else None, _ptr(target.normals) if target.has_normal() else None,
            nn.indices.ptr, nn.distances.ptr, _hostf(t16), float(mc * mc), float(scale), _hostf(H), _hostf(b),
            C.byref(err), C.byref(inl)))
        return LinearizedResult(H.reshape(6, 6), b, err.value, inl.value)

    def _error(self, source, target, nn: KNNResult, T, scale):
        err, inl = C.c_float(), C.c_uint32()
        mc = np.float32(self.params.max_correspondence_distance)
        t16 = _T16(T)
        self._genz()
        check(_lib.lib().spx_error(
            self.queue.handle, int(self.params.reg_type), self._loss(), source.points.ptr,
            _ptr(source.covs) if source.has_cov() else None, source.size(), target.points.ptr,
            _ptr(target.covs) if target.has_cov() else None, _ptr(target.normals) if target.has_normal() else None,
            nn.indices.ptr, nn.distances.ptr, _hostf(t16), float(mc * mc), float(scale), C.byref(err),
            C.byref(inl)))
        return err.value, inl.value

    def compute_linearized_result(self, source, target, target_knn: KNNBase, pose,
                                  options: ExecutionOptions | None = None, initial_pose=None) -> LinearizedResult:
        """Registration::compute_linearized_result (registration.hpp:312-331); with `initial_pose` the overload
        that applies the degenerate regularisation relative to it (:312-323)."""
        target_knn.nearest_neighbor_search_async(source, self._neighbors, None, pose)
        lin = self._linearize(source, target, self._neighbors, pose, self._scale(options))
        if initial_pose is not None and self.params.degenerate_reg.type != DegenerateRegularizationType.none:
            a = self.params.addons_c()
            H = np.ascontiguousarray(lin.H, np.float32).reshape(36).copy()
            b = np.ascontiguousarray(lin.b, np.float32).reshape(6).copy()
            check(_lib.lib().spx_degenerate_regularize(C.byref(a), _hostf(H), _hostf(b), int(lin.inlier),
                                                       _hostf(_T16(pose)), _hostf(_T16(initial_pose))))
            lin.H, lin.b = H.reshape(6, 6), b
        return lin

    def compute_error_frozen(self, source, target, pose, options: ExecutionOptions | None = None):
        """Registration::compute_error_frozen (registration.hpp:350-359)."""
        return self._error(source, target, self._neighbors, pose, self._scale(options))

    def compute_icp_robust_weights(self, source, target, target_knn: KNNBase, pose, robust_scale: float) -> np.ndarray:
        """Registration::compute_icp_robust_weights (registration.hpp:279-294)."""
        n = source.size()
        if n == 0:
            return np.zeros(0, np.float32)
        target_knn.nearest_neighbor_search_async(source, self._neighbors, None, pose)
        w = DeviceArray(self.queue, (n,), np.float32)
        mc = np.float32(self.params.max_correspondence_distance)
        t16 = _T16(pose)
        self._genz()
        check(_lib.lib().spx_robust_weights(
            self.queue.handle, int(self.params.reg_type), self._loss(), source.points.ptr,
            _ptr(source.covs) if source.has_cov() else None, n, target.points.ptr,
            _ptr(target.covs) if target.has_cov() else None, _ptr(target.normals) if target.has_normal() else None,
            self._neighbors.indices.ptr, self._neighbors.distances.ptr, _hostf(t16), float(mc * mc),
            float(robust_scale), w.ptr))
        return w.download()

    def _align_injected_knn(self, source, target, knn: KNNBase, T0, options, trace) -> RegistrationResult:
        """The reference loop (registration.hpp:227-272, 803-964) with a user KNNBase: correspondences
        come from the injected object, linearise / error run on the GPU, the 6x6 step on the host."""
        P = self.params
        res = RegistrationResult(T=T0.copy())
        scale = self._scale(options)
        lam = P.lm.init_lambda
        radius = P.dogleg.initial_trust_region_radius
        conv = lambda d: (np.linalg.norm(d[:3]) < P.criteria.rotation and  # noqa: E731
                          np.linalg.norm(d[3:]) < P.criteria.translation)
        clampr = lambda r: min(max(r, P.dogleg.min_trust_region_radius), P.dogleg.max_trust_region_radius)  # noqa
        poses = []
        for it in range(P.max_iterations):
            knn.nearest_neighbor_search_async(source, self._neighbors, None, res.T)
            lin = self._linearize(source, target, self._neighbors, res.T, scale)
            res.H_raw, res.b_raw, res.error_raw = lin.H, lin.b, lin.error
            if P.optimization_method == OptimizationMethod.GAUSS_NEWTON:
                ok, d = solve_6x6(lin.H, lin.b, P.gn.lambda_)
                res.converged = bool(ok and conv(d))
                res.T = (res.T @ se3_exp(d)).astype(np.float32)
                res.iterations, res.H, res.b, res.error, res.inlier = it, lin.H, lin.b, lin.error, lin.inlier
            elif P.optimization_method == OptimizationMethod.LEVENBERG_MARQUARDT:
                last = FLT_MAX
                for _ in range(P.lm.max_inner_iterations):
                    ok, d = solve_6x6(lin.H, lin.b, lam)
                    res.converged = bool(ok and conv(d))
                    Tn = (res.T @ se3_exp(d)).astype(np.float32)
                    ne, ni = self._error(source, target, self._neighbors, Tn, scale)
                    if ne <= lin.error:
                        res.converged, res.T, res.error, res.inlier = bool(conv(d)), Tn, ne, ni
                        lam = min(max(lam / P.lm.lambda_factor, P.lm.min_lambda), P.lm.max_lambda)
                        break
                    elif abs(ne - last) <= 1e-6:
                        res.converged, res.T, res.error, res.inlier = bool(conv(d)), Tn, ne, ni
                        break
                    else:
                        lam = min(max(lam * P.lm.lambda_factor, P.lm.min_lambda), P.lm.max_lambda)
                    last = ne
                res.iterations, res.H, res.b = it, lin.H, lin.b
            else:
                res.H, res.b, res.error, res.inlier, res.iterations = lin.H, lin.b, lin.error, lin.inlier, it
                radius = clampr(radius)
                p, step_norm, pred = dogleg_step(lin.H, lin.b, radius)
                if pred <= 0.0:
                    radius = clampr(radius * P.dogleg.gamma_decrease)
                else:
                    Tn = (res.T @ se3_exp(p)).astype(np.float32)
                    ne, ni = self._error(source, target, self._neighbors, Tn, scale)
                    rho = (lin.error - ne) / pred
                    if rho < P.dogleg.eta1:
                        radius = clampr(radius * P.dogleg.gamma_decrease)
                    else:
                        res.converged, res.T, res.error, res.inlier = bool(conv(p)), Tn, ne, ni
                        if rho > P.dogleg.eta2 and step_norm >= radius * 0.99:
                            radius = clampr(radius * P.dogleg.gamma_increase)
            poses.append(res.T.copy())
            if res.converged:
                break
        if trace:
            while len(poses) < max(P.max_iterations, 1):
                poses.append(poses[-1] if poses else res.T.copy())
            res.trace = np.stack(poses)
        return res


# ------------------------------------------------------------------ pipeline wrappers
@dataclass
class RandomSamplingParams:  # registration_pipeline_params.hpp:11-16
    enable: bool = True
    num: int = 1000
    use_intensities: bool = False
    weighted_ratio: float = 0.8


@dataclass
class RobustScheduleParams:  # registration_pipeline_params.hpp:18-25
    auto_scale: bool = False
    init_scale: float = 10.0
    min_scale: float = 0.5
    rotation_init_scale: float = 10.0
    rotation_min_scale: float = 0.5
    auto_scaling_iter: int = 4


class BatchAligner:
    """spx_align_batch (include/spx.h): P RAW scan pairs -> P registration results in one call (BASELINE
    config 5).  Per cloud voxel grid -> index -> KNN k -> covariances on `lanes` concurrent internal queues, then
    one batched Registration::align.  Reference semantics per pair: voxel_downsampling.hpp:50-79,
    covariance.hpp:260-311, registration.hpp:201-276."""

    def __init__(self, queue: DeviceQueue, params: "RegistrationParams | None" = None, voxel_size: float = 0.25,
                 k_correspondences: int = 10, lanes: int = 0):
        if voxel_size <= 0.0:
            raise ValueError("voxel_size must be positive")
        self.queue = queue
        self.params = params if params is not None else RegistrationParams()
        h = C.c_void_p()
        Pc = self.params.to_c()
        check(_lib.lib().spx_batch_create(queue.handle, C.byref(Pc), float(voxel_size), int(k_correspondences), int(lanes),
                                          C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().spx_batch_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def align(self, pairs):
        """pairs: sequence of (source_raw, target_raw[, initial_guess]) with raw clouds as PointCloudShared.
        Returns (results, n_src_after_voxel, n_tgt_after_voxel)."""
        pairs = list(pairs)
        n = len(pairs)
        if n == 0:
            return [], np.zeros(0, np.uint32), np.zeros(0, np.uint32)
        Pc = self.params.to_c()
        check(_lib.lib().spx_batch_set_params(self._h, C.byref(Pc)))
        arr = (_lib.ScanPairC * n)()
        keep = []
        for j, pr in enumerate(pairs):
            src, tgt = pr[0], pr[1]
            T0 = None if len(pr) < 3 or pr[2] is None else _T16(np.asarray(pr[2], np.float32))
            keep.append(T0)
            arr[j].src_raw = _addr(src.points.ptr) if src.size() else None
            arr[j].n_src = src.size()
            arr[j].tgt_raw = _addr(tgt.points.ptr) if tgt.size() else None
            arr[j].n_tgt = tgt.size()
            arr[j].T_init_host = _hostf(T0)
        R = (RegistrationResultC * n)()
        ns, nt = np.zeros(n, np.uint32), np.zeros(n, np.uint32)
        check(_lib.lib().spx_align_batch(self._h, n, arr, R, ns.ctypes.data_as(C.c_void_p), nt.ctypes.data_as(C.c_void_p)))
        return [RegistrationResult.from_c(R[j]) for j in range(n)], ns, nt

    def last_timing(self) -> dict:
        ms, it = C.c_float(), C.c_int32()
        check(_lib.lib().spx_batch_last_timing(self._h, C.byref(ms), C.byref(it)))
        return dict(align_ms=ms.value, iterations=it.value)


@dataclass
class VelocityUpdateParams:  # registration_pipeline_params.hpp:27-30
    enable: bool = False
    iter: int = 1


@dataclass
class RegistrationPipelineParams:  # registration_pipeline_params.hpp:32-41
    registration: RegistrationParams = field(default_factory=RegistrationParams)
    random_sampling: RandomSamplingParams = field(default_factory=RandomSamplingParams)
    robust: RobustScheduleParams = field(default_factory=RobustScheduleParams)
    velocity_update: VelocityUpdateParams = field(default_factory=VelocityUpdateParams)


class VelocityUpdateAligner:
    """pipeline::VelocityUpdateAligner (pipeline/velocity_update.hpp:16-104): deskew the source with the current
    pose estimate under a constant-velocity model (options.prev_pose, options.dt), align, repeat."""

    def __init__(self, aligner, velocity_update_iter: int, verbose: bool = False):
        self._aligner = aligner.align if isinstance(aligner, Registration) else aligner
        self.velocity_update_iter = velocity_update_iter
        self.verbose = verbose
        self._deskewed = None

    def get_deskewed_point_cloud(self):
        return self._deskewed

    def align(self, source, target, target_knn, initial_guess=None, options: "ExecutionOptions | None" = None):
        options = options if options is not None else ExecutionOptions()
        T0 = np.eye(4, dtype=np.float32) if initial_guess is None else np.asarray(initial_guess, np.float32)
        result = RegistrationResult(T=T0.copy())
        if source.size() == 0:
            return result
        if not source.has_timestamps():
            self._deskewed = transform.transform_copy(source, np.eye(4, dtype=np.float32))
            return self._aligner(self._deskewed, target, target_knn, result.T, options)
        self._deskewed = PointCloudShared(source.queue)
        for _ in range(max(1, self.velocity_update_iter)):
            deskew.deskew_point_cloud_constant_velocity(source, self._deskewed, options.prev_pose, result.T, options.dt)
            result = self._aligner(self._deskewed, target, target_knn, result.T, options)
        return result


def robust_scale_schedule(init_scale: float, min_scale: float, levels: int) -> list[float]:
    """pipeline/robust.hpp:84-87,106-110: s_{l+1} = s_l * (min/init)^(1/(L-1)), in fp32 like the reference."""
    f = np.float32(1.0)
    if levels > 1:
        f = np.float32(np.power(np.float32(min_scale) / np.float32(init_scale),
                                np.float32(1.0) / np.float32(levels - 1), dtype=np.float32))
    out, s = [], np.float32(init_scale)
    for _ in range(levels):
        out.append(float(s))
        s = np.float32(s * f)
    return out


class RegistrationPipeline:
    """registration::RegistrationPipeline (registration_pipeline.hpp:17-151) with the robust-scale
    annealing wrapper (pipeline/robust.hpp:42-114).  `aligner` may be any callable with the
    RegistrationAligner signature (pipeline/aligner.hpp:13-15) — the reference's tests pass lambdas.
    Random sampling (default ON in the reference, 1000 points, registration_pipeline.hpp:127-140) draws
    from the library's persistent std::mt19937(1234) exactly as the reference does."""

    def __init__(self, queue_or_aligner, pipeline_params: RegistrationPipelineParams | None = None):
        self.pipeline_params = pipeline_params if pipeline_params is not None else RegistrationPipelineParams()
        if callable(queue_or_aligner):
            self.registration = None
            self._aligner = queue_or_aligner
        else:
            self.registration = Registration(queue_or_aligner, self.pipeline_params.registration)
            self._aligner = self.registration.align
        self._velocity = None
        vu = self.pipeline_params.velocity_update
        if vu.enable:  # registration_pipeline.hpp:99-110: robust -> velocity update -> base aligner
            self._velocity = VelocityUpdateAligner(self._aligner, vu.iter, self.pipeline_params.registration.verbose)
            self._aligner = self._velocity.align
        self._input = None
        self._filter = None

    def get_registration_input_point_cloud(self):
        return self._input

    def get_deskewed_point_cloud(self):
        return self._velocity.get_deskewed_point_cloud() if self._velocity is not None else self._input

    def align(self, source, target, target_knn, initial_guess=None, options: ExecutionOptions | None = None):
        rs = self.pipeline_params.random_sampling
        if rs.enable and source.size() > rs.num:
            if self._filter is None:
                self._filter = PreprocessFilter(source.queue)
            if rs.use_intensities and source.has_intensity():  # registration_pipeline.hpp:131-134
                source = self._filter.mixed_random_sampling(source, source.intensities, rs.num, rs.weighted_ratio,
                                                            PointCloudShared(source.queue))
            else:
                source = self._filter.random_sampling(source, rs.num, PointCloudShared(source.queue))
        self._input = source
        options = options if options is not None else ExecutionOptions()
        T0 = np.eye(4, dtype=np.float32) if initial_guess is None else np.asarray(initial_guess, np.float32)
        if not self.pipeline_params.robust.auto_scale:  # registration_pipeline.hpp:118-121
            return self._aligner(source, target, target_knn, T0, options)
        return self._robust_align(source, target, target_knn, T0, options)

    def _robust_align(self, source, target, target_knn, T0, options):
        # pipeline/robust.hpp:42-114
        pp = self.pipeline_params.robust
        reg = self.pipeline_params.registration
        result = RegistrationResult(T=T0.copy())
        if source.size() == 0:
            return result
        fixed = options.robust_scale > 0.0 or options.rotation_robust_scale > 0.0
        auto = (not fixed) and reg.robust.type != RobustLossType.NONE and pp.auto_scale
        if auto and (pp.min_scale <= 0.0 or pp.min_scale >= pp.init_scale):
            print("[Caution] `pipeline.robust.min_scale` must be greater than zero and less than "
                  "`pipeline.robust.init_scale`.")
            auto = False
        if auto and pp.auto_scaling_iter == 0:
            print("[Caution] `pipeline.robust.auto_scaling_iter` must be greater than zero. Disable auto scaling.")
            auto = False
        levels = max(1, pp.auto_scaling_iter) if auto else 1
        if options.robust_scale > 0.0:
            scales = [options.robust_scale] * levels
        elif auto:
            scales = robust_scale_schedule(pp.init_scale, pp.min_scale, levels)
        else:
            scales = [reg.robust.default_scale]
        rot = robust_scale_schedule(pp.rotation_init_scale, pp.rotation_min_scale, levels) if auto else \
            [options.rotation_robust_scale if options.rotation_robust_scale > 0 else 10.0] * levels
        for lvl in range(levels):
            o = ExecutionOptions(robust_scale=scales[lvl], rotation_robust_scale=rot[lvl], dt=options.dt,
                                 prev_pose=options.prev_pose)
            result = self._aligner(source, target, target_knn, result.T, o)
        return result
