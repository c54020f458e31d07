"""ctypes binding of libspx.so — the C-ABI declared in include/spx.h.

There is no CPU fallback: if the library is missing it is rebuilt with nvcc, and if that fails the
import raises; every call checks the returned status and raises SpxError with spx_last_error().
"""
from __future__ import annotations

import ctypes as C
import os
import re

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(HERE, "libspx.so")
HEADER = os.path.join(HERE, "..", "include", "spx.h")

SPX_SUMS_LEN = 32


class SpxError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(msg)
        self.code = code


class SpxInvalidArgument(SpxError, ValueError):
    """SPX_ERR_INVALID_ARGUMENT: std::invalid_argument / std::runtime_error in the reference."""


class RegistrationParamsC(C.Structure):
    """struct spx_registration_params (include/spx.h)."""
    _fields_ = [
        ("reg_type", C.c_int32), ("robust_loss", C.c_int32), ("optimization_method", C.c_int32),
        ("max_iterations", C.c_int32), ("max_correspondence_distance", C.c_float),
        ("robust_default_scale", C.c_float), ("criteria_translation", C.c_float), ("criteria_rotation", C.c_float),
        ("gn_lambda", C.c_float), ("lm_max_inner_iterations", C.c_int32), ("lm_lambda_factor", C.c_float),
        ("lm_init_lambda", C.c_float), ("lm_max_lambda", C.c_float), ("lm_min_lambda", C.c_float),
        ("dogleg_initial_trust_region_radius", C.c_float), ("dogleg_min_trust_region_radius", C.c_float),
        ("dogleg_max_trust_region_radius", C.c_float), ("dogleg_eta1", C.c_float), ("dogleg_eta2", C.c_float),
        ("dogleg_gamma_decrease", C.c_float), ("dogleg_gamma_increase", C.c_float), ("max_grid_blocks", C.c_int32),
        ("genz_planarity_threshold", C.c_float), ("rotation_constraint_enable", C.c_int32),
        ("rotation_constraint_weight", C.c_float), ("rotation_constraint_robust_scale", C.c_float), ("reserved", C.c_int32 * 3),
    ]


class RegistrationResultC(C.Structure):
    """struct spx_registration_result (include/spx.h)."""
    _fields_ = [
        ("T", C.c_float * 16), ("converged", C.c_int32), ("iterations", C.c_int32), ("H", C.c_float * 36),
        ("b", C.c_float * 6), ("error", C.c_float), ("H_raw", C.c_float * 36), ("b_raw", C.c_float * 6),
        ("error_raw", C.c_float), ("inlier", C.c_uint32),
    ]


class RegistrationAddonsC(C.Structure):
    """struct spx_registration_addons (include/spx.h)."""
    _fields_ = [("degenerate_type", C.c_int32), ("rot_eigenvalue_threshold", C.c_float),
                ("trans_eigenvalue_threshold", C.c_float), ("base_factor", C.c_float), ("map_prior_enabled", C.c_int32),
                ("rot_vel_sigma", C.c_float), ("trans_vel_sigma", C.c_float), ("rot_base_sigma", C.c_float),
                ("trans_base_sigma", C.c_float)]


class AlignPairC(C.Structure):
    """struct spx_align_pair (include/spx.h)."""
    _fields_ = [
        ("src_points", C.c_void_p), ("src_covs", C.c_void_p), ("ns", C.c_size_t), ("tgt_points", C.c_void_p),
        ("tgt_covs", C.c_void_p), ("tgt_normals", C.c_void_p), ("nt", C.c_size_t), ("target_index", C.c_void_p),
        ("T_init_host", C.POINTER(C.c_float)), ("robust_scale", C.c_float),
    ]


class ScanPairC(C.Structure):
    """struct spx_scan_pair (include/spx.h)."""
    _fields_ = [("src_raw", C.c_void_p), ("n_src", C.c_size_t), ("tgt_raw", C.c_void_p), ("n_tgt", C.c_size_t),
                ("T_init_host", C.POINTER(C.c_float))]


def declared_symbols() -> list[str]:
    """Every function include/spx.h declares (the exported-symbol test walks this list)."""
    with open(HEADER) as f:
        text = f.read()
    return sorted(set(re.findall(r"SPX_API\s+[\w\s\*]+?\b(spx_\w+)\s*\(", text)))


_lib = None


def _load() -> C.CDLL:
    if not os.path.exists(SO_PATH):
        from . import build as _build
        _build.build()
    if not os.path.exists(SO_PATH):
        raise ImportError(f"libspx.so not found at {SO_PATH} and could not be built (nvcc missing?) — "
                          "sycl_points_b200 has no CPU fallback")
    return C.CDLL(SO_PATH)


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    L = _load()
    vp, sz, f32p, i32p, u32p = C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p
    hostf = C.POINTER(C.c_float)
    sig = {
        "spx_last_error": (C.c_char_p, []),
        "spx_abi_version": (C.c_int, []),
        "spx_device_count": (C.c_int, [C.POINTER(C.c_int)]),
        "spx_device_info": (C.c_int, [C.c_int, C.c_char_p, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                      C.POINTER(C.c_size_t), C.POINTER(C.c_int)]),
        "spx_queue_create": (C.c_int, [C.c_int, C.POINTER(vp)]),
        "spx_queue_create_with_priority": (C.c_int, [C.c_int, C.c_int, C.POINTER(vp)]),
        "spx_queue_create_on_stream": (C.c_int, [C.c_int, vp, C.POINTER(vp)]),
        "spx_queue_destroy": (C.c_int, [vp]),
        "spx_queue_sync": (C.c_int, [vp]),
        "spx_queue_set_blocking_sync": (C.c_int, [vp, C.c_int]),
        "spx_queue_device": (C.c_int, [vp, C.POINTER(C.c_int)]),
        "spx_kernel_launch_count": (C.c_uint64, []),
        "spx_profiler_range": (C.c_int, [C.c_int]),
        "spx_malloc": (C.c_int, [vp, sz, C.POINTER(vp)]),
        "spx_free": (C.c_int, [vp, vp]),
        "spx_malloc_host": (C.c_int, [sz, C.POINTER(vp)]),
        "spx_free_host": (C.c_int, [vp]),
        "spx_memcpy_h2d": (C.c_int, [vp, vp, vp, sz]),
        "spx_memcpy_d2h": (C.c_int, [vp, vp, vp, sz]),
        "spx_memcpy_d2d": (C.c_int, [vp, vp, vp, sz]),
        "spx_memset": (C.c_int, [vp, vp, C.c_int, sz]),
        "spx_event_create": (C.c_int, [C.POINTER(vp)]),
        "spx_event_destroy": (C.c_int, [vp]),
        "spx_event_record": (C.c_int, [vp, vp]),
        "spx_queue_wait_event": (C.c_int, [vp, vp]),
        "spx_event_elapsed_ms": (C.c_int, [vp, vp, C.POINTER(C.c_float)]),
        "spx_knn_bruteforce": (C.c_int, [vp, f32p, sz, f32p, sz, C.c_int, hostf, i32p, f32p]),
        "spx_index_build": (C.c_int, [vp, f32p, sz, C.c_float, C.POINTER(vp)]),
        "spx_index_build_hinted": (C.c_int, [vp, f32p, sz, hostf, hostf, C.c_float, C.c_float, C.POINTER(vp)]),
        "spx_voxel_last_box": (C.c_int, [vp, hostf, hostf, C.POINTER(C.c_float)]),
        "spx_index_destroy": (C.c_int, [vp]),
        "spx_index_knn": (C.c_int, [vp, f32p, sz, C.c_int, hostf, i32p, f32p]),
        "spx_index_radius": (C.c_int, [vp, f32p, sz, C.c_int, C.c_float, hostf, i32p, f32p]),
        "spx_index_remove_by_flags": (C.c_int, [vp, vp, i32p, sz, sz]),
        "spx_index_info": (C.c_int, [vp, C.POINTER(C.c_float), C.POINTER(C.c_int32), C.POINTER(C.c_int64),
                                     C.POINTER(C.c_int64)]),
        "spx_index_nn_stats": (C.c_int, [vp, f32p, sz, hostf, C.c_float, u32p]),
        "spx_index_levels": (C.c_int, [vp, C.POINTER(C.c_int32)]),
        "spx_deskew_constant_velocity": (C.c_int, [vp, f32p, f32p, f32p, f32p, sz, hostf, C.c_float, f32p, f32p, f32p]),
        "spx_se3_log": (C.c_int, [hostf, hostf]),
        "spx_covariance": (C.c_int, [vp, f32p, sz, i32p, C.c_int, f32p]),
        "spx_covariance_robust": (C.c_int, [vp, f32p, sz, i32p, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, f32p]),
        "spx_normals": (C.c_int, [vp, f32p, sz, i32p, C.c_int, f32p]),
        "spx_normals_from_covs": (C.c_int, [vp, f32p, f32p, sz, f32p]),
        "spx_points_from_xyz": (C.c_int, [vp, f32p, sz, f32p]),
        "spx_eigen3": (C.c_int, [vp, f32p, sz, f32p, f32p]),
        "spx_covariance_update_plane": (C.c_int, [vp, f32p, sz]),
        "spx_transform": (C.c_int, [vp, f32p, f32p, f32p, sz, hostf]),
        "spx_voxel_downsample": (C.c_int, [vp, f32p, sz, C.c_float, sz, f32p, C.POINTER(C.c_size_t)]),
        "spx_voxel_downsample_attrs": (C.c_int, [vp, f32p, sz, C.c_float, sz, f32p, f32p, f32p, f32p, f32p, f32p, f32p,
                                                 C.POINTER(C.c_size_t)]),
        "spx_polar_downsample_attrs": (C.c_int, [vp, f32p, sz, C.c_float, C.c_float, C.c_float, C.c_int, sz, f32p, f32p, f32p,
                                                 f32p, f32p, f32p, f32p, C.POINTER(C.c_size_t)]),
        "spx_box_filter": (C.c_int, [vp, f32p, sz, C.c_float, C.c_float, f32p, C.POINTER(C.c_size_t)]),
        "spx_spd_function": (C.c_int, [vp, f32p, sz, C.c_int, C.c_float, f32p]),
        "spx_voxelmap_create": (C.c_int, [vp, C.c_float, C.POINTER(vp)]),
        "spx_voxelmap_destroy": (C.c_int, [vp]),
        "spx_voxelmap_set_params": (C.c_int, [vp, C.c_float, C.c_uint32, C.c_uint32, C.c_float, C.c_uint32]),
        "spx_voxelmap_clear": (C.c_int, [vp]),
        "spx_voxelmap_add": (C.c_int, [vp, f32p, f32p, f32p, f32p, sz, hostf]),
        "spx_voxelmap_remove_old": (C.c_int, [vp]),
        "spx_voxelmap_info": (C.c_int, [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint32),
                                        C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
        "spx_voxelmap_downsample": (C.c_int, [vp, hostf, C.c_float, f32p, f32p, f32p, f32p, vp, sz,
                                              C.POINTER(C.c_size_t)]),
        "spx_voxelmap_overlap_ratio": (C.c_int, [vp, f32p, sz, hostf, C.POINTER(C.c_float)]),
        "spx_box_filter_indices": (C.c_int, [vp, f32p, sz, C.c_float, C.c_float, i32p, C.POINTER(C.c_size_t)]),
        "spx_linearize": (C.c_int, [vp, C.c_int, C.c_int, f32p, f32p, sz, f32p, f32p, f32p, i32p, f32p, hostf,
                                    C.c_float, C.c_float, hostf, hostf, C.POINTER(C.c_float),
                                    C.POINTER(C.c_uint32)]),
        "spx_error": (C.c_int, [vp, C.c_int, C.c_int, f32p, f32p, sz, f32p, f32p, f32p, i32p, f32p, hostf, C.c_float,
                                C.c_float, C.POINTER(C.c_float), C.POINTER(C.c_uint32)]),
        "spx_robust_weights": (C.c_int, [vp, C.c_int, C.c_int, f32p, f32p, sz, f32p, f32p, f32p, i32p, f32p, hostf,
                                         C.c_float, C.c_float, f32p]),
        "spx_default_registration_params": (None, [C.POINTER(RegistrationParamsC)]),
        "spx_set_genz_planarity_threshold": (C.c_int, [C.c_float]),
        "spx_set_rotation_constraint": (C.c_int, [C.c_int, C.c_float, C.c_float]),
        "spx_solve_6x6": (C.c_int, [hostf, hostf, C.c_float, hostf, C.POINTER(C.c_int)]),
        "spx_se3_exp": (C.c_int, [hostf, hostf]),
        "spx_dogleg_step": (C.c_int, [hostf, hostf, C.c_float, hostf, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
        "spx_registration_create": (C.c_int, [vp, C.POINTER(RegistrationParamsC), C.POINTER(vp)]),
        "spx_registration_destroy": (C.c_int, [vp]),
        "spx_registration_set_params": (C.c_int, [vp, C.POINTER(RegistrationParamsC)]),
        "spx_default_registration_addons": (None, [C.POINTER(RegistrationAddonsC)]),
        "spx_registration_set_addons": (C.c_int, [vp, C.POINTER(RegistrationAddonsC)]),
        "spx_registration_set_map_prior_state": (C.c_int, [vp, C.POINTER(RegistrationResultC), hostf, C.POINTER(C.c_int),
                                                           hostf]),
        "spx_degenerate_regularize": (C.c_int, [C.POINTER(RegistrationAddonsC), hostf, hostf, C.c_uint32, hostf, hostf]),
        "spx_registration_align": (C.c_int, [vp, f32p, f32p, sz, f32p, f32p, f32p, sz, vp, hostf, C.c_float,
                                             C.POINTER(RegistrationResultC), hostf]),
        "spx_registration_align_batch": (C.c_int, [vp, sz, C.POINTER(AlignPairC), C.POINTER(RegistrationResultC)]),
        "spx_batch_create": (C.c_int, [vp, C.POINTER(RegistrationParamsC), C.c_float, C.c_int, C.c_int, C.POINTER(vp)]),
        "spx_batch_destroy": (C.c_int, [vp]),
        "spx_batch_set_params": (C.c_int, [vp, C.POINTER(RegistrationParamsC)]),
        "spx_align_batch": (C.c_int, [vp, sz, C.POINTER(ScanPairC), C.POINTER(RegistrationResultC), u32p, u32p]),
        "spx_batch_last_timing": (C.c_int, [vp, C.POINTER(C.c_float), C.POINTER(C.c_int32)]),
        "spx_registration_kept_correspondences": (C.c_int, [vp, C.POINTER(C.c_uint64)]),
        "spx_registration_last_timing": (C.c_int, [vp, C.POINTER(C.c_float), C.POINTER(C.c_int32),
                                                   C.POINTER(C.c_int32)]),
        "spx_registration_phase_times": (C.c_int, [vp, C.c_int, vp, C.c_int]),
        "spx_registration_neighbors": (C.c_int, [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(C.c_size_t)]),
        "spx_registration_shard_begin": (C.c_int, [vp, f32p, f32p, sz, f32p, f32p, f32p, sz, vp, hostf, C.c_float]),
        "spx_registration_shard_linearize": (C.c_int, [vp, vp]),
        "spx_registration_shard_update": (C.c_int, [vp, vp]),
        "spx_registration_shard_finish": (C.c_int, [vp, C.POINTER(RegistrationResultC)]),
        "spx_malloc_managed": (C.c_int, [sz, C.POINTER(vp)]),
        "spx_free_managed": (C.c_int, [vp]),
        "spx_managed_trim": (C.c_int, []),
        "spx_prefetch": (C.c_int, [vp, vp, sz, C.c_int]),
        "spx_rng_create": (C.c_int, [C.c_uint32, C.POINTER(vp)]),
        "spx_rng_seed": (C.c_int, [vp, C.c_uint32]),
        "spx_rng_destroy": (C.c_int, [vp]),
        "spx_random_sampling": (C.c_int, [vp, vp, sz, sz, i32p, C.POINTER(C.c_size_t)]),
        "spx_gather": (C.c_int, [vp, vp, sz, i32p, sz, vp]),
        "spx_weighted_random_sampling": (C.c_int, [vp, vp, f32p, sz, sz, i32p, C.POINTER(C.c_size_t)]),
        "spx_rng_uniform_index": (C.c_int, [vp, sz, C.POINTER(C.c_size_t)]),
        "spx_farthest_point_sampling": (C.c_int, [vp, f32p, sz, sz, sz, i32p, C.POINTER(C.c_size_t)]),
        "spx_mixed_random_sampling": (C.c_int, [vp, vp, f32p, sz, sz, C.c_float, i32p, C.POINTER(C.c_size_t)]),
        "spx_angle_incidence_indices": (C.c_int, [vp, f32p, f32p, f32p, sz, C.c_float, C.c_float, i32p,
                                                  C.POINTER(C.c_size_t)]),
        "spx_statistical_outlier_indices": (C.c_int, [vp, f32p, sz, C.c_int, C.c_float, f32p, i32p, C.POINTER(C.c_size_t)]),
        "spx_radius_outlier_indices": (C.c_int, [vp, f32p, sz, C.c_float, C.c_uint32, i32p, C.POINTER(C.c_size_t)]),
        "spx_euclidean_clusters": (C.c_int, [vp, f32p, sz, C.c_float, C.c_uint32, C.c_uint32, i32p, i32p, u32p,
                                             C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
        "spx_plane_segment": (C.c_int, [vp, f32p, sz, C.c_float, C.c_uint32, C.c_uint64, f32p, C.c_double, C.c_int, f32p,
                                        i32p, i32p, C.POINTER(C.c_size_t), i32p, u32p]),
        "spx_fpfh": (C.c_int, [vp, f32p, f32p, sz, i32p, f32p, C.c_int, f32p]),
        "spx_feature_correspondences": (C.c_int, [vp, f32p, sz, f32p, sz, C.c_int, i32p, i32p, C.POINTER(C.c_size_t)]),
        "spx_ransac_registration": (C.c_int, [vp, f32p, sz, f32p, sz, i32p, i32p, sz, C.c_float, C.c_uint32, C.c_uint64,
                                              C.c_float, C.c_int, f32p, C.POINTER(C.c_int32), i32p,
                                              C.POINTER(C.c_size_t), u32p]),
        "spx_comm_create": (C.c_int, [vp, C.c_int, C.c_int, C.POINTER(vp)]),
        "spx_comm_destroy": (C.c_int, [vp]),
        "spx_comm_ipc_handle": (C.c_int, [vp, C.c_char_p]),
        "spx_comm_connect_ipc": (C.c_int, [vp, C.c_char_p]),
        "spx_comm_connect_local": (C.c_int, [C.POINTER(vp), C.c_int]),
        "spx_registration_align_sharded_launch": (C.c_int, [vp, vp, f32p, f32p, sz, f32p, f32p, f32p, sz, vp, hostf,
                                                            C.c_float]),
        "spx_registration_align_sharded_finish": (C.c_int, [vp, C.POINTER(RegistrationResultC)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)  # AttributeError here = header/library mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    if L.spx_abi_version() != 1:
        raise ImportError("libspx.so ABI version mismatch; rebuild with python -m sycl_points_b200.build --force")
    _lib = L
    return L


def check(rc: int) -> None:
    if rc == 0:
        return
    msg = lib().spx_last_error().decode("utf-8", "replace")
    if rc == -1:
        raise SpxInvalidArgument(rc, msg)
    raise SpxError(rc, msg)
