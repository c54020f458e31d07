"""sycl_points_b200 — B200 (sm_100a) implementation of the per-iteration registration hot path of
fateshelled/sycl_points behind the C-ABI in include/spx.h.  See DESIGN.md.

The package contains only what that path needs: csrc/ (hand-written CUDA kernels + the C-ABI),
_lib.py (ctypes binding), api.py (host-side mirror of the reference interface).  There is no CPU
fallback; importing works without a GPU (the library loads), computing does not."""
from ._lib import SpxError, SpxInvalidArgument, declared_symbols, lib  # noqa: F401
from .api import *  # noqa: F401,F403
from .api import (BatchAligner, DeviceArray, DeviceQueue, EuclideanClustering, EuclideanClusters,  # noqa: F401
                  Event, ExecutionOptions, FPFHEstimation, KDTree, KNNBase, KNNResult, LinearizedResult, OptimizationMethod,
                  OutlierRemoval, PinnedArray, PlaneModel, PlaneSegmentation, PointCloudShared, PreprocessFilter,
                  RANSACRegistration, RANSACResult, RegType, Registration, RegistrationParams, RegistrationPipeline, RegistrationPipelineParams,
                  RegistrationResult, RobustLossType, VoxelGrid, covariance, device_count, kernel_launch_count,
                  knn_search_bruteforce, match_features, robust_scale_schedule, transform)
