/*
 * spx.h — C-ABI of libspx.so, the B200 (sm_100a) implementation of the per-iteration
 * registration hot path of fateshelled/sycl_points.
 *
 * The reference is a header-only C++20/SYCL library with no FFI of its own (SURVEY.md §8(b));
 * this ABI replaces its SYCL queue / USM layer (I/utils/sycl_utils.hpp) and the kernels behind
 * its public C++ entry points.  Each function cites the reference interface it stands in for:
 *     I/ = cpp/include/sycl_points/     (paths inside fateshelled/sycl_points)
 *
 * Conventions
 *  - every function returns 0 (SPX_OK) or a negative spx_status; spx_last_error() gives the
 *    thread-local message.  CUDA errors are surfaced, never swallowed.
 *  - all array arguments are DEVICE pointers obtained from spx_malloc (or any CUDA device
 *    pointer on the queue's device) unless the name ends in _host.
 *  - points / normals: float[n][4] (xyz1 / xyz0, I/points/types.hpp:11-13)
 *    covariances:      float[n][16], column-major 4x4 with zero 4th row/col (types.hpp:12)
 *    transforms:       float[16] HOST memory, column-major (Eigen::Matrix4f::data() order)
 *    KNN result:       int32 idx[nq][k], float dist[nq][k] squared distances, ascending by
 *                      (dist, idx); unfilled = -1 / FLT_MAX (I/algorithms/knn/result.hpp:12-34)
 *  - work is enqueued on the queue's CUDA stream; functions that return values to the host
 *    synchronise that stream, the others are asynchronous (call spx_queue_sync).
 *  - a queue and the handles created from it are single-threaded, like the reference's
 *    Registration / VoxelGrid / KDTree instances; distinct queues may run concurrently.
 */
#ifndef SPX_H_
#define SPX_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPX_ABI_VERSION 1

#if defined(__GNUC__)
#define SPX_API __attribute__((visibility("default")))
#else
#define SPX_API
#endif

typedef enum spx_status {
    SPX_OK = 0,
    SPX_ERR_INVALID_ARGUMENT = -1, /* std::invalid_argument / std::runtime_error in the reference */
    SPX_ERR_CUDA = -2,
    SPX_ERR_UNSUPPORTED = -3,
    SPX_ERR_INTERNAL = -4
} spx_status;

/* I/algorithms/registration/factor.hpp:18-32 (same numeric values) */
typedef enum spx_reg_type {
    SPX_REG_POINT_TO_POINT = 0,
    SPX_REG_POINT_TO_PLANE = 1,
    SPX_REG_POINT_TO_DISTRIBUTION = 2,
    SPX_REG_GICP = 3,
    SPX_REG_GENZ = 4 /* factor.hpp:378-449: plane factor x alpha / point factor x (1 - alpha), alpha recounted per linearisation */
} spx_reg_type;

/* I/algorithms/robust/robust.hpp:14-20 */
typedef enum spx_robust_loss {
    SPX_LOSS_NONE = 0,
    SPX_LOSS_HUBER = 1,
    SPX_LOSS_TUKEY = 2,
    SPX_LOSS_CAUCHY = 3,
    SPX_LOSS_GEMAN_MCCLURE = 4
} spx_robust_loss;

/* I/algorithms/registration/registration_params.hpp:17-21 */
typedef enum spx_optimization_method {
    SPX_OPT_GAUSS_NEWTON = 0,
    SPX_OPT_LEVENBERG_MARQUARDT = 1,
    SPX_OPT_POWELL_DOGLEG = 2
} spx_optimization_method;

typedef struct spx_queue_s* spx_queue_t;               /* sycl_utils::DeviceQueue, sycl_utils.hpp:491-626 */
typedef struct spx_event_s* spx_event_t;               /* sycl_utils::events,      sycl_utils.hpp:234-280 */
typedef struct spx_index_s* spx_index_t;               /* knn::KDTree (as a KNNBase), kdtree.hpp:142-280 */
typedef struct spx_registration_s* spx_registration_t; /* registration::Registration, registration.hpp:88-965 */

/* RegistrationParams, I/algorithms/registration/registration_params.hpp:41-114 (defaults there). */
typedef struct spx_registration_params {
    int32_t reg_type;           /* spx_reg_type, default GICP */
    int32_t robust_loss;        /* spx_robust_loss, default NONE */
    int32_t optimization_method;/* spx_optimization_method, default GN */
    int32_t max_iterations;     /* 20 */
    float max_correspondence_distance; /* 2.0 */
    float robust_default_scale; /* 10.0 */
    float criteria_translation; /* 1e-3 m */
    float criteria_rotation;    /* 1e-3 rad */
    float gn_lambda;            /* 1.0 */
    int32_t lm_max_inner_iterations; /* 10 */
    float lm_lambda_factor;     /* 2 */
    float lm_init_lambda;       /* 1 */
    float lm_max_lambda;        /* 1e3 */
    float lm_min_lambda;        /* 1e-6 */
    float dogleg_initial_trust_region_radius; /* 1 */
    float dogleg_min_trust_region_radius;     /* 1e-4 */
    float dogleg_max_trust_region_radius;     /* 10 */
    float dogleg_eta1;          /* .25 */
    float dogleg_eta2;          /* .75 */
    float dogleg_gamma_decrease;/* .25 */
    float dogleg_gamma_increase;/* 2 */
    int32_t max_grid_blocks;    /* cap on the align kernel's persistent grid (blocks, 0 = auto: one full wave) */
    float genz_planarity_threshold; /* RegistrationParams::genz.planarity_threshold, 0.2 (registration_params.hpp:51-53) */
    int32_t rotation_constraint_enable;       /* RegistrationParams::rotation_constraint (registration_params.hpp:54-62), off */
    float rotation_constraint_weight;         /* 1 */
    float rotation_constraint_robust_scale;   /* 10; a positive ExecutionOptions::rotation_robust_scale goes here (registration.hpp:219-221) */
    int32_t reserved[3];        /* must be zero */
} spx_registration_params;

/* RegistrationResult, I/algorithms/registration/result.hpp:13-28.  `iterations` keeps the
 * reference's meaning: the 0-based index of the last iteration run (registration.hpp:815). */
typedef struct spx_registration_result {
    float T[16];       /* column-major */
    int32_t converged;
    int32_t iterations;
    float H[36];
    float b[6];
    float error;
    float H_raw[36];
    float b_raw[6];
    float error_raw;
    uint32_t inlier;
} spx_registration_result;

/* Solver add-ons of Registration (both default-off; host-side 6x6 arithmetic between the device linearisation and the
 * step, exactly where the reference applies them: registration.hpp:248-253):
 *   DegenerateRegularizationParams (degenerate_regularization.hpp:35-40): nl-reg — for every eigen-direction of the
 *     rotation / translation 3x3 block of H whose eigenvalue / inlier is below its threshold, H += lambda v v^T and
 *     b += lambda v v^T Log(T_initial^-1 T), lambda = base_factor * inlier (:58-112);
 *   MapPriorParams (map_prior.hpp:15-21): a Gaussian prior around the predicted pose whose information is the previous
 *     frame's calibrated Hessian inflated by velocity-proportional process noise (:30-117); adds Omega to H,
 *     Omega Log(T_pred^-1 T) to b and 1/2 e^T Omega e to the error (:119-139). */
typedef struct spx_registration_addons {
    int32_t degenerate_type;          /* 0 none, 1 nl_reg */
    float rot_eigenvalue_threshold;   /* 10 */
    float trans_eigenvalue_threshold; /* 1 */
    float base_factor;                /* 1 */
    int32_t map_prior_enabled;        /* 0 */
    float rot_vel_sigma;              /* 1 */
    float trans_vel_sigma;            /* 1 */
    float rot_base_sigma;             /* 3.16e-2 */
    float trans_base_sigma;           /* 1e-2 */
} spx_registration_addons;

/* ------------------------------------------------------------------ runtime (replaces sycl_utils.hpp) */
SPX_API const char* spx_last_error(void);
SPX_API int spx_abi_version(void);
SPX_API int spx_device_count(int* count);
/* name: >= 256 bytes; sm = major*10+minor (100 on B200) */
SPX_API int spx_device_info(int device, char* name, int* sm, int* sm_count, size_t* global_mem_bytes, int* l2_bytes);

/* DeviceQueue(device) — sycl_utils.hpp:491-529.  Owns one in-order CUDA stream + scratch arena. */
SPX_API int spx_queue_create(int device, spx_queue_t* out);
/* The same with a scheduling hint (sycl::ext::oneapi::property::queue::priority_high / _low in the reference's
 * runtime): priority > 0 = the device's most urgent stream priority, < 0 = the least urgent, 0 = default.  When
 * two queues have work pending, the blocks of the more urgent one are placed first. */
SPX_API int spx_queue_create_with_priority(int device, int priority, spx_queue_t* out);
/* Same, on a caller-owned cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream). */
SPX_API int spx_queue_create_on_stream(int device, void* cuda_stream, spx_queue_t* out);
SPX_API int spx_queue_destroy(spx_queue_t q);
SPX_API int spx_queue_sync(spx_queue_t q); /* events.wait_and_throw(), sycl_utils.hpp:262-270 */
SPX_API int spx_queue_device(spx_queue_t q, int* device);
/* how spx_queue_sync (and every call that returns values to the host) waits: 0 = spin (lowest
 * latency, default), 1 = block on an OS primitive (frees the core: many queues / ranks per host) */
SPX_API int spx_queue_set_blocking_sync(spx_queue_t q, int blocking);
/* Kernels launched by this library since load (all queues): bench.py's `gpu_launches`. */
SPX_API uint64_t spx_kernel_launch_count(void);

/* tuning aid: cudaProfilerStart / cudaProfilerStop (ncu --profile-from-start off captures only the range) */
SPX_API int spx_profiler_range(int start);

/* shared_vector<T> storage — sycl_utils.hpp:630-635 (USM shared -> explicit device memory) */
SPX_API int spx_malloc(spx_queue_t q, size_t bytes, void** out);
SPX_API int spx_free(spx_queue_t q, void* ptr);
SPX_API int spx_malloc_host(size_t bytes, void** out); /* pinned */
SPX_API int spx_free_host(void* ptr);
SPX_API int spx_memcpy_h2d(spx_queue_t q, void* dst, const void* src_host, size_t bytes); /* async on the stream */
SPX_API int spx_memcpy_d2h(spx_queue_t q, void* dst_host, const void* src, size_t bytes); /* async on the stream */
SPX_API int spx_memcpy_d2d(spx_queue_t q, void* dst, const void* src, size_t bytes);
SPX_API int spx_memset(spx_queue_t q, void* dst, int value, size_t bytes);

/* USM *shared* semantics for the C++ facade's shared_vector<T> (host-dereferenceable, device-usable):
 * CUDA managed memory + explicit prefetch (the reference's mem_advise hints, sycl_utils.hpp:283-364). */
SPX_API int spx_malloc_managed(size_t bytes, void** out);
SPX_API int spx_free_managed(void* ptr); /* returns the block to a size-class cache (no device sync) */
SPX_API int spx_managed_trim(void);      /* releases every cached idle block */
SPX_API int spx_prefetch(spx_queue_t q, const void* ptr, size_t bytes, int to_device); /* to_device 0 = to host */

SPX_API int spx_event_create(spx_event_t* out);
SPX_API int spx_event_destroy(spx_event_t e);
SPX_API int spx_event_record(spx_queue_t q, spx_event_t e);
SPX_API int spx_event_elapsed_ms(spx_event_t start, spx_event_t stop, float* ms); /* synchronises on stop */
/* work enqueued on q after this call starts only once e has completed (handler::depends_on across queues) */
SPX_API int spx_queue_wait_event(spx_queue_t q, spx_event_t e);

/* ------------------------------------------------------------------ KNN
 * knn_search_bruteforce(queue, queries, targets, k) — I/algorithms/knn/bruteforce.hpp:24-96.
 * Tile scan of all targets; dist = fma(dz,dz,fma(dy,dy,dx*dx)); result ordered by (dist, idx).
 * T_host (nullable, 16 floats): transform applied to each query first — the reference's
 * brute force takes none (pass NULL); KNNBase::knn_search_async does (knn.hpp:22-24).
 * 1 <= k <= 128. */
SPX_API int spx_knn_bruteforce(spx_queue_t q, const float* queries, size_t nq, const float* targets, size_t nt, int k,
                       const float* T_host, int32_t* idx, float* dist);

/* KDTree::build(queue, cloud, leaf) — kdtree.hpp:165-180,292-413.  Builds a GPU-resident exact
 * index (uniform cell grid, counting-sorted on device) over `targets`; cell_size <= 0 picks one
 * from the point density.  The index keeps its own sorted copy; `targets` may be freed after. */
SPX_API int spx_index_build(spx_queue_t q, const float* targets, size_t nt, float cell_size, spx_index_t* out);
/* The same index from a caller that already knows a box containing the points and the cell edges it wants — e.g. a
 * cloud that just came out of the voxel grid (spx_voxel_last_box; ~1.85 x voxel_size holds ~3 points per occupied
 * cell on LiDAR surfaces, ~2.4 x voxel_size ~5 for the k >= 2 first-pass grid).  Skips the build's bounding-box /
 * occupancy pass and its host round trip: fully asynchronous.  A box that misses points costs speed, never exactness
 * (cell coordinates clamp into the grid).  knn_cell_size <= cell_size: no extra k-NN grid. */
SPX_API int spx_index_build_hinted(spx_queue_t q, const float* targets, size_t nt, const float* lo3_host, const float* hi3_host,
                           float cell_size, float knn_cell_size, spx_index_t* out);
SPX_API int spx_index_destroy(spx_index_t index);
/* KNNBase::knn_search_async(queries, k, result, depends, transT) — knn.hpp:22-24,
 * kdtree.hpp:203-224,424-562.  Exact: identical to spx_knn_bruteforce on the same inputs
 * (ring search with a proven stop bound over a hierarchy of grids, DESIGN.md §index).
 * 1 <= k <= 128 (the reference throws above 100, kdtree.hpp:221-223).  Asynchronous. */
SPX_API int spx_index_knn(spx_index_t index, const float* queries, size_t nq, int k, const float* T_host, int32_t* idx,
                  float* dist);
/* KDTree::radius_search_async(queries, max_k, radius, result, depends, transT) — kdtree.hpp:226-280,564-720: the
 * max_k nearest targets within `radius` (dist^2 <= radius^2), ascending by (dist, idx), the rest -1 / FLT_MAX. */
SPX_API int spx_index_radius(spx_index_t index, const float* queries, size_t nq, int max_k, float radius, const float* T_host,
                     int32_t* idx, float* dist);
/* KDTree::remove_nodes_by_flags(flags, indices) — kdtree.hpp:282-284,721-760: points whose flag is not INCLUDE (1) leave
 * the index, the others are re-numbered new_index[old] (device arrays of n entries; n_kept = number of kept points =
 * 1 + the largest new index).  The grid is rebuilt over the kept points; searches then report the new numbers. */
SPX_API int spx_index_remove_by_flags(spx_index_t index, const uint8_t* flags, const int32_t* new_index, size_t n, size_t n_kept);
/* introspection for tests / DESIGN.md: cell size, grid dims[3], occupied cells, points */
SPX_API int spx_index_info(spx_index_t index, float* cell_size, int32_t* dims3, int64_t* occupied_cells, int64_t* n_points);
/* tuning aid: per-query work counters of the k = 1 search, stats4[q] = {segments, candidate points,
 * shells, last level}; max_radius <= 0 = unbounded */
SPX_API int spx_index_nn_stats(spx_index_t index, const float* queries, size_t nq, const float* T_host, float max_radius,
                       uint32_t* stats4);
/* number of grid levels (each 8x coarser than the previous) the index keeps */
SPX_API int spx_index_levels(spx_index_t index, int32_t* n_levels);

/* ------------------------------------------------------------------ features
 * covariance::estimate_async(queue, neighbors, points, covs) — I/algorithms/feature/covariance.hpp:16-47,260-292 */
SPX_API int spx_covariance(spx_queue_t q, const float* points, size_t n, const int32_t* knn_idx, int k, float* covs);
/* covariance::estimate_robust_async(queue, neighbors, points, covs, robust_type, mad_scale, min_robust_scale,
 * robust_max_iterations) — covariance.hpp:97-134,143-250,323-373: M-estimated covariances (weights from the squared
 * Mahalanobis distances at scale mad_scale x median, floored at min_robust_scale).  robust_loss NONE = the plain
 * estimate; k <= 64 (the reference's MAX_K).  Reference defaults: CAUCHY, 1.0, 1.0, 1 iteration. */
SPX_API int spx_covariance_robust(spx_queue_t q, const float* points, size_t n, const int32_t* knn_idx, int k, int robust_loss,
                          float mad_scale, float min_robust_scale, int robust_max_iterations, float* covs);
/* covariance::estimate_normals_async(neighbors, points) — covariance.hpp:49-65,417-445 */
SPX_API int spx_normals(spx_queue_t q, const float* points, size_t n, const int32_t* knn_idx, int k, float* normals);
/* covariance::extract_normals_async(points) — covariance.hpp:467-495 */
SPX_API int spx_normals_from_covs(spx_queue_t q, const float* points, const float* covs, size_t n, float* normals);

/* PointCloudShared(queue, PointCloudCPU) — I/points/point_cloud.hpp:110-198 copies Vector4f points (xyz1, 16 B) to the
 * device.  A LiDAR driver delivers packed xyz: this expands float[n][3] (device) to float[n][4] with w = 1 on the
 * device, so that the host-to-device copy of a raw scan carries 12 instead of 16 bytes per point.  Asynchronous. */
SPX_API int spx_points_from_xyz(spx_queue_t q, const float* xyz, size_t n, float* points);

/* eigen_utils::symmetric_eigen_decomposition_3x3 — I/utils/eigen_utils.hpp:443-562 — applied to the
 * upper-left 3x3 of n stored covariances (which must be symmetric, as covariance::estimate writes
 * them: the upper triangle is read).  evals[n][3] ascending; evecs[n][9] row-major 3x3 whose column
 * k is eigenvector k.  cos / acos / cbrt are correctly rounded (DESIGN.md §4).  Asynchronous. */
SPX_API int spx_eigen3(spx_queue_t q, const float* covs, size_t n, float* evals, float* evecs);
/* covariance::kernel::update_covariance_plane — covariance.hpp:67-74 — C <- V diag(1e-3, 1, 1) V^T,
 * in place on n covariances: the per-point GICP regularisation (factor.hpp:250-255) that
 * spx_registration_align applies once per cloud per align.  Asynchronous. */
SPX_API int spx_covariance_update_plane(spx_queue_t q, float* covs, size_t n);

/* transform::transform_async(cloud, trans) — I/algorithms/common/transform.hpp:45-104: in place,
 * points T p, covariances T C T^T (nullable), normals T n (nullable; not re-normalised, as the
 * reference's kernel).  Asynchronous. */
SPX_API int spx_transform(spx_queue_t q, float* points, float* covs, float* normals, size_t n, const float* T_host);

/* deskew::deskew_point_cloud_constant_velocity (algorithms/deskew/relative_pose_deskew.hpp:36-178): every point is
 * moved by se3_exp(tau * twist), tau = clamp(timestamp_offset_ms * 1e-3 / scan_duration_s, 0, 1); normals and
 * covariances (both nullable, in and out together) are rotated by the rotation of that motion.  twist6_host =
 * se3_log(previous_pose^-1 * current_pose) as [rx ry rz tx ty tz] (spx_se3_log).  Outputs may alias the inputs. */
SPX_API int spx_deskew_constant_velocity(spx_queue_t q, const float* points, const float* normals, const float* covs,
                                         const float* timestamp_offsets_ms, size_t n, const float* twist6_host,
                                         float scan_duration_s, float* points_out, float* normals_out, float* covs_out);
/* eigen_utils::lie::se3_log (utils/eigen_utils.hpp:991-1034; spx_se3_exp below is its inverse): host arithmetic,
 * column-major 4x4 -> [rx ry rz tx ty tz].  No device work, no queue. */
SPX_API int spx_se3_log(const float* T_host, float* twist6_host);


/* ------------------------------------------------------------------ filters
 * filter::VoxelGrid::downsampling(points, result) — I/algorithms/filter/voxel_downsampling.hpp:50-62,
 * key = I/algorithms/common/voxel_constants.hpp:36-62.  Device radix sort by (key, index), fp32
 * running sum per voxel in that order, mean = sum / sum.w, voxels with sum.w < min_voxel_count
 * dropped, output ascending key.  out_points must hold n points; *m_host receives the count
 * (synchronises).  voxel_size <= 0 -> SPX_ERR_INVALID_ARGUMENT (voxel_downsampling.hpp:23-25). */
SPX_API int spx_voxel_downsample(spx_queue_t q, const float* points, size_t n, float voxel_size, size_t min_voxel_count,
                         float* out_points, size_t* m_host);
/* Metric box [lo, hi] that contains every point the LAST spx_voxel_downsample* call on this queue produced (from the
 * voxel coordinates' bounding box the sort already needed; one voxel of slack): the hint of spx_index_build_hinted. */
SPX_API int spx_voxel_last_box(spx_queue_t q, float* lo3_host, float* hi3_host, float* voxel_size);
/* filter::VoxelGrid::downsampling(cloud, result) — voxel_downsampling.hpp:64-79,220-288: the cloud
 * overload also aggregates per-point attributes over each voxel in the same order: mean RGBA
 * (float[n][4]), MEDIAN intensity (float[n], :82-98), mean timestamp offset (float[n]).  Any
 * attribute input may be NULL (then its output is ignored). */
SPX_API int spx_voxel_downsample_attrs(spx_queue_t q, const float* points, size_t n, float voxel_size,
                               size_t min_voxel_count, const float* rgb, const float* intensity,
                               const float* timestamps, float* out_points, float* out_rgb, float* out_intensity,
                               float* out_timestamps, size_t* m_host);

/* filter::PolarGrid::downsampling (algorithms/filter/polar_downsampling.hpp:30-108 key, :341-452 aggregation): the
 * same sort-and-aggregate pass as the voxel grid with cells in (range, elevation, azimuth) — key = range cell
 * (lowest digits), elevation cell, azimuth cell (highest); points at the origin or on the polar axis are dropped.
 * Output in ascending key order; attributes as spx_voxel_downsample_attrs. */
#define SPX_COORD_LIDAR 0  /* x forward, y left, z up    (common/coordinate_system.hpp) */
#define SPX_COORD_CAMERA 1 /* x right, y down, z forward */
SPX_API int spx_polar_downsample_attrs(spx_queue_t q, const float* points, size_t n, float distance_voxel_size,
                                       float elevation_voxel_size, float azimuth_voxel_size, int coordinate_system,
                                       size_t min_voxel_count, const float* rgb, const float* intensity,
                                       const float* timestamps, float* out_points, float* out_rgb, float* out_intensity,
                                       float* out_timestamps, size_t* m_host);
/* PreprocessFilter::box_filter(cloud, min, max) — preprocess_operator/box_filter_operator.hpp:19-54,
 * common.hpp:15-25, common/filter_by_flags.hpp:43-49 (order-preserving).  Synchronises. */
SPX_API int spx_box_filter(spx_queue_t q, const float* points, size_t n, float min_distance, float max_distance,
                   float* out_points, size_t* m_host);

/* The same filter returning the KEPT INDICES (ascending, device int32[<= n]) instead of the points: what
 * common/filter_by_flags.hpp:29-57 applies to every attribute the cloud carries (covariances, normals, rgb,
 * intensities, timestamp offsets) — run each through spx_gather.  Synchronises. */
SPX_API int spx_box_filter_indices(spx_queue_t q, const float* points, size_t n, float min_distance, float max_distance,
                           int32_t* idx_out, size_t* m_host);

/* PreprocessFilter::random_sampling(source, output, n) — preprocess_operator/random_sampling_operator.hpp:15-58:
 * partial Fisher-Yates over 0..n-1 with a persistent std::mt19937 (seed 1234) and
 * std::uniform_int_distribution<size_t>(i, n-1) (libstdc++), then ORDER-PRESERVING compaction.
 * spx_random_sampling writes the m = min(n, sampling_num) selected indices in ascending order to
 * idx_out (device, int32[m]); spx_gather applies them to any per-point attribute (elem_bytes a
 * multiple of 4: 16 = points/normals, 64 = covariances, 4 = intensities). */
typedef struct spx_rng_s* spx_rng_t;
SPX_API int spx_rng_create(uint32_t seed, spx_rng_t* out);
SPX_API int spx_rng_seed(spx_rng_t rng, uint32_t seed);
SPX_API int spx_rng_destroy(spx_rng_t rng);
SPX_API int spx_random_sampling(spx_queue_t q, spx_rng_t rng, size_t n, size_t sampling_num, int32_t* idx_out, size_t* m_host);
SPX_API int spx_gather(spx_queue_t q, const void* src, size_t elem_bytes, const int32_t* idx, size_t m, void* dst);
/* PreprocessFilter::mixed_random_sampling(source, output, weights, n, weighted_ratio) —
 * preprocess_operator/mixed_random_sampling_operator.hpp:29-107: floor(n * ratio) points by weighted reservoir keys
 * log(u) / w (the robust ICP weights of registration.hpp:412-462), the rest uniformly from the remainder; same
 * persistent mt19937 stream and libstdc++ distributions as the reference.  weights: device float[n].  Kept indices
 * ascending in idx_out (device int32[min(n, sampling_num)]); apply them with spx_gather.  Synchronises. */
SPX_API int spx_mixed_random_sampling(spx_queue_t q, spx_rng_t rng, const float* weights, size_t n, size_t sampling_num,
                                      float weighted_ratio, int32_t* idx_out, size_t* m_host);
/* PreprocessFilter::weighted_random_sampling(source, output, weights, n) —
 * preprocess_operator/weighted_sampling_operator.hpp:29-96: n points by weighted reservoir keys over the points of
 * positive weight; SPX_ERR_INVALID_ARGUMENT for negative / non-finite weights, no positive weight, or n larger than
 * the number of positive weights.  Kept indices ascending.  Synchronises. */
SPX_API int spx_weighted_random_sampling(spx_queue_t q, spx_rng_t rng, const float* weights, size_t n, size_t sampling_num,
                                         int32_t* idx_out, size_t* m_host);
/* PreprocessFilter::farthest_point_sampling(source, output, n) —
 * preprocess_operator/farthest_point_sampling_operator.hpp:27-94: starting from `first_index` (the reference draws it
 * with uniform_int_distribution<size_t>(0, N-1) on the operator's mt19937: spx_rng_uniform_index), repeatedly takes the
 * point farthest from everything selected so far (squared distance over xyzw, ties to the lower index).  One cooperative
 * launch for the whole selection.  Kept indices ascending (device int32[min(n, sampling_num)]).  Synchronises. */
SPX_API int spx_rng_uniform_index(spx_rng_t rng, size_t n, size_t* out);
SPX_API int spx_farthest_point_sampling(spx_queue_t q, const float* points, size_t n, size_t sampling_num,
                                        size_t first_index, int32_t* idx_out, size_t* m_host);
/* PreprocessFilter::angle_incidence_filter(source, output, min_angle, max_angle) —
 * preprocess_operator/angle_incidence_filter_operator.hpp:23-111: keep the points whose incidence angle (between the
 * ray from the sensor and the surface normal; normals, or the smallest-eigenvalue direction of covs when normals is
 * NULL) lies in [min_angle, max_angle] (0 <= min < max <= pi/2, else SPX_ERR_INVALID_ARGUMENT).  Kept indices
 * ascending in idx_out (device int32[<= n]).  Synchronises. */
SPX_API int spx_angle_incidence_indices(spx_queue_t q, const float* points, const float* normals, const float* covs,
                                        size_t n, float min_angle, float max_angle, int32_t* idx_out, size_t* m_host);
/* filter::OutlierRemoval (I/algorithms/filter/outlier_removal_filter.hpp; semantics of PCL's StatisticalOutlierRemoval /
 * RadiusOutlierRemoval, DESIGN.md §3.3) on an index built over `points` (n must equal the index's point count, else
 * SPX_ERR_INVALID_ARGUMENT).  d^2 = fma(dz,dz,fma(dy,dy,dx*dx)); a point with a non-finite coordinate is removed; the
 * "others" of point i are every j != i by index, exact duplicates included.  Kept indices ascending in idx_out (device
 * int32[<= n]); apply them to every attribute with spx_gather.  Synchronises once (the count).
 *   statistical: d_i = mean of sqrtf(d^2) over the k nearest others (the k+1 nearest neighbours minus i itself, or
 *     minus the last when i is not listed; fp32, rank order, entries without a neighbour or with an overflowed d^2
 *     skipped; no entry left = invalid, removed).  mu, sigma = mean and sample deviation of the valid d_i (fp64,
 *     fixed fold order, variance clamped at 0); keep i iff (double)d_i <= mu + stddev_mul * sigma, every valid point
 *     when at most one is valid.  1 <= mean_k <= 127, stddev_mul finite.  mean_dist_out (nullable, device float[n])
 *     receives d_i, NaN for invalid points.
 *   radius: keep i iff at least min_neighbors others lie at d^2 <= radius * radius (fp32); radius finite, >= 0. */
SPX_API int spx_statistical_outlier_indices(spx_index_t index, const float* points, size_t n, int mean_k, float stddev_mul,
                                            float* mean_dist_out, int32_t* idx_out, size_t* m_host);
SPX_API int spx_radius_outlier_indices(spx_index_t index, const float* points, size_t n, float radius,
                                       uint32_t min_neighbors, int32_t* idx_out, size_t* m_host);
/* Euclidean cluster extraction (semantics of PCL's EuclideanClusterExtraction, DESIGN.md §3.4) on an index built over
 * `points` (n must equal the index's point count, else SPX_ERR_INVALID_ARGUMENT).  Points i != j are adjacent iff both
 * are finite and d^2 = fma(dz,dz,fma(dy,dy,dx*dx)) <= tolerance * tolerance (fp32; exact duplicates are adjacent at
 * tolerance 0).  A cluster is a connected component of that graph; a point with a non-finite coordinate belongs to
 * none and bridges none.  A component is kept iff min_cluster_size <= size <= max_cluster_size (larger ones are
 * dropped, not split).  The C kept clusters are ordered by size descending, ties by smallest member ascending:
 * labels_out (nullable, device int32[n]) receives each point's cluster rank, -1 for non-finite points and dropped
 * components; indices_out (device int32[>= n_members]) the members of cluster 0, 1, ... each in ascending index order;
 * offsets_out (device uint32[>= C + 1]) the exclusive prefix of the cluster sizes, offsets_out[C] = n_members.
 * tolerance finite and >= 0, 1 <= min_cluster_size <= max_cluster_size, n < 2^31.  The result is a pure function of
 * the input (runs repeat bit for bit).  n = 0 gives 0 clusters, writes nothing and launches nothing.  Synchronises
 * once (the counts).  Unlike the radius filter the search has no early stop: the cost grows with the number of
 * neighbours within tolerance of each point. */
SPX_API int spx_euclidean_clusters(spx_index_t index, const float* points, size_t n, float tolerance,
                                   uint32_t min_cluster_size, uint32_t max_cluster_size, int32_t* labels_out,
                                   int32_t* indices_out, uint32_t* offsets_out, size_t* n_clusters_host,
                                   size_t* n_members_host);
/* RANSAC plane segmentation (semantics of PCL's SACSegmentation with SACMODEL_PLANE / SACMODEL_PERPENDICULAR_PLANE and
 * SAC_RANSAC, DESIGN.md §3.5) of the n points (float4 xyz1, 16-byte aligned).  F = the indices of the points whose
 * x, y and z are finite, ascending; n_f = |F|.  Hypothesis h in [0, max_iterations) samples F[j_s], s = 0, 1, 2, with
 * j_s = ((r >> 32) * n_f) >> 32 and r = splitmix64(seed + (3h + s + 1) * 0x9E3779B97F4A7C15) (counter-based: no
 * state, no host RNG), and builds the plane through the three points in fp64 (the fma chain of §3.5).  It is invalid
 * when two of its j_s are equal, n_f < 3, the cross product is degenerate (l^2 <= 1e-12 |u|^2 |v|^2), or axis3_host
 * (nullable, 3 floats, finite and nonzero) is given and |n . axis| < cos(eps_angle).  Its fp32 coefficients
 * (n_x, n_y, n_z, d) count point i as an inlier iff fabsf(fmaf(n_z,z,fmaf(n_y,y,fmaf(n_x,x,d)))) < threshold (strict);
 * non-finite points never are.  The best hypothesis is the valid one with most inliers, ties to the lowest h.  With
 * optimize != 0 and >= 3 inliers its plane is refitted to them (the smallest-eigenvalue direction of their fp64
 * covariance, oriented like the hypothesis normal, through their centroid; kept only when finite) and the inliers are
 * selected again.  coeffs4_host receives the final plane (NaN without a model), hypothesis_host the best h (-1 without
 * a model), inliers_out (device int32[>= n_inliers]) the inliers ascending, n_inliers_host their count, remainder_out
 * (nullable, device int32[>= n - n_inliers]) every other index ascending (non-finite rows included), counts_out
 * (nullable, device uint32[max_iterations]) every hypothesis's inlier count, 0xFFFFFFFF for an invalid one.
 * threshold finite and > 0, 1 <= max_iterations <= 2^20, eps_angle in [0, pi/2], n < 2^31, else
 * SPX_ERR_INVALID_ARGUMENT.  Without refinement the result is a pure function of the input; with it runs still repeat
 * bit for bit.  n = 0 gives no model and launches nothing.  Synchronises once. */
SPX_API int spx_plane_segment(spx_queue_t q, const float* points, size_t n, float threshold, uint32_t max_iterations,
                              uint64_t seed, const float* axis3_host, double eps_angle, int optimize,
                              float* coeffs4_host, int32_t* hypothesis_host, int32_t* inliers_out,
                              size_t* n_inliers_host, int32_t* remainder_out, uint32_t* counts_out);
/* FPFH descriptors (Rusu et al. 2009, with the point's own SPFH term; DESIGN.md §3.6) of the n points (float4 xyz1)
 * with their normals (float4 xyz0, oriented as spx_normals writes them) over the radius neighbours nn_idx int32[n][k] /
 * nn_dist float[n][k] exactly as spx_index_radius returns them (1 <= k <= 128).  A point is valid iff x, y, z and the
 * normal's xyz are finite; N(i) = the listed j >= 0, j != i, j valid, listed d^2 > 0, in rank order.  The pair feature,
 * its three 11-bin histograms (f1 = atan2 decided by exact-in-sign tests against the ten boundary rays), SPFH_i = bin
 * counts x (100 / pairs counted) and F_i[b] = acc[b] (100 / sum_g) + SPFH_i[b] with acc[b] = sum over N(i) of
 * SPFH_j[b] / d^2_ij are pinned op for op in §3.6.  features: device float[n][33], bins 0-10 f1, 11-21 f2, 22-32 f3;
 * an invalid point's row is NaN.  points, normals and features 16-byte aligned; n < 2^31.  The result is a pure
 * function of the input.  n = 0 launches nothing.  Asynchronous. */
SPX_API int spx_fpfh(spx_queue_t q, const float* points, const float* normals, size_t n, const int32_t* nn_idx,
                     const float* nn_dist, int k, float* features);
/* Nearest-feature correspondences (DESIGN.md §3.6): nn(i) = the target row t with the lowest (D(i, t), t) over the
 * targets with D not NaN, D = fma(d_32, d_32, ... fma(d_1, d_1, d_0 d_0)), d_b = s_b - t_b (fp32).  A source row with
 * no such target has no correspondence.  mutual != 0 keeps (i, nn(i)) only if the reverse search from nn(i) picks i.
 * src_idx_out / tgt_idx_out (device int32[>= n_source]) receive the pairs ascending in i, m_host their count.  Rows
 * are float[33]; counts < 2^31.  Synchronises once. */
SPX_API int spx_feature_correspondences(spx_queue_t q, const float* source_features, size_t n_source,
                                        const float* target_features, size_t n_target, int mutual, int32_t* src_idx_out,
                                        int32_t* tgt_idx_out, size_t* m_host);
/* RANSAC registration over the m correspondences (src_idx[k], tgt_idx[k]) between source and target points (float4,
 * 16-byte aligned; DESIGN.md §3.6).  A correspondence with an index out of range or a non-finite coordinate is never
 * an inlier and makes every hypothesis that samples it invalid.  Hypothesis h in [0, max_iterations) samples
 * correspondences c_s = ((r >> 32) m) >> 32, r = splitmix64(seed + (3h + s + 1) 0x9E3779B97F4A7C15) (the stream of
 * spx_plane_segment).  It is invalid when m < 3, two c_s are equal, an edge fails ds^2 >= tau^2 dt^2 and
 * dt^2 >= tau^2 ds^2 (fp64, tau = edge_length_similarity) or a triangle is degenerate (l^2 <= 1e-12 |u|^2 |v|^2); its
 * pose is the closed-form triad R = F_q F_p^T, t = c_q - R c_p in fp64, rounded to fp32.  Correspondence k is an inlier
 * iff dot(R p + t - q) < eps * eps (fp32 chain of §3.6, strict).  The best hypothesis is the valid one with most
 * inliers, ties to the lowest h.  With optimize != 0 and >= 3 inliers the pose is refitted to them by least squares
 * (fp64 moments in a fixed order; a coplanar set is fine; kept only when finite) and the inliers are selected again.
 * T4x4_host receives the pose column-major (NaN without a model), hypothesis_host the best h (-1 without a model),
 * inliers_out (device int32[>= m]) the inlier positions ascending, n_inliers_host their count, counts_out (nullable,
 * device uint32[max_iterations]) every hypothesis's count, 0xFFFFFFFF for an invalid one.
 * eps finite and > 0, 1 <= max_iterations <= 2^20, 0 < edge_length_similarity <= 1, m < 2^31, else
 * SPX_ERR_INVALID_ARGUMENT.  Without refinement the result is a pure function of the input; with it runs still repeat
 * bit for bit.  m = 0 gives no model and launches no kernel (counts_out, when given, is set to 0xFFFFFFFF by a memset).
 * Synchronises once. */
SPX_API int spx_ransac_registration(spx_queue_t q, const float* source_points, size_t n_source,
                                    const float* target_points, size_t n_target, const int32_t* src_idx,
                                    const int32_t* tgt_idx, size_t m, float max_correspondence_distance,
                                    uint32_t max_iterations, uint64_t seed, float edge_length_similarity, int optimize,
                                    float* T4x4_host, int32_t* hypothesis_host, int32_t* inliers_out,
                                    size_t* n_inliers_host, uint32_t* counts_out);

/* ------------------------------------------------------------------ submap: mapping::VoxelHashMap
 * I/algorithms/mapping/voxel_hash_map.hpp:22-1066 — a device hash table keyed by the voxel key of
 * voxel_constants.hpp:36-62 (open addressing, double hashing :607-612, <= 100 probes :498, capacities from the
 * reference's list of primes :481-482).  A slot accumulates sum xyz + count, the sum of the log-Euclidean images
 * of the covariances rotated into the map frame (:420-476), sum rgba, sum intensity and the call number of its last
 * update.  The accumulation order inside a call is unspecified (fp32 atomics, as in the reference): sums agree
 * with a sequential evaluation to rounding.
 *   create       VoxelHashMap(queue, voxel_size) :29-36; voxel_size <= 0 -> SPX_ERR_INVALID_ARGUMENT (:41-43)
 *   set_params   set_voxel_size / set_max_staleness (100) / set_remove_old_data_cycle (10) /
 *                set_rehash_threshold (0.7) / set_min_num_point (1) :40-80
 *   clear        :83-112
 *   add          add_point_cloud(cloud, sensor_pose) :117-140: rehash when voxel_num / capacity > threshold, insert the
 *                points transformed by sensor_pose (column-major 4x4, NULL = identity; covs float[n][16], rgb
 *                float[n][4], intensities float[n], each nullable), every remove_old_data_cycle-th call drop the
 *                voxels not updated for more than max_staleness calls, ++call counter.  Synchronises (voxel count).
 *   remove_old   remove_old_data() :248,794-845
 *   info         capacity, voxel_num, call counter, which attributes the map holds
 *   downsample   downsampling(result, center, distance) :146-188,936-1065: voxels with count >= min_num_point whose
 *                centroid lies in [center - distance, center + distance]^3, in slot order: centroid (w = 1),
 *                exp(mean log-covariance) as float[16], mean rgba, mean intensity; out_keys (nullable) receives the
 *                voxel key of every row.  Outputs must hold voxel_num rows (out_capacity); attribute outputs the map
 *                does not hold are left untouched.  *m_host = rows written.  Synchronises.
 *   overlap_ratio compute_overlap_ratio(cloud, sensor_pose) :194-246: fraction of the points whose voxel exists with
 *                count >= min_num_point.  Synchronises. */
/* eigen_utils::log_spd_3x3(A, min_eigenvalue) / exp_spd_3x3(A) — I/utils/eigen_utils.hpp:646-677 — on n
 * column-major 3x3 matrices (device or managed float[n][9]); asynchronous. */
SPX_API int spx_spd_function(spx_queue_t q, const float* mats, size_t n, int is_log, float min_eigenvalue, float* out);
typedef struct spx_voxelmap_s* spx_voxelmap_t;
SPX_API int spx_voxelmap_create(spx_queue_t q, float voxel_size, spx_voxelmap_t* out);
SPX_API int spx_voxelmap_destroy(spx_voxelmap_t m);
SPX_API int spx_voxelmap_set_params(spx_voxelmap_t m, float voxel_size, uint32_t max_staleness,
                                    uint32_t remove_old_data_cycle, float rehash_threshold, uint32_t min_num_point);
SPX_API int spx_voxelmap_clear(spx_voxelmap_t m);
SPX_API int spx_voxelmap_add(spx_voxelmap_t m, const float* points, const float* covs, const float* rgb,
                             const float* intensities, size_t n, const float* sensor_pose16);
SPX_API int spx_voxelmap_remove_old(spx_voxelmap_t m);
SPX_API int spx_voxelmap_info(spx_voxelmap_t m, uint64_t* capacity, uint64_t* voxel_num, uint32_t* staleness_counter,
                              int* has_cov, int* has_rgb, int* has_intensity);
SPX_API int spx_voxelmap_downsample(spx_voxelmap_t m, const float* center3, float distance, float* out_points,
                                    float* out_covs, float* out_rgb, float* out_intensities, uint64_t* out_keys,
                                    size_t out_capacity, size_t* m_host);
SPX_API int spx_voxelmap_overlap_ratio(spx_voxelmap_t m, const float* points, size_t n, const float* sensor_pose16,
                                       float* ratio);

/* ------------------------------------------------------------------ registration
 * Registration::compute_linearized_result / linearize — registration.hpp:312-331,513-676:
 * per source i: skip if dist[i] > max_corr_sq; factor (factor.hpp:130-278) on
 * (src[i], tgt[idx[i]]); robust weight/rho (robust.hpp:56-114); sum to 6x6 H, 6 b, error,
 * inlier.  src_covs/tgt_covs NULL -> identity, tgt_normals NULL -> zero (registration.hpp:589-592).
 * Outputs are HOST pointers (H 36 floats, symmetric); synchronises like the reference (:674). */
SPX_API int spx_linearize(spx_queue_t q, int reg_type, int robust_loss, const float* src_points, const float* src_covs,
                  size_t ns, const float* tgt_points, const float* tgt_covs, const float* tgt_normals,
                  const int32_t* nn_idx, const float* nn_dist, const float* T_host, float max_corr_sq,
                  float robust_scale, float* H_host, float* b_host, float* error_host, uint32_t* inlier_host);
/* Registration::compute_error_frozen / compute_error — registration.hpp:350-359,678-789 */
SPX_API int spx_error(spx_queue_t q, int reg_type, int robust_loss, const float* src_points, const float* src_covs, size_t ns,
              const float* tgt_points, const float* tgt_covs, const float* tgt_normals, const int32_t* nn_idx,
              const float* nn_dist, const float* T_host, float max_corr_sq, float robust_scale, float* error_host,
              uint32_t* inlier_host);
/* Registration::compute_icp_robust_weights — registration.hpp:279-294,412-462; weights[ns] device. */
SPX_API int spx_robust_weights(spx_queue_t q, int reg_type, int robust_loss, const float* src_points, const float* src_covs,
                       size_t ns, const float* tgt_points, const float* tgt_covs, const float* tgt_normals,
                       const int32_t* nn_idx, const float* nn_dist, const float* T_host, float max_corr_sq,
                       float robust_scale, float* weights);

/* host-side pieces of the optimiser, exported so a caller that injects its own KNN (the
 * reference's tests subclass KNNBase) can drive the loop: registration.hpp:791-801 (LDLT solve
 * of (H + lambda I) delta = -b, fp64 inside), eigen_utils.hpp:909-943 (se3_exp, column-major
 * out), dogleg_step.hpp:34-102. */
SPX_API void spx_default_registration_params(spx_registration_params* p);
/* GenZ planarity threshold used by the stateless entry points below and above (spx_linearize, spx_error,
 * spx_robust_weights), which take no parameter struct; thread-local, default 0.2.  Registration handles use
 * spx_registration_params::genz_planarity_threshold. */
SPX_API int spx_set_genz_planarity_threshold(float threshold);
/* RegistrationParams::rotation_constraint for the same stateless entry points (thread-local, default off): the
 * Jensen-Bregman LogDet term of I/algorithms/registration/rotation_constraint.hpp:15-121 added to every correspondence
 * (registration.hpp:629-649,757-764). */
SPX_API int spx_set_rotation_constraint(int enable, float weight, float robust_scale);
SPX_API int spx_solve_6x6(const float* H_host, const float* b_host, float lambda, float* delta_host, int* success);
SPX_API int spx_se3_exp(const float* twist6_host, float* T_host);
SPX_API int spx_dogleg_step(const float* H_host, const float* g_host, float radius, float* p_host, float* step_norm,
                    float* predicted_reduction);

/* Registration(queue, params) — registration.hpp:105-114 */
SPX_API int spx_registration_create(spx_queue_t q, const spx_registration_params* params, spx_registration_t* out);
SPX_API int spx_registration_destroy(spx_registration_t reg);
SPX_API int spx_registration_set_params(spx_registration_t reg, const spx_registration_params* params);
/* Registration(queue, params) with params.degenerate_reg / params.map_prior (registration.hpp:112-113); setting them
 * drops a stored prior (MapPrior::set_params, map_prior.hpp:25-28). */
SPX_API void spx_default_registration_addons(spx_registration_addons* a);
SPX_API int spx_registration_set_addons(spx_registration_t reg, const spx_registration_addons* a);
/* Registration::set_map_prior_state(prev_result, T_pred) — registration.hpp:124-126, MapPrior::update map_prior.hpp:30-117
 * (T_pred column-major 4x4).  *active_out (nullable): whether a prior is now in force. */
SPX_API int spx_registration_set_map_prior_state(spx_registration_t reg, const spx_registration_result* prev_result,
                                                 const float* T_pred16, int* active_out, float* omega36_out);
/* DegenerateRegularization::regularize on host H (36, symmetric) / b (6) in place — degenerate_regularization.hpp:58-112;
 * what compute_linearized_result(…, pose, initial_pose, …) applies to its raw result (registration.hpp:312-323). */
SPX_API int spx_degenerate_regularize(const spx_registration_addons* a, float* H36, float* b6, uint32_t inlier,
                                      const float* T_current16, const float* T_initial16);


/* Registration::align(source, target, target_knn, initial_guess, options) — registration.hpp:201-276
 * with the target's spx_index as the KNNBase.  GN runs as a device-resident loop (nearest
 * neighbour + linearise + reduce + 6x6 solve + pose update in one kernel per iteration, no host
 * round trip until the end); LM / dog-leg take one host decision per trial step (:830-964).
 * robust_scale <= 0 selects params.robust_default_scale (:217-218).  Missing inputs raise the
 * reference's validate_params errors (:129-193).  T_trace_host (nullable): max_iterations*16
 * floats, pose after each outer iteration.  Synchronises. */
SPX_API int spx_registration_align(spx_registration_t reg, const float* src_points, const float* src_covs, size_t ns,
                           const float* tgt_points, const float* tgt_covs, const float* tgt_normals, size_t nt,
                           spx_index_t target_index, const float* T_init_host, float robust_scale,
                           spx_registration_result* result_host, float* T_trace_host);
/* Batched Registration::align — BASELINE config 5 / SURVEY.md §8(b) `spx_align_batch`, §8(e) "all pairs share
 * launches via a pair-id segment key": n_pairs independent (source, target, index, initial guess) tuples are
 * aligned by ONE set-up launch and ONE persistent cooperative launch (Gauss-Newton; LM / dog-leg fall back to
 * one align after the other).  Every pair's result is bit for bit what spx_registration_align returns for that
 * pair alone (the per-pair sums are folded in an order that depends on the pair's own size only).  Reference
 * semantics per pair: registration.hpp:201-276.  pairs_host / results_host are HOST arrays; the pointers inside
 * a pair are device pointers as for spx_registration_align.  Synchronises once. */
typedef struct spx_align_pair {
    const float* src_points;
    const float* src_covs;
    size_t ns;
    const float* tgt_points;
    const float* tgt_covs;
    const float* tgt_normals;
    size_t nt;
    spx_index_t target_index;
    const float* T_init_host; /* 16 floats column-major, NULL = identity */
    float robust_scale;       /* <= 0: params.robust_default_scale */
} spx_align_pair;
SPX_API int spx_registration_align_batch(spx_registration_t reg, size_t n_pairs, const spx_align_pair* pairs_host,
                                 spx_registration_result* results_host);
/* spx_align_batch — SURVEY.md §8(b), BASELINE config 5 ("batched odometry: independent scan pairs: voxel
 * downsample + covariance + GICP"): n_pairs RAW scan pairs to registration results in one call.  Per cloud:
 * VoxelGrid::downsampling(voxel_size) -> KDTree::build -> knn_search(k) -> covariance::estimate
 * (voxel_downsampling.hpp:50-79, kdtree.hpp:165-224, covariance.hpp:260-311), spread over `lanes` internal queues
 * (streams) driven by as many host threads; then ONE batched Registration::align for all pairs
 * (spx_registration_align_batch).  A cloud that appears in several pairs (same pointer and size) is processed once.
 * lanes <= 0: SPX_BATCH_LANES or 8.  Results are bit for bit those of the single-pair entry points.
 * n_src_out / n_tgt_out (nullable, HOST uint32[n_pairs]): points after the voxel grid.  Synchronises. */
typedef struct spx_batch_s* spx_batch_t;
typedef struct spx_scan_pair {
    const float* src_raw; /* device float[n_src][4] */
    size_t n_src;
    const float* tgt_raw;
    size_t n_tgt;
    const float* T_init_host; /* 16 floats column-major, NULL = identity */
} spx_scan_pair;
SPX_API int spx_batch_create(spx_queue_t q, const spx_registration_params* params, float voxel_size, int k_correspondences,
                     int lanes, spx_batch_t* out);
SPX_API int spx_batch_destroy(spx_batch_t batch);
SPX_API int spx_batch_set_params(spx_batch_t batch, const spx_registration_params* params);
SPX_API int spx_align_batch(spx_batch_t batch, size_t n_pairs, const spx_scan_pair* pairs_host,
                    spx_registration_result* results_host, uint32_t* n_src_out, uint32_t* n_tgt_out);
/* CUDA-event time of the batched align kernel of the last spx_align_batch and the most iterations any pair ran */
SPX_API int spx_batch_last_timing(spx_batch_t batch, float* align_ms, int32_t* iterations);
/* CUDA-event time of the iteration kernels of the last align on this handle (from just before the
 * first iteration launch to just after the last), the number of iteration kernels launched and
 * the number of outer iterations that did work: bench.py's live per-launch duration. */
SPX_API int spx_registration_last_timing(spx_registration_t reg, float* loop_ms, int32_t* launches, int32_t* iterations);
/* Tuning aid: correspondences of the last align that were KEPT without a search, summed over its iterations.  The
 * split-kernel Gauss-Newton loop (large clouds) and the sharded one-launch align keep a query's nearest neighbour
 * while the query has moved less than half the margin its last search certified between the nearest and every other
 * target point — the same index and the same distance find_correspondences (registration.hpp:576-604 ->
 * kdtree.hpp:463-553) would return.
 * SPX_KEEP_FRAC < 0 in the environment searches every query in every iteration. */
SPX_API int spx_registration_kept_correspondences(spx_registration_t reg, uint64_t* kept);
/* tuning aid: per-iteration phase timestamps of the cooperative align kernel (globaltimer ns, latest
 * block to reach each phase): times_host[it][8] = {start, first-pass search done, cooperative search done,
 * accumulate done, partials written, grid barrier passed, fold done, solve done}.  enable != 0 allocates the buffer (affects later
 * aligns on this handle), enable == 0 frees it; times_host nullable. */
SPX_API int spx_registration_phase_times(spx_registration_t reg, int enable, uint64_t* times_host, int max_iterations);
/* neighbours cached by the last align / linearise on this handle (registration.hpp:365), device
 * pointers valid until the next call: used by compute_error_frozen-style callers */
SPX_API int spx_registration_neighbors(spx_registration_t reg, const int32_t** nn_idx, const float** nn_dist, size_t* n);

/* ------------------------------------------------------------------ multi-GPU building blocks
 * Source points are sharded across ranks, the target + index replicated (SURVEY.md §8(e)).
 * One outer GN iteration on a shard = nearest neighbour + linearise + block reduce into
 * sums_dev[SPX_SUMS_LEN] doubles (21 upper-triangle H terms, 6 b, error, inlier count, 3 pad) with
 * NO host sync; the caller all-reduces sums_dev (NCCL, same stream) and then calls
 * spx_registration_shard_update on every rank, which solves and advances the device-resident
 * pose identically everywhere. */
#define SPX_SUMS_LEN 32
SPX_API int spx_registration_shard_begin(spx_registration_t reg, const float* src_points, const float* src_covs, size_t ns,
                                 const float* tgt_points, const float* tgt_covs, const float* tgt_normals, size_t nt,
                                 spx_index_t target_index, const float* T_init_host, float robust_scale);
SPX_API int spx_registration_shard_linearize(spx_registration_t reg, double* sums_dev);
SPX_API int spx_registration_shard_update(spx_registration_t reg, const double* sums_dev);
SPX_API int spx_registration_shard_finish(spx_registration_t reg, spx_registration_result* result_host);

/* ------------------------------------------------------------------ multi-GPU: fused linearise + exchange
 * The same sharding (source split, target + index replicated), but the exchange of the sums row
 * happens INSIDE the iteration kernel over NVLink peer memory instead of a separate NCCL call:
 * every rank's align kernel stores its 32-double partial row into every peer's mailbox, waits for
 * the peers' rows, folds them in rank order (bitwise identical everywhere) and takes the same
 * Gauss-Newton step — one cooperative launch per align per GPU, no host round trip, no collective
 * launch per iteration.  The reference has no multi-device path (SURVEY.md §2.2); this is the
 * B200-native replacement of what would be an all-reduce after registration.hpp:576-661.
 *
 * One communicator per rank.  Two ways to wire the mailboxes:
 *  - one process per GPU (torch.distributed): spx_comm_ipc_handle on every rank, all-gather the
 *    64-byte handles with any host-side transport, spx_comm_connect_ipc, then a host barrier;
 *  - one process driving several GPUs: spx_comm_connect_local on the array of communicators. */
typedef struct spx_comm_s* spx_comm_t;
#define SPX_IPC_HANDLE_BYTES 64
#define SPX_MAX_WORLD 8
SPX_API int spx_comm_create(spx_queue_t q, int rank, int world, spx_comm_t* out);
SPX_API int spx_comm_destroy(spx_comm_t comm);
SPX_API int spx_comm_ipc_handle(spx_comm_t comm, uint8_t* handle64_host);
/* handles_host: world * SPX_IPC_HANDLE_BYTES bytes, rank-major (own entry ignored) */
SPX_API int spx_comm_connect_ipc(spx_comm_t comm, const uint8_t* handles_host);
SPX_API int spx_comm_connect_local(spx_comm_t* comms, int world);
/* Gauss-Newton align of this rank's source shard against the replicated target; every rank must
 * call launch (asynchronous) with the same params / initial guess, then finish (synchronises,
 * result identical on every rank; H, b, error, inlier are the GLOBAL sums).  A peer that does not
 * answer within ~5 s aborts the kernel and finish returns SPX_ERR_INTERNAL. */
SPX_API int spx_registration_align_sharded_launch(spx_registration_t reg, spx_comm_t comm, const float* src_points,
                                          const float* src_covs, size_t ns, const float* tgt_points,
                                          const float* tgt_covs, const float* tgt_normals, size_t nt,
                                          spx_index_t target_index, const float* T_init_host, float robust_scale);
SPX_API int spx_registration_align_sharded_finish(spx_registration_t reg, spx_registration_result* result_host);

#ifdef __cplusplus
}
#endif
#endif /* SPX_H_ */
