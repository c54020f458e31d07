// Statistical and radius outlier removal on the exact grid index (I/algorithms/filter/outlier_removal_filter.hpp in
// the reference; semantics of PCL's StatisticalOutlierRemoval / RadiusOutlierRemoval, pinned in DESIGN.md §3.3).
//
// Statistical: the k+1 nearest neighbours of every point in its own cloud come from the index's k-NN (spx_index_knn,
// "brute force, ties by index"), in chunks of queries so that the neighbour lists never need more than
// OR_CHUNK_ENTRIES entries of scratch.  One kernel per chunk turns each list into the point's mean distance to its k
// nearest others and writes per-block fp64 partials of (sum, sum of squares, count); the last block of the last
// chunk folds every partial in block order (deterministic) into mu, sigma and the threshold.  A flag pass, the
// device-wide scan and compact_index_kernel produce the kept indices in ascending order.
//
// Radius: a counting search per point on ONE grid level whose cell edge is comparable to the radius — grid_search
// with a policy that counts the other points within r^2 and stops once the count reaches min_neighbors.  The bounded
// search visits every cell that can hold a point within its max_radius (the margin argument of spx_grid.cuh; cell
// coordinates clamp, so points outside a hinted box sit in the boundary cells, whose slabs extend to infinity).
#include <cmath>

#include "spx_grid.cuh"
#include "spx_scan.cuh"

using namespace spx;

namespace {

constexpr int OR_THREADS = 256;
constexpr int OR_WARPS = OR_THREADS / 32;
constexpr size_t OR_CHUNK_ENTRIES = (size_t)1 << 25;  // neighbour entries per k-NN chunk (256 MB of idx + dist)
constexpr size_t OR_CHUNK_MAX = (size_t)1 << 20;      // queries per chunk

struct SorStats {
    double mu, sigma, thr;  // thr = mu + alpha sigma (+inf when at most one point is valid)
    unsigned long long n_valid;
    unsigned int ticket;
};

__device__ __forceinline__ bool finite3(const float4 p) { return isfinite(p.x) && isfinite(p.y) && isfinite(p.z); }

// Mean distance of each query of the chunk to its k nearest OTHER points, from its k+1 nearest neighbours in the
// cloud (kk = k + 1 entries per row, ascending by (dist, idx)): the entry whose index is the query itself is dropped,
// or the last one when the query is not listed (more than k exact duplicates with lower indices).  Entries without a
// neighbour (idx < 0) or with an overflowed distance are skipped; sum of sqrtf(d^2) in rank order, fp32, / count.
// Per-block fp64 partials (S1, S2, N) over the valid points; LAST: the last block folds all `n_partials` partials of
// this and the earlier chunks in block order and writes the threshold.
__global__ void __launch_bounds__(OR_THREADS) sor_mean_kernel(const float4* __restrict__ pts, uint32_t base, uint32_t nq,
                                                              const int32_t* __restrict__ idx, const float* __restrict__ dist,
                                                              int kk, float* __restrict__ mean, double* __restrict__ partials,
                                                              uint32_t block_base, uint32_t n_partials, int last, double alpha,
                                                              SorStats* __restrict__ st) {
    const uint32_t t = blockIdx.x * OR_THREADS + threadIdx.x;
    double s1 = 0.0, s2 = 0.0;
    uint32_t cnt = 0;
    if (t < nq) {
        const uint32_t i = base + t;
        float dbar = __int_as_float(0x7fc00000);  // NaN: removed as invalid
        if (finite3(__ldg(pts + i))) {
            const int32_t* irow = idx + (size_t)t * kk;
            const float* drow = dist + (size_t)t * kk;
            int drop = kk - 1;
            for (int j = 0; j < kk; ++j)
                if (irow[j] == (int32_t)i) {
                    drop = j;
                    break;
                }
            float sum = 0.0f;
            int c = 0;
            for (int j = 0; j < kk; ++j) {
                if (j == drop) continue;
                const float d = drow[j];
                if (irow[j] < 0 || !isfinite(d)) continue;
                sum = __fadd_rn(sum, __fsqrt_rn(d));
                ++c;
            }
            if (c > 0) {
                dbar = __fdiv_rn(sum, (float)c);
                const double v = (double)dbar;
                s1 = v;
                s2 = __dmul_rn(v, v);
                cnt = 1;
            }
        }
        mean[i] = dbar;
    }
    // fixed-order block reduction: warp butterflies, then the warps in order
    __shared__ double red[3][OR_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    s1 = warp_sum(s1);
    s2 = warp_sum(s2);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (lane == 0) {
        red[0][warp] = s1;
        red[1][warp] = s2;
        red[2][warp] = (double)cnt;
    }
    __syncthreads();
    if (threadIdx.x < 3) {
        double s = 0.0;
        for (int w = 0; w < OR_WARPS; ++w) s += red[threadIdx.x][w];
        __stcg(partials + (size_t)(block_base + blockIdx.x) * 3 + threadIdx.x, s);
    }
    if (!last) return;
    __shared__ bool is_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) is_last = atomicAdd(&st->ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    // every thread folds its stride of the partials in order, then the threads are folded in order
    __shared__ double fold[3][OR_THREADS];
    double a = 0.0, b = 0.0, c = 0.0;
    for (uint32_t p = threadIdx.x; p < n_partials; p += OR_THREADS) {
        a += __ldcg(partials + (size_t)p * 3);
        b += __ldcg(partials + (size_t)p * 3 + 1);
        c += __ldcg(partials + (size_t)p * 3 + 2);
    }
    fold[0][threadIdx.x] = a;
    fold[1][threadIdx.x] = b;
    fold[2][threadIdx.x] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        double S1 = 0.0, S2 = 0.0, N = 0.0;
        for (int u = 0; u < OR_THREADS; ++u) {
            S1 += fold[0][u];
            S2 += fold[1][u];
            N += fold[2][u];
        }
        const double INF = __longlong_as_double(0x7ff0000000000000ll);
        double mu = 0.0, sigma = 0.0, thr = INF;
        if (N > 0.0) mu = __ddiv_rn(S1, N);
        if (N > 1.0) {
            // PCL's formula; a variance that rounds below zero (all means equal) is zero
            const double var = __ddiv_rn(__dsub_rn(S2, __ddiv_rn(__dmul_rn(S1, S1), N)), __dsub_rn(N, 1.0));
            sigma = sqrt(fmax(var, 0.0));
            thr = __dadd_rn(mu, __dmul_rn(alpha, sigma));
        }
        st->mu = mu;
        st->sigma = sigma;
        st->thr = thr;
        st->n_valid = (unsigned long long)N;
        st->ticket = 0u;
    }
}

__global__ void __launch_bounds__(OR_THREADS) sor_flag_kernel(const float* __restrict__ mean, uint32_t n,
                                                              const SorStats* __restrict__ st, uint32_t* __restrict__ flags) {
    const uint32_t i = blockIdx.x * OR_THREADS + threadIdx.x;
    if (i >= n) return;
    const float d = mean[i];
    flags[i] = (!isnan(d) && (double)d <= st->thr) ? 1u : 0u;
}

// grid_search policy: counts the points other than `self` with d^2 <= r2; once `need` is reached worst() drops below
// every bound, which prunes the remaining rows and ends the search at the next stop test.
struct CountWithin {
    float r2;
    int self;
    uint32_t need, cnt;
    __device__ __forceinline__ float worst() const { return cnt >= need ? -1.0f : FLT_MAX; }
    __device__ __forceinline__ void offer(float ds, int idx, uint32_t) { cnt += (ds <= r2 && idx != self) ? 1u : 0u; }
};

__global__ void __launch_bounds__(OR_THREADS) ror_flag_kernel(const GridView g, const float4* __restrict__ pts, uint32_t n,
                                                              float reach, float r2, uint32_t min_neighbors,
                                                              uint32_t* __restrict__ flags) {
    const uint32_t i = blockIdx.x * OR_THREADS + threadIdx.x;
    if (i >= n) return;
    const float4 p = __ldg(pts + i);
    uint32_t keep = 0u;
    if (finite3(p)) {
        if (min_neighbors == 0u) {
            keep = 1u;
        } else {
            CountWithin c{r2, (int)i, min_neighbors, 0u};
            // r_begin 1: the first pass is the 3x3x3 block; unbounded shell count (the stop test ends it)
            grid_search(g, p.x, p.y, p.z, c, reach, 1, 1 << 20);
            keep = c.cnt >= min_neighbors ? 1u : 0u;
        }
    }
    flags[i] = keep;
}

// flags -> ascending kept indices in idx_out, *m_host (the call's one synchronisation)
void compact_and_count(spx_queue_t q, const uint32_t* flags, uint32_t* pos, uint32_t* scan_tmp, uint32_t* total_dev,
                       uint32_t n, int32_t* idx_out, size_t* m_host) {
    cudaStream_t st = q->stream;
    exclusive_scan_u32(st, flags, pos, n, scan_tmp, total_dev);
    compact_index_kernel<<<div_up(n, COMPACT_THREADS), COMPACT_THREADS, 0, st>>>(flags, pos, n, idx_out);
    SPX_LAUNCH_CHECK();
    uint32_t* htotal = static_cast<uint32_t*>(q->pinned_get(64));
    SPX_CUDA(cudaMemcpyAsync(htotal, total_dev, 4, cudaMemcpyDeviceToHost, st));
    q->sync();
    *m_host = *htotal;
}

}  // namespace

extern "C" {

int spx_statistical_outlier_indices(spx_index_t index, const float* points, size_t n_in, int mean_k, float stddev_mul,
                                    float* mean_dist_out, int32_t* idx_out, size_t* m_host) {
    return guard([&] {
        SPX_REQUIRE(index && m_host, "[OutlierRemoval::statistical] null argument");
        SPX_REQUIRE(n_in == index->n_total, "[OutlierRemoval::statistical] the index was not built over these points");
        SPX_REQUIRE(mean_k >= 1 && mean_k <= 127, "[OutlierRemoval::statistical] `mean_k` must be in [1, 127]");
        SPX_REQUIRE(std::isfinite(stddev_mul), "[OutlierRemoval::statistical] `stddev_mul` must be finite");
        *m_host = 0;
        if (n_in == 0) return;
        SPX_REQUIRE(points && idx_out, "[OutlierRemoval::statistical] null pointer");
        spx_queue_t q = index->q;
        DeviceGuard dg(q->device);
        cudaStream_t st = q->stream;
        const uint32_t n = (uint32_t)n_in;
        if (index->n == 0) {  // no finite point: every point is invalid, nothing is kept
            if (mean_dist_out) SPX_CUDA(cudaMemsetAsync(mean_dist_out, 0xff, (size_t)n * 4, st));  // (all-ones bits: NaN)
            q->sync();
            return;
        }
        const int kk = mean_k + 1;
        const size_t chunk = std::min<size_t>(
            n, std::min(OR_CHUNK_MAX, std::max<size_t>(OR_THREADS, OR_CHUNK_ENTRIES / (size_t)kk / OR_THREADS * OR_THREADS)));
        const size_t n_chunks = (n + chunk - 1) / chunk;
        const uint32_t blocks_per_chunk = (uint32_t)div_up(chunk, OR_THREADS);
        const uint32_t n_partials = (uint32_t)div_up(n, OR_THREADS);  // every chunk but the last is whole blocks
        // scratch outside the queue arena (the k-NN calls reset it): neighbour lists of one chunk, the mean distances
        // when the caller does not want them, the partials and the statistics; returned to the stream's pool at the end
        const size_t b_idx = align_up(chunk * kk * 4, 256), b_dist = b_idx, b_mean = mean_dist_out ? 0 : align_up((size_t)n * 4, 256);
        const size_t b_part = align_up((size_t)n_partials * 3 * 8, 256);
        char* scratch = nullptr;
        SPX_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&scratch), b_idx + b_dist + b_mean + b_part + sizeof(SorStats), st));
        struct Free {
            char* p;
            cudaStream_t s;
            ~Free() { cudaFreeAsync(p, s); }
        } release{scratch, st};
        int32_t* nn_idx = reinterpret_cast<int32_t*>(scratch);
        float* nn_dist = reinterpret_cast<float*>(scratch + b_idx);
        float* mean = mean_dist_out ? mean_dist_out : reinterpret_cast<float*>(scratch + b_idx + b_dist);
        double* partials = reinterpret_cast<double*>(scratch + b_idx + b_dist + b_mean);
        SorStats* stats = reinterpret_cast<SorStats*>(scratch + b_idx + b_dist + b_mean + b_part);
        SPX_CUDA(cudaMemsetAsync(stats, 0, sizeof(SorStats), st));
        const float4* pts = reinterpret_cast<const float4*>(points);
        for (size_t c = 0; c < n_chunks; ++c) {
            const size_t base = c * chunk;
            const uint32_t nq = (uint32_t)std::min(chunk, (size_t)n - base);
            if (spx_index_knn(index, points + base * 4, nq, kk, nullptr, nn_idx, nn_dist) != SPX_OK)
                throw Error(SPX_ERR_INTERNAL, spx_last_error());
            sor_mean_kernel<<<div_up(nq, OR_THREADS), OR_THREADS, 0, st>>>(
                pts, (uint32_t)base, nq, nn_idx, nn_dist, kk, mean, partials, (uint32_t)(c * blocks_per_chunk), n_partials,
                c + 1 == n_chunks, (double)stddev_mul, stats);
            SPX_LAUNCH_CHECK();
        }
        q->arena_reset();
        q->arena_reserve((size_t)n * 8 + scan_scratch_elems(n) * 4 + 4096);
        uint32_t* flags = q->take<uint32_t>(n);
        uint32_t* pos = q->take<uint32_t>(n);
        uint32_t* scan_tmp = q->take<uint32_t>(scan_scratch_elems(n));
        uint32_t* total_dev = q->take<uint32_t>(16);
        sor_flag_kernel<<<div_up(n, OR_THREADS), OR_THREADS, 0, st>>>(mean, n, stats, flags);
        SPX_LAUNCH_CHECK();
        compact_and_count(q, flags, pos, scan_tmp, total_dev, n, idx_out, m_host);
    });
}

int spx_radius_outlier_indices(spx_index_t index, const float* points, size_t n_in, float radius, uint32_t min_neighbors,
                               int32_t* idx_out, size_t* m_host) {
    return guard([&] {
        SPX_REQUIRE(index && m_host, "[OutlierRemoval::radius] null argument");
        SPX_REQUIRE(n_in == index->n_total, "[OutlierRemoval::radius] the index was not built over these points");
        SPX_REQUIRE(std::isfinite(radius) && radius >= 0.0f, "[OutlierRemoval::radius] `radius` must be finite and >= 0");
        *m_host = 0;
        if (n_in == 0) return;
        SPX_REQUIRE(points && idx_out, "[OutlierRemoval::radius] null pointer");
        spx_queue_t q = index->q;
        DeviceGuard dg(q->device);
        cudaStream_t st = q->stream;
        const uint32_t n = (uint32_t)n_in;
        q->arena_reset();
        q->arena_reserve((size_t)n * 8 + scan_scratch_elems(n) * 4 + 4096);
        uint32_t* flags = q->take<uint32_t>(n);
        uint32_t* pos = q->take<uint32_t>(n);
        uint32_t* scan_tmp = q->take<uint32_t>(scan_scratch_elems(n));
        uint32_t* total_dev = q->take<uint32_t>(16);
        // (an index with no finite point: every finite query counts 0)
        const GridView g = radius_search_level(index->levels, radius);
        // r^2 as spx_index_radius computes it; the search reach gets a relative allowance for the rounding of the fp32
        // distance (a point counted at d^2 <= r^2 can lie a few ulps beyond r)
        const float r2 = radius * radius;
        const float reach = radius + radius * 1.0e-5f;
        if (index->n == 0 && min_neighbors > 0u) {
            SPX_CUDA(cudaMemsetAsync(flags, 0, (size_t)n * 4, st));
        } else {
            ror_flag_kernel<<<div_up(n, OR_THREADS), OR_THREADS, 0, st>>>(g, reinterpret_cast<const float4*>(points), n, reach,
                                                                          r2, min_neighbors, flags);
            SPX_LAUNCH_CHECK();
        }
        compact_and_count(q, flags, pos, scan_tmp, total_dev, n, idx_out, m_host);
    });
}

}  // extern "C"
