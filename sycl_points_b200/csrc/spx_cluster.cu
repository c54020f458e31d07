// Euclidean cluster extraction on the exact grid index (semantics of PCL's EuclideanClusterExtraction, pinned in
// DESIGN.md §3.4): the connected components of the graph that joins two finite points at d^2 <= t^2.
//
// Link: one thread per finite point i runs grid_search on ONE level (radius_search_level, as the radius outlier
// filter) with a policy that never stops early, and unions i with every j < i within t.  Union-find is lock-free
// over the original indices: a root is only ever linked below a smaller root, so the trees have no cycles and the
// final root of a component is its minimum index whatever order the unions ran in.  Flatten + an integer atomicAdd
// count the component sizes; a flag pass, the device scan and a compaction list the clusters that pass the size
// filter in root order (the call's one synchronisation, for C and the member count).  Two stable LSD radix sorts
// (spx_sort.cuh) then order the clusters by size descending (ties: root, i.e. smallest member, ascending) and the
// kept points by cluster, members ascending.  Every step is a pure function of the input: runs repeat bit for bit.
#include <cmath>

#include "spx_grid.cuh"
#include "spx_sort.cuh"

using namespace spx;

namespace {

constexpr int CL_THREADS = 256;

__device__ __forceinline__ bool finite3(const float4 p) { return isfinite(p.x) && isfinite(p.y) && isfinite(p.z); }

// Root of x with path halving.  parent[] is read and written through volatile accesses: other threads link roots and
// halve paths while this one walks, so no load may come from a non-coherent cache.  Writing the grandparent is always
// safe, since an ancestor of x stays one.
__device__ __forceinline__ int uf_find(volatile int* parent, int x) {
    int p = parent[x];
    while (p != x) {
        const int g = parent[p];
        if (g == p) return p;
        parent[x] = g;
        x = g;
        p = parent[x];
    }
    return x;
}

// Joins the trees of a and b: the larger root is CAS-linked below the smaller one.  A failed CAS means that root has
// just been linked elsewhere; both roots are found again and the join retried.
__device__ __forceinline__ void uf_union(int* parent, int a, int b) {
    volatile int* vp = parent;
    for (;;) {
        a = uf_find(vp, a);
        b = uf_find(vp, b);
        if (a == b) return;  // in a dense region almost every pair is already joined: no CAS
        const int hi = max(a, b), lo = min(a, b);
        const int old = atomicCAS(parent + hi, hi, lo);
        if (old == hi) return;
        a = old;
        b = lo;
    }
}

// grid_search policy: worst() stays at FLT_MAX (no early stop), so every point within the search reach is offered.
// Each edge is joined once, from its higher endpoint.  That sees every edge because the fp32 chain
// fma(dz,dz,fma(dy,dy,dx*dx)) is bitwise symmetric in i and j: (-d)^2 == d^2 exactly, so d^2(i, j) == d^2(j, i).
struct UnionWithin {
    float t2;
    int self;
    int* parent;
    __device__ __forceinline__ float worst() const { return FLT_MAX; }
    __device__ __forceinline__ void offer(float ds, int idx, uint32_t) {
        if (idx < self && ds <= t2) uf_union(parent, self, idx);
    }
};

// parent[i] = i for finite points, -1 for the others (they belong to no cluster); sizes zeroed
__global__ void __launch_bounds__(CL_THREADS) cl_init_kernel(const float4* __restrict__ pts, uint32_t n,
                                                             int* __restrict__ parent, uint32_t* __restrict__ size) {
    const uint32_t i = blockIdx.x * CL_THREADS + threadIdx.x;
    if (i >= n) return;
    parent[i] = finite3(__ldg(pts + i)) ? (int)i : -1;
    size[i] = 0u;
}

__global__ void __launch_bounds__(CL_THREADS) cl_link_kernel(const GridView g, const float4* __restrict__ pts, uint32_t n,
                                                             float reach, float t2, int* parent) {
    const uint32_t i = blockIdx.x * CL_THREADS + threadIdx.x;
    if (i >= n) return;
    const float4 p = __ldg(pts + i);
    if (!finite3(p)) return;
    UnionWithin u{t2, (int)i, parent};
    // r_begin 1: the first pass is the 3x3x3 block; the search ends once everything within `reach` has been seen
    grid_search(g, p.x, p.y, p.z, u, reach, 1, 1 << 20);
}

// root[i] = root of i (-1 for non-finite points); size[root] counts the component.  The roots go to their own array:
// other threads still halve paths through parent[i] while this one walks, and such a write can replace a root just
// stored in parent[i] by an ancestor that is not the root.
__global__ void __launch_bounds__(CL_THREADS) cl_flatten_kernel(uint32_t n, int* parent, int* __restrict__ root,
                                                                uint32_t* __restrict__ size) {
    const uint32_t i = blockIdx.x * CL_THREADS + threadIdx.x;
    if (i >= n) return;
    volatile int* vp = parent;
    const int r = vp[i] < 0 ? -1 : uf_find(vp, (int)i);
    root[i] = r;
    if (r >= 0) atomicAdd(size + r, 1u);
}

// flags[i] = 1 for the roots whose component passes the size filter; counters[0] += their sizes (the member count)
__global__ void __launch_bounds__(CL_THREADS) cl_select_kernel(uint32_t n, const int* __restrict__ root,
                                                               const uint32_t* __restrict__ size, uint32_t min_size,
                                                               uint32_t max_size, uint32_t* __restrict__ flags,
                                                               uint32_t* __restrict__ counters) {
    const uint32_t i = blockIdx.x * CL_THREADS + threadIdx.x;
    uint32_t keep = 0u, members = 0u;
    if (i < n) {
        const uint32_t s = size[i];
        keep = (root[i] == (int)i && s >= min_size && s <= max_size) ? 1u : 0u;
        members = keep ? s : 0u;
        flags[i] = keep;
    }
    members = __reduce_add_sync(0xffffffffu, members);
    if ((threadIdx.x & 31) == 0 && members) atomicAdd(counters, members);
}

// the kept roots in ascending order, keyed by n - size (ascending key = descending size)
__global__ void __launch_bounds__(CL_THREADS) cl_root_compact_kernel(const uint32_t* __restrict__ flags,
                                                                     const uint32_t* __restrict__ pos,
                                                                     const uint32_t* __restrict__ size, uint32_t n,
                                                                     uint32_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    const uint32_t i = blockIdx.x * CL_THREADS + threadIdx.x;
    if (i >= n || !flags[i]) return;
    keys[pos[i]] = n - size[i];
    vals[pos[i]] = i;
}

// cluster c = the c-th sorted root: rank[root] = c, sizes[c] = its size
__global__ void __launch_bounds__(CL_THREADS) cl_rank_kernel(uint32_t c_count, uint32_t n, const uint32_t* __restrict__ keys,
                                                             const uint32_t* __restrict__ roots, uint32_t* __restrict__ rank,
                                                             uint32_t* __restrict__ sizes) {
    const uint32_t c = blockIdx.x * CL_THREADS + threadIdx.x;
    if (c >= c_count) return;
    rank[roots[c]] = c;
    sizes[c] = n - keys[c];
}

// labels[i] = rank of i's cluster or -1; keep[i] = labels[i] >= 0
__global__ void __launch_bounds__(CL_THREADS) cl_label_kernel(uint32_t n, const int* __restrict__ root,
                                                              const uint32_t* __restrict__ flags,
                                                              const uint32_t* __restrict__ rank, int32_t* __restrict__ labels,
                                                              uint32_t* __restrict__ keep) {
    const uint32_t i = blockIdx.x * CL_THREADS + threadIdx.x;
    if (i >= n) return;
    const int r = root[i];
    const int32_t lab = (r >= 0 && flags[r]) ? (int32_t)rank[r] : -1;
    labels[i] = lab;
    keep[i] = lab >= 0 ? 1u : 0u;
}

// the kept points in ascending index order, keyed by their label
__global__ void __launch_bounds__(CL_THREADS) cl_member_compact_kernel(const uint32_t* __restrict__ keep,
                                                                       const uint32_t* __restrict__ pos,
                                                                       const int32_t* __restrict__ labels, uint32_t n,
                                                                       uint32_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    const uint32_t i = blockIdx.x * CL_THREADS + threadIdx.x;
    if (i >= n || !keep[i]) return;
    keys[pos[i]] = (uint32_t)labels[i];
    vals[pos[i]] = i;
}

int radix_passes(unsigned long long max_key) { return std::max(1, (bits_for(max_key) + RADIX_BITS - 1) / RADIX_BITS); }

}  // namespace

extern "C" {

int spx_euclidean_clusters(spx_index_t index, const float* points, size_t n_in, float tolerance, uint32_t min_cluster_size,
                           uint32_t max_cluster_size, int32_t* labels_out, int32_t* indices_out, uint32_t* offsets_out,
                           size_t* n_clusters_host, size_t* n_members_host) {
    return guard([&] {
        SPX_REQUIRE(index && n_clusters_host && n_members_host, "[EuclideanClustering] null argument");
        SPX_REQUIRE(n_in == index->n_total, "[EuclideanClustering] the index was not built over these points");
        SPX_REQUIRE(n_in < (1ull << 31), "[EuclideanClustering] at most 2^31 - 1 points");
        SPX_REQUIRE(std::isfinite(tolerance) && tolerance >= 0.0f, "[EuclideanClustering] `tolerance` must be finite and >= 0");
        SPX_REQUIRE(min_cluster_size >= 1u && min_cluster_size <= max_cluster_size,
                    "[EuclideanClustering] need 1 <= min_cluster_size <= max_cluster_size");
        *n_clusters_host = 0;
        *n_members_host = 0;
        if (n_in == 0) return;
        SPX_REQUIRE(points && indices_out && offsets_out, "[EuclideanClustering] null pointer");
        spx_queue_t q = index->q;
        DeviceGuard dg(q->device);
        cudaStream_t st = q->stream;
        const uint32_t n = (uint32_t)n_in;
        const size_t words = align_up(n, 64);
        q->arena_reset();
        q->arena_reserve((11 * words + scan_scratch_elems(n) + radix_sort_scratch_elems(n) + 64) * 4 + 16 * 256);
        int* parent = q->take<int>(n);
        int* root = q->take<int>(n);
        uint32_t* size = q->take<uint32_t>(n);
        uint32_t* flags = q->take<uint32_t>(n);
        uint32_t* pos = q->take<uint32_t>(n);
        uint32_t* keep = q->take<uint32_t>(n);
        int32_t* labels = labels_out ? labels_out : q->take<int32_t>(n);
        uint32_t* keys_a = q->take<uint32_t>(n);
        uint32_t* keys_b = q->take<uint32_t>(n);
        uint32_t* vals_in = q->take<uint32_t>(n);
        uint32_t* vals_tmp = q->take<uint32_t>(n);
        uint32_t* scan_tmp = q->take<uint32_t>(scan_scratch_elems(n));
        uint32_t* sort_tmp = q->take<uint32_t>(radix_sort_scratch_elems(n));
        uint32_t* counters = q->take<uint32_t>(16);  // {members, clusters}
        const float4* pts = reinterpret_cast<const float4*>(points);
        const int blocks = div_up(n, CL_THREADS);

        // t^2 as spx_radius_outlier_indices computes it; the reach allows for the rounding of the fp32 distance
        const float t2 = tolerance * tolerance;
        const float reach = tolerance + tolerance * 1.0e-5f;
        SPX_CUDA(cudaMemsetAsync(counters, 0, 16 * 4, st));
        cl_init_kernel<<<blocks, CL_THREADS, 0, st>>>(pts, n, parent, size);
        SPX_LAUNCH_CHECK();
        cl_link_kernel<<<blocks, CL_THREADS, 0, st>>>(radius_search_level(index->levels, tolerance), pts, n, reach, t2,
                                                      parent);
        SPX_LAUNCH_CHECK();
        cl_flatten_kernel<<<blocks, CL_THREADS, 0, st>>>(n, parent, root, size);
        SPX_LAUNCH_CHECK();
        cl_select_kernel<<<blocks, CL_THREADS, 0, st>>>(n, root, size, min_cluster_size, max_cluster_size, flags,
                                                        counters);
        SPX_LAUNCH_CHECK();
        exclusive_scan_u32(st, flags, pos, n, scan_tmp, counters + 1);
        cl_root_compact_kernel<<<blocks, CL_THREADS, 0, st>>>(flags, pos, size, n, keys_a, vals_in);
        SPX_LAUNCH_CHECK();
        uint32_t* hcount = static_cast<uint32_t*>(q->pinned_get(64));
        SPX_CUDA(cudaMemcpyAsync(hcount, counters, 8, cudaMemcpyDeviceToHost, st));
        q->sync();
        const uint32_t n_members = hcount[0], n_clusters = hcount[1];

        if (n_clusters == 0) {
            SPX_CUDA(cudaMemsetAsync(offsets_out, 0, 4, st));
            SPX_CUDA(cudaMemsetAsync(labels, 0xff, (size_t)n * 4, st));  // (all-ones bits: -1)
        } else {
            // clusters by n - size: stable, so equal sizes keep root (= smallest member) order
            const int rp = radix_passes(n - min_cluster_size);
            uint32_t* const rkeys[2] = {keys_a, keys_b};
            uint32_t* const rvals[2] = {vals_tmp, keep};
            radix_sort_pairs<uint32_t>(st, n_clusters, rp, rkeys, vals_in, rvals, sort_tmp);
            uint32_t* sizes = vals_in;  // (free again)
            cl_rank_kernel<<<div_up(n_clusters, CL_THREADS), CL_THREADS, 0, st>>>(n_clusters, n, rkeys[rp & 1],
                                                                                  rvals[(rp - 1) & 1], pos, sizes);
            SPX_LAUNCH_CHECK();
            exclusive_scan_u32(st, sizes, offsets_out, n_clusters, scan_tmp, offsets_out + n_clusters);
            cl_label_kernel<<<blocks, CL_THREADS, 0, st>>>(n, root, flags, pos, labels, keep);
            SPX_LAUNCH_CHECK();
            uint32_t* mpos = size;  // (free again)
            exclusive_scan_u32(st, keep, mpos, n, scan_tmp, nullptr);
            cl_member_compact_kernel<<<blocks, CL_THREADS, 0, st>>>(keep, mpos, labels, n, keys_a, vals_in);
            SPX_LAUNCH_CHECK();
            // members by label: stable, so each cluster's members stay ascending; the last pass writes indices_out
            const int mp = radix_passes(n_clusters - 1);
            uint32_t* const mvals[2] = {(mp & 1) ? reinterpret_cast<uint32_t*>(indices_out) : vals_tmp,
                                        (mp & 1) ? vals_tmp : reinterpret_cast<uint32_t*>(indices_out)};
            radix_sort_pairs<uint32_t>(st, n_members, mp, rkeys, vals_in, mvals, sort_tmp);
        }
        *n_clusters_host = n_clusters;
        *n_members_host = n_members;
    });
}

}  // extern "C"
