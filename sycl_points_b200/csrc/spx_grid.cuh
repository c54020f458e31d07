// Device-side view of the exact nearest-neighbour index (uniform cell grid, points counting-
// sorted by cell) and the ring search over it.  Shared by the KNN entry points (spx_knn.cu) and
// the fused nearest-neighbour + linearise kernels (spx_registration.cu).
//
// Exactness argument (DESIGN.md §index): cells are visited in Chebyshev shells r = 0,1,2,...
// around the query's (clamped) cell c.  Every point NOT yet visited after shell r lies in a cell
// whose index differs from c by more than r on some axis a, so |p_a - q_a| >= gap_a(r), the
// distance from q_a to the slab [o_a + (c_a-r) h, o_a + (c_a+r+1) h] (infinite on a side where the
// slab already touches the grid boundary: there are no cells, hence no points, beyond it).  The
// fp32 distance fma(dz,dz,fma(dy,dy,dx*dx)) is monotone in each |d_a|, so every unvisited point
// has dist >= (min_a gap_a(r))^2 up to rounding; the search stops once the current k-th best is
// STRICTLY below (bound - margin)^2, margin covering the rounding of cell assignment and of the
// slab coordinates.  Strictness + the (dist, index) insertion order make ties resolve to the
// lowest index no matter in which order cells are visited — the brute-force contract.
#pragma once

#include "spx_common.cuh"

namespace spx {

constexpr int GRID_MAX_LEVELS = 6;
constexpr int GRID_LEVEL_FACTOR = 4;   // cell edge ratio between consecutive levels
constexpr int GRID_LEVEL_RINGS = 2;    // shells (beyond the query's own cell) searched on a level before moving
                                       // to the next coarser one: empty space is crossed in coarse steps, so a
                                       // query with nothing nearby costs a few dozen row look-ups per level

struct GridView {
    float ox, oy, oz;    // grid origin (bbox min of the indexed points)
    float cell, inv;     // cell edge and its reciprocal
    float margin;        // slab-coordinate / cell-assignment rounding allowance
    int dx, dy, dz;      // grid dimensions
    const uint32_t* __restrict__ start;  // [dx*dy*dz + 1] first sorted position of each cell
    const float4* __restrict__ pts;      // sorted points, w = original index (int bits)
    uint32_t n;                          // indexed (finite) points
};

// LiDAR clouds span three orders of magnitude in density (ground rings metres apart at range,
// centimetres near the sensor), so one cell size cannot serve every query: the index keeps up to
// GRID_MAX_LEVELS independent grids over the same points, each GRID_LEVEL_FACTOR coarser than the
// previous one.  A query runs the ring search on the finest level for a few shells and, if the stop
// bound has not been met, starts over on the next level (the candidate list carries over; re-offered
// points are recognised by their index).  The coarsest level is searched until its whole grid has
// been seen, so every query terminates with the exact answer and no brute-force pass is needed.
struct GridLevels {
    int n_levels;
    GridView lv[GRID_MAX_LEVELS];
};

// The one level a fixed-radius search (radius outlier removal, Euclidean clustering) runs on: the finest whose cell
// edge is at least radius / 2 (at most three shells), else the coarsest.  An index with no finite point has a 1-cell
// level 0 and no points.
inline GridView radius_search_level(const GridLevels& L, float radius) {
    for (int l = 0; l < L.n_levels; ++l)
        if (L.lv[l].cell * 2.0f >= radius) return L.lv[l];
    return L.lv[L.n_levels - 1];
}

#ifdef __CUDACC__

__device__ __forceinline__ int grid_coord(float q, float o, float inv, int dim) {
    // identical expression for build and query: floor((q - o) * inv), clamped into the grid
    float g = floorf(__fmul_rn(__fsub_rn(q, o), inv));
    g = fminf(fmaxf(g, 0.0f), (float)(dim - 1));
    return (int)g;
}

// distance from q to the slab of cell index ci on one axis (0 inside); >= 0.  The two boundary cells of an axis also
// hold the points that lie BEYOND the grid on their side (cell coordinates clamp), so their slabs extend to
// infinity outward: a query outside the grid must not be told that the boundary cell is far away.
__device__ __forceinline__ float axis_gap(float q, float o, float cell, int ci, int dim) {
    const float INF = __int_as_float(0x7f800000);
    const float lo = ci > 0 ? __fmaf_rn((float)ci, cell, o) : -INF;
    const float hi = ci < dim - 1 ? __fmaf_rn((float)(ci + 1), cell, o) : INF;
    return fmaxf(fmaxf(lo - q, q - hi), 0.0f);
}

// Lower bound on |p_a - q_a| for points in cells farther than r from c on axis a (see header).
__device__ __forceinline__ float shell_bound_axis(float q, float o, float cell, int c, int r, int dim) {
    const float INF = __int_as_float(0x7f800000);
    const float lo = (c - r > 0) ? q - __fmaf_rn((float)(c - r), cell, o) : INF;
    const float hi = (c + r < dim - 1) ? __fmaf_rn((float)(c + r + 1), cell, o) - q : INF;
    return fminf(lo, hi);
}

// One candidate list per thread.  K1: a register pair.  General k: the thread's row of the output
// arrays (global memory, L1/L2-resident; touched only on insertion, which is rare once warm).
struct Best1 {
    static constexpr bool MARGIN = false;
    float d;
    int i;      // original index
    __device__ __forceinline__ void init() { d = FLT_MAX; i = -1; }
    __device__ __forceinline__ float worst() const { return d; }
    __device__ __forceinline__ void offer(float ds, int idx, uint32_t) {
        if (ds < d || (ds == d && (i < 0 || idx < i))) { d = ds; i = idx; }
    }
};

// Best1 + what the ICP loop's keep test needs (spx_registration.cu): a lower bound on the distance of every OTHER
// target point.  d2 = smallest squared distance among the other points the search looked at and among the pruning
// bounds it applied (a cell or row left out because it lies beyond sqrt(lim2) counts as a point at lim2); u = the
// radius (metres) the last block scanned certifies — nothing unseen lies closer.  min(sqrt(d2), u) - sqrt(d) is how
// far apart the nearest and the second nearest are at least: a query that moves by less than half of that keeps its
// correspondence, bit for bit what a new search would return.  A point met twice (the warm start inside the block,
// or on two levels) is recognised by its index.
struct Best1M {
    static constexpr bool MARGIN = true;
    float d;
    int i;
    float d2;
    float u;
    __device__ __forceinline__ void init() { d = FLT_MAX; i = -1; d2 = FLT_MAX; u = 0.0f; }
    __device__ __forceinline__ float worst() const { return d; }
    __device__ __forceinline__ void offer(float ds, int idx, uint32_t) {
        const bool other = idx != i;
        const bool better = other && (ds < d || (ds == d && (i < 0 || idx < i)));
        d2 = better ? d : (other ? fminf(d2, ds) : d2);
        d = better ? ds : d;
        i = better ? idx : i;
    }
};

struct BestK {
    float* d;   // element j at d[j * stride]
    int* i;
    int k;
    int stride;
    float wd;   // cached k-th best
    int wi;
    __device__ __forceinline__ void init() {
        for (int j = 0; j < k; ++j) { d[j * stride] = FLT_MAX; i[j * stride] = -1; }
        wd = FLT_MAX; wi = -1;
    }
    __device__ __forceinline__ float worst() const { return wd; }
    __device__ __forceinline__ void offer(float ds, int idx, uint32_t) {
        if (!lex_less(ds, idx, wd, wi)) return;
        int pos = k - 1;
        while (pos > 0 && lex_less(ds, idx, d[(pos - 1) * stride], i[(pos - 1) * stride])) --pos;
        // the same point offered again by a coarser level lands right behind its own entry
        if (pos > 0 && i[(pos - 1) * stride] == idx) return;
        for (int j = k - 1; j > pos; --j) {
            d[j * stride] = d[(j - 1) * stride];
            i[j * stride] = i[(j - 1) * stride];
        }
        d[pos * stride] = ds;
        i[pos * stride] = idx;
        wd = d[(k - 1) * stride];
        wi = i[(k - 1) * stride];
    }
};

// Small k (<= K): the sorted candidate list lives in REGISTERS as packed 64-bit keys
//   key = ((dist bits) << 32 | index) + 1          (dist >= 0, so its bits order like the value;
//                                                   the index in the low word breaks ties -> (dist, index))
// and an insertion is K predicated compare-exchanges — no memory traffic, no data-dependent loop, so
// lanes of a warp never diverge inside it.  Lists shorter than K are padded at the FRONT with key 0
// (below every real key), which keeps the k-th best in the fixed register key[K-1].
template <int K>
struct BestR {
    unsigned long long key[K];
    bool dedup;  // a coarser level re-offers points the finer one has already seen
    static constexpr unsigned long long EMPTY = ((0x7f7fffffull << 32) | 0xffffffffull) + 1ull;  // FLT_MAX, -1
    __device__ __forceinline__ void init(int k) {
#pragma unroll
        for (int j = 0; j < K; ++j) key[j] = (j < K - k) ? 0ull : EMPTY;
        dedup = false;
    }
    __device__ __forceinline__ float worst() const { return __uint_as_float((uint32_t)((key[K - 1] - 1ull) >> 32)); }
    __device__ __forceinline__ void offer(float ds, int idx, uint32_t) {
        unsigned long long c = (((unsigned long long)__float_as_uint(ds) << 32) | (unsigned long long)(uint32_t)idx) + 1ull;
        if (c >= key[K - 1]) return;
        if (dedup) {  // rare path (levels >= 1): is this exact (dist, index) already listed?
            bool seen = false;
#pragma unroll
            for (int j = 0; j < K; ++j) seen |= (c == key[j]);
            if (seen) return;
        }
        // K compare-exchanges, 2 ISETP + 4 SEL each: the new key sinks to its place, the old k-th falls off
#pragma unroll
        for (int j = 0; j < K; ++j) {
            const bool lt = c < key[j];
            const unsigned long long lo = lt ? c : key[j];
            const unsigned long long hi = lt ? key[j] : c;
            key[j] = lo;
            c = hi;
        }
    }
    __device__ __forceinline__ float dist_at(int j) const { return __uint_as_float((uint32_t)((key[j] - 1ull) >> 32)); }
    __device__ __forceinline__ int idx_at(int j) const { return (int)(uint32_t)((key[j] - 1ull) & 0xffffffffull); }
};

template <typename Best>
__device__ __forceinline__ void best_set_dedup(Best&, bool) {}
template <int K>
__device__ __forceinline__ void best_set_dedup(BestR<K>& b, bool v) { b.dedup = v; }

constexpr int GRID_SEG_CHUNK = 9;  // the merged first pass (3x3 rows) fits one chunk
constexpr int GRID_BATCH = 4;  // candidate loads in flight per thread

// optional per-query work counters (spx_index_knn_stats, used to tune the index); the default
// policy compiles to nothing
struct NoStats {
    __device__ __forceinline__ void segment(uint32_t) {}
    __device__ __forceinline__ void shell() {}
    __device__ __forceinline__ void level(int) {}
};
struct CountStats {
    uint32_t segs = 0, cands = 0, shells = 0, last_level = 0;
    __device__ __forceinline__ void segment(uint32_t n) { ++segs; cands += n; }
    __device__ __forceinline__ void shell() { ++shells; }
    __device__ __forceinline__ void level(int l) { last_level = l; }
};

// Ring search.  max_radius: stop expanding once every point within it has been seen (ICP use:
// correspondences farther than max_correspondence_distance are rejected anyway,
// registration.hpp:584); pass +inf for an unbounded exact search.  r_max: shells after which an
// unbounded search gives up (returns false -> caller falls back to a full scan).
template <typename Best, typename Stats = NoStats>
__device__ __forceinline__ bool grid_search(const GridView& g, float qx, float qy, float qz, Best& best, float max_radius,
                                         int r_begin, int r_max, Stats* stats = nullptr) {
    const int cx = grid_coord(qx, g.ox, g.inv, g.dx);
    const int cy = grid_coord(qy, g.oy, g.inv, g.dy);
    const int cz = grid_coord(qz, g.oz, g.inv, g.dz);
    const float INF = __int_as_float(0x7f800000);
    // rounding allowance: grid part (build) + the query's own magnitude (q - slab coordinate)
    const float margin = g.margin + 1e-6f * fmaxf(fmaxf(fabsf(qx), fabsf(qy)), fabsf(qz));
    // bounded searches never need anything beyond max_radius (+ allowance): prune against it too
    const float reach = max_radius + margin;
    const float reach2 = reach < 1.8e19f ? __fmul_rn(reach, reach) : INF;

    uint32_t seg_lo[GRID_SEG_CHUNK], seg_hi[GRID_SEG_CHUNK];
    int nseg = 0;

    // Two-phase processing of up to GRID_SEG_CHUNK cell ranges: (1) all `start` look-ups are issued
    // back to back, (2) the candidate points of ALL ranges are walked as one flat stream in batches
    // of GRID_BATCH loads issued before any distance is evaluated.  A query's time is a chain of
    // L2 round trips, so the number of dependent trips — not the arithmetic — is what is minimised.
    auto flush = [&]() {
        uint32_t ls[GRID_SEG_CHUNK], le[GRID_SEG_CHUNK];
#pragma unroll
        for (int t = 0; t < GRID_SEG_CHUNK; ++t) {
            uint32_t a = 0, b = 0;
            if (t < nseg) {
                a = __ldg(g.start + seg_lo[t]);
                b = __ldg(g.start + seg_hi[t] + 1);
            }
            ls[t] = a;
            le[t] = b;
        }
        int t = 0;
        uint32_t j = ls[0], end = le[0];
        if (stats)
            for (int u = 0; u < nseg; ++u) stats->segment(le[u] - ls[u]);
        while (t < nseg) {
            uint32_t addr[GRID_BATCH];
            float4 p[GRID_BATCH];
#pragma unroll
            for (int u = 0; u < GRID_BATCH; ++u) {
                while (t < nseg && j >= end) {
                    ++t;
                    if (t < nseg) {
                        j = ls[t];
                        end = le[t];
                    }
                }
                addr[u] = 0xffffffffu;
                if (t < nseg) addr[u] = j++;
            }
#pragma unroll
            for (int u = 0; u < GRID_BATCH; ++u)
                if (addr[u] != 0xffffffffu) p[u] = __ldg(g.pts + addr[u]);
#pragma unroll
            for (int u = 0; u < GRID_BATCH; ++u)
                if (addr[u] != 0xffffffffu)
                    best.offer(dist_sq(qx, qy, qz, p[u].x, p[u].y, p[u].z), __float_as_int(p[u].w), addr[u]);
        }
        nseg = 0;
    };

    // The first pass covers shells 0 and 1 together (the 3x3 block of rows around the query's cell,
    // each row one contiguous range of 3 cells): for the dense part of a cloud that is the whole
    // search, with a fixed trip count and no pruning arithmetic.  Later passes add one shell each
    // and prune rows / trim their x range against the best distance known so far.
    for (int r = r_begin;; ++r) {
        const bool merged = (r == 1);
        const int z0 = max(cz - r, 0), z1 = min(cz + r, g.dz - 1);
        const int y0 = max(cy - r, 0), y1 = min(cy + r, g.dy - 1);
        for (int zz = z0; zz <= z1; ++zz) {
            const bool ez = (zz - cz == r) || (cz - zz == r);
            for (int yy = y0; yy <= y1; ++yy) {
                const bool edge = merged || ez || (yy - cy == r) || (cy - yy == r);
                int xa = max(cx - r, 0), xb = min(cx + r, g.dx - 1);
                const float lim2 = fminf(best.worst(), reach2);
                if (lim2 < 1.0e30f) {
                    // prune rows that cannot hold anything better than the current k-th best, and
                    // cells of the row farther along x than sqrt(lim2 - gap^2) (+ allowance)
                    const float gz = axis_gap(qz, g.oz, g.cell, zz, g.dz);
                    const float gy = axis_gap(qy, g.oy, g.cell, yy, g.dy);
                    const float gyz = fmaxf(sqrtf(__fmaf_rn(gz, gz, __fmul_rn(gy, gy))) - margin, 0.0f);
                    const float gyz2 = __fmul_rn(gyz, gyz);
                    if (gyz2 > lim2) continue;
                    const float w = sqrtf(lim2 - gyz2) + margin;
                    xa = max(xa, grid_coord(qx - w, g.ox, g.inv, g.dx));
                    xb = min(xb, grid_coord(qx + w, g.ox, g.inv, g.dx));
                    if (xa > xb) continue;
                }
                const uint32_t row = ((uint32_t)zz * (uint32_t)g.dy + (uint32_t)yy) * (uint32_t)g.dx;
                if (edge) {
                    seg_lo[nseg] = row + xa;
                    seg_hi[nseg] = row + xb;
                    if (++nseg == GRID_SEG_CHUNK) flush();
                } else {
                    // interior row of a later shell: only the two end cells are new
                    if (cx - r >= xa) {
                        seg_lo[nseg] = seg_hi[nseg] = row + (cx - r);
                        if (++nseg == GRID_SEG_CHUNK) flush();
                    }
                    if (cx + r <= xb) {
                        seg_lo[nseg] = seg_hi[nseg] = row + (cx + r);
                        if (++nseg == GRID_SEG_CHUNK) flush();
                    }
                }
            }
        }
        if (nseg) flush();
        if (stats) stats->shell();

        const float bound = fminf(fminf(shell_bound_axis(qx, g.ox, g.cell, cx, r, g.dx),
                                        shell_bound_axis(qy, g.oy, g.cell, cy, r, g.dy)),
                                  shell_bound_axis(qz, g.oz, g.cell, cz, r, g.dz));
        if (bound == INF) return true;  // whole grid visited
        const float bs = bound - margin;
        if (bs > 0.0f && best.worst() < __fmul_rn(bs, bs)) return true;
        if (bs >= max_radius) return true;  // everything within max_radius has been seen
        if (r >= r_max) return false;
    }
}

// First pass on the finest level: the 3x3x3 block of cells around the query's cell, i.e. 9 rows of
// 3 contiguous cells.  No pruning arithmetic, fixed trip counts, all 18 `start` look-ups issued at
// once; for queries inside the dense part of a cloud this is the entire search.  Returns true when
// the stop bound of shell 1 is already met.
template <typename Best, typename Stats = NoStats>
__device__ __forceinline__ bool grid_first_pass(const GridView& g, float qx, float qy, float qz, Best& best,
                                                float max_radius, Stats* stats = nullptr) {
    const int cx = grid_coord(qx, g.ox, g.inv, g.dx);
    const int cy = grid_coord(qy, g.oy, g.inv, g.dy);
    const int cz = grid_coord(qz, g.oz, g.inv, g.dz);
    const int xa = max(cx - 1, 0), xb = min(cx + 1, g.dx - 1);
    uint32_t ls[9], le[9];
    // rows in order of proximity (the query's own row, the four edge neighbours, the four corners):
    // the k-th best tightens early and most later candidates are rejected by one compare
    constexpr int ORDER[9] = {4, 1, 3, 5, 7, 0, 2, 6, 8};
#pragma unroll
    for (int s = 0; s < 9; ++s) {
        const int t = ORDER[s];
        const int zz = cz + (t / 3) - 1, yy = cy + (t % 3) - 1;
        const bool ok = zz >= 0 && zz < g.dz && yy >= 0 && yy < g.dy;
        const uint32_t row = ((uint32_t)zz * (uint32_t)g.dy + (uint32_t)yy) * (uint32_t)g.dx;
        ls[s] = ok ? __ldg(g.start + row + xa) : 0u;
        le[s] = ok ? __ldg(g.start + row + xb + 1) : 0u;
    }
#pragma unroll
    for (int t = 0; t < 9; ++t) {
        if (stats) stats->segment(le[t] - ls[t]);
        for (uint32_t j = ls[t]; j < le[t]; j += 4) {
            float4 p[4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (j + u < le[t]) p[u] = __ldg(g.pts + j + u);
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (j + u < le[t])
                    best.offer(dist_sq(qx, qy, qz, p[u].x, p[u].y, p[u].z), __float_as_int(p[u].w), j + u);
        }
    }
    if (stats) stats->shell();
    const float INF = __int_as_float(0x7f800000);
    const float margin = g.margin + 1e-6f * fmaxf(fmaxf(fabsf(qx), fabsf(qy)), fabsf(qz));
    const float bound = fminf(fminf(shell_bound_axis(qx, g.ox, g.cell, cx, 1, g.dx),
                                    shell_bound_axis(qy, g.oy, g.cell, cy, 1, g.dy)),
                              shell_bound_axis(qz, g.oz, g.cell, cz, 1, g.dz));
    if (bound == INF) return true;
    const float bs = bound - margin;
    return (bs > 0.0f && best.worst() < __fmul_rn(bs, bs)) || bs >= max_radius;
}

// Exact search over the level hierarchy (see GridLevels).  With level_limit >= n_levels it always
// terminates with the full answer (returns true); with a smaller limit it gives up after the last
// allowed level's shells and returns false (the caller hands the query to a heavier path).
template <typename Best, typename Stats = NoStats>
__device__ __forceinline__ bool grid_search_levels(const GridLevels& g, float qx, float qy, float qz, Best& best,
                                                   float max_radius, Stats* stats = nullptr,
                                                   int level_limit = GRID_MAX_LEVELS, bool first_pass_done = false,
                                                   int rings0 = GRID_LEVEL_RINGS) {
    if (stats) stats->level(0);
    // first_pass_done: `best` already holds the outcome of an unsuccessful first pass (another kernel ran it)
    if (!first_pass_done && grid_first_pass(g.lv[0], qx, qy, qz, best, max_radius, stats)) return true;
    const int nl = min(g.n_levels, level_limit);
    for (int l = 0; l < nl; ++l) {
        const bool last = (l == g.n_levels - 1);
        if (l == 1) best_set_dedup(best, true);
        if (stats) stats->level(l);
        if (grid_search(g.lv[l], qx, qy, qz, best, max_radius, l == 0 ? 2 : 1,
                        last ? (1 << 20) : (l == 0 ? rings0 : GRID_LEVEL_RINGS), stats))
            return true;
    }
    return false;
}

// ---- warp-cooperative k-NN for the rare queries whose k-th neighbour is far away (isolated
// points: a scan edge, a bird).  One query per warp.  Rows of a shell are enumerated uniformly, the
// candidates of a row are taken with stride 32, every lane keeps its own register list, and the
// warp-wide k-th best — the pruning / stopping bound — comes from a k-round merge of the 32 lists
// after every shell.  A single lane walking tens of thousands of candidates on the coarse levels
// was a 0.4 ms tail on a 0.17 ms kernel.
template <int K>
__device__ __forceinline__ unsigned long long warp_merge_topk(const BestR<K>& mine, int k, unsigned long long* out /*[K] or null*/) {
    const unsigned FULL = 0xffffffffu;
    unsigned long long cur[K];
#pragma unroll
    for (int j = 0; j < K; ++j) cur[j] = mine.key[j];
    unsigned long long kth = BestR<K>::EMPTY;
    for (int t = 0; t < k; ++t) {
        // the lane's smallest unconsumed real entry sits at slot K - k (front padding is key 0)
        unsigned long long h = BestR<K>::EMPTY;
#pragma unroll
        for (int j = 0; j < K; ++j)
            if (j == K - k) h = cur[j];
        unsigned long long m = h;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long v = __shfl_xor_sync(FULL, m, o);
            m = v < m ? v : m;
        }
        if (h == m && m != BestR<K>::EMPTY) {  // every lane holding this exact (dist, index) pops it: duplicates vanish
#pragma unroll
            for (int j = 0; j < K - 1; ++j)
                if (j >= K - k) cur[j] = cur[j + 1];
            cur[K - 1] = BestR<K>::EMPTY;
        }
        if (out) {
#pragma unroll
            for (int j = 0; j < K; ++j)
                if (j == K - k + t) out[j] = m;
        }
        kth = m;
    }
    return kth;
}

template <int K>
static __device__ __noinline__ void knn_coop_search(const GridLevels& gl, float qx, float qy, float qz, int k,
                                                    int32_t* __restrict__ irow, float* __restrict__ drow) {
    const int lane = threadIdx.x & 31;
    const float INF = __int_as_float(0x7f800000);
    BestR<K> mine;
    mine.init(k);
    mine.dedup = true;
    float kth_d = FLT_MAX;  // warp-wide k-th best squared distance so far
    bool done = false;
    for (int l = 0; l < gl.n_levels && !done; ++l) {
        const GridView& g = gl.lv[l];
        const bool last = (l == gl.n_levels - 1);
        const int cx = grid_coord(qx, g.ox, g.inv, g.dx);
        const int cy = grid_coord(qy, g.oy, g.inv, g.dy);
        const int cz = grid_coord(qz, g.oz, g.inv, g.dz);
        const float margin = g.margin + 1e-6f * fmaxf(fmaxf(fabsf(qx), fabsf(qy)), fabsf(qz));
        // more shells per level than the per-lane searches take: a shell here costs one or two round trips
        // when it is empty, while the next level's first block scans every point of 27 cells 4x the size
        const int r_max = last ? (1 << 20) : 4;
        for (int r = 1;; ++r) {
            const bool merged = (r == 1);
            const int z0 = max(cz - r, 0), z1 = min(cz + r, g.dz - 1);
            const int y0 = max(cy - r, 0), y1 = min(cy + r, g.dy - 1);
            // 32 rows (z, y) of the shell at a time: every lane prunes ONE row and looks up its cell
            // range(s), all in one round trip; the warp then strides the candidates of the rows that
            // hold any.  Around an isolated query whole shells are empty: one trip each instead of one
            // per row (25 rows x 2 shells x every level was most of this kernel's time).
            const int ny = y1 - y0 + 1, nrows = (z1 - z0 + 1) * ny;
            for (int row0 = 0; row0 < nrows; row0 += 32) {
                uint32_t s0 = 0, e0 = 0, s1 = 0, e1 = 0;
                const int ri = row0 + lane;
                if (ri < nrows) {
                    const int zz = z0 + ri / ny, yy = y0 + ri % ny;
                    const bool edge = merged || (zz - cz == r) || (cz - zz == r) || (yy - cy == r) || (cy - yy == r);
                    int xa = max(cx - r, 0), xb = min(cx + r, g.dx - 1);
                    bool ok = true;
                    if (kth_d < 1.0e30f) {
                        const float gz = axis_gap(qz, g.oz, g.cell, zz, g.dz);
                        const float gy = axis_gap(qy, g.oy, g.cell, yy, g.dy);
                        const float gyz = fmaxf(sqrtf(__fmaf_rn(gz, gz, __fmul_rn(gy, gy))) - margin, 0.0f);
                        const float gyz2 = __fmul_rn(gyz, gyz);
                        ok = !(gyz2 > kth_d);
                        if (ok) {
                            const float w = sqrtf(kth_d - gyz2) + margin;
                            xa = max(xa, grid_coord(qx - w, g.ox, g.inv, g.dx));
                            xb = min(xb, grid_coord(qx + w, g.ox, g.inv, g.dx));
                            ok = xa <= xb;
                        }
                    }
                    if (ok) {
                        const uint32_t row = ((uint32_t)zz * (uint32_t)g.dy + (uint32_t)yy) * (uint32_t)g.dx;
                        // up to two ranges: the whole row on the shell's faces, its two end cells otherwise
                        if (edge) {
                            s0 = __ldg(g.start + row + xa);
                            e0 = __ldg(g.start + row + xb + 1);
                        } else {
                            if (cx - r >= xa) {
                                s0 = __ldg(g.start + row + (cx - r));
                                e0 = __ldg(g.start + row + (cx - r) + 1);
                            }
                            if (cx + r <= xb) {
                                s1 = __ldg(g.start + row + (cx + r));
                                e1 = __ldg(g.start + row + (cx + r) + 1);
                            }
                        }
                    }
                }
                unsigned m = __ballot_sync(0xffffffffu, e0 > s0 || e1 > s1);
                while (m) {
                    const int src = __ffs(m) - 1;
                    m &= m - 1;
                    const uint32_t a0 = __shfl_sync(0xffffffffu, s0, src), b0 = __shfl_sync(0xffffffffu, e0, src);
                    const uint32_t a1 = __shfl_sync(0xffffffffu, s1, src), b1 = __shfl_sync(0xffffffffu, e1, src);
                    // 8 loads in flight per lane: on a coarse level a row holds thousands of points
                    for (uint32_t j = a0 + lane; j < b0; j += 32 * 8) {
                        float4 p[8];
#pragma unroll
                        for (int u = 0; u < 8; ++u)
                            if (j + 32 * u < b0) p[u] = __ldg(g.pts + j + 32 * u);
#pragma unroll
                        for (int u = 0; u < 8; ++u)
                            if (j + 32 * u < b0)
                                mine.offer(dist_sq(qx, qy, qz, p[u].x, p[u].y, p[u].z), __float_as_int(p[u].w), j + 32 * u);
                    }
                    for (uint32_t j = a1 + lane; j < b1; j += 32) {
                        const float4 p = __ldg(g.pts + j);
                        mine.offer(dist_sq(qx, qy, qz, p.x, p.y, p.z), __float_as_int(p.w), j);
                    }
                }
            }
            const unsigned long long kth = warp_merge_topk<K>(mine, k, nullptr);
            kth_d = __uint_as_float((uint32_t)((kth - 1ull) >> 32));
            const float bound = fminf(fminf(shell_bound_axis(qx, g.ox, g.cell, cx, r, g.dx),
                                            shell_bound_axis(qy, g.oy, g.cell, cy, r, g.dy)),
                                      shell_bound_axis(qz, g.oz, g.cell, cz, r, g.dz));
            if (bound == INF) {
                done = true;
                break;
            }
            const float bs = bound - margin;
            if (bs > 0.0f && kth_d < __fmul_rn(bs, bs)) {
                done = true;
                break;
            }
            if (r >= r_max) break;
        }
    }
    unsigned long long outk[K];
#pragma unroll
    for (int j = 0; j < K; ++j) outk[j] = BestR<K>::EMPTY;
    warp_merge_topk<K>(mine, k, outk);
    if (lane == 0) {
#pragma unroll
        for (int j = 0; j < K; ++j)
            if (j >= K - k) {
                irow[j - (K - k)] = (int)(uint32_t)((outk[j] - 1ull) & 0xffffffffull);
                drow[j - (K - k)] = __uint_as_float((uint32_t)((outk[j] - 1ull) >> 32));
            }
    }
}

// ------------------------------------------------------------------ ICP nearest neighbour
// k = 1 search of the registration loop (kdtree.hpp:463-553 with k = 1, bounded by
// max_correspondence_distance: registration.hpp:584 rejects anything farther).  Same exactness
// argument as grid_search; three additions that matter for the iteration kernel:
//  * warm start: the previous iteration's correspondence is offered first.  It is a real target
//    point, so it only tightens the pruning bound — the answer is unchanged — and after the first
//    iteration most queries touch one or two cells instead of 27;
//  * first pass = the 3x3 rows around the query's cell, rows and x-ranges pruned against the bound,
//    every `start` look-up issued at once: a typical query is 3-4 dependent L2 round trips;
//  * queries the first pass cannot finish (nothing nearby: scan edges, sparse far range; ~8 % of a
//    LiDAR scan, and spatially clustered, i.e. concentrated in a few warps) are NOT continued by
//    their lane.  The iteration kernel appends them to a work list and, after a grid barrier, all
//    warps of the grid drain it: one query per warp at a time, shell rows and candidates scanned 32
//    wide (load-balanced by a prefix sum over the rows' candidate counts).  The tail the whole grid
//    used to wait for — one warp owning dozens of expensive queries — is spread over every SM.

constexpr uint32_t ICP_LANE_CANDS = 64;  // most candidates a single lane scans on a coarser level

__device__ __forceinline__ unsigned long long best_key(float d, int i) {
    return ((unsigned long long)__float_as_uint(d) << 32) | (unsigned long long)(uint32_t)i;  // i = -1 sorts last
}

// One pruned pass over the 3x3x3 block of `g` around the query.  Valid on ANY level (every level
// indexes all points): afterwards every point closer than min(bound, current best) has been seen.
// Returns 1 when `best` is final, 0 when not proven, -1 when the rows hold more than max_cands
// candidates (nothing scanned: the caller leaves dense blocks to the cooperative search).
// B = Best1M: the pruning bound is the candidate's distance PLUS `infl` metres, so that the pass also proves how far
// away everything else is (see Best1M).
template <class B>
__device__ __forceinline__ int icp_first_pass(const GridView& g, float qx, float qy, float qz, B& best,
                                              float max_radius, uint32_t max_cands = 0xffffffffu, float infl = 0.0f) {
    const int cx = grid_coord(qx, g.ox, g.inv, g.dx);
    const int cy = grid_coord(qy, g.oy, g.inv, g.dy);
    const int cz = grid_coord(qz, g.oz, g.inv, g.dz);
    const float INF = __int_as_float(0x7f800000);
    const float margin = g.margin + 1e-6f * fmaxf(fmaxf(fabsf(qx), fabsf(qy)), fabsf(qz));
    const float reach = max_radius + margin;
    const float reach2 = reach < 1.8e19f ? __fmul_rn(reach, reach) : INF;
    float lim2 = fminf(best.d, reach2);
    if constexpr (B::MARGIN) {
        if (best.d < reach2) {
            const float r = sqrtf(best.d) + infl;
            lim2 = fminf(fmaxf(__fmul_rn(r, r), best.d), reach2);
        }
    }
    // Row (y, z) can hold something better than the bound only if its distance g_yz to the query
    // satisfies g_yz <= sqrt(lim2) + margin =: L, and then only in cells within
    // w = sqrt(L^2 - g_yz^2) + margin of the query along x (w is never smaller than grid_search's
    // sqrt(lim2 - (g_yz - margin)^2) + margin: 2 margin (sqrt(lim2) + margin - g_yz) >= 0).  Pruning
    // arithmetic only pays when the bound is tighter than the block being looked at.
    const bool prune = lim2 < __fmul_rn(4.0f, __fmul_rn(g.cell, g.cell));
    const float L = prune ? sqrtf(lim2) + margin : INF;
    const float L2 = prune ? __fmul_rn(L, L) : INF;
    float gy2[3], gz2[3];
#pragma unroll
    for (int v = 0; v < 3; ++v) {
        const float a = prune ? axis_gap(qy, g.oy, g.cell, cy + v - 1, g.dy) : 0.0f;
        const float b = prune ? axis_gap(qz, g.oz, g.cell, cz + v - 1, g.dz) : 0.0f;
        gy2[v] = __fmul_rn(a, a);
        gz2[v] = __fmul_rn(b, b);
    }
    uint32_t ls[9], le[9];
#pragma unroll
    for (int t = 0; t < 9; ++t) {
        const int zz = cz + (t / 3) - 1, yy = cy + (t % 3) - 1;
        bool ok = zz >= 0 && zz < g.dz && yy >= 0 && yy < g.dy;
        int xa = max(cx - 1, 0), xb = min(cx + 1, g.dx - 1);
        if (prune) {
            const float g2 = __fadd_rn(gy2[t % 3], gz2[t / 3]);
            ok = ok && g2 <= L2;
            if (ok) {
                const float w = sqrtf(fmaxf(L2 - g2, 0.0f)) + margin;
                xa = max(xa, grid_coord(qx - w, g.ox, g.inv, g.dx));
                xb = min(xb, grid_coord(qx + w, g.ox, g.inv, g.dx));
                ok = xa <= xb;
            }
        }
        const uint32_t row = ((uint32_t)zz * (uint32_t)g.dy + (uint32_t)yy) * (uint32_t)g.dx;
        ls[t] = ok ? __ldg(g.start + row + xa) : 0u;
        le[t] = ok ? __ldg(g.start + row + xb + 1) : 0u;
    }
    if (max_cands != 0xffffffffu) {
        uint32_t total = 0;
#pragma unroll
        for (int t = 0; t < 9; ++t) total += le[t] - ls[t];
        if (total > max_cands) return -1;
    }
#pragma unroll
    for (int t = 0; t < 9; ++t) {
        for (uint32_t j = ls[t]; j < le[t]; j += 4) {
            float4 p[4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (j + u < le[t]) p[u] = __ldg(g.pts + j + u);
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (j + u < le[t])
                    best.offer(dist_sq(qx, qy, qz, p[u].x, p[u].y, p[u].z), __float_as_int(p[u].w), j + u);
        }
    }
    const float bound = fminf(fminf(shell_bound_axis(qx, g.ox, g.cell, cx, 1, g.dx),
                                    shell_bound_axis(qy, g.oy, g.cell, cy, 1, g.dy)),
                              shell_bound_axis(qz, g.oz, g.cell, cz, 1, g.dz));
    if constexpr (B::MARGIN) {
        if (prune) best.d2 = fminf(best.d2, lim2);
        best.u = bound == INF ? INF : fmaxf(bound - margin, 0.0f);
    }
    if (bound == INF) return 1;
    const float bs = bound - margin;
    return ((bs > 0.0f && best.worst() < __fmul_rn(bs, bs)) || bs >= max_radius) ? 1 : 0;
}

// Warp-cooperative continuation for ONE query (all arguments warp-uniform, every lane calls it).  `best` holds what
// the per-lane first pass left: usually a real candidate (the warm start or a point of the 3x3x3 block), whose
// distance bounds the answer.  Instead of walking shell after shell, the warp picks the finest (level, ring radius)
// whose block CERTIFIES that bound — everything outside is farther than min(best, max_radius) — and finishes the
// query with ONE scan of it: rows (z, y) spread over the lanes and pruned against the bound, x-ranges trimmed, the
// ring-1 cells of the finest level (covered by the first pass) skipped, candidates of all rows scanned 32 wide.
// A query without any candidate and without a radius bound first grows its block until it holds a point (counted
// from the cell ranges, nothing scanned).  `best` is warp-uniform on entry and exit.
constexpr int ICP_RMAX = 5;  // growth sequence: largest ring radius on a level that is not the coarsest (11 cells < the next level's 12)
// Certifying block: a finer level with a larger ring costs more row look-ups ((2r+1)^2, two loads each) but scans
// fewer candidates — its cells hug the bound's sphere.  It matters most for queries WITHOUT a neighbour inside
// max_radius (dense clouds that overlap only partly): the sphere they must prove empty is cut out of 0.4 m cells
// (a few hundred boundary points) instead of 1.5 m ones (up to 10^5).
#ifndef SPX_ICP_RMAX_CERT
#define SPX_ICP_RMAX_CERT 15
#endif
constexpr int ICP_RMAX_CERT = SPX_ICP_RMAX_CERT;

// B = Best1M: the block has to certify the candidate's distance plus `infl` metres, and rows / cells are pruned
// against that inflated bound (see Best1M); the stop test stays the plain one.
template <class B>
static __device__ __noinline__ void icp_coop_search(const GridLevels& gl, float qx, float qy, float qz, B& best,
                                                    float max_radius, uint32_t* dbg = nullptr, float infl = 0.0f) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const float INF = __int_as_float(0x7f800000);
    int l_min = 0, r_done = 1;  // level 0: the first pass covered ring 1
    for (;;) {
        int L = l_min, R = r_done + 1;
        bool found = false;
        // A candidate's distance is what a block has to certify.  Without a candidate the block first GROWS until it
        // holds a point (or has covered max_radius): certifying the bare radius instead would scan every point
        // within max_radius of each such query — in the first iteration of a dense, misaligned pair that is a quarter
        // of the source at thousands of candidates each (8 ms instead of 0.5 at 1.6 M points).
        float cert_d = best.d;  // squared distance the block has to certify
        if constexpr (B::MARGIN) {
            if (best.d < 1.0e30f) {
                const float r = sqrtf(best.d) + infl;
                cert_d = fmaxf(__fmul_rn(r, r), best.d);
            }
        }
        if (best.d < 1.0e30f) {
            for (int l = l_min; l < gl.n_levels && !found; ++l) {
                const GridView& g = gl.lv[l];
                const bool last = l == gl.n_levels - 1;
                const int cx = grid_coord(qx, g.ox, g.inv, g.dx);
                const int cy = grid_coord(qy, g.oy, g.inv, g.dy);
                const int cz = grid_coord(qz, g.oz, g.inv, g.dz);
                const float margin = g.margin + 1e-6f * fmaxf(fmaxf(fabsf(qx), fabsf(qy)), fabsf(qz));
                const int r_first = (l == l_min) ? r_done + 1 : 1;
                const int r_last = last ? (1 << 20) : ICP_RMAX_CERT;
                for (int r = r_first; r <= r_last; ++r) {
                    const float bound = fminf(fminf(shell_bound_axis(qx, g.ox, g.cell, cx, r, g.dx),
                                                    shell_bound_axis(qy, g.oy, g.cell, cy, r, g.dy)),
                                              shell_bound_axis(qz, g.oz, g.cell, cz, r, g.dz));
                    const float bs = bound - margin;
                    if (bound == INF || (bs > 0.0f && cert_d < __fmul_rn(bs, bs)) || bs >= max_radius) {
                        L = l;
                        R = r;
                        found = true;
                        break;
                    }
                }
            }
        }
        if (!found) {
            // no candidate and no radius: the smallest block of the growth sequence that holds a point at all
            int l = l_min, r = r_done;
            for (;;) {
                const bool last = l == gl.n_levels - 1;
                if (last || r < ICP_RMAX) {
                    ++r;
                } else {
                    ++l;
                    r = 1;
                }
                const GridView& g = gl.lv[l];
                const int cx = grid_coord(qx, g.ox, g.inv, g.dx);
                const int cy = grid_coord(qy, g.oy, g.inv, g.dy);
                const int cz = grid_coord(qz, g.oz, g.inv, g.dz);
                const int z0 = max(cz - r, 0), z1 = min(cz + r, g.dz - 1);
                const int y0 = max(cy - r, 0), y1 = min(cy + r, g.dy - 1);
                const int xa = max(cx - r, 0), xb = min(cx + r, g.dx - 1);
                const int ny = y1 - y0 + 1, nrows = (z1 - z0 + 1) * ny;
                uint32_t c = 0;
                for (int t = lane; t < nrows; t += 32) {
                    const uint32_t row = ((uint32_t)(z0 + t / ny) * (uint32_t)g.dy + (uint32_t)(y0 + t % ny)) * (uint32_t)g.dx;
                    c += __ldg(g.start + row + xb + 1) - __ldg(g.start + row + xa);
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(FULL, c, o);
                const bool whole = z0 == 0 && y0 == 0 && xa == 0 && z1 == g.dz - 1 && y1 == g.dy - 1 && xb == g.dx - 1;
                if (c > 0u || whole) break;
                if (max_radius < 1.8e19f) {  // nothing inside max_radius: the (empty) block that proves it ends the search
                    const float margin = g.margin + 1e-6f * fmaxf(fmaxf(fabsf(qx), fabsf(qy)), fabsf(qz));
                    const float bound = fminf(fminf(shell_bound_axis(qx, g.ox, g.cell, cx, r, g.dx),
                                                    shell_bound_axis(qy, g.oy, g.cell, cy, r, g.dy)),
                                              shell_bound_axis(qz, g.oz, g.cell, cz, r, g.dz));
                    if (bound - margin >= max_radius) break;
                }
            }
            L = l;
            R = r;
        }
        // ---- one scan of block (L, R), cells within ring r_skip of the same level excluded
        const GridView& g = gl.lv[L];
        const int r_skip = (L == l_min) ? r_done : -1;
        const int cx = grid_coord(qx, g.ox, g.inv, g.dx);
        const int cy = grid_coord(qy, g.oy, g.inv, g.dy);
        const int cz = grid_coord(qz, g.oz, g.inv, g.dz);
        const float margin = g.margin + 1e-6f * fmaxf(fmaxf(fabsf(qx), fabsf(qy)), fabsf(qz));
        // what has to be beaten: the current candidate, or the search radius (+ allowance)
        const float reach = max_radius + margin;
        const float lim2 = fminf(cert_d, reach < 1.8e19f ? __fmul_rn(reach, reach) : INF);
        const int z0 = max(cz - R, 0), z1 = min(cz + R, g.dz - 1);
        const int y0 = max(cy - R, 0), y1 = min(cy + R, g.dy - 1);
        const int ny = y1 - y0 + 1;
        const int nrows = (z1 - z0 + 1) * ny;
        B mine = best;  // per-lane candidate, merged after the scan
        if (dbg) {
            dbg[1] += 1;
            dbg[2] += (uint32_t)nrows;
        }
        for (int base = 0; base < nrows; base += 32) {
            const int t = base + lane;
            uint32_t sA = 0, eA = 0, sB = 0, eB = 0;
            if (t < nrows) {
                const int zz = z0 + t / ny, yy = y0 + t % ny;
                const bool outer = max(abs(zz - cz), abs(yy - cy)) > r_skip;
                int xa = max(cx - R, 0), xb = min(cx + R, g.dx - 1);
                bool ok = true;
                if (lim2 < 1.0e30f) {
                    const float gz = axis_gap(qz, g.oz, g.cell, zz, g.dz);
                    const float gy = axis_gap(qy, g.oy, g.cell, yy, g.dy);
                    const float gyz = fmaxf(sqrtf(__fmaf_rn(gz, gz, __fmul_rn(gy, gy))) - margin, 0.0f);
                    const float gyz2 = __fmul_rn(gyz, gyz);
                    ok = gyz2 <= lim2;
                    const float w = sqrtf(fmaxf(lim2 - gyz2, 0.0f)) + margin;
                    xa = max(xa, grid_coord(qx - w, g.ox, g.inv, g.dx));
                    xb = min(xb, grid_coord(qx + w, g.ox, g.inv, g.dx));
                    ok = ok && xa <= xb;
                }
                if (ok) {
                    const uint32_t row = ((uint32_t)zz * (uint32_t)g.dy + (uint32_t)yy) * (uint32_t)g.dx;
                    if (outer) {
                        sA = __ldg(g.start + row + xa);
                        eA = __ldg(g.start + row + xb + 1);
                    } else {  // only the cells beyond the ring already covered: the two ends of the row
                        const int la = xa, lb = min(xb, cx - r_skip - 1);
                        const int ra = max(xa, cx + r_skip + 1), rb = xb;
                        if (la <= lb) {
                            sA = __ldg(g.start + row + la);
                            eA = __ldg(g.start + row + lb + 1);
                        }
                        if (ra <= rb) {
                            sB = __ldg(g.start + row + ra);
                            eB = __ldg(g.start + row + rb + 1);
                        }
                    }
                }
            }
            const uint32_t cA = eA - sA, cnt = cA + (eB - sB);
            uint32_t inc = cnt;  // inclusive prefix sum of the candidate counts over the lanes
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t v = __shfl_up_sync(FULL, inc, o);
                if (lane >= o) inc += v;
            }
            const uint32_t total = __shfl_sync(FULL, inc, 31);
            if (dbg) dbg[3] += total;
            for (uint32_t cb = 0; cb < total; cb += 32) {
                const uint32_t kk = cb + lane;
                const bool live = kk < total;
                const uint32_t key = live ? kk : 0u;
                int owner = 0;  // number of lanes whose inclusive sum is <= key
#pragma unroll
                for (int sft = 16; sft > 0; sft >>= 1) {
                    const uint32_t v = __shfl_sync(FULL, inc, owner + sft - 1);
                    if (v <= key) owner += sft;
                }
                owner = min(owner, 31);
                const uint32_t o_inc = __shfl_sync(FULL, inc, owner);
                const uint32_t o_cnt = __shfl_sync(FULL, cnt, owner);
                const uint32_t o_cA = __shfl_sync(FULL, cA, owner);
                const uint32_t o_sA = __shfl_sync(FULL, sA, owner);
                const uint32_t o_sB = __shfl_sync(FULL, sB, owner);
                if (live) {
                    const uint32_t jj = key - (o_inc - o_cnt);
                    const uint32_t pos = jj < o_cA ? o_sA + jj : o_sB + (jj - o_cA);
                    const float4 p = __ldg(g.pts + pos);
                    mine.offer(dist_sq(qx, qy, qz, p.x, p.y, p.z), __float_as_int(p.w), pos);
                }
            }
        }
        // merge the lanes' candidates: minimum by (dist, index)
        unsigned long long k = best_key(mine.d, mine.i);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long v = __shfl_xor_sync(FULL, k, o);
            k = v < k ? v : k;
        }
        const unsigned win = __ballot_sync(FULL, best_key(mine.d, mine.i) == k);
        const int wl = __ffs(win) - 1;
        best.d = __shfl_sync(FULL, mine.d, wl);
        best.i = __shfl_sync(FULL, mine.i, wl);
        l_min = L;
        r_done = R;
        // stop test of the block just completed (grid_search's)
        const float bound = fminf(fminf(shell_bound_axis(qx, g.ox, g.cell, cx, R, g.dx),
                                        shell_bound_axis(qy, g.oy, g.cell, cy, R, g.dy)),
                                  shell_bound_axis(qz, g.oz, g.cell, cz, R, g.dz));
        if constexpr (B::MARGIN) {
            // every point but the winner: a lane whose candidate IS the winner contributes its runner-up
            float o = mine.i == best.i ? mine.d2 : mine.d;
#pragma unroll
            for (int sft = 16; sft > 0; sft >>= 1) o = fminf(o, __shfl_xor_sync(FULL, o, sft));
            best.d2 = lim2 < 1.0e30f ? fminf(o, lim2) : o;
            best.u = bound == INF ? INF : fmaxf(bound - margin, 0.0f);
        }
        if (bound == INF) return;  // whole grid visited
        const float bs = bound - margin;
        if (bs > 0.0f && best.worst() < __fmul_rn(bs, bs)) return;
        if (bs >= max_radius) return;  // everything within max_radius has been seen
    }
}

// Per-lane part of the search: warm start (warm_idx >= 0 offers that target point first, read from the target cloud
// in its original order — a correspondence found on a coarser level has no position in the finest level's array) +
// pruned first pass.  Returns true when `best` is final; otherwise `best` holds the bound reached so far and the query
// goes to the cooperative continuation.
template <class B>
__device__ __forceinline__ bool icp_fast(const GridLevels& gl, float qx, float qy, float qz, int warm_idx,
                                         const float4* __restrict__ tgt_pts, float max_radius, B& best, float infl = 0.0f) {
    const GridView& g = gl.lv[0];
    best.init();
    if (warm_idx >= 0) {
        const float4 p = __ldg(tgt_pts + warm_idx);
        best.offer(dist_sq(qx, qy, qz, p.x, p.y, p.z), warm_idx, 0u);
    }
    // (A per-lane pass on the next coarser level for the unproven, sparse-neighbourhood queries was
    // measured: it halves the cooperative phase but doubles this one — those queries cluster in the
    // same warps — for a net loss; icp_first_pass keeps its max_cands hook for that experiment.)
    return icp_first_pass(g, qx, qy, qz, best, max_radius, 0xffffffffu, infl) == 1;
}

// What a finished search leaves for the keep test: metres the query may still move (summed over the iterations) before
// its correspondence has to be searched again; 0 = search every time.  The allowance covers the rounding of the fp32
// distances the search compares (1e-7 relative on coordinates of magnitude qinf).
__device__ __forceinline__ float icp_keep_slack(const Best1M& b, float qinf, float max_corr_sq) {
    if (b.i < 0 || !(b.d <= max_corr_sq)) return 0.0f;
    const float m = fminf(sqrtf(b.d2), b.u) - sqrtf(b.d);
    return fmaxf(m - (1.0e-3f + 1.0e-5f * qinf), 0.0f);
}

#endif  // __CUDACC__

}  // namespace spx

// host-side handle
struct spx_index_s {
    spx_queue_t q = nullptr;
    size_t n_total = 0;   // points given to build
    uint32_t n = 0;       // finite points indexed
    float4* sorted[spx::GRID_MAX_LEVELS] = {};
    uint32_t* start[spx::GRID_MAX_LEVELS] = {};
    size_t ncells[spx::GRID_MAX_LEVELS] = {};
    unsigned long long* occ_dev = nullptr;  // occupied cells of the finest level (device counter)
    cudaEvent_t ready = nullptr;            // recorded on q's stream when the build's last kernel is queued: users on
                                            // OTHER queues wait on it (KDTree::build is synchronous in the reference)
    spx::GridLevels levels{};      // k = 1 searches and the registration kernels
    spx::GridLevels levels_knn{};  // k >= 2 searches: an extra, coarser first grid + the regular levels above the finest
};
