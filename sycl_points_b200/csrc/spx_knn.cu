// KNN on the device: the brute-force tile scan (I/algorithms/knn/bruteforce.hpp:24-96) and the
// GPU-resident exact index that stands in for knn::KDTree (kdtree.hpp:142-562) behind the same
// KNNBase contract (knn.hpp:14-61).
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <cstring>

#include <algorithm>
#include <vector>

#include "spx_grid.cuh"
#include "spx_scan.cuh"
#include "spx_tma.cuh"

using namespace spx;

namespace {

// ------------------------------------------------------------------ brute force
constexpr int BF_THREADS = 256;
constexpr int BF_TILE = 2048;  // float4 targets staged per step (32 KB of shared memory)

// One thread owns QPT queries and streams every target tile out of shared memory (one broadcast
// LDS.128 per target feeds QPT distance evaluations).  Candidate lists live in the thread's rows of
// the output arrays; only the k-th best is cached in registers.  Targets are tested BF_BATCH at a
// time with no branch per pair: the steady state is 3 sub + 1 mul + 2 fma + 1 predicated compare
// per (query, target) pair and one branch per BF_BATCH x QPT pairs; a batch with a hit (rare once the
// lists are warm: ~k ln(N/k) inserts per query in total) replays its pairs in index order with a
// strict '<', which yields exactly the (dist, index) order of bruteforce.hpp:71-83.
// PACKED: two queries share one packed-FP32 instruction stream (sm_100 FADD2 / FMUL2 / FFMA2 via
// sub/mul/fma.rn.f32x2 — IEEE round-to-nearest per element, so results stay bit-identical).
constexpr int BF_BATCH = 4;

// fma(dz,dz,fma(dy,dy,dx*dx)) for two queries at once against one target
__device__ __forceinline__ unsigned long long dist_sq2(unsigned long long qx, unsigned long long qy, unsigned long long qz,
                                                       float px, float py, float pz) {
    const unsigned long long PX = pack2(px, px), PY = pack2(py, py), PZ = pack2(pz, pz);
    unsigned long long dx, dy, dz, r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(dx) : "l"(qx), "l"(PX));
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(dy) : "l"(qy), "l"(PY));
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(dz) : "l"(qz), "l"(PZ));
    asm("mul.rn.f32x2 %0, %1, %1;" : "=l"(r) : "l"(dx));
    asm("fma.rn.f32x2 %0, %1, %1, %2;" : "=l"(r) : "l"(dy), "l"(r));
    asm("fma.rn.f32x2 %0, %1, %1, %2;" : "=l"(r) : "l"(dz), "l"(r));
    return r;
}

// Measured and rejected (r2h): a persistent grid whose warps take their queries by ticket, against the tail of the
// 2.2-wave grid — 13 % SLOWER: blocks that start every pass together stay in lockstep, so nothing overlaps their
// staging phases, while the hardware's own block scheduler already fills the tail.
template <int QPT, bool PACKED, bool TMA, int BATCH = BF_BATCH>
__global__ void __launch_bounds__(BF_THREADS) knn_bruteforce_kernel(const float4* __restrict__ queries, uint32_t nq,
                                                                    const float4* __restrict__ targets, uint32_t nt,
                                                                    int k, Xform T, int has_T,
                                                                    int32_t* __restrict__ idx,
                                                                    float* __restrict__ dist) {
    static_assert(!PACKED || QPT % 2 == 0, "packed variant pairs queries");
    // (static shared memory: 2 x 16 KB with TMA staging, 1 x 32 KB without)
    constexpr int TILE = TMA ? BF_TILE / 2 : BF_TILE;
    __shared__ __align__(128) float4 tiles[TMA ? 2 : 1][TILE];
    __shared__ __align__(8) unsigned long long bars[2];
    const uint32_t first = (blockIdx.x * BF_THREADS + threadIdx.x) * QPT;

    float qx[QPT], qy[QPT], qz[QPT], wd[QPT];
    float* drow[QPT];
    int32_t* irow[QPT];
#pragma unroll
    for (int u = 0; u < QPT; ++u) {
        const uint32_t qi = first + u;
        const bool live = qi < nq;
        float4 q = live ? __ldg(queries + qi) : make_float4(0.f, 0.f, 0.f, 1.f);
        if (has_T) q = transform_point(T, q);
        qx[u] = q.x; qy[u] = q.y; qz[u] = q.z;
        drow[u] = dist + (size_t)(live ? qi : 0) * k;
        irow[u] = idx + (size_t)(live ? qi : 0) * k;
        if (live) {
            for (int j = 0; j < k; ++j) { drow[u][j] = FLT_MAX; irow[u][j] = -1; }
            wd[u] = FLT_MAX;
        } else {
            wd[u] = -1.0f;  // nothing compares below it: the slot never inserts
        }
    }
    unsigned long long qx2[QPT / 2 + 1], qy2[QPT / 2 + 1], qz2[QPT / 2 + 1];
    if (PACKED) {
#pragma unroll
        for (int u = 0; u < QPT / 2; ++u) {
            qx2[u] = pack2(qx[2 * u], qx[2 * u + 1]);
            qy2[u] = pack2(qy[2 * u], qy[2 * u + 1]);
            qz2[u] = pack2(qz[2 * u], qz[2 * u + 1]);
        }
    }

    if (TMA) {
        if (threadIdx.x == 0) {
            mbar_init(&bars[0], 1);
            mbar_init(&bars[1], 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncthreads();
        if (threadIdx.x == 0 && nt > 0) {
            const uint32_t bytes = min((uint32_t)TILE, nt) * (uint32_t)sizeof(float4);
            mbar_expect_tx(&bars[0], bytes);
            bulk_g2s(&tiles[0][0], targets, bytes, &bars[0]);
        }
    }
    uint32_t it = 0;
    for (uint32_t base = 0; base < nt; base += TILE, ++it) {
        const int lim = min((uint32_t)TILE, nt - base);
        const int limb = (lim + BATCH - 1) / BATCH * BATCH;  // sentinels cover the padding
        const float4* tile;
        if (TMA) {
            const uint32_t buf = it & 1u;
            // the other buffer was read in the previous iteration, which ended in a block barrier: refill it now
            if (threadIdx.x == 0 && base + TILE < nt) {
                const uint32_t bytes = min((uint32_t)TILE, nt - base - TILE) * (uint32_t)sizeof(float4);
                mbar_expect_tx(&bars[buf ^ 1u], bytes);
                bulk_g2s(&tiles[buf ^ 1u][0], targets + base + TILE, bytes, &bars[buf ^ 1u]);
            }
            mbar_wait(&bars[buf], (it >> 1) & 1u);
            if (lim < limb) {  // (last tile only) sentinels beyond the end: squares overflow to +inf, never a k-th best
                if (threadIdx.x < (unsigned)(limb - lim))
                    tiles[buf][lim + threadIdx.x] = make_float4(FLT_MAX, FLT_MAX, FLT_MAX, 1.0f);
                __syncthreads();
            }
            tile = tiles[buf];
        } else {
            __syncthreads();
#pragma unroll
            for (int t = threadIdx.x; t < TILE; t += BF_THREADS) {
                const uint32_t j = base + t;
                tiles[0][t] = j < nt ? __ldg(targets + j) : make_float4(FLT_MAX, FLT_MAX, FLT_MAX, 1.0f);
            }
            __syncthreads();
            tile = tiles[0];
        }
#pragma unroll 2
        for (int t = 0; t < limb; t += BATCH) {
            float ds[BATCH][QPT];
            bool any = false;
#pragma unroll
            for (int v = 0; v < BATCH; ++v) {
                const float4 p = tile[t + v];
                if (PACKED) {
#pragma unroll
                    for (int u = 0; u < QPT / 2; ++u)
                        unpack2(dist_sq2(qx2[u], qy2[u], qz2[u], p.x, p.y, p.z), ds[v][2 * u], ds[v][2 * u + 1]);
                } else {
#pragma unroll
                    for (int u = 0; u < QPT; ++u) ds[v][u] = dist_sq(qx[u], qy[u], qz[u], p.x, p.y, p.z);
                }
#pragma unroll
                for (int u = 0; u < QPT; ++u) any |= ds[v][u] < wd[u];
            }
            // A target that beats some query's k-th best is rare (k (1 + ln(N / k)) of N per query) but divergent:
            // handled per lane, the sorted insertion — a chain of dependent loads and stores on the query's result
            // row — ran with one lane in 32 and took a quarter of the kernel's issue slots (24 of 32 lanes active on
            // average, profiles/r2g_ncu_bf_p4.txt).  Here the WARP inserts for the lane: each lane holds one slot of
            // the row (k <= 128: up to four), the position is a ballot count, the shift one coalesced load and store.
            if (__any_sync(0xffffffffu, any)) {
                const int lane = threadIdx.x & 31;
#pragma unroll
                for (int u = 0; u < QPT; ++u) {
#pragma unroll
                    for (int v = 0; v < BATCH; ++v) {
                        const float d1 = ds[v][u];
                        unsigned m = __ballot_sync(0xffffffffu, d1 < wd[u]);
                        while (m) {
                            const int src = __ffs(m) - 1;
                            m &= m - 1;
                            const float dd = __shfl_sync(0xffffffffu, d1, src);
                            const uint32_t qi = first + (uint32_t)((src - lane) * QPT + u);  // src's query (a live one)
                            float* d = dist + (size_t)qi * k;
                            int32_t* id = idx + (size_t)qi * k;
                            // pos = entries with dist <= dd (strict '<' insertion: behind its equals, bruteforce.hpp:71-83)
                            int pos = 0;
                            float pd[4];
                            int32_t pi[4];
#pragma unroll
                            for (int e = 0; e < 4; ++e) {
                                const int j = e * 32 + lane;
                                pd[e] = 0.f;
                                pi[e] = 0;
                                if (e * 32 < k) {
                                    const bool in = j < k;
                                    const float cd = in ? d[j] : FLT_MAX;
                                    pos += __popc(__ballot_sync(0xffffffffu, in && cd <= dd));
                                    if (in && j > 0) {
                                        pd[e] = d[j - 1];
                                        pi[e] = id[j - 1];
                                    }
                                }
                            }
                            const float tail = k >= 2 ? d[k - 2] : dd;  // (same address in every lane)
                            __syncwarp();  // every load of the old row is done before any slot is overwritten
#pragma unroll
                            for (int e = 0; e < 4; ++e) {
                                const int j = e * 32 + lane;
                                if (e * 32 < k && j < k && j >= pos) {
                                    d[j] = j == pos ? dd : pd[e];
                                    id[j] = j == pos ? (int)(base + t + v) : pi[e];
                                }
                            }
                            __syncwarp();  // the row is consistent before the next insertion reads it
                            if (lane == src) wd[u] = pos == k - 1 ? dd : tail;
                        }
                    }
                }
            }
        }
        if (TMA) __syncthreads();  // every thread is done with this buffer before the next iteration refills it
    }
}

// ------------------------------------------------------------------ index build
__device__ __forceinline__ int float_ordered(float f) {
    const int i = __float_as_int(f);
    return i ^ ((i >> 31) & 0x7fffffff);
}
// The box is accumulated with atomicMax only, in an encoding whose empty state is all zero bits (the head is
// initialised by the memset that clears the occupancy bitmaps, not by a kernel): with u(x) = the
// order-preserving unsigned image of a finite float, mx[a] = max u(x) and mn[a] = max ~u(x).
struct BBoxAcc {
    uint32_t mn[3];
    uint32_t mx[3];
    uint32_t finite;
    uint32_t done_blocks;  // ticket: the last block of bbox_kernel derives the occupancy plan
};
struct OccPlan {
    float lo[3];
    float c0;        // volume-heuristic cell edge the candidates are multiples of
    float ext[3];
    float max_abs;
};
constexpr int OCC_CANDS = 8;
// everything the host reads back from the first phase of the build, contiguous: ONE device-to-host copy
struct BuildHead {
    BBoxAcc acc;
    OccPlan plan;
    unsigned int ones[OCC_CANDS];
};
__device__ void occ_plan(const volatile BBoxAcc* acc, OccPlan* plan);

// accumulators are initialised by a kernel, not by a host-to-device copy: a small H2D copy queues
// behind whatever bulk upload another queue has in flight on the same copy engine (measured: the
// streamed end-to-end step lost 0.6 ms to exactly that)
__global__ void bbox_kernel(const float4* __restrict__ pts, uint32_t n, BuildHead* head) {
    BBoxAcc* acc = &head->acc;
    int mn[3] = {INT_MAX, INT_MAX, INT_MAX}, mx[3] = {INT_MIN, INT_MIN, INT_MIN};
    uint32_t cnt = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float4 p = __ldg(pts + i);
        if (isfinite(p.x) && isfinite(p.y) && isfinite(p.z)) {
            mn[0] = min(mn[0], float_ordered(p.x)); mx[0] = max(mx[0], float_ordered(p.x));
            mn[1] = min(mn[1], float_ordered(p.y)); mx[1] = max(mx[1], float_ordered(p.y));
            mn[2] = min(mn[2], float_ordered(p.z)); mx[2] = max(mx[2], float_ordered(p.z));
            ++cnt;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            mn[a] = min(mn[a], __shfl_xor_sync(0xffffffffu, mn[a], o));
            mx[a] = max(mx[a], __shfl_xor_sync(0xffffffffu, mx[a], o));
        }
        cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    }
    // one set of atomics per BLOCK (per-warp atomics on seven shared addresses serialise)
    __shared__ uint32_t smn[3], smx[3];
    __shared__ uint32_t scnt;
    if (threadIdx.x == 0) {
        for (int a = 0; a < 3; ++a) smn[a] = smx[a] = 0u;
        scnt = 0;
    }
    __syncthreads();
    if ((threadIdx.x & 31) == 0 && cnt) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            atomicMax(&smn[a], ~((uint32_t)mn[a] ^ 0x80000000u));
            atomicMax(&smx[a], (uint32_t)mx[a] ^ 0x80000000u);
        }
        atomicAdd(&scnt, cnt);
    }
    __syncthreads();
    if (threadIdx.x == 0 && scnt) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            atomicMax(&acc->mn[a], smn[a]);
            atomicMax(&acc->mx[a], smx[a]);
        }
        atomicAdd(&acc->finite, scnt);
    }
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(&acc->done_blocks, 1u) == gridDim.x - 1) {
            __threadfence();
            occ_plan(acc, &head->plan);
        }
    }
}

struct GridGeom {
    float ox, oy, oz, inv;
    int dx, dy, dz;
};

__device__ __forceinline__ uint32_t cell_of(const GridGeom& g, const float4 p) {
    const int cx = grid_coord(p.x, g.ox, g.inv, g.dx);
    const int cy = grid_coord(p.y, g.oy, g.inv, g.dy);
    const int cz = grid_coord(p.z, g.oz, g.inv, g.dz);
    return ((uint32_t)cz * (uint32_t)g.dy + (uint32_t)cy) * (uint32_t)g.dx + (uint32_t)cx;
}

// ---- cell-size selection without a host round trip per attempt
// The finest cell edge is chosen so that an occupied cell holds ~3 points.  Occupancy as a function
// of the cell edge is measured for OCC_CANDS candidate edges in ONE pass: every point sets one bit
// per candidate in a hashed bitmap of M bits, and the number of occupied cells follows from the
// fraction of zero bits (linear counting: n_occ ~ -M ln(zeros / M), within ~1 % at the loads used).
__constant__ float OCC_FACTOR[OCC_CANDS] = {0.35f, 0.5f, 0.7071f, 1.0f, 1.4142f, 2.0f, 2.8284f, 4.0f};

// written by the last block of bbox_kernel, read by occ_mark_kernel and by the host
__device__ void occ_plan(const volatile BBoxAcc* acc, OccPlan* plan) {
    float lo[3], ext[3], max_ext = 0.0f, max_abs = 0.0f;
    for (int a = 0; a < 3; ++a) {
        const int ol = (int)(~acc->mn[a] ^ 0x80000000u), oh = (int)(acc->mx[a] ^ 0x80000000u);
        lo[a] = __int_as_float(ol ^ ((ol >> 31) & 0x7fffffff));
        const float hi = __int_as_float(oh ^ ((oh >> 31) & 0x7fffffff));
        ext[a] = hi - lo[a];
        max_ext = fmaxf(max_ext, ext[a]);
        max_abs = fmaxf(max_abs, fmaxf(fabsf(lo[a]), fabsf(hi)));
    }
    if (!(max_ext > 0.0f)) max_ext = 1.0f;
    double vol = 1.0;
    for (int a = 0; a < 3; ++a) vol *= (double)fmaxf(ext[a], 0.02f * max_ext);
    float c0 = (float)cbrt(vol / (2.0 * (double)max((uint32_t)acc->finite, 1u)));
    c0 = fmaxf(c0, 1e-6f * fmaxf(max_abs, 1.0f));
    for (int a = 0; a < 3; ++a) {
        plan->lo[a] = lo[a];
        plan->ext[a] = ext[a];
    }
    plan->c0 = c0;
    plan->max_abs = max_abs;
}

__global__ void occ_mark_kernel(const float4* __restrict__ pts, uint32_t n, const OccPlan* __restrict__ plan,
                                uint32_t* __restrict__ bitmaps, uint32_t words_per_map) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 p = __ldg(pts + i);
    if (!(isfinite(p.x) && isfinite(p.y) && isfinite(p.z))) return;
    const float rx = p.x - plan->lo[0], ry = p.y - plan->lo[1], rz = p.z - plan->lo[2];
    const float c0 = plan->c0;
    const uint32_t mask = words_per_map * 32u - 1u;
#pragma unroll
    for (int j = 0; j < OCC_CANDS; ++j) {
        const float inv = 1.0f / (c0 * OCC_FACTOR[j]);
        const uint32_t ix = (uint32_t)fminf(rx * inv, 4.0e9f), iy = (uint32_t)fminf(ry * inv, 4.0e9f),
                       iz = (uint32_t)fminf(rz * inv, 4.0e9f);
        uint32_t h = ix * 73856093u ^ iy * 19349663u ^ iz * 83492791u;
        h ^= h >> 16; h *= 0x85ebca6bu; h ^= h >> 13; h *= 0xc2b2ae35u; h ^= h >> 16;
        h &= mask;
        atomicOr(bitmaps + (size_t)j * words_per_map + (h >> 5), 1u << (h & 31u));
    }
}

__global__ void occ_count_kernel(const uint32_t* __restrict__ bitmaps, uint32_t words_per_map,
                                 unsigned int* __restrict__ ones) {
    const int j = blockIdx.y;
    unsigned int c = 0;
    for (uint32_t w = blockIdx.x * blockDim.x + threadIdx.x; w < words_per_map; w += gridDim.x * blockDim.x)
        c += __popc(bitmaps[(size_t)j * words_per_map + w]);
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(ones + j, c);
}

// occupied cells of a finished level = cells whose range in `start` is not empty
__global__ void occupied_from_start_kernel(const uint32_t* __restrict__ start, size_t ncells, unsigned long long* occupied) {
    unsigned long long c = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < ncells; i += (size_t)gridDim.x * blockDim.x)
        c += start[i + 1] != start[i];
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(occupied, c);
}

// Stable order: a point's slot inside its cell must be its rank among the cell's points in ORIGINAL
// index order, so that the sorted copy (and therefore the visiting order) is deterministic run to
// run.  The scatter below hands out slots with atomics (arrival order); each cell's slice of the
// finest level is then ordered by original index in a second pass (cells are tiny).  Points arrive
// spatially sorted (voxel order), so the lanes of a warp mostly share a handful of cells — on the
// coarse levels a single one: one atomic per distinct cell per warp (__match_any_sync) instead of one
// per point (120 k atomics on six addresses took 30 us per coarse level).
// ---- all levels in one pass
// The levels are independent counting sorts of the same points, so they share launches: one count
// kernel, ONE scan over the concatenated per-level count arrays, one scatter kernel.  Level l's
// counts start at cell_base[l]; every level sums to n, so the scanned value of level l's cell c is
// l*n + (position inside the level): the levels' sorted copies are laid out back to back in one
// array and `start` values index it directly (GridView::pts is the common base pointer).
struct LevelSet {
    int n_levels;  // incl. the extra k-NN grid (always the last entry) when the index has one
    GridGeom geom[GRID_MAX_LEVELS + 1];
    uint32_t cell_base[GRID_MAX_LEVELS + 2];
};

__global__ void levels_count_kernel(const float4* __restrict__ pts, uint32_t n, LevelSet ls, uint32_t* __restrict__ counts) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
    bool ok = false;
    if (i < n) {
        p = __ldg(pts + i);
        ok = isfinite(p.x) && isfinite(p.y) && isfinite(p.z);
    }
    for (int l = 0; l < ls.n_levels; ++l) {
        const uint32_t c = ok ? ls.cell_base[l] + cell_of(ls.geom[l], p) : 0xffffffffu;
        const unsigned peers = __match_any_sync(0xffffffffu, c);
        if (ok && lane == __ffs(peers) - 1) atomicAdd(counts + c, (uint32_t)__popc(peers));
    }
}

__global__ void levels_scatter_kernel(const float4* __restrict__ pts, uint32_t n, LevelSet ls,
                                      const uint32_t* __restrict__ start, uint32_t* __restrict__ remaining,
                                      float4* __restrict__ sorted) {
    // `remaining` holds the per-cell counts of levels_count_kernel: a warp's group of points takes its
    // slots off the END of the cell's range (no second zeroed cursor array); the order inside a cell is free
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
    bool ok = false;
    if (i < n) {
        p = __ldg(pts + i);
        ok = isfinite(p.x) && isfinite(p.y) && isfinite(p.z);
    }
    const float4 rec = make_float4(p.x, p.y, p.z, __int_as_float((int)i));
    for (int l = 0; l < ls.n_levels; ++l) {
        const uint32_t c = ok ? ls.cell_base[l] + cell_of(ls.geom[l], p) : 0xffffffffu;
        const unsigned peers = __match_any_sync(0xffffffffu, c);
        const int leader = __ffs(peers) - 1;
        uint32_t base = 0;
        if (ok && lane == leader) {
            const uint32_t g = (uint32_t)__popc(peers);
            base = __ldg(start + c) + atomicSub(remaining + c, g) - g;
        }
        base = __shfl_sync(0xffffffffu, base, leader);
        if (ok) sorted[base + __popc(peers & ((1u << lane) - 1u))] = rec;
    }
}


// ------------------------------------------------------------------ index search
constexpr int GRID_THREADS = 128;

// k == 1: the candidate is a register pair.  k > 1: each thread's sorted candidate list lives in
// shared memory, element j of thread t at [j * GRID_THREADS + t] (conflict-free), and the block
// writes its [queries][k] result tile out cooperatively so the global stores coalesce.
template <bool K1>
__global__ void __launch_bounds__(GRID_THREADS) grid_knn_kernel(const GridLevels g, const float4* __restrict__ queries,
                                                                 uint32_t nq, int k, Xform T, int has_T,
                                                                 int32_t* __restrict__ idx, float* __restrict__ dist) {
    extern __shared__ float smem_lists[];
    const uint32_t q0 = blockIdx.x * GRID_THREADS;
    const uint32_t qi = q0 + threadIdx.x;
    const float INF = __int_as_float(0x7f800000);
    float4 q = make_float4(0.f, 0.f, 0.f, 1.f);
    if (qi < nq) {
        q = __ldg(queries + qi);
        if (has_T) q = transform_point(T, q);
    }
    const bool searchable = qi < nq && isfinite(q.x) && isfinite(q.y) && isfinite(q.z) && g.lv[0].n > 0;
    if (K1) {
        Best1 best;
        best.init();
        if (searchable) grid_search_levels(g, q.x, q.y, q.z, best, INF);
        if (qi < nq) {
            idx[qi] = best.i;
            dist[qi] = best.d;
        }
    } else {
        BestK best;
        best.d = smem_lists + threadIdx.x;
        best.i = reinterpret_cast<int*>(smem_lists + (size_t)k * GRID_THREADS) + threadIdx.x;
        best.k = k;
        best.stride = GRID_THREADS;
        best.init();
        if (searchable) grid_search_levels(g, q.x, q.y, q.z, best, INF);
        __syncthreads();
        const float* sd = smem_lists;
        const int* si = reinterpret_cast<const int*>(smem_lists + (size_t)k * GRID_THREADS);
        const uint32_t live = min((uint32_t)GRID_THREADS, nq - q0);
        for (uint32_t e = threadIdx.x; e < live * (uint32_t)k; e += GRID_THREADS) {
            const uint32_t ql = e / (uint32_t)k, j = e - ql * (uint32_t)k;
            dist[(size_t)q0 * k + e] = sd[j * GRID_THREADS + ql];
            idx[(size_t)q0 * k + e] = si[j * GRID_THREADS + ql];
        }
    }
}

// k == 1, two passes (same split as the registration kernels, spx_registration.cu nn_search_grid):
// pass 1, one lane per query: first pass over the 3x3x3 block; unfinished queries go to a work list.
// pass 2, one warp per listed query: cooperative continuation over shells and coarser levels.
__global__ void __launch_bounds__(GRID_THREADS) grid_nn1_fast_kernel(const GridLevels g, const float4* __restrict__ queries,
                                                                     uint32_t nq, Xform T, int has_T, float max_radius,
                                                                     int32_t* __restrict__ idx, float* __restrict__ dist,
                                                                     uint32_t* __restrict__ worklist,
                                                                     unsigned int* __restrict__ wl_count) {
    const uint32_t qi = blockIdx.x * GRID_THREADS + threadIdx.x;
    const int lane = threadIdx.x & 31;
    bool pending = false;
    if (qi < nq) {
        float4 q = __ldg(queries + qi);
        if (has_T) q = transform_point(T, q);
        Best1 best;
        best.init();
        if (isfinite(q.x) && isfinite(q.y) && isfinite(q.z) && g.lv[0].n > 0)
            pending = !icp_fast(g, q.x, q.y, q.z, -1, nullptr, max_radius, best);
        idx[qi] = best.i;
        dist[qi] = best.d;
    }
    const unsigned m = __ballot_sync(0xffffffffu, pending);
    if (m) {
        unsigned int slot = 0;
        if (lane == __ffs(m) - 1) slot = atomicAdd(wl_count, (unsigned int)__popc(m));
        slot = __shfl_sync(0xffffffffu, slot, __ffs(m) - 1);
        if (pending) worklist[slot + __popc(m & ((1u << lane) - 1u))] = qi;
    }
}

__global__ void __launch_bounds__(GRID_THREADS) grid_nn1_coop_kernel(const GridLevels g, const float4* __restrict__ queries,
                                                                     Xform T, int has_T, float max_radius,
                                                                     int32_t* __restrict__ idx, float* __restrict__ dist,
                                                                     const uint32_t* __restrict__ worklist,
                                                                     const unsigned int* __restrict__ wl_count,
                                                                     unsigned int* __restrict__ wl_cursor) {
    const int lane = threadIdx.x & 31;
    const unsigned int n_slow = *wl_count;
    for (;;) {
        unsigned int k = 0;
        if (lane == 0) k = atomicAdd(wl_cursor, 1u);
        k = __shfl_sync(0xffffffffu, k, 0);
        if (k >= n_slow) break;
        const uint32_t qi = worklist[k];
        float4 q = __ldg(queries + qi);
        if (has_T) q = transform_point(T, q);
        Best1 best;
        best.i = idx[qi];
        best.d = dist[qi];
        icp_coop_search(g, q.x, q.y, q.z, best, max_radius);
        if (lane == 0) {
            idx[qi] = best.i;
            dist[qi] = best.d;
        }
    }
}

// 1 < k <= K: register-resident lists (BestR); the block stages its [queries][k] tile in shared
// memory and writes it out cooperatively so the global stores coalesce.
template <int K>
__global__ void __launch_bounds__(GRID_THREADS) grid_knn_reg_kernel(const GridLevels g, const float4* __restrict__ queries,
                                                                     uint32_t nq, int k, Xform T, int has_T,
                                                                     int32_t* __restrict__ idx, float* __restrict__ dist) {
    __shared__ float sd[K * GRID_THREADS];
    __shared__ int si[K * GRID_THREADS];
    const uint32_t q0 = blockIdx.x * GRID_THREADS;
    const uint32_t qi = q0 + threadIdx.x;
    const float INF = __int_as_float(0x7f800000);
    float4 q = make_float4(0.f, 0.f, 0.f, 1.f);
    if (qi < nq) {
        q = __ldg(queries + qi);
        if (has_T) q = transform_point(T, q);
    }
    BestR<K> best;
    best.init(k);
    if (qi < nq && isfinite(q.x) && isfinite(q.y) && isfinite(q.z) && g.lv[0].n > 0)
        grid_search_levels(g, q.x, q.y, q.z, best, INF);
    // slots K-k .. K-1 hold the k results in ascending order; row layout [j][thread] is conflict-free
#pragma unroll
    for (int j = 0; j < K; ++j) {
        if (j >= K - k) {
            sd[(j - (K - k)) * GRID_THREADS + threadIdx.x] = best.dist_at(j);
            si[(j - (K - k)) * GRID_THREADS + threadIdx.x] = best.idx_at(j);
        }
    }
    __syncthreads();
    const uint32_t live = min((uint32_t)GRID_THREADS, nq - q0);
    for (uint32_t e = threadIdx.x; e < live * (uint32_t)k; e += GRID_THREADS) {
        const uint32_t ql = e / (uint32_t)k, j = e - ql * (uint32_t)k;
        dist[(size_t)q0 * k + e] = sd[j * GRID_THREADS + ql];
        idx[(size_t)q0 * k + e] = si[j * GRID_THREADS + ql];
    }
}

// 1 < k <= K in two launches, the split the k = 1 search and the registration kernels use: queries
// the first pass cannot certify (not enough neighbours inside the 3x3x3 block: sparse regions,
// clustered in a few blocks) go to a work list and are searched again — from scratch, registers
// only — by a second kernel whose warps take 32 listed queries at a time, so the expensive queries
// are packed densely into warps (no idle lanes next to them) and spread over every SM.
template <int K>
__global__ void __launch_bounds__(GRID_THREADS) grid_knn_reg_first_kernel(const GridLevels g, const float4* __restrict__ queries,
                                                                           uint32_t nq, int k, Xform T, int has_T,
                                                                           int32_t* __restrict__ idx, float* __restrict__ dist,
                                                                           uint32_t* __restrict__ worklist,
                                                                           unsigned int* __restrict__ wl_count,
                                                                           unsigned long long* __restrict__ carry,
                                                                           unsigned int* __restrict__ wl_count_back) {
    const uint32_t qi = blockIdx.x * GRID_THREADS + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const float INF = __int_as_float(0x7f800000);
    bool pending = false;
    BestR<K> best;
    best.init(k);
    if (qi < nq) {
        float4 q = __ldg(queries + qi);
        if (has_T) q = transform_point(T, q);
        if (isfinite(q.x) && isfinite(q.y) && isfinite(q.z) && g.lv[0].n > 0)
            pending = !grid_first_pass(g.lv[0], q.x, q.y, q.z, best, INF);
        if (!pending) {
            int32_t* irow = idx + (size_t)qi * k;
            float* drow = dist + (size_t)qi * k;
#pragma unroll
            for (int j = 0; j < K; ++j)
                if (j >= K - k) {
                    irow[j - (K - k)] = best.idx_at(j);
                    drow[j - (K - k)] = best.dist_at(j);
                }
        }
    }
    // wl_count_back != null: queries that do not even HAVE k candidates yet (sparse surroundings: the expensive ones)
    // are listed from the front, the others from the back of the same array, and the list kernel drains front first
    // — the long queries start at once instead of forming the kernel's tail
    const bool sparse = pending && best.key[K - 1] == BestR<K>::EMPTY;
    const bool to_back = pending && wl_count_back != nullptr && !sparse;
    const bool to_front = pending && !to_back;
    const unsigned mf = __ballot_sync(0xffffffffu, to_front), mb = __ballot_sync(0xffffffffu, to_back);
    unsigned int w = 0;
    if (mf) {
        unsigned int slot = 0;
        if (lane == __ffs(mf) - 1) slot = atomicAdd(wl_count, (unsigned int)__popc(mf));
        slot = __shfl_sync(0xffffffffu, slot, __ffs(mf) - 1);
        if (to_front) w = slot + __popc(mf & ((1u << lane) - 1u));
    }
    if (mb) {
        unsigned int slot = 0;
        if (lane == __ffs(mb) - 1) slot = atomicAdd(wl_count_back, (unsigned int)__popc(mb));
        slot = __shfl_sync(0xffffffffu, slot, __ffs(mb) - 1);
        if (to_back) w = nq - 1u - (slot + __popc(mb & ((1u << lane) - 1u)));
    }
    if (pending) {
        // the list kernel resumes from this state instead of repeating the first pass
        worklist[w] = qi;
#pragma unroll
        for (int j = 0; j < K; ++j) carry[(size_t)j * nq + w] = best.key[j];
    }
}

constexpr int LIST_LANES = 16;
template <int K>
__global__ void __launch_bounds__(GRID_THREADS) grid_knn_reg_list_kernel(const GridLevels g, const float4* __restrict__ queries,
                                                                          uint32_t nq, int k, Xform T, int has_T,
                                                                          int32_t* __restrict__ idx, float* __restrict__ dist,
                                                                          const uint32_t* __restrict__ worklist,
                                                                          const unsigned int* __restrict__ wl_count,
                                                                          unsigned int* __restrict__ wl_cursor,
                                                                          uint32_t* __restrict__ far_list,
                                                                          unsigned int* __restrict__ far_count,
                                                                          const unsigned long long* __restrict__ carry,
                                                                          int list_levels, int list_rings0) {
    const int lane = threadIdx.x & 31;
    const float INF = __int_as_float(0x7f800000);
    const unsigned int n_slow = *wl_count;
    for (;;) {
        // LIST_LANES queries per warp and turn: fewer than 32 because a warp lasts as long as its slowest
        // lane and the list is short (a third of the queries) — more, shorter warps fill the machine better
        unsigned int base = 0;
        if (lane == 0) base = atomicAdd(wl_cursor, (unsigned int)LIST_LANES);
        base = __shfl_sync(0xffffffffu, base, 0);
        if (base >= n_slow) break;
        if (lane < LIST_LANES && base + lane < n_slow) {
            const uint32_t w = base + lane;
            const uint32_t qi = worklist[w];
            float4 q = __ldg(queries + qi);
            if (has_T) q = transform_point(T, q);
            BestR<K> best;
            best.dedup = false;
#pragma unroll
            for (int j = 0; j < K; ++j) best.key[j] = carry[(size_t)j * nq + w];
            // per lane, from where the earlier stages stopped, up to level `list_levels`; a query still
            // open after that has its k-th neighbour several coarse cells away and goes to the
            // warp-cooperative kernel
            if (grid_search_levels(g, q.x, q.y, q.z, best, INF, (NoStats*)nullptr, list_levels, true, list_rings0)) {
                int32_t* irow = idx + (size_t)qi * k;
                float* drow = dist + (size_t)qi * k;
#pragma unroll
                for (int j = 0; j < K; ++j)
                    if (j >= K - k) {
                        irow[j - (K - k)] = best.idx_at(j);
                        drow[j - (K - k)] = best.dist_at(j);
                    }
            } else {
                far_list[atomicAdd(far_count, 1u)] = qi;
            }
        }
    }
}

template <int K>
__global__ void __launch_bounds__(GRID_THREADS) grid_knn_far_kernel(const GridLevels g, const float4* __restrict__ queries, int k,
                                                                    Xform T, int has_T, int32_t* __restrict__ idx,
                                                                    float* __restrict__ dist, const uint32_t* __restrict__ far_list,
                                                                    const unsigned int* __restrict__ far_count,
                                                                    unsigned int* __restrict__ far_cursor) {
    const int lane = threadIdx.x & 31;
    const unsigned int n_far = *far_count;
    for (;;) {
        unsigned int t = 0;
        if (lane == 0) t = atomicAdd(far_cursor, 1u);
        t = __shfl_sync(0xffffffffu, t, 0);
        if (t >= n_far) break;
        const uint32_t qi = far_list[t];
        float4 q = __ldg(queries + qi);
        if (has_T) q = transform_point(T, q);
        knn_coop_search<K>(g, q.x, q.y, q.z, k, idx + (size_t)qi * k, dist + (size_t)qi * k);
    }
}

// ---- the queries the first pass could not certify, ONE WARP per query, bound-driven.
// The first pass leaves such a query with the candidates of its 3x3x3 block (its k-th best distance d_k, when it
// has k of them, is an UPPER bound of the answer's k-th distance).  Instead of walking shell after shell, the warp
//   * picks the finest (level, ring radius) whose scanned block certifies d_k — every point outside it is farther
//     than sqrt(d_k) — so that ONE scan finishes the query; a query with fewer than k candidates first grows its
//     block (ring 2, then the next coarser level's 3x3x3, ...) until it has k;
//   * looks up the (z, y) rows of that block 32 at a time (rows and x-ranges pruned against d_k, cells a finer ring
//     of the same level has already covered skipped), and scans their candidates 32 wide, load-balanced by a prefix
//     sum over the rows' counts;
//   * keeps a candidate only if (dist, index) sorts before the current k-th entry — few do — in a small
//     shared-memory buffer, and merges buffer and list by k rounds of a warp-wide minimum (equal (dist, index) keys,
//     i.e. the same point offered by two levels, leave together: duplicates vanish).
// The list lives one 64-bit key per lane ((dist bits << 32 | index) + 1, BestR's encoding): lanes K-k .. K-1 hold the k
// entries in ascending order.  Exactness: the stop test is grid_search's (k-th best strictly inside the scanned
// block's certified radius, or the whole grid seen), ties resolve by index through the key order.
constexpr int COOP_BUF = 64;
constexpr int COOP_U = 2;     // 32-candidate batches in flight per step
constexpr int COOP_RMAX = 5;  // largest ring radius on a level that is not the coarsest (11 cells < the next level's 12)

template <int K>
__global__ void __launch_bounds__(GRID_THREADS) grid_knn_coop_list_kernel(const GridLevels gl, const float4* __restrict__ queries,
                                                                          uint32_t nq, int k, Xform T, int has_T,
                                                                          int32_t* __restrict__ idx, float* __restrict__ dist,
                                                                          const uint32_t* __restrict__ worklist,
                                                                          const unsigned int* __restrict__ wl_count,
                                                                          unsigned int* __restrict__ wl_cursor,
                                                                          const unsigned long long* __restrict__ carry,
                                                                          const unsigned int* __restrict__ wl_count_back,
                                                                          uint32_t* __restrict__ dbg) {
    constexpr unsigned long long EMPTY = BestR<K>::EMPTY;
    const unsigned FULL = 0xffffffffu;
    const float INF = __int_as_float(0x7f800000);
    __shared__ unsigned long long sbuf[GRID_THREADS / 32][COOP_BUF];
    const int lane = threadIdx.x & 31;
    unsigned long long* buf = sbuf[threadIdx.x >> 5];
    const unsigned int n_front = *wl_count, n_slow = n_front + *wl_count_back;
    const int first = K - k;  // lane of the list's smallest entry
    for (;;) {
        unsigned int w = 0;
        if (lane == 0) w = atomicAdd(wl_cursor, 1u);
        w = __shfl_sync(FULL, w, 0);
        if (w >= n_slow) break;
        if (w >= n_front) w = nq - 1u - (w - n_front);  // the back part of the list
        const uint32_t qi = worklist[w];
        float4 q = __ldg(queries + qi);
        if (has_T) q = transform_point(T, q);
        unsigned long long mykey = (lane < K) ? carry[(size_t)lane * nq + w] : EMPTY;
        if (lane < first) mykey = 0ull;
        int nb = 0;  // accepted candidates waiting in the buffer
        uint32_t d_cands = 0, d_scans = 0, d_merges = 0, d_last = 0;
        const long long d_t0 = dbg ? clock64() : 0;

        auto merge = [&]() {
            // candidates of this lane: its list entry and up to two buffer entries
            unsigned long long c0 = (lane >= first && lane < K) ? mykey : EMPTY;
            unsigned long long c1 = lane < nb ? buf[lane] : EMPTY;
            unsigned long long c2 = lane + 32 < nb ? buf[lane + 32] : EMPTY;
            unsigned long long out = EMPTY;
            for (int t = 0; t < k; ++t) {
                unsigned long long m = c0 < c1 ? c0 : c1;
                m = c2 < m ? c2 : m;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const unsigned long long v = __shfl_xor_sync(FULL, m, o);
                    m = v < m ? v : m;
                }
                if (m != EMPTY) {  // every copy of this exact (dist, index) leaves
                    if (c0 == m) c0 = EMPTY;
                    if (c1 == m) c1 = EMPTY;
                    if (c2 == m) c2 = EMPTY;
                }
                if (lane == first + t) out = m;
            }
            mykey = lane < first ? 0ull : (lane < K ? out : EMPTY);
            nb = 0;
            ++d_merges;
            __syncwarp();
        };

        // scan every cell within Chebyshev radius r of the query's cell on level l that lies farther than r_done
        // (cells a previous scan of this level has covered; -1: none)
        auto scan = [&](const GridView& g, int r, int r_done) {
            const int cx = grid_coord(q.x, g.ox, g.inv, g.dx);
            const int cy = grid_coord(q.y, g.oy, g.inv, g.dy);
            const int cz = grid_coord(q.z, g.oz, g.inv, g.dz);
            const float margin = g.margin + 1e-6f * fmaxf(fmaxf(fabsf(q.x), fabsf(q.y)), fabsf(q.z));
            // rows (z, y) in CENTRE-OUT order (ring 0, ring 1, ...): near rows first, so the k-th best tightens early
            // and the far rows are pruned or rejected by one compare (a sweep from one face of the block offers
            // candidates in decreasing distance: half of them would enter the list)
            const int nrows = (2 * r + 1) * (2 * r + 1);
            for (int base = 0; base < nrows; base += 32) {
                unsigned long long kth = __shfl_sync(FULL, mykey, K - 1);
                const float lim2 = kth != EMPTY ? __uint_as_float((uint32_t)((kth - 1ull) >> 32)) : INF;
                const int t = base + lane;
                uint32_t sA = 0, eA = 0, sB = 0, eB = 0;
                int ddz = 0, ddy = 0;
                if (t > 0 && t < nrows) {
                    int rr = 1;
                    while ((2 * rr + 1) * (2 * rr + 1) <= t) ++rr;
                    const int pp = t - (2 * rr - 1) * (2 * rr - 1), side = 2 * rr, edge = pp / side, o = pp - edge * side;
                    ddz = edge == 0 ? -rr : (edge == 1 ? -rr + o : (edge == 2 ? rr : rr - o));
                    ddy = edge == 0 ? -rr + o : (edge == 1 ? rr : (edge == 2 ? rr - o : -rr));
                }
                const int zz = cz + ddz, yy = cy + ddy;
                if (t < nrows && zz >= 0 && zz < g.dz && yy >= 0 && yy < g.dy) {
                    const bool outer = max(abs(zz - cz), abs(yy - cy)) > r_done;  // no cell of this row seen before
                    int xa = max(cx - r, 0), xb = min(cx + r, g.dx - 1);
                    bool ok = true;
                    if (lim2 < 1.0e30f) {
                        const float gz = axis_gap(q.z, g.oz, g.cell, zz, g.dz);
                        const float gy = axis_gap(q.y, g.oy, g.cell, yy, g.dy);
                        const float gyz = fmaxf(sqrtf(__fmaf_rn(gz, gz, __fmul_rn(gy, gy))) - margin, 0.0f);
                        const float gyz2 = __fmul_rn(gyz, gyz);
                        ok = gyz2 <= lim2;
                        const float wd = sqrtf(fmaxf(lim2 - gyz2, 0.0f)) + margin;
                        xa = max(xa, grid_coord(q.x - wd, g.ox, g.inv, g.dx));
                        xb = min(xb, grid_coord(q.x + wd, g.ox, g.inv, g.dx));
                        ok = ok && xa <= xb;
                    }
                    if (ok) {
                        const uint32_t row = ((uint32_t)zz * (uint32_t)g.dy + (uint32_t)yy) * (uint32_t)g.dx;
                        if (outer) {
                            sA = __ldg(g.start + row + xa);
                            eA = __ldg(g.start + row + xb + 1);
                        } else {  // only the cells beyond the ring already covered: two ends of the row
                            const int la = xa, lb = min(xb, cx - r_done - 1);
                            const int ra = max(xa, cx + r_done + 1), rb = xb;
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
                // LONG rows (coarse levels: a row can hold thousands of points) are strided by the whole warp, four
                // loads per lane in flight, no per-candidate bookkeeping; the others share the prefix-sum path below
                {
                    unsigned longm = __ballot_sync(FULL, (eA - sA) + (eB - sB) >= 128u);
                    while (longm) {
                        const int src = __ffs(longm) - 1;
                        longm &= longm - 1;
#pragma unroll
                        for (int seg = 0; seg < 2; ++seg) {
                            const uint32_t a0 = __shfl_sync(FULL, seg ? sB : sA, src), b0 = __shfl_sync(FULL, seg ? eB : eA, src);
                            d_cands += b0 - a0;
                            for (uint32_t jb = a0; jb < b0; jb += 128) {  // warp-uniform trip count
                                const uint32_t j = jb + lane;
                                float4 p4[4];
#pragma unroll
                                for (int u = 0; u < 4; ++u)
                                    if (j + 32 * u < b0) p4[u] = __ldg(g.pts + j + 32 * u);
#pragma unroll
                                for (int u = 0; u < 4; ++u) {
                                    if (jb + 32 * u >= b0) continue;  // warp-uniform
                                    if (nb > COOP_BUF - 32) merge();
                                    const unsigned long long kth4 = __shfl_sync(FULL, mykey, K - 1);
                                    bool take = false;
                                    unsigned long long c4 = EMPTY;
                                    if (j + 32 * u < b0) {
                                        const float ds = dist_sq(q.x, q.y, q.z, p4[u].x, p4[u].y, p4[u].z);
                                        c4 = (((unsigned long long)__float_as_uint(ds) << 32) |
                                              (unsigned long long)(uint32_t)__float_as_int(p4[u].w)) + 1ull;
                                        take = c4 < kth4;
                                    }
                                    const unsigned m = __ballot_sync(FULL, take);
                                    if (take) buf[nb + __popc(m & ((1u << lane) - 1u))] = c4;
                                    nb += __popc(m);
                                    __syncwarp();
                                }
                            }
                        }
                        if (lane == src) sA = eA = sB = eB = 0u;
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
                d_cands += total;
                // COOP_U x 32 candidates per step, their loads issued together: a coarse block can hold thousands of
                // candidates, and one load per step is one L2 round trip per 32 of them
                for (uint32_t cb = 0; cb < total; cb += 32 * COOP_U) {
                    unsigned long long ck[COOP_U];
                    float4 pp[COOP_U];
                    bool live[COOP_U];
#pragma unroll
                    for (int u = 0; u < COOP_U; ++u) {
                        const uint32_t kk = cb + u * 32 + lane;
                        live[u] = kk < total;
                        pp[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (cb + u * 32 >= total) continue;  // warp-uniform
                        const uint32_t key = live[u] ? kk : 0u;
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
                        if (live[u]) {
                            const uint32_t jj = key - (o_inc - o_cnt);
                            const uint32_t pos = jj < o_cA ? o_sA + jj : o_sB + (jj - o_cA);
                            pp[u] = __ldg(g.pts + pos);
                        }
                    }
#pragma unroll
                    for (int u = 0; u < COOP_U; ++u) {
                        const float ds = dist_sq(q.x, q.y, q.z, pp[u].x, pp[u].y, pp[u].z);
                        ck[u] = live[u] ? (((unsigned long long)__float_as_uint(ds) << 32) |
                                           (unsigned long long)(uint32_t)__float_as_int(pp[u].w)) + 1ull
                                        : EMPTY;
                    }
#pragma unroll
                    for (int u = 0; u < COOP_U; ++u) {
                        if (cb + u * 32 >= total) continue;  // warp-uniform
                        if (nb > COOP_BUF - 32) merge();
                        kth = __shfl_sync(FULL, mykey, K - 1);
                        const bool take = ck[u] < kth;
                        const unsigned m = __ballot_sync(FULL, take);
                        if (take) buf[nb + __popc(m & ((1u << lane) - 1u))] = ck[u];
                        nb += __popc(m);
                        __syncwarp();
                    }
                }
            }
            if (nb) merge();
        };

        int l_min = 0;      // never go back to a finer level
        int r_done = 1;     // level 0: the first pass covered ring 1 completely
        for (;;) {
            const unsigned long long kth = __shfl_sync(FULL, mykey, K - 1);
            const bool full = kth != EMPTY;
            const float d_k = full ? __uint_as_float((uint32_t)((kth - 1ull) >> 32)) : INF;
            int L = l_min, R = r_done + 1;
            bool found = false;
            if (full) {
                // the finest block that certifies d_k
                for (int l = l_min; l < gl.n_levels && !found; ++l) {
                    const GridView& g = gl.lv[l];
                    const bool last = l == gl.n_levels - 1;
                    const int cx = grid_coord(q.x, g.ox, g.inv, g.dx);
                    const int cy = grid_coord(q.y, g.oy, g.inv, g.dy);
                    const int cz = grid_coord(q.z, g.oz, g.inv, g.dz);
                    const float margin = g.margin + 1e-6f * fmaxf(fmaxf(fabsf(q.x), fabsf(q.y)), fabsf(q.z));
                    const int r_first = (l == l_min) ? r_done + 1 : 1;
                    const int r_last = last ? (1 << 20) : COOP_RMAX;
                    for (int r = r_first; r <= r_last; ++r) {
                        const float bound = fminf(fminf(shell_bound_axis(q.x, g.ox, g.cell, cx, r, g.dx),
                                                        shell_bound_axis(q.y, g.oy, g.cell, cy, r, g.dy)),
                                                  shell_bound_axis(q.z, g.oz, g.cell, cz, r, g.dz));
                        const float bs = bound - margin;
                        if (bound == INF || (bs > 0.0f && d_k < __fmul_rn(bs, bs))) {
                            L = l;
                            R = r;
                            found = true;
                            break;
                        }
                    }
                }
            }
            if (!found) {
                // fewer than k candidates so far: the smallest block of the growth sequence (rings r_done+1 .. COOP_RMAX
                // of this level, then rings 1 .. COOP_RMAX of the next coarser one, ...; the coarsest level grows until
                // the grid is covered) that HOLDS at least k points — counted from the rows' cell ranges, one round trip
                // per 32 rows, nothing scanned: an isolated query crosses empty space without touching a point
                int l = l_min, r = r_done;
                for (;;) {
                    const bool last = l == gl.n_levels - 1;
                    if (last || r < COOP_RMAX) {
                        ++r;
                    } else {
                        ++l;
                        r = 1;
                    }
                    const GridView& g = gl.lv[l];
                    const int cx = grid_coord(q.x, g.ox, g.inv, g.dx);
                    const int cy = grid_coord(q.y, g.oy, g.inv, g.dy);
                    const int cz = grid_coord(q.z, g.oz, g.inv, g.dz);
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
                    if (c >= (uint32_t)k || whole) break;
                }
                L = l;
                R = r;
            }
            const GridView& g = gl.lv[L];
            ++d_scans;
            d_last = (uint32_t)(L * 100 + R) + (full ? 0u : 10000u);
            scan(g, R, L == l_min ? r_done : -1);
            l_min = L;
            r_done = R;
            // stop test of the block just completed (grid_search's)
            {
                const int cx = grid_coord(q.x, g.ox, g.inv, g.dx);
                const int cy = grid_coord(q.y, g.oy, g.inv, g.dy);
                const int cz = grid_coord(q.z, g.oz, g.inv, g.dz);
                const float margin = g.margin + 1e-6f * fmaxf(fmaxf(fabsf(q.x), fabsf(q.y)), fabsf(q.z));
                const float bound = fminf(fminf(shell_bound_axis(q.x, g.ox, g.cell, cx, R, g.dx),
                                                shell_bound_axis(q.y, g.oy, g.cell, cy, R, g.dy)),
                                          shell_bound_axis(q.z, g.oz, g.cell, cz, R, g.dz));
                if (bound == INF) break;  // whole grid visited
                const unsigned long long kth2 = __shfl_sync(FULL, mykey, K - 1);
                const float bs = bound - margin;
                if (kth2 != EMPTY && bs > 0.0f && __uint_as_float((uint32_t)((kth2 - 1ull) >> 32)) < __fmul_rn(bs, bs)) break;
            }
        }
        if (dbg && lane == 0) {
            dbg[(size_t)w * 6 + 0] = d_cands;
            dbg[(size_t)w * 6 + 1] = d_scans;
            dbg[(size_t)w * 6 + 2] = d_merges;
            dbg[(size_t)w * 6 + 3] = (uint32_t)(clock64() - d_t0);
            dbg[(size_t)w * 6 + 4] = d_last;
            dbg[(size_t)w * 6 + 5] = qi;
        }
        if (lane >= first && lane < K) {
            idx[(size_t)qi * k + (lane - first)] = (int)(uint32_t)((mykey - 1ull) & 0xffffffffull);
            dist[(size_t)qi * k + (lane - first)] = __uint_as_float((uint32_t)((mykey - 1ull) >> 32));
        }
    }
}

template <int K>
void launch_knn_reg(spx_index_t index, spx_queue_t q, const float4* qs, uint32_t nq, int k, const Xform& T, int has_T,
                    int32_t* idx, float* dist) {
    const GridLevels& levels = index->levels_knn;  // k >= 2: the first level is the k-NN grid
    q->arena_reset();
    q->arena_reserve((size_t)nq * (8 + 8 * K) + 8192);
    uint32_t* worklist = q->take<uint32_t>(nq);
    uint32_t* far_list = q->take<uint32_t>(nq);
    unsigned long long* carry = q->take<unsigned long long>((size_t)nq * K);  // [K][nq]: first-pass lists of the pending
    int list_levels = 2, list_rings0 = GRID_LEVEL_RINGS;  // tuning aids
    if (const char* e = std::getenv("SPX_KNN_LIST_LEVELS")) list_levels = std::atoi(e);
    if (const char* e = std::getenv("SPX_KNN_LIST_RINGS0")) list_rings0 = std::atoi(e);
    unsigned int* counters = q->take<unsigned int>(16);  // {list count, list cursor, far count, far cursor, back count}
    SPX_CUDA(cudaMemsetAsync(counters, 0, 8 * sizeof(unsigned int), q->stream));
    static const bool legacy = std::getenv("SPX_KNN_LEGACY_LIST") != nullptr;  // tuning aid: the per-lane list + far kernels
    grid_knn_reg_first_kernel<K><<<div_up(nq, GRID_THREADS), GRID_THREADS, 0, q->stream>>>(levels, qs, nq, k, T, has_T, idx,
                                                                                         dist, worklist, counters, carry, legacy ? nullptr : counters + 4);
    SPX_LAUNCH_CHECK();
    if (!legacy) {
        // one warp per unfinished query, bound-driven (resident grid: the warps pull queries off the list)
        uint32_t* dbg = nullptr;
        static const bool debug = std::getenv("SPX_KNN_DEBUG") != nullptr;  // tuning aid: per-query work of the list kernel
        if (debug) {
            SPX_CUDA(cudaMalloc(&dbg, (size_t)nq * 6 * sizeof(uint32_t)));
            SPX_CUDA(cudaMemsetAsync(dbg, 0, (size_t)nq * 6 * sizeof(uint32_t), q->stream));
        }
        grid_knn_coop_list_kernel<K><<<q->sm_count * 16, GRID_THREADS, 0, q->stream>>>(levels, qs, nq, k, T, has_T, idx, dist,
                                                                                   worklist, counters, counters + 1, carry, counters + 4, dbg);
        if (debug) {
            SPX_LAUNCH_CHECK();
            std::vector<uint32_t> h((size_t)nq * 6);
            unsigned int hc[4];
            SPX_CUDA(cudaMemcpyAsync(h.data(), dbg, h.size() * 4, cudaMemcpyDeviceToHost, q->stream));
            SPX_CUDA(cudaMemcpyAsync(hc, counters, sizeof(hc), cudaMemcpyDeviceToHost, q->stream));
            SPX_CUDA(cudaStreamSynchronize(q->stream));
            cudaFree(dbg);
            std::vector<size_t> order(nq);
            for (size_t i = 0; i < order.size(); ++i) order[i] = i;
            std::sort(order.begin(), order.end(), [&](size_t a, size_t b) { return h[a * 6 + 3] > h[b * 6 + 3]; });
            unsigned long long tc = 0, tcy = 0;
            for (size_t i = 0; i < order.size(); ++i) { tc += h[i * 6]; tcy += h[i * 6 + 3]; }
            fprintf(stderr, "[knn debug] nq %u listed %u total cands %llu mean cycles %llu\n", nq, hc[0], tc, order.empty() ? 0ull : tcy / order.size());
            for (size_t i = 0; i < std::min<size_t>(12, order.size()); ++i) {
                const uint32_t* e = &h[order[i] * 6];
                fprintf(stderr, "   q %u: cands %u scans %u merges %u cycles %u last(L*100+R,+10000 notfull) %u\n", e[5], e[0], e[1], e[2], e[3], e[4]);
            }
        }
        return;
    }
    grid_knn_reg_list_kernel<K><<<q->sm_count * 16, GRID_THREADS, 0, q->stream>>>(
        levels, qs, nq, k, T, has_T, idx, dist, worklist, counters, counters + 1, far_list, counters + 2, carry,
        list_levels, list_rings0);
    SPX_LAUNCH_CHECK();
    grid_knn_far_kernel<K><<<q->sm_count, GRID_THREADS, 0, q->stream>>>(levels, qs, k, T, has_T, idx, dist, far_list,
                                                                       counters + 2, counters + 3);
}

// work counters of the k = 1 search (tuning aid): stats[q] = {segments, candidates, shells, last level}
__global__ void __launch_bounds__(GRID_THREADS) grid_nn_stats_kernel(const GridLevels g, const float4* __restrict__ queries,
                                                                      uint32_t nq, Xform T, int has_T, float max_radius,
                                                                      uint4* __restrict__ stats) {
    const uint32_t qi = blockIdx.x * GRID_THREADS + threadIdx.x;
    if (qi >= nq) return;
    float4 q = __ldg(queries + qi);
    if (has_T) q = transform_point(T, q);
    Best1 best;
    best.init();
    CountStats cs;
    if (isfinite(q.x) && isfinite(q.y) && isfinite(q.z) && g.lv[0].n > 0)
        grid_search_levels(g, q.x, q.y, q.z, best, max_radius, &cs);
    stats[qi] = make_uint4(cs.segs, cs.cands, cs.shells, cs.last_level);
}

// radius search = the max_k nearest within the radius: entries farther than radius^2 become unfilled (-1 / FLT_MAX),
// kdtree.hpp:564-720 (dist_sq <= radius_sq is kept, :663,678)
__global__ void __launch_bounds__(256) radius_mask_kernel(int32_t* __restrict__ idx, float* __restrict__ dist, size_t n,
                                                          float radius_sq) {
    const size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    if (!(dist[i] <= radius_sq)) {
        idx[i] = -1;
        dist[i] = FLT_MAX;
    }
}

// remove_nodes_by_flags — kdtree.hpp:282-284,721-760: the kept points, re-numbered by `new_index`, gathered out of the
// index's own sorted copy (level 0 holds every finite point once, its original index in w)
__global__ void __launch_bounds__(256) index_kept_points_kernel(const float4* __restrict__ sorted, uint32_t n,
                                                                const uint8_t* __restrict__ flags,
                                                                const int32_t* __restrict__ new_index, size_t n_flags,
                                                                float4* __restrict__ out) {
    const uint32_t j = blockIdx.x * 256 + threadIdx.x;
    if (j >= n) return;
    const float4 p = __ldg(sorted + j);
    const int orig = __float_as_int(p.w);
    if (orig < 0 || (size_t)orig >= n_flags) return;
    if (flags[orig] == 1) {  // filter::INCLUDE_FLAG
        const int ni = new_index[orig];
        if (ni >= 0) out[ni] = make_float4(p.x, p.y, p.z, 1.0f);
    }
}

void launch_bruteforce(spx_queue_t q, const float4* queries, uint32_t nq, const float4* targets, uint32_t nt, int k,
                       const Xform& T, int has_T, int32_t* idx, float* dist) {
    if (nq == 0) return;
    // Two queries per thread as ONE packed-FP32 stream, the k-th-best test every two targets: measured best on
    // 1 M x 1 M, k = 20 (profiles/r2k_bf_variants.txt, r2l: p2/batch 2 257 ms; p4/batch 2 305; p2/batch 4 278;
    // p4/batch 4 404; scalar q2 343, q1 359) — more queries per thread or a longer batch make the (rare, but
    // warp-wide) insertion path fire more often than the saved shared-memory reads are worth.  Small query sets keep
    // one query per thread so the grid still covers the SMs.  SPX_BF_VARIANT (tuning): "q1", "q2", "q4", "q8", "p2",
    // "p4", "p8" force a variant, SPX_BF_BATCH the number of targets per k-th-best test.
    int qpt = nq >= (uint32_t)q->sm_count * BF_THREADS * 4 ? 2 : 1;
    bool packed = qpt >= 2;
    if (const char* e = std::getenv("SPX_BF_VARIANT")) {
        packed = e[0] == 'p';
        qpt = e[1] == '8' ? 8 : (e[1] == '4' ? 4 : (e[1] == '2' ? 2 : 1));
        if (qpt == 1) packed = false;
    }
    const unsigned blocks = (unsigned)div_up(nq, (size_t)BF_THREADS * qpt);
    // TMA-staged, double-buffered tiles (2 x 1024 targets of shared memory per block) whenever the targets are 16-byte aligned
    // — every cudaMalloc'ed cloud is; SPX_BF_TMA=0 keeps the synchronous staging (tuning aid)
    static const bool allow_tma = !(std::getenv("SPX_BF_TMA") && std::getenv("SPX_BF_TMA")[0] == '0');
    const bool tma = allow_tma && (reinterpret_cast<uintptr_t>(targets) % 16 == 0);
#define SPX_BF_LAUNCH(Q, P)                                                                                              \
    do {                                                                                                                 \
        if (tma)                                                                                                         \
            knn_bruteforce_kernel<Q, P, true><<<blocks, BF_THREADS, 0, q->stream>>>(queries, nq, targets, nt, k, T, has_T, \
                                                                                    idx, dist);                         \
        else                                                                                                             \
            knn_bruteforce_kernel<Q, P, false><<<blocks, BF_THREADS, 0, q->stream>>>(queries, nq, targets, nt, k, T,      \
                                                                                     has_T, idx, dist);                 \
    } while (0)
    int batch = (packed && qpt == 2) ? 2 : BF_BATCH;
    if (const char* e = std::getenv("SPX_BF_BATCH")) batch = std::atoi(e);  // tuning aid (packed TMA variants only)
#define SPX_BF_LAUNCH_B(Q, B)                                                                                        \
    knn_bruteforce_kernel<Q, true, true, B><<<blocks, BF_THREADS, 0, q->stream>>>(queries, nq, targets, nt, k, T, has_T, \
                                                                                  idx, dist)
    if (tma && packed && qpt == 2 && batch == 1) SPX_BF_LAUNCH_B(2, 1);
    else if (tma && packed && qpt == 4 && batch == 1) SPX_BF_LAUNCH_B(4, 1);
    else if (tma && packed && qpt == 2 && batch == 2) SPX_BF_LAUNCH_B(2, 2);
    else if (tma && packed && qpt == 2 && batch == 8) SPX_BF_LAUNCH_B(2, 8);
    else if (tma && packed && qpt == 4 && batch == 2) SPX_BF_LAUNCH_B(4, 2);
    else if (tma && packed && qpt == 4 && batch == 8) SPX_BF_LAUNCH_B(4, 8);
    else if (qpt == 8 && packed) SPX_BF_LAUNCH(8, true);
    else if (qpt == 8) SPX_BF_LAUNCH(8, false);
    else if (qpt == 4 && packed) SPX_BF_LAUNCH(4, true);
    else if (qpt == 4) SPX_BF_LAUNCH(4, false);
    else if (qpt == 2 && packed) SPX_BF_LAUNCH(2, true);
    else if (qpt == 2) SPX_BF_LAUNCH(2, false);
    else SPX_BF_LAUNCH(1, false);
#undef SPX_BF_LAUNCH_B
#undef SPX_BF_LAUNCH
    SPX_LAUNCH_CHECK();
}

// dense-grid budget of the finest level: 64 cells per point, at least 2^24, at most 2^28 (the `start`
// array is 4 B per cell — 1 GiB at the cap, against 180 GB of HBM).  LiDAR clouds are surfaces in a
// mostly empty bounding box, so the cell count grows much faster than the point count as the cell
// edge shrinks; a budget that is too small forces cells with tens of points each (measured on the
// 1.5 M-point config-4 cloud: 10 points per occupied cell at 2^24 cells).
inline size_t max_cells_for(size_t n) {
    return std::min<size_t>((size_t)1 << 28, std::max<size_t>((size_t)1 << 24, n * 64));
}

}  // namespace

extern "C" {

int spx_knn_bruteforce(spx_queue_t q, const float* queries, size_t nq, const float* targets, size_t nt, int k,
                       const float* T_host, int32_t* idx, float* dist) {
    return guard([&] {
        SPX_REQUIRE(q, "[knn_search_bruteforce] null queue");
        SPX_REQUIRE(k >= 1 && k <= 128, "[knn_search_bruteforce] `k` must be in [1, 128]");
        SPX_REQUIRE(nq < (1ull << 31) && nt < (1ull << 31), "[knn_search_bruteforce] too many points");
        if (nq == 0) return;
        SPX_REQUIRE(queries && idx && dist && (targets || nt == 0), "[knn_search_bruteforce] null pointer");
        DeviceGuard g(q->device);
        const Xform T = T_host ? xform_from_colmajor(T_host) : xform_identity();
        launch_bruteforce(q, reinterpret_cast<const float4*>(queries), (uint32_t)nq,
                          reinterpret_cast<const float4*>(targets), (uint32_t)nt, k, T, T_host != nullptr, idx, dist);
    });
}

namespace {
// a caller that already knows a box containing the points (e.g. the voxel box of a down-sampled cloud) and the cell
// edges it wants skips the build's first phase — bounding box, occupancy curve, and the host round trip that sizes
// the grid.  A box that misses points is harmless for exactness (cell coordinates clamp into the grid, and every bound
// of the searches is a lower bound on clamped points), it only costs speed.
struct BuildHint {
    float lo[3], hi[3];
    float cell, cell_knn;
};
int index_build_impl(spx_queue_t q, const float* targets, size_t nt, float cell_size, const BuildHint* hint, spx_index_t* out);
}  // namespace

int spx_index_build(spx_queue_t q, const float* targets, size_t nt, float cell_size, spx_index_t* out) {
    return index_build_impl(q, targets, nt, cell_size, nullptr, out);
}

int spx_index_build_hinted(spx_queue_t q, const float* targets, size_t nt, const float* lo3_host, const float* hi3_host,
                           float cell_size, float knn_cell_size, spx_index_t* out) {
    if (!lo3_host || !hi3_host || !(cell_size > 0.0f)) {
        set_last_error("[KDTree::build] hinted build needs a box and a positive cell size");
        return SPX_ERR_INVALID_ARGUMENT;
    }
    BuildHint h;
    for (int a = 0; a < 3; ++a) {
        h.lo[a] = lo3_host[a];
        h.hi[a] = hi3_host[a];
        if (!(h.hi[a] >= h.lo[a]) || !std::isfinite(h.lo[a]) || !std::isfinite(h.hi[a])) {
            set_last_error("[KDTree::build] hinted build: the box is empty or not finite");
            return SPX_ERR_INVALID_ARGUMENT;
        }
    }
    h.cell = cell_size;
    h.cell_knn = knn_cell_size;
    return index_build_impl(q, targets, nt, cell_size, &h, out);
}

namespace {
int index_build_impl(spx_queue_t q, const float* targets, size_t nt, float cell_size, const BuildHint* hint, spx_index_t* out) {
    if (out) *out = nullptr;
    return guard([&] {
        SPX_REQUIRE(q && out, "[KDTree::build] null argument");
        SPX_REQUIRE(nt < (1ull << 31), "[KDTree::build] too many points");
        SPX_REQUIRE(targets || nt == 0, "[KDTree::build] null points");
        DeviceGuard dg(q->device);
        // the handle reaches the caller only when the build succeeded: a throw below (budget checks, allocation
        // failures) releases what was allocated so far instead of leaking a half-built index
        struct Holder {
            spx_index_s* p;
            spx_index_t* out;
            bool done = false;
            ~Holder() {
                if (done) {
                    if (!p->ready) cudaEventCreateWithFlags(&p->ready, cudaEventDisableTiming);
                    if (p->ready) cudaEventRecord(p->ready, p->q->stream);
                    *out = p;
                    return;
                }
                for (int l = 0; l < GRID_MAX_LEVELS; ++l) {
                    if (p->sorted[l]) cudaFreeAsync(p->sorted[l], p->q->stream);
                    if (p->start[l]) cudaFreeAsync(p->start[l], p->q->stream);
                }
                if (p->occ_dev) cudaFreeAsync(p->occ_dev, p->q->stream);
                delete p;
            }
        };
        auto* ix = new spx_index_s();
        ix->q = q;
        ix->n_total = nt;
        Holder holder{ix, out};
        GridLevels& L = ix->levels;
        L = GridLevels{};
        L.n_levels = 1;
        L.lv[0].dx = L.lv[0].dy = L.lv[0].dz = 1;
        L.lv[0].cell = 1.0f;
        L.lv[0].inv = 1.0f;
        ix->levels_knn = L;
        if (nt == 0) {  // empty tree: every search returns -1 / FLT_MAX (kdtree.hpp:296-300)
            holder.done = true;
            return;
        }
        const float4* pts = reinterpret_cast<const float4*>(targets);
        const uint32_t n = (uint32_t)nt;
        cudaStream_t st = q->stream;

        const size_t MAX_CELLS = max_cells_for(n);
        // scratch: bbox accumulator, occupancy plan + bitmaps + counters, per-point cell ids, per-cell counts
        uint32_t map_bits = 1u << 16;
        while (map_bits < 8u * n && map_bits < (1u << 30)) map_bits <<= 1;
        const uint32_t words_per_map = map_bits / 32u;
        q->arena_reset();
        q->arena_reserve(sizeof(BuildHead) + 1024 + (size_t)OCC_CANDS * words_per_map * 4 +
                         (2 * MAX_CELLS + MAX_CELLS / 32 + MAX_CELLS / 1024 + 384) * 4 + 8192);
        BuildHead* head = q->take<BuildHead>(1);
        OccPlan* plan = &head->plan;
        unsigned int* ones = head->ones;
        uint32_t* bitmaps = q->take<uint32_t>((size_t)OCC_CANDS * words_per_map);
        uint32_t* counts = q->take<uint32_t>(2 * MAX_CELLS + MAX_CELLS / 32 + MAX_CELLS / 1024 + 384);

        BuildHead* hhead = static_cast<BuildHead*>(q->pinned_get(1024));
        unsigned int* hones = hhead->ones;
        const bool adaptive = !(cell_size > 0.0f);
        if (hint) {
            // everything the first phase would have measured, from the caller's box: no kernel, no round trip
            std::memset(hhead, 0, sizeof(BuildHead));
            hhead->acc.finite = n;  // (non-finite points are skipped by the counting kernels; only capacities use this)
            float max_abs = 0.0f;
            for (int a = 0; a < 3; ++a) {
                hhead->plan.lo[a] = hint->lo[a];
                hhead->plan.ext[a] = hint->hi[a] - hint->lo[a];
                max_abs = std::max(max_abs, std::max(std::fabs(hint->lo[a]), std::fabs(hint->hi[a])));
            }
            hhead->plan.max_abs = max_abs;
            hhead->plan.c0 = hint->cell;
        } else {
        // accumulators, ticket and counters start as zero bits: one memset clears them together with the
        // occupancy bitmaps behind them; the bounding-box kernel's last block derives the occupancy plan
        SPX_CUDA(cudaMemsetAsync(head, 0,
                                 adaptive ? (size_t)(reinterpret_cast<char*>(bitmaps + (size_t)OCC_CANDS * words_per_map) -
                                                     reinterpret_cast<char*>(head))
                                          : sizeof(BuildHead),
                                 st));
        bbox_kernel<<<std::min(div_up(n, 256), q->sm_count * 8), 256, 0, st>>>(pts, n, head);
        SPX_LAUNCH_CHECK();
        if (adaptive) {
            occ_mark_kernel<<<div_up(n, 256), 256, 0, st>>>(pts, n, plan, bitmaps, words_per_map);
            SPX_LAUNCH_CHECK();
            occ_count_kernel<<<dim3(std::min(div_up(words_per_map, 256), 64), OCC_CANDS), 256, 0, st>>>(bitmaps, words_per_map,
                                                                                                       ones);
            SPX_LAUNCH_CHECK();
        }
        SPX_CUDA(cudaMemcpyAsync(hhead, head, sizeof(BuildHead), cudaMemcpyDeviceToHost, st));
        q->sync();  // the only host round trip of the build: grid dimensions size the allocations
        }
        const BBoxAcc bb = hhead->acc;
        const OccPlan pl = hhead->plan;
        ix->n = bb.finite;
        L.lv[0].n = bb.finite;
        if (bb.finite == 0) {
            holder.done = true;
            return;
        }

        float lo[3], ext[3];
        float max_ext = 0.0f;
        const float max_abs = pl.max_abs;
        for (int a = 0; a < 3; ++a) {
            lo[a] = pl.lo[a];
            ext[a] = pl.ext[a];
            max_ext = std::max(max_ext, ext[a]);
        }
        if (!(max_ext > 0.0f)) max_ext = 1.0f;

        auto dims_for = [&](float cell, int dims[3]) {
            double nc = 1.0;
            for (int a = 0; a < 3; ++a) {
                const double d = std::floor((double)ext[a] / (double)cell) + 1.0;
                dims[a] = (int)std::min(d, 2.0e9);
                nc *= d;
            }
            return nc;
        };
        // finest level: the cell edge at which an occupied cell holds ~3 points (measured optimum on
        // LiDAR-shaped clouds for both the k = 10 and the warm-started k = 1 searches: smaller cells
        // send more queries past the first pass, larger ones add candidates to every query), read off
        // the measured occupancy curve by log-log interpolation between the candidates
        // occupancy curve -> cell edge at which an occupied cell holds `want` points
        auto cell_for = [&](double want) {
            double avg[OCC_CANDS];
            for (int j = 0; j < OCC_CANDS; ++j) {
                const double zeros = (double)map_bits - (double)hones[j];
                const double occ = zeros >= 1.0 ? -(double)map_bits * std::log(zeros / (double)map_bits)
                                                : (double)map_bits * std::log((double)map_bits);
                avg[j] = (double)bb.finite / std::max(occ, 1.0);
            }
            static const double F[OCC_CANDS] = {0.35, 0.5, 0.7071, 1.0, 1.4142, 2.0, 2.8284, 4.0};
            double f = F[OCC_CANDS - 1];
            if (avg[0] >= want) {
                f = F[0];
            } else {
                for (int j = 0; j + 1 < OCC_CANDS; ++j)
                    if (avg[j] < want && avg[j + 1] >= want) {
                        const double t = (std::log(want) - std::log(avg[j])) / std::max(std::log(avg[j + 1]) - std::log(avg[j]), 1e-9);
                        f = std::exp(std::log(F[j]) + t * (std::log(F[j + 1]) - std::log(F[j])));
                        break;
                    }
            }
            if (bb.finite <= 8) f = 1.0;
            float c = (float)(pl.c0 * f);
            return std::max(c, 1e-6f * std::max(max_abs, 1.0f));
        };
        float cell = cell_size;
        float cell_knn = 0.0f;  // edge of the extra first-pass grid of the k >= 2 searches (0: none)
        if (hint) {
            cell_knn = hint->cell_knn;
        } else if (adaptive) {
            double want = 3.0, want_knn = 5.0;
            if (const char* e = std::getenv("SPX_CELL_TARGET")) want = std::max(0.5, std::atof(e));          // tuning aids
            if (const char* e = std::getenv("SPX_KNN_CELL_TARGET")) want_knn = std::max(0.0, std::atof(e));
            cell = cell_for(want);
            // A k-nearest-neighbour search (k ~ 10-20: the covariance stage) wants larger cells than the k = 1 search
            // of the registration loop: with ~3 points per occupied cell a third of the k = 10 queries cannot be
            // certified from their 3x3x3 block, with ~5 almost all can (measured: 0.19 -> 0.12 ms at 120 k points),
            // while the registration iteration slows down by 15 % on such cells.  The index therefore carries ONE
            // more grid, used only as the first level of the k >= 2 searches.
            if (want_knn > want * 1.05 && bb.finite > 64) cell_knn = cell_for(want_knn);
        }
        int dims[3];
        for (;;) {  // respect the dense-grid budget
            const double nc = dims_for(cell, dims);
            if (nc <= (double)MAX_CELLS) break;
            cell *= (float)std::cbrt(nc / (double)MAX_CELLS) * 1.02f;
        }
        // level geometry: the finest grid, then grids GRID_LEVEL_FACTOR x coarser until only a few cells wide
        LevelSet ls{};
        float cells[GRID_MAX_LEVELS];
        int level = 0;
        size_t total_cells = 0;
        for (;;) {
            ls.geom[level] = GridGeom{lo[0], lo[1], lo[2], 1.0f / cell, dims[0], dims[1], dims[2]};
            ls.cell_base[level] = (uint32_t)total_cells;
            cells[level] = cell;
            ix->ncells[level] = (size_t)dims[0] * dims[1] * dims[2];
            total_cells += ix->ncells[level];
            if (level + 1 >= GRID_MAX_LEVELS || std::max(dims[0], std::max(dims[1], dims[2])) <= 4) break;
            ++level;
            cell *= (float)GRID_LEVEL_FACTOR;
            dims_for(cell, dims);
        }
        const int n_regular = level + 1;
        ls.n_levels = n_regular;
        int knn_dims[3] = {0, 0, 0};
        if (cell_knn > cells[0] * 1.02f && (n_regular < 2 || cell_knn < cells[1] * 0.9f)) {
            dims_for(cell_knn, knn_dims);
            ls.geom[n_regular] = GridGeom{lo[0], lo[1], lo[2], 1.0f / cell_knn, knn_dims[0], knn_dims[1], knn_dims[2]};
            ls.cell_base[n_regular] = (uint32_t)total_cells;
            total_cells += (size_t)knn_dims[0] * knn_dims[1] * knn_dims[2];
            ls.n_levels = n_regular + 1;
        } else {
            cell_knn = 0.0f;
        }
        ls.cell_base[ls.n_levels] = (uint32_t)total_cells;
        SPX_REQUIRE((unsigned long long)ls.n_levels * bb.finite < (1ull << 32) && total_cells + 1 < (1ull << 32),
                    "[KDTree::build] cloud too large for 32-bit index positions");
        // (counts / scan scratch were sized for MAX_CELLS of the finest level + the coarser ones: <= 1/63 more)
        SPX_REQUIRE(total_cells + 1 <= 2 * MAX_CELLS + MAX_CELLS / 32 + 64, "[KDTree::build] internal: cell budget exceeded");

        SPX_CUDA(cudaMallocAsync(&ix->start[0], (total_cells + 1) * 4, st));
        SPX_CUDA(cudaMallocAsync(&ix->sorted[0], (size_t)ls.n_levels * bb.finite * sizeof(float4), st));
        // per-cell counts and, right behind them, the zeroed ticket + status words of the one-launch scan
        const size_t scan_at = align_up(total_cells + 1, 2);
        SPX_REQUIRE(scan_at + scan_lookback_words(total_cells + 1) <= 2 * MAX_CELLS + MAX_CELLS / 32 + MAX_CELLS / 1024 + 384,
                    "[KDTree::build] internal: count buffer too small");
        SPX_CUDA(cudaMemsetAsync(counts, 0, (scan_at + scan_lookback_words(total_cells + 1)) * 4, st));
        levels_count_kernel<<<div_up(n, 256), 256, 0, st>>>(pts, n, ls, counts);
        SPX_LAUNCH_CHECK();
        exclusive_scan_u32_onepass(st, counts, ix->start[0], total_cells + 1, counts + scan_at, nullptr);
        levels_scatter_kernel<<<div_up(n, 256), 256, 0, st>>>(pts, n, ls, ix->start[0], counts, ix->sorted[0]);
        SPX_LAUNCH_CHECK();
        // (the points of a cell stay in the order the scatter's atomics handed out: every search orders its
        // candidates by (distance, original index), so no result depends on it)
        for (int l = 0; l < ls.n_levels; ++l) {
            const bool extra = l >= n_regular;  // the k-NN first-pass grid
            GridView knn_view{};
            GridView& v = extra ? knn_view : L.lv[l];
            const float cl = extra ? cell_knn : cells[l];
            v.ox = lo[0]; v.oy = lo[1]; v.oz = lo[2];
            v.cell = cl;
            v.inv = ls.geom[l].inv;
            v.dx = ls.geom[l].dx; v.dy = ls.geom[l].dy; v.dz = ls.geom[l].dz;
            v.margin = 1e-3f * cl + 2e-6f * (max_abs + max_ext);
            v.start = ix->start[0] + ls.cell_base[l];
            v.pts = ix->sorted[0];  // common base: `start` values of level l already include l * n
            v.n = bb.finite;
            if (extra) ix->levels_knn.lv[0] = knn_view;
        }
        L.n_levels = n_regular;
        // the level list of the k >= 2 searches: the extra grid first, then the regular levels above the finest
        if (cell_knn > 0.0f) {
            ix->levels_knn.n_levels = n_regular;
            for (int l = 1; l < n_regular; ++l) ix->levels_knn.lv[l] = L.lv[l];
        } else {
            ix->levels_knn = L;
        }
        // no final sync: everything above is ordered on the queue's stream, and so is every search on it; users on
        // other queues wait on `ready` (recorded by the holder)
        holder.done = true;
    });
}
}  // namespace

int spx_index_destroy(spx_index_t index) {
    return guard([&] {
        if (!index) return;
        if (queue_is_live(index->q)) {
            DeviceGuard g(index->q->device);
            for (int l = 0; l < GRID_MAX_LEVELS; ++l) {
                if (index->sorted[l]) cudaFreeAsync(index->sorted[l], index->q->stream);
                if (index->start[l]) cudaFreeAsync(index->start[l], index->q->stream);
            }
            if (index->occ_dev) cudaFreeAsync(index->occ_dev, index->q->stream);
        } else {  // the queue was destroyed first: synchronous frees
            for (int l = 0; l < GRID_MAX_LEVELS; ++l) {
                if (index->sorted[l]) cudaFree(index->sorted[l]);
                if (index->start[l]) cudaFree(index->start[l]);
            }
            if (index->occ_dev) cudaFree(index->occ_dev);
        }
        if (index->ready) cudaEventDestroy(index->ready);
        delete index;
    });
}

int spx_index_info(spx_index_t index, float* cell_size, int32_t* dims3, int64_t* occupied_cells, int64_t* n_points) {
    return guard([&] {
        SPX_REQUIRE(index, "[spx_index_info] null index");
        const GridView& v = index->levels.lv[0];
        if (cell_size) *cell_size = v.cell;
        if (dims3) {
            dims3[0] = v.dx;
            dims3[1] = v.dy;
            dims3[2] = v.dz;
        }
        if (occupied_cells) {
            *occupied_cells = 0;
            if (index->start[0] && index->n > 0) {  // counted on demand: nothing on the search path needs it
                spx_queue_t q = index->q;
                DeviceGuard g(q->device);
                if (!index->occ_dev) {
                    SPX_CUDA(cudaMallocAsync(&index->occ_dev, sizeof(unsigned long long), q->stream));
                    SPX_CUDA(cudaMemsetAsync(index->occ_dev, 0, sizeof(unsigned long long), q->stream));
                    occupied_from_start_kernel<<<std::min(div_up(index->ncells[0], 256), q->sm_count * 8), 256, 0, q->stream>>>(
                        index->start[0], index->ncells[0], index->occ_dev);
                    SPX_LAUNCH_CHECK();
                }
                unsigned long long* h = static_cast<unsigned long long*>(q->pinned_get(64));
                SPX_CUDA(cudaMemcpyAsync(h, index->occ_dev, sizeof(unsigned long long), cudaMemcpyDeviceToHost, q->stream));
                q->sync();
                *occupied_cells = (int64_t)*h;
            }
        }
        if (n_points) *n_points = index->n;
    });
}

int spx_index_levels(spx_index_t index, int32_t* n_levels) {
    return guard([&] {
        SPX_REQUIRE(index && n_levels, "[spx_index_levels] null argument");
        *n_levels = index->levels.n_levels;
    });
}

int spx_index_nn_stats(spx_index_t index, const float* queries, size_t nq, const float* T_host, float max_radius,
                       uint32_t* stats4) {
    return guard([&] {
        SPX_REQUIRE(index && queries && stats4, "[spx_index_nn_stats] null argument");
        spx_queue_t q = index->q;
        DeviceGuard g(q->device);
        const Xform T = T_host ? xform_from_colmajor(T_host) : xform_identity();
        const float r = max_radius > 0.0f ? max_radius : INFINITY;
        grid_nn_stats_kernel<<<div_up(nq, GRID_THREADS), GRID_THREADS, 0, q->stream>>>(
            index->levels, reinterpret_cast<const float4*>(queries), (uint32_t)nq, T, T_host != nullptr, r,
            reinterpret_cast<uint4*>(stats4));
        SPX_LAUNCH_CHECK();
    });
}

int spx_index_radius(spx_index_t index, const float* queries, size_t nq, int max_k, float radius, const float* T_host,
                     int32_t* idx, float* dist) {
    const int rc = spx_index_knn(index, queries, nq, max_k, T_host, idx, dist);
    if (rc != SPX_OK || nq == 0) return rc;
    return guard([&] {
        spx_queue_t q = index->q;
        DeviceGuard g(q->device);
        const size_t n = nq * (size_t)max_k;
        radius_mask_kernel<<<div_up(n, 256), 256, 0, q->stream>>>(idx, dist, n, radius * radius);
        SPX_LAUNCH_CHECK();
    });
}

int spx_index_remove_by_flags(spx_index_t index, const uint8_t* flags, const int32_t* new_index, size_t n, size_t n_kept) {
    return guard([&] {
        SPX_REQUIRE(index, "[KDTree::remove_nodes_by_flags] null index");
        SPX_REQUIRE(flags && new_index, "[KDTree::remove_nodes_by_flags_impl] null flags / indices");
        spx_queue_t q = index->q;
        DeviceGuard g(q->device);
        float4* kept = nullptr;
        SPX_CUDA(cudaMallocAsync(&kept, std::max<size_t>(n_kept, 1) * sizeof(float4), q->stream));
        // slots no kept point lands on (indices that skip numbers) hold NaN: the rebuilt index ignores them
        SPX_CUDA(cudaMemsetAsync(kept, 0xff, std::max<size_t>(n_kept, 1) * sizeof(float4), q->stream));
        if (index->n > 0) {
            index_kept_points_kernel<<<div_up(index->n, 256), 256, 0, q->stream>>>(index->sorted[0], index->n, flags, new_index,
                                                                                 n, kept);
            SPX_LAUNCH_CHECK();
        }
        spx_index_t fresh = nullptr;
        if (spx_index_build(q, reinterpret_cast<const float*>(kept), n_kept, 0.0f, &fresh) != SPX_OK) {
            cudaFreeAsync(kept, q->stream);
            throw Error(SPX_ERR_INTERNAL, spx_last_error());
        }
        SPX_CUDA(cudaFreeAsync(kept, q->stream));  // the index keeps its own sorted copy
        // the handle the caller holds now IS the rebuilt index
        for (int l = 0; l < GRID_MAX_LEVELS; ++l) {
            if (index->sorted[l]) cudaFreeAsync(index->sorted[l], q->stream);
            if (index->start[l]) cudaFreeAsync(index->start[l], q->stream);
        }
        if (index->occ_dev) cudaFreeAsync(index->occ_dev, q->stream);
        if (index->ready) cudaEventDestroy(index->ready);  // (the rebuilt index brings its own)
        *index = *fresh;
        delete fresh;
    });
}

int spx_index_knn(spx_index_t index, const float* queries, size_t nq, int k, const float* T_host, int32_t* idx,
                  float* dist) {
    return guard([&] {
        SPX_REQUIRE(index, "[KDTree::knn_search_async] null index");
        SPX_REQUIRE(k >= 1 && k <= 128, "[KDTree::knn_search_async] `k` is too large. not support.");
        SPX_REQUIRE(nq < (1ull << 31), "[KDTree::knn_search_async] too many queries");
        if (nq == 0) return;  // empty query -> empty result (kdtree.hpp:429-436)
        SPX_REQUIRE(queries && idx && dist, "[KDTree::knn_search_async] null pointer");
        spx_queue_t q = index->q;
        DeviceGuard g(q->device);
        const Xform T = T_host ? xform_from_colmajor(T_host) : xform_identity();
        const int has_T = T_host != nullptr;
        const unsigned blocks = (unsigned)div_up(nq, GRID_THREADS);
        const float4* qs = reinterpret_cast<const float4*>(queries);
        if (k == 1) {
            q->arena_reset();
            q->arena_reserve(nq * 4 + 4096);
            uint32_t* worklist = q->take<uint32_t>(nq);
            unsigned int* counters = q->take<unsigned int>(16);
            SPX_CUDA(cudaMemsetAsync(counters, 0, 2 * sizeof(unsigned int), q->stream));
            grid_nn1_fast_kernel<<<blocks, GRID_THREADS, 0, q->stream>>>(index->levels, qs, (uint32_t)nq, T, has_T, INFINITY,
                                                                        idx, dist, worklist, counters);
            SPX_LAUNCH_CHECK();
            // the drain kernel sizes itself to the device, not to the (unknown on the host) list length
            grid_nn1_coop_kernel<<<q->sm_count * 8, GRID_THREADS, 0, q->stream>>>(index->levels, qs, T, has_T, INFINITY, idx,
                                                                                 dist, worklist, counters, counters + 1);
        } else if (k <= 20 && std::getenv("SPX_KNN_ONEPASS")) {  // tuning aid: the single-launch variant
            if (k <= 5)
                grid_knn_reg_kernel<5><<<blocks, GRID_THREADS, 0, q->stream>>>(index->levels, qs, (uint32_t)nq, k, T, has_T, idx, dist);
            else if (k <= 10)
                grid_knn_reg_kernel<10><<<blocks, GRID_THREADS, 0, q->stream>>>(index->levels, qs, (uint32_t)nq, k, T, has_T, idx, dist);
            else
                grid_knn_reg_kernel<20><<<blocks, GRID_THREADS, 0, q->stream>>>(index->levels, qs, (uint32_t)nq, k, T, has_T, idx, dist);
        } else if (k <= 5) {
            launch_knn_reg<5>(index, q, qs, (uint32_t)nq, k, T, has_T, idx, dist);
        } else if (k <= 10) {
            launch_knn_reg<10>(index, q, qs, (uint32_t)nq, k, T, has_T, idx, dist);
        } else if (k <= 20) {
            launch_knn_reg<20>(index, q, qs, (uint32_t)nq, k, T, has_T, idx, dist);
        } else {
            const size_t smem = (size_t)k * GRID_THREADS * 8;
            // the attribute belongs to the (function, device) pair: one process may drive several GPUs
            static std::atomic<unsigned long long> attr_set{0ull};
            const unsigned long long bit = 1ull << (q->device & 63);
            if (!(attr_set.load(std::memory_order_acquire) & bit)) {
                SPX_CUDA(cudaFuncSetAttribute(grid_knn_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                              128 * GRID_THREADS * 8));
                attr_set.fetch_or(bit, std::memory_order_release);
            }
            grid_knn_kernel<false><<<blocks, GRID_THREADS, smem, q->stream>>>(index->levels_knn, qs, (uint32_t)nq, k, T,
                                                                             has_T, idx, dist);
        }
        SPX_LAUNCH_CHECK();
    });
}

}  // extern "C"
