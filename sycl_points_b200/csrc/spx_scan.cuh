// Device-wide exclusive prefix sum over uint32 (counting sort of the cell grid, radix-sort digit
// offsets, voxel compaction).  Three-phase reduce / scan / down-sweep; the middle phase recurses
// on the per-block totals, so any n up to 2^32-1 elements works with O(log_{4096} n) levels.
// The reference does this on the device too, with its own three kernels
// (I/algorithms/common/prefix_sum.hpp:30-166); this is an independent shared-memory design.
#pragma once

#include "spx_common.cuh"

namespace spx {

constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 16;  // per thread
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

// block-level exclusive scan of one value per thread; returns the exclusive prefix, total in *total
__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* smem_warp /*[32]*/, uint32_t* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) smem_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const int nw = blockDim.x >> 5;
        uint32_t w = lane < nw ? smem_warp[lane] : 0u;
        uint32_t winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc += t;
        }
        smem_warp[lane] = winc - w;  // exclusive warp offsets
        if (lane == 31) smem_warp[32] = winc;
    }
    __syncthreads();
    const uint32_t off = smem_warp[warp];
    if (total) *total = smem_warp[32];
    return off + inc - v;
}

// phase 1: per-tile totals
static __global__ void __launch_bounds__(SCAN_THREADS) scan_tile_totals_kernel(const uint32_t* __restrict__ in, size_t n,
                                                                        uint32_t* __restrict__ totals) {
    __shared__ uint32_t sw[33];
    const size_t base = (size_t)blockIdx.x * SCAN_TILE + (size_t)threadIdx.x * SCAN_ITEMS;
    uint32_t s = 0;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        const size_t j = base + i;
        if (j < n) s += in[j];
    }
    uint32_t total;
    block_exclusive_scan(s, sw, &total);
    if (threadIdx.x == 0) totals[blockIdx.x] = total;
}

// phase 3 (also the whole job when n fits one tile): scan inside the tile + tile offset.
// RAW_TOTALS: `tile_offsets` holds the un-scanned per-tile totals and every block sums its
// predecessors itself (a few KB of L2 reads) — saves the middle launch for up to SCAN_TILE tiles.
template <bool RAW_TOTALS>
static __global__ void __launch_bounds__(SCAN_THREADS) scan_tile_apply_kernel(const uint32_t* __restrict__ in, size_t n,
                                                                       const uint32_t* __restrict__ tile_offsets,
                                                                       uint32_t* __restrict__ out,
                                                                       uint32_t* __restrict__ grand_total) {
    __shared__ uint32_t sw[33];
    __shared__ uint32_t tile_off;
    uint32_t my_off = 0;
    if (RAW_TOTALS) {
        uint32_t part = 0;
        for (uint32_t t = threadIdx.x; t < blockIdx.x; t += SCAN_THREADS) part += tile_offsets[t];
        uint32_t tot;
        block_exclusive_scan(part, sw, &tot);
        if (threadIdx.x == 0) tile_off = tot;
        __syncthreads();
        my_off = tile_off;
        __syncthreads();  // sw is reused below
    } else if (tile_offsets) {
        my_off = tile_offsets[blockIdx.x];
    }
    const size_t base = (size_t)blockIdx.x * SCAN_TILE + (size_t)threadIdx.x * SCAN_ITEMS;
    uint32_t v[SCAN_ITEMS];
    uint32_t s = 0;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        const size_t j = base + i;
        v[i] = j < n ? in[j] : 0u;
        s += v[i];
    }
    uint32_t total;
    uint32_t run = block_exclusive_scan(s, sw, &total) + my_off;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        const size_t j = base + i;
        if (j < n) out[j] = run;
        run += v[i];
    }
    if (grand_total && blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) *grand_total = my_off + total;
}

// ---- decoupled look-back over per-tile counts (chained scan): used by the one-launch scan below and by
// the voxel grid's fused mean + compaction kernel.  A status word = flag (2 bits) | value (62 bits).
constexpr int LB_THREADS = 256;  // block size of every kernel that calls block_lookback
constexpr unsigned long long LB_LOCAL = 1ull << 62, LB_INCL = 1ull << 63, LB_VALUE = LB_LOCAL - 1ull;

// Exclusive prefix of `count` over the tiles before `tile`; called by every thread of the block.
// Each round reads the LB_WIN nearest predecessors not yet accounted for, all at once: when a whole
// wave of tiles publishes together, hardly any of them is inclusive yet and the walk is long — with
// one warp's 32 entries per L2 round trip it was the largest part of the kernel.
constexpr int LB_PER = 4;
constexpr uint32_t LB_WIN = LB_THREADS * LB_PER;
__device__ __forceinline__ void lookback_publish(volatile unsigned long long* status, uint32_t tile,
                                                 unsigned long long count) {
    if (threadIdx.x == 0) status[tile] = (tile == 0 ? LB_INCL : LB_LOCAL) | count;
}
__device__ __forceinline__ unsigned long long block_lookback(volatile unsigned long long* status, uint32_t tile,
                                                             unsigned long long count, uint32_t* s_min /*[2]*/,
                                                             unsigned long long* s_sum) {
    const uint32_t t = threadIdx.x;
    if (tile == 0) return 0ull;
    unsigned long long prev = 0;
    long long p = (long long)tile - 1;
    for (;;) {
        __syncthreads();
        if (t == 0) {
            s_min[0] = LB_WIN;  // nearest inclusive entry of the window
            s_min[1] = LB_WIN;  // nearest entry not published yet
            *s_sum = 0ull;
        }
        __syncthreads();
        unsigned long long v[LB_PER];
#pragma unroll
        for (int u = 0; u < LB_PER; ++u) {  // entry e of the window is tile p - e
            const long long idx = p - (long long)(u * LB_THREADS + t);
            v[u] = LB_INCL;  // before the first tile: an inclusive zero
            if (idx >= 0) v[u] = status[idx];
        }
        uint32_t f = LB_WIN, un = LB_WIN;
#pragma unroll
        for (int u = LB_PER - 1; u >= 0; --u) {
            const uint32_t e = u * LB_THREADS + t;
            if (v[u] & LB_INCL) f = e;
            if ((v[u] >> 62) == 0) un = e;
        }
        if (f < LB_WIN) atomicMin(&s_min[0], f);
        if (un < LB_WIN) atomicMin(&s_min[1], un);
        __syncthreads();
        const uint32_t F = s_min[0], U = s_min[1];
        if (U < F) continue;  // a tile the sum needs has not published yet (it runs: tickets are ordered)
        unsigned long long x = 0;
#pragma unroll
        for (int u = 0; u < LB_PER; ++u)
            if ((uint32_t)(u * LB_THREADS + t) <= F) x += v[u] & LB_VALUE;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        if ((t & 31) == 0 && x) atomicAdd(s_sum, x);
        __syncthreads();
        prev += *s_sum;
        if (F < LB_WIN) break;
        p -= LB_WIN;
    }
    if (t == 0) status[tile] = LB_INCL | (prev + count);
    return prev;
}


// One-launch exclusive scan: tiles taken by ticket, tile offsets by look-back.  `status` (tiles words of
// 64 bits) and `ticket` must be zero at launch.
static __global__ void __launch_bounds__(SCAN_THREADS) scan_lookback_kernel(const uint32_t* __restrict__ in, size_t n,
                                                                            uint32_t* __restrict__ out,
                                                                            unsigned long long* status, uint32_t* ticket,
                                                                            uint32_t* __restrict__ grand_total) {
    static_assert(SCAN_THREADS == LB_THREADS, "block_lookback is written for LB_THREADS threads");
    __shared__ uint32_t sw[33];
    __shared__ uint32_t s_tile, s_min[2];
    __shared__ unsigned long long s_sum;
    if (threadIdx.x == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const size_t base = (size_t)tile * SCAN_TILE + (size_t)threadIdx.x * SCAN_ITEMS;
    uint32_t v[SCAN_ITEMS];
    uint32_t s = 0;
    // a thread's 16 items are 64 contiguous bytes: four 16-byte accesses when the tile is whole and the arrays
    // are 16-byte aligned (the index build's are), scalar otherwise
    const bool vec = base + SCAN_ITEMS <= n && ((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
    if (vec) {
#pragma unroll
        for (int i = 0; i < SCAN_ITEMS / 4; ++i) {
            const uint4 x = __ldg(reinterpret_cast<const uint4*>(in + base) + i);
            v[4 * i] = x.x;
            v[4 * i + 1] = x.y;
            v[4 * i + 2] = x.z;
            v[4 * i + 3] = x.w;
        }
#pragma unroll
        for (int i = 0; i < SCAN_ITEMS; ++i) s += v[i];
    } else {
#pragma unroll
        for (int i = 0; i < SCAN_ITEMS; ++i) {
            const size_t j = base + i;
            v[i] = j < n ? in[j] : 0u;
            s += v[i];
        }
    }
    uint32_t total;
    uint32_t run = block_exclusive_scan(s, sw, &total);
    lookback_publish(status, tile, total);
    const unsigned long long off = block_lookback(status, tile, total, s_min, &s_sum);
    run += (uint32_t)off;
    if (vec) {
#pragma unroll
        for (int i = 0; i < SCAN_ITEMS / 4; ++i) {
            uint4 x;
            x.x = run;
            run += v[4 * i];
            x.y = run;
            run += v[4 * i + 1];
            x.z = run;
            run += v[4 * i + 2];
            x.w = run;
            run += v[4 * i + 3];
            reinterpret_cast<uint4*>(out + base)[i] = x;
        }
    } else {
#pragma unroll
        for (int i = 0; i < SCAN_ITEMS; ++i) {
            const size_t j = base + i;
            if (j < n) out[j] = run;
            run += v[i];
        }
    }
    if (grand_total && (size_t)(tile + 1) * SCAN_TILE >= n && threadIdx.x == 0) *grand_total = (uint32_t)off + total;
}
inline size_t scan_lookback_words(size_t n) {  // uint32 words of zeroed scratch: [ticket 2][status 2 x tiles]
    return 2 + 2 * ((n + SCAN_TILE - 1) / SCAN_TILE);
}
// out may alias in
inline void exclusive_scan_u32_onepass(cudaStream_t st, const uint32_t* in, uint32_t* out, size_t n,
                                       uint32_t* zeroed_scratch, uint32_t* grand_total) {
    if (n == 0) {
        if (grand_total) SPX_CUDA(cudaMemsetAsync(grand_total, 0, sizeof(uint32_t), st));
        return;
    }
    const size_t tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    scan_lookback_kernel<<<(unsigned)tiles, SCAN_THREADS, 0, st>>>(in, n, out, reinterpret_cast<unsigned long long*>(zeroed_scratch + 2),
                                                                  zeroed_scratch, grand_total);
    SPX_LAUNCH_CHECK();
}

inline size_t scan_scratch_elems(size_t n) {
    size_t total = 0;
    while (n > SCAN_TILE) {
        n = (n + SCAN_TILE - 1) / SCAN_TILE;
        total += align_up(n, 64);
    }
    return total + 64;
}

// out may alias in.  scratch: scan_scratch_elems(n) uint32.  grand_total (device, nullable) gets sum(in).
inline void exclusive_scan_u32(cudaStream_t st, const uint32_t* in, uint32_t* out, size_t n, uint32_t* scratch,
                               uint32_t* grand_total) {
    if (n == 0) {
        if (grand_total) SPX_CUDA(cudaMemsetAsync(grand_total, 0, sizeof(uint32_t), st));
        return;
    }
    const size_t tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    if (tiles == 1) {
        scan_tile_apply_kernel<false><<<1, SCAN_THREADS, 0, st>>>(in, n, nullptr, out, grand_total);
        SPX_LAUNCH_CHECK();
        return;
    }
    uint32_t* totals = scratch;
    scan_tile_totals_kernel<<<(unsigned)tiles, SCAN_THREADS, 0, st>>>(in, n, totals);
    SPX_LAUNCH_CHECK();
    if (tiles <= (size_t)SCAN_TILE) {  // two launches: each apply block sums its predecessors' totals itself
        scan_tile_apply_kernel<true><<<(unsigned)tiles, SCAN_THREADS, 0, st>>>(in, n, totals, out, grand_total);
        SPX_LAUNCH_CHECK();
        return;
    }
    exclusive_scan_u32(st, totals, totals, tiles, scratch + align_up(tiles, 64), nullptr);
    scan_tile_apply_kernel<false><<<(unsigned)tiles, SCAN_THREADS, 0, st>>>(in, n, totals, out, grand_total);
    SPX_LAUNCH_CHECK();
}

// order-preserving compaction to indices: out[pos[i]] = i for every flagged i (pos = exclusive scan of flags).  The
// index-producing filters (box, angle of incidence, farthest point sampling, outlier removal) end with it.
constexpr int COMPACT_THREADS = 256;
static __global__ void __launch_bounds__(COMPACT_THREADS) compact_index_kernel(const uint32_t* __restrict__ flags,
                                                                               const uint32_t* __restrict__ pos, uint32_t n,
                                                                               int32_t* __restrict__ out) {
    const uint32_t i = blockIdx.x * COMPACT_THREADS + threadIdx.x;
    if (i >= n) return;
    if (flags[i]) out[pos[i]] = (int32_t)i;
}

}  // namespace spx
