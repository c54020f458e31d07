// Stable LSD radix sort of (key, uint32 value) pairs, one 8-bit digit per pass: histogram -> device-wide scan
// (spx_scan.cuh) -> scatter.  Used by the voxel grid for counts too large for its one-launch passes and by the
// Euclidean cluster extraction to order clusters and their members.
#pragma once

#include "spx_scan.cuh"

namespace spx {

constexpr int RS_THREADS = 256;
constexpr int RS_ITEMS = 8;  // keys per thread
constexpr int RS_TILE = RS_THREADS * RS_ITEMS;
constexpr int RS_WARPS = RS_THREADS / 32;
constexpr int RADIX_BITS = 8;
constexpr int RADIX = 1 << RADIX_BITS;

inline int bits_for(unsigned long long v) {  // bits needed to represent values in [0, v]
    int b = 0;
    while (v) {
        ++b;
        v >>= 1;
    }
    return b;
}

template <typename KeyT>
__global__ void __launch_bounds__(RS_THREADS) radix_hist_kernel(const KeyT* __restrict__ keys, uint32_t n, int shift,
                                                                uint32_t nblocks, uint32_t* __restrict__ ghist) {
    __shared__ uint32_t h[RADIX];
    h[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t base = blockIdx.x * RS_TILE;
#pragma unroll
    for (int it = 0; it < RS_ITEMS; ++it) {
        const uint32_t i = base + it * RS_THREADS + threadIdx.x;
        if (i < n) atomicAdd(&h[(uint32_t)(keys[i] >> shift) & (RADIX - 1)], 1u);
    }
    __syncthreads();
    ghist[(size_t)threadIdx.x * nblocks + blockIdx.x] = h[threadIdx.x];
}

// Each warp owns a contiguous 256-key slice of the tile and walks it 32 keys at a time, so
// "earlier in the input" == "earlier (warp, chunk, lane)".  __match_any_sync groups equal digits
// inside a chunk; the per-warp digit counters give the rank inside the warp; a per-digit prefix
// over the warps (seeded with the scanned global histogram) gives the final, stable position.
template <typename KeyT>
__global__ void __launch_bounds__(RS_THREADS) radix_scatter_kernel(const KeyT* __restrict__ keys_in,
                                                                   const uint32_t* __restrict__ vals_in,
                                                                   KeyT* __restrict__ keys_out,
                                                                   uint32_t* __restrict__ vals_out,
                                                                   const uint32_t* __restrict__ goffs, uint32_t n,
                                                                   int shift, uint32_t nblocks) {
    __shared__ uint32_t wcnt[RS_WARPS][RADIX];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int t = threadIdx.x; t < RS_WARPS * RADIX; t += RS_THREADS) (&wcnt[0][0])[t] = 0;
    __syncthreads();

    KeyT key[RS_ITEMS];
    uint32_t val[RS_ITEMS], rank[RS_ITEMS];
    const uint32_t wbase = blockIdx.x * RS_TILE + warp * (32 * RS_ITEMS);
#pragma unroll
    for (int c = 0; c < RS_ITEMS; ++c) {
        const uint32_t i = wbase + c * 32 + lane;
        const bool live = i < n;
        const unsigned act = __ballot_sync(0xffffffffu, live);
        rank[c] = 0;
        key[c] = 0;
        val[c] = 0;
        if (live) {
            key[c] = keys_in[i];
            val[c] = vals_in ? vals_in[i] : i;
            const uint32_t digit = (uint32_t)(key[c] >> shift) & (RADIX - 1);
            const unsigned peers = __match_any_sync(act, digit);
            const uint32_t before = __popc(peers & ((1u << lane) - 1));
            const uint32_t prev = wcnt[warp][digit];
            __syncwarp(act);
            if (before == 0) wcnt[warp][digit] = prev + __popc(peers);
            __syncwarp(act);
            rank[c] = prev + before;
        }
    }
    __syncthreads();
    {
        const int d = threadIdx.x;  // RS_THREADS == RADIX
        uint32_t run = goffs[(size_t)d * nblocks + blockIdx.x];
#pragma unroll
        for (int w = 0; w < RS_WARPS; ++w) {
            const uint32_t t = wcnt[w][d];
            wcnt[w][d] = run;
            run += t;
        }
    }
    __syncthreads();
#pragma unroll
    for (int c = 0; c < RS_ITEMS; ++c) {
        const uint32_t i = wbase + c * 32 + lane;
        if (i < n) {
            const uint32_t digit = (uint32_t)(key[c] >> shift) & (RADIX - 1);
            const uint32_t dst = wcnt[warp][digit] + rank[c];
            keys_out[dst] = key[c];
            vals_out[dst] = val[c];
        }
    }
}

// uint32 words of scratch radix_sort_pairs needs for n pairs: the per-block digit histograms and their scan
inline size_t radix_sort_scratch_elems(size_t n) {
    const size_t h = (size_t)RADIX * (size_t)div_up(n, RS_TILE);
    return align_up(h + 64, 64) + scan_scratch_elems(h);
}

// `passes` passes over the digits of keys[0] (pass p sorts by bits [8p, 8p + 8)), ping-ponging between keys[0] and
// keys[1] and writing the values to vals[0], vals[1], vals[0], ...; vals_in == nullptr takes each pair's position as
// its value.  After the call the sorted keys are in keys[passes & 1] and the values in vals[(passes - 1) & 1].
template <typename KeyT>
inline void radix_sort_pairs(cudaStream_t st, uint32_t n, int passes, KeyT* const keys[2], const uint32_t* vals_in,
                             uint32_t* const vals[2], uint32_t* scratch) {
    if (n == 0) return;
    const uint32_t nblocks = (uint32_t)div_up(n, RS_TILE);
    uint32_t* ghist = scratch;
    uint32_t* scan_tmp = scratch + align_up((size_t)RADIX * nblocks + 64, 64);
    const uint32_t* vin = vals_in;
    for (int p = 0; p < passes; ++p) {
        const int shift = p * RADIX_BITS;
        radix_hist_kernel<KeyT><<<nblocks, RS_THREADS, 0, st>>>(keys[p & 1], n, shift, nblocks, ghist);
        SPX_LAUNCH_CHECK();
        exclusive_scan_u32(st, ghist, ghist, (size_t)RADIX * nblocks, scan_tmp, nullptr);
        radix_scatter_kernel<KeyT><<<nblocks, RS_THREADS, 0, st>>>(keys[p & 1], vin, keys[(p + 1) & 1], vals[p & 1],
                                                                    ghist, n, shift, nblocks);
        SPX_LAUNCH_CHECK();
        vin = vals[p & 1];
    }
}

}  // namespace spx
