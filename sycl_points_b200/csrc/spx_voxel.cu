// Voxel-grid downsampling and the box filter on the device.
//
// Reference: filter::VoxelGrid::downsampling (I/algorithms/filter/voxel_downsampling.hpp:50-62) —
// only the key computation runs on the device there (:114-144); the sort (:146-179, host std::sort)
// and the per-voxel mean (:181-218, host sweep) are host code.  Here all three are kernels:
//   1. voxel coordinates per point (voxel_constants.hpp:36-62) + their bounding box,
//   2. an order-preserving compact key  ((z-zmin)·ny + (y-ymin))·nx + (x-xmin)  — same ordering as
//      the reference's 63-bit key but only ceil(log2(nx·ny·nz)) significant bits, so the LSD radix
//      sort needs 3-4 eight-bit passes instead of 8,
//   3. a stable LSD radix sort of (key, original index) — stability gives the (key, index) order the
//      oracle defines for the order the reference leaves to std::sort,
//   4. one thread per voxel run: fp32 running sum in that order, mean = sum / sum.w, drop runs with
//      sum.w < min_voxel_count (:204), stream-compact to ascending-key output.
#include <cmath>

#include <cooperative_groups.h>

#include "spx_math.cuh"
#include "spx_sort.cuh"

using namespace spx;

namespace {

constexpr int VX_THREADS = 256;

struct CoordAcc {
    int mn[3];
    int mx[3];
    uint32_t valid;
    uint32_t pad;
};

// How a point becomes three integer grid coordinates (the key's digits, c[2] most significant):
//   voxel grid  c = floor(p * inv) per axis (compute_voxel_bit, voxel_constants.hpp:36-53);
//   polar grid  c = floor(range * inv[0]), floor(elevation * inv[1]), floor(azimuth * inv[2])
//               (compute_polar_bit, filter/polar_downsampling.hpp:30-108; DISTANCE lowest, AZIMUTH highest).
struct CoordMap {
    float inv[3];
    int polar;  // 0 voxel grid, 1 polar LIDAR frame, 2 polar CAMERA frame
};

// Returns false for the points the reference maps to invalid_coord (non-finite, outside the 21-bit range; for
// the polar grid also the origin and the points on the polar axis).  atan2 is evaluated in fp64 and cast — the
// library's rule for transcendentals — and the squared sums are plain fp32 multiplies and adds, left to right.
template <bool POLAR>
__device__ __forceinline__ bool voxel_coords(const float4 p, const CoordMap& cm, int c[3]) {
    if (!isfinite(p.x) || !isfinite(p.y) || !isfinite(p.z)) return false;
    float fx, fy, fz;
    if constexpr (!POLAR) {
        fx = floorf(__fmul_rn(p.x, cm.inv[0]));
        fy = floorf(__fmul_rn(p.y, cm.inv[1]));
        fz = floorf(__fmul_rn(p.z, cm.inv[2]));
    } else {
        const float xx = __fmul_rn(p.x, p.x), yy = __fmul_rn(p.y, p.y), zz = __fmul_rn(p.z, p.z);
        const float r = sqrtf(__fadd_rn(__fadd_rn(xx, yy), zz));
        if (r == 0.0f) return false;
        float azimuth, elevation;
        if (cm.polar == 1) {
            const float x2y2 = __fadd_rn(xx, yy);
            if (x2y2 == 0.0f) return false;
            azimuth = (float)atan2((double)p.y, (double)p.x);
            elevation = (float)atan2((double)p.z, (double)sqrtf(x2y2));
        } else {
            const float x2z2 = __fadd_rn(xx, zz);
            if (x2z2 == 0.0f) return false;
            azimuth = (float)atan2((double)p.x, (double)p.z);
            elevation = (float)atan2((double)-p.y, (double)sqrtf(x2z2));
        }
        fx = floorf(__fmul_rn(r, cm.inv[0]));
        fy = floorf(__fmul_rn(elevation, cm.inv[1]));
        fz = floorf(__fmul_rn(azimuth, cm.inv[2]));
    }
    const float lim = 1048576.0f;  // 2^20: coord + offset must land in [0, 2^21 - 1]
    if (!(fx >= -lim && fx < lim && fy >= -lim && fy < lim && fz >= -lim && fz < lim)) return false;
    c[0] = (int)fx + (1 << 20);
    c[1] = (int)fy + (1 << 20);
    c[2] = (int)fz + (1 << 20);
    return true;
}

// On the device the box is accumulated with atomicMax only, in an encoding whose empty state is all zero
// bits (so the accumulator is initialised by the memset that zeroes the rest of the scratch, not by a kernel):
// mn[a] holds max(2^21 - c), mx[a] holds max(c + 1) over the valid points' voxel coordinates c in [0, 2^21).
// coord_acc_decode turns the copy that reached the host back into plain min / max.
inline void coord_acc_decode(CoordAcc* h) {
    for (int a = 0; a < 3; ++a) {
        h->mn[a] = h->valid ? (1 << 21) - h->mn[a] : INT_MAX;
        h->mx[a] = h->valid ? h->mx[a] - 1 : INT_MIN;
    }
}

// per-thread box + count of valid points -> the block's -> the cloud's (one set of global atomics per
// block: per-warp atomics on seven shared addresses serialise).  Called by every thread of the block.
__device__ __forceinline__ void coord_acc_commit(int mn[3], int mx[3], uint32_t cnt, CoordAcc* acc) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            mn[a] = min(mn[a], __shfl_xor_sync(0xffffffffu, mn[a], o));
            mx[a] = max(mx[a], __shfl_xor_sync(0xffffffffu, mx[a], o));
        }
        cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    }
    __shared__ int smn[3], smx[3];
    __shared__ uint32_t scnt;
    if (threadIdx.x == 0) {
        for (int a = 0; a < 3; ++a) smn[a] = smx[a] = 0;
        scnt = 0;
    }
    __syncthreads();
    if ((threadIdx.x & 31) == 0 && cnt) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            atomicMax(&smn[a], (1 << 21) - mn[a]);
            atomicMax(&smx[a], mx[a] + 1);
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
        atomicAdd(&acc->valid, scnt);
    }
}

template <bool POLAR>
__global__ void __launch_bounds__(VX_THREADS) voxel_bbox_kernel(const float4* __restrict__ pts, uint32_t n, CoordMap cm,
                                                                CoordAcc* acc) {
    int mn[3] = {INT_MAX, INT_MAX, INT_MAX}, mx[3] = {INT_MIN, INT_MIN, INT_MIN};
    uint32_t cnt = 0;
    for (uint32_t i = blockIdx.x * VX_THREADS + threadIdx.x; i < n; i += gridDim.x * VX_THREADS) {
        int c[3];
        if (voxel_coords<POLAR>(__ldg(pts + i), cm, c)) {
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                mn[a] = min(mn[a], c[a]);
                mx[a] = max(mx[a], c[a]);
            }
            ++cnt;
        }
    }
    coord_acc_commit(mn, mx, cnt, acc);
}

struct KeyGeom {
    int mn[3];
    int mx[3];                   // last voxel coordinate the key covers (checked when the box was guessed)
    unsigned long long nx, nxy;  // strides of the compact key
    unsigned long long invalid;  // key given to dropped points (sorts after every valid key)
};

template <typename KeyT, bool POLAR>
__global__ void __launch_bounds__(VX_THREADS) voxel_key_kernel(const float4* __restrict__ pts, uint32_t n, CoordMap cm,
                                                               KeyGeom g, KeyT* __restrict__ keys) {
    const uint32_t i = blockIdx.x * VX_THREADS + threadIdx.x;
    if (i >= n) return;
    int c[3];
    unsigned long long key = g.invalid;
    if (voxel_coords<POLAR>(__ldg(pts + i), cm, c))
        key = (unsigned long long)(c[2] - g.mn[2]) * g.nxy + (unsigned long long)(c[1] - g.mn[1]) * g.nx +
              (unsigned long long)(c[0] - g.mn[0]);
    keys[i] = (KeyT)key;
}

// ---- the same sort as ONE kernel per digit ("onesweep": chained scan with decoupled look-back).
// The digit histograms of every pass come out of the key kernel; a pass then needs no separate
// histogram and no device-wide scan: a tile publishes its per-digit counts in `status`, walks back
// over its predecessors' entries until it meets an inclusive one, and scatters.  Tiles are taken by
// ticket, so a tile only ever waits for tiles that already run.  Used while counts fit the 30 value
// bits of a status word; above that the three-kernel passes above take over.
constexpr uint32_t OS_LOCAL = 1u << 30;  // status word = flag | count
constexpr uint32_t OS_INCL = 2u << 30;
constexpr uint32_t OS_VALUE = OS_LOCAL - 1u;
constexpr int OS_MAX_PASSES = 8;
template <typename KeyT>
struct OsItems {
    static constexpr int value = sizeof(KeyT) == 4 ? 16 : 8;  // keys per thread (tile staged in 32 / 24 KB of smem)
};

template <typename KeyT, bool POLAR>
__global__ void __launch_bounds__(VX_THREADS) voxel_key_hist_kernel(const float4* __restrict__ pts, uint32_t n,
                                                                    CoordMap cm, KeyGeom g, KeyT* __restrict__ keys,
                                                                    int passes, uint32_t* __restrict__ ghist,
                                                                    uint32_t* __restrict__ outside, CoordAcc* acc) {
    // acc != null (the box in `g` is a guess): this cloud's own box and valid count are accumulated here,
    // in the same read of the points, instead of by voxel_bbox_kernel
    int bmn[3] = {INT_MAX, INT_MAX, INT_MAX}, bmx[3] = {INT_MIN, INT_MIN, INT_MIN};
    uint32_t bcnt = 0;
    __shared__ uint32_t h[OS_MAX_PASSES * RADIX];
    for (int t = threadIdx.x; t < passes * RADIX; t += VX_THREADS) h[t] = 0;
    __syncthreads();
    constexpr int KH = 4;  // points per thread and step, their loads in flight together
    for (uint32_t i0 = blockIdx.x * (VX_THREADS * KH) + threadIdx.x; i0 < n; i0 += gridDim.x * (VX_THREADS * KH)) {
        float4 pt[KH];
#pragma unroll
        for (int u = 0; u < KH; ++u) pt[u] = __ldg(pts + min(i0 + u * VX_THREADS, n - 1));
#pragma unroll
        for (int u = 0; u < KH; ++u) {
            const uint32_t i = i0 + u * VX_THREADS;
            if (i >= n) break;
            int c[3];
            unsigned long long key = g.invalid;
            if (voxel_coords<POLAR>(pt[u], cm, c)) {
#pragma unroll
                for (int a = 0; a < 3; ++a) {
                    bmn[a] = min(bmn[a], c[a]);
                    bmx[a] = max(bmx[a], c[a]);
                }
                ++bcnt;
                if (c[0] < g.mn[0] || c[0] > g.mx[0] || c[1] < g.mn[1] || c[1] > g.mx[1] || c[2] < g.mn[2] || c[2] > g.mx[2])
                    *outside = 1u;  // only possible with a guessed box: the host starts over with the exact one
                else
                    key = (unsigned long long)(c[2] - g.mn[2]) * g.nxy + (unsigned long long)(c[1] - g.mn[1]) * g.nx +
                          (unsigned long long)(c[0] - g.mn[0]);
            }
            keys[i] = (KeyT)key;
            for (int p = 0; p < passes; ++p)
                atomicAdd(&h[p * RADIX + ((uint32_t)(key >> (p * RADIX_BITS)) & (RADIX - 1))], 1u);
        }
    }
    __syncthreads();
    for (int t = threadIdx.x; t < passes * RADIX; t += VX_THREADS)
        if (h[t]) atomicAdd(ghist + t, h[t]);
    if (acc) coord_acc_commit(bmn, bmx, bcnt, acc);
}

template <typename KeyT>
__global__ void __launch_bounds__(RS_THREADS, 4) onesweep_kernel(const KeyT* __restrict__ keys_in,
                                                              const uint32_t* __restrict__ vals_in,
                                                              KeyT* __restrict__ keys_out, uint32_t* __restrict__ vals_out,
                                                              const uint32_t* __restrict__ ghist /*[RADIX], this pass*/,
                                                              uint32_t* status /*[tiles][RADIX], zeroed*/,
                                                              uint32_t* ticket /*zeroed*/, uint32_t n, int shift) {
    constexpr int ITEMS = OsItems<KeyT>::value;
    constexpr uint32_t TILE = RS_THREADS * ITEMS;
    __shared__ uint32_t wcnt[RS_WARPS][RADIX];
    __shared__ uint32_t dig_excl[RADIX];  // first tile-sorted position of each digit
    __shared__ uint32_t gbase[RADIX];     // global position of tile-sorted element e of digit d = gbase[d] + e
    __shared__ uint32_t sw_a[33], sw_b[33];
    __shared__ uint32_t s_tile;
    __shared__ KeyT skey[TILE];
    __shared__ uint32_t sval[TILE];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_tile = atomicAdd(ticket, 1u);
    for (int t = threadIdx.x; t < RS_WARPS * RADIX; t += RS_THREADS) (&wcnt[0][0])[t] = 0;
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint32_t tbase = tile * TILE;

    KeyT key[ITEMS];
    uint32_t val[ITEMS], rank[ITEMS];
    const uint32_t wbase = tbase + warp * (32 * ITEMS);
#pragma unroll
    for (int c = 0; c < ITEMS; ++c) {  // loads first: all ITEMS requests of a thread are in flight together
        const uint32_t i = wbase + c * 32 + lane;
        key[c] = 0;
        if (i < n) key[c] = keys_in[i];
    }
#pragma unroll
    for (int c = 0; c < ITEMS; ++c) {  // stable rank inside the warp's slice, as in radix_scatter_kernel
        const uint32_t i = wbase + c * 32 + lane;
        const bool live = i < n;
        const unsigned act = __ballot_sync(0xffffffffu, live);
        rank[c] = 0;
        if (live) {
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
#pragma unroll
    for (int c = 0; c < ITEMS; ++c) {  // the payload is fetched while the look-back below waits
        const uint32_t i = wbase + c * 32 + lane;
        val[c] = i;
        if (vals_in && i < n) val[c] = vals_in[i];
    }
    uint32_t my_count, my_excl;
    {
        const int d = threadIdx.x;  // RS_THREADS == RADIX: one digit per thread
        uint32_t count = 0;
#pragma unroll
        for (int w = 0; w < RS_WARPS; ++w) {
            const uint32_t t = wcnt[w][d];
            wcnt[w][d] = count;
            count += t;
        }
        my_count = count;
        *(volatile uint32_t*)(status + (size_t)tile * RADIX + d) = (tile == 0 ? OS_INCL : OS_LOCAL) | count;
        my_excl = block_exclusive_scan(count, sw_a, nullptr);
        dig_excl[d] = my_excl;
    }
    __syncthreads();
#pragma unroll
    for (int c = 0; c < ITEMS; ++c) {  // the tile in digit order, in shared memory
        const uint32_t i = wbase + c * 32 + lane;
        if (i < n) {
            const uint32_t digit = (uint32_t)(key[c] >> shift) & (RADIX - 1);
            const uint32_t pos = dig_excl[digit] + wcnt[warp][digit] + rank[c];
            skey[pos] = key[c];
            sval[pos] = val[c];
        }
    }
    {
        // look-back, now that the registers of the tile are free: thread d walks back over the
        // predecessors' entries of digit d, OS_LOOK of them in flight per round trip (when every tile of a
        // one-wave launch publishes at once the walk is long: it is a chain of L2 latencies).  Entries are
        // consumed strictly in order; an unpublished one (flag 0: that tile runs, tickets are ordered)
        // restarts the batch at its position.
        const int d = threadIdx.x;
        const uint32_t gstart = block_exclusive_scan(ghist[d], sw_b, nullptr);
        uint32_t prev = 0;
        if (tile > 0) {
            constexpr int OS_LOOK = 32;
            int p = (int)tile - 1;
            bool done = false;
            while (!done) {
                uint32_t v[OS_LOOK];
#pragma unroll
                for (int u = 0; u < OS_LOOK; ++u)
                    v[u] = *(volatile const uint32_t*)(status + (size_t)max(p - u, 0) * RADIX + d);
#pragma unroll
                for (int u = 0; u < OS_LOOK; ++u) {
                    if (done || (v[u] >> 30) == 0) break;
                    prev += v[u] & OS_VALUE;
                    done = (v[u] & OS_INCL) != 0;
                    --p;
                }
            }
            *(volatile uint32_t*)(status + (size_t)tile * RADIX + d) = OS_INCL | (prev + my_count);
        }
        gbase[d] = gstart + prev - my_excl;
    }
    __syncthreads();
    const uint32_t cnt = min(TILE, n - tbase);
    for (uint32_t e = threadIdx.x; e < cnt; e += RS_THREADS) {  // digit runs leave as contiguous stores
        const KeyT k = skey[e];
        const uint32_t dst = gbase[(uint32_t)(k >> shift) & (RADIX - 1)] + e;
        keys_out[dst] = k;
        vals_out[dst] = sval[e];
    }
}

// ---- per-voxel mean
// optional per-point attributes aggregated with the points (voxel_downsampling.hpp:220-288): mean
// RGBA, median intensity (:82-98), mean timestamp offset — all over the voxel's points in the same
// stable (key, index) order
struct VoxAttrs {
    const float4* rgb;
    const float* intensity;
    const float* timestamps;
    float4* rgb_mean;    // per sorted position (run head), compacted afterwards
    float* intensity_med;
    float* ts_mean;
};

__device__ __forceinline__ uint32_t float_key(float f) {  // order-preserving float -> uint
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_float(uint32_t k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}
// rank-th smallest (0-based) intensity of the run [j0, j1) by radix selection on the ordered bits:
// 32 passes over the run, no scratch, exact for any run length (what nth_element returns)
__device__ float run_select(const float* __restrict__ v, const uint32_t* __restrict__ svals, uint32_t j0, uint32_t j1,
                            uint32_t rank) {
    uint32_t prefix = 0, mask = 0;
    for (int bit = 31; bit >= 0; --bit) {
        const uint32_t b = 1u << bit;
        uint32_t zeros = 0;
        for (uint32_t j = j0; j < j1; ++j) {
            const uint32_t k = float_key(__ldg(v + svals[j]));
            zeros += ((k & mask) == prefix) && !(k & b);
        }
        if (rank >= zeros) {
            rank -= zeros;
            prefix |= b;
        }
        mask |= b;
    }
    return key_float(prefix);
}

// ---- per-voxel mean + stream compaction in one kernel.
// A tile of the sorted (key, index) list is staged in shared memory — keys and indices with
// coalesced loads, the points gathered through the indices — and the heads of the voxel runs are
// compacted so that CONSECUTIVE threads walk consecutive runs (one thread per element left ~4 of
// 32 lanes busy and made the kernel issue-bound).  The sum over a run stays strictly sequential in
// (key, index) order; a run that leaves the tile continues in global memory.  Kept voxels are
// counted per tile, the tile's output offset comes from a decoupled look-back over the tiles'
// counts (tiles taken by ticket), and the means go straight to their final, ascending-key place.
constexpr int VR_THREADS = LB_THREADS;
template <typename KeyT>
struct VrTile {
    static constexpr int value = sizeof(KeyT) == 4 ? 1024 : 512;
};
constexpr int VR_HALO = 256;  // elements staged past the tile so that its last run rarely leaves shared memory

// one run: strictly sequential fp32 sum over [l, ...) while the key matches — voxel_downsampling.hpp:193-201.
// Returns the global end of the run; sum.w is the divisor of every mean of this voxel.
template <typename KeyT>
__device__ __forceinline__ uint32_t walk_run(const KeyT* sk, const float4* sp, uint32_t l, uint32_t staged, uint32_t base,
                                             const float4* __restrict__ pts, const KeyT* __restrict__ skeys,
                                             const uint32_t* __restrict__ svals, uint32_t n_valid, float4& sum) {
    const KeyT key = sk[l];
    float sx = 0.f, sy = 0.f, sz = 0.f, sw = 0.f;
    // four elements per step, their shared-memory loads issued together and ahead of the key tests: one
    // element at a time is a chain of two dependent loads, a compare and a branch (~100 cycles each)
    bool open = true;
    while (open && l < staged) {
        KeyT kq[4];
        float4 pq[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const uint32_t ll = min(l + u, staged - 1);
            kq[u] = sk[ll];
            pq[u] = sp[ll];
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (open && l < staged && kq[u] == key) {
                sx = __fadd_rn(sx, pq[u].x); sy = __fadd_rn(sy, pq[u].y); sz = __fadd_rn(sz, pq[u].z);
                sw = __fadd_rn(sw, pq[u].w);
                ++l;
            } else {
                open = false;
            }
        }
    }
    // a run longer than the halo goes on in global memory: 8 independent loads in flight per step,
    // the adds stay in (key, index) order
    uint32_t j = base + l;
    open = (l == staged);
    while (open && j < n_valid) {
        KeyT kb[8];
        float4 pb[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const uint32_t jj = min(j + u, n_valid - 1);
            kb[u] = skeys[jj];
            pb[u] = __ldg(pts + svals[jj]);
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            if (open && j < n_valid && kb[u] == key) {
                sx = __fadd_rn(sx, pb[u].x); sy = __fadd_rn(sy, pb[u].y); sz = __fadd_rn(sz, pb[u].z);
                sw = __fadd_rn(sw, pb[u].w);
                ++j;
            } else {
                open = false;
            }
        }
    }
    sum = make_float4(sx, sy, sz, sw);
    return j;
}

// EARLY: the tile publishes its number of RUNS as soon as it knows them, before the walks, and every
// run is written at its run rank.  The look-back after the walks then never waits (a tile that has
// to wait for the slowest tile before it keeps its slot on the SM: publishing after the walks made a
// wave of tiles last as long as its slowest one, 10 of 22 us per tile).  A run that fails the
// min_voxel_count test cannot be compacted away in this mode: it is counted in `dropped`, and the
// host runs the kernel again with EARLY = false (counts published after the walks, only kept runs
// ranked).  With min_voxel_count <= 1 and w == 1 — the reference's homogeneous points — nothing is
// ever dropped.
template <typename KeyT, bool EARLY>
__global__ void __launch_bounds__(VR_THREADS) voxel_reduce_kernel(const float4* __restrict__ pts,
                                                                  const KeyT* __restrict__ skeys,
                                                                  const uint32_t* __restrict__ svals, uint32_t n_valid_arg,
                                                                  const uint32_t* __restrict__ n_valid_dev,
                                                                  float min_count, unsigned long long* status,
                                                                  uint32_t* ticket, float4* __restrict__ out,
                                                                  uint32_t* __restrict__ total_out /*[0] total, [1] dropped*/,
                                                                  VoxAttrs at) {
    // n_valid_dev: the host launched before it knew how many points are valid (guessed key geometry):
    // the grid covers all points and the tiles past the valid ones leave at once
    const uint32_t n_valid = n_valid_dev ? *n_valid_dev : n_valid_arg;
    constexpr int TILE = VrTile<KeyT>::value;
    constexpr int RPT = TILE / VR_THREADS;
    constexpr int WARPS = VR_THREADS / 32;
    __shared__ KeyT sk[TILE + VR_HALO];
    __shared__ float4 sp[TILE + VR_HALO];  // the points; a finished run leaves its mean at its head
    __shared__ uint16_t heads[TILE];       // tile-local start of run r
    __shared__ uint16_t ranks[TILE];       // rank of run r among the tile's kept runs
    __shared__ uint8_t keepf[TILE];
    __shared__ uint32_t sw[33];
    __shared__ uint32_t s_tile, s_min[2];
    __shared__ unsigned long long s_sum;
    __shared__ KeyT s_prev_key;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    if (t == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint32_t base = tile * (uint32_t)TILE;
    if (base >= n_valid) return;
    const uint32_t cnt = min((uint32_t)TILE, n_valid - base);                 // elements owned by the tile
    const uint32_t staged = min((uint32_t)(TILE + VR_HALO), n_valid - base);  // elements in shared memory
    {
        // index loads first, then every gather of the thread in flight together (two round trips per tile
        // instead of two per element)
        constexpr int SPT = (TILE + VR_HALO) / VR_THREADS;
        uint32_t si[SPT];
        KeyT kk[SPT];
        float4 pp[SPT];
        if (t == 0) s_prev_key = base > 0 ? skeys[base - 1] : (KeyT)0;
#pragma unroll
        for (int u = 0; u < SPT; ++u) {
            const uint32_t l = u * VR_THREADS + t;
            si[u] = 0;
            kk[u] = 0;
            if (l < staged) {
                si[u] = svals[base + l];
                kk[u] = skeys[base + l];
            }
        }
#pragma unroll
        for (int u = 0; u < SPT; ++u) pp[u] = __ldg(pts + si[u]);
#pragma unroll
        for (int u = 0; u < SPT; ++u) {
            const uint32_t l = u * VR_THREADS + t;
            if (l < staged) {
                sk[l] = kk[u];
                sp[l] = pp[u];
            }
        }
    }
    __syncthreads();

    // heads of the runs that start in this tile, in order: thread t owns elements RPT*t .. RPT*t + RPT-1
    uint32_t hmask = 0;
#pragma unroll
    for (int u = 0; u < RPT; ++u) {
        const uint32_t l = (uint32_t)t * RPT + u;
        if (l < cnt) {
            const bool head = l > 0 ? sk[l - 1] != sk[l] : (base == 0 || s_prev_key != sk[0]);
            hmask |= (head ? 1u : 0u) << u;
        }
    }
    uint32_t n_heads;
    uint32_t hpos = block_exclusive_scan(__popc(hmask), sw, &n_heads);
#pragma unroll
    for (int u = 0; u < RPT; ++u)
        if (hmask >> u & 1u) heads[hpos++] = (uint16_t)(t * RPT + u);
    if (EARLY) lookback_publish(status, tile, n_heads);
    __syncthreads();

    // the runs are dealt to the warps in slices of m consecutive lanes: packed enough that the walk is
    // not issue-bound, spread enough that every warp takes part and the longest run in a warp is short
    const uint32_t m = min(32u, max(1u, (n_heads + WARPS - 1) / WARPS));
    for (uint32_t r0 = 0; r0 < n_heads; r0 += WARPS * m) {
        const uint32_t r = r0 + warp * m + lane;
        if ((uint32_t)lane < m && r < n_heads) {
            const uint32_t l = heads[r];
            float4 sum;
            walk_run<KeyT>(sk, sp, l, staged, base, pts, skeys, svals, n_valid, sum);
            const bool kept = sum.w >= min_count;  // :204
            keepf[r] = kept ? 1 : 0;
            // only this run's walker ever reads the run's elements, so its head can take the result
            if (kept)
                sp[l] = make_float4(__fdiv_rn(sum.x, sum.w), __fdiv_rn(sum.y, sum.w), __fdiv_rn(sum.z, sum.w),
                                    __fdiv_rn(sum.w, sum.w));
        }
    }
    __syncthreads();
    uint32_t n_keep = n_heads;
    if (!EARLY) {
        uint32_t mine = 0;
#pragma unroll
        for (int u = 0; u < RPT; ++u) {
            const uint32_t r = (uint32_t)t * RPT + u;
            if (r < n_heads) mine += keepf[r];
        }
        uint32_t rank = block_exclusive_scan(mine, sw, &n_keep);
#pragma unroll
        for (int u = 0; u < RPT; ++u) {
            const uint32_t r = (uint32_t)t * RPT + u;
            if (r < n_heads) {
                ranks[r] = (uint16_t)rank;
                rank += keepf[r];
            }
        }
        lookback_publish(status, tile, n_keep);
    } else {
        uint32_t lost = 0;
#pragma unroll
        for (int u = 0; u < RPT; ++u) {
            const uint32_t r = (uint32_t)t * RPT + u;
            if (r < n_heads) {
                ranks[r] = (uint16_t)r;
                lost += keepf[r] ? 0u : 1u;
            }
        }
        if (lost) atomicAdd(total_out + 1, lost);
    }
    const unsigned long long off = block_lookback(status, tile, n_keep, s_min, &s_sum);
    if (t == 0 && base + cnt == n_valid) *total_out = (uint32_t)(off + n_keep);
#pragma unroll
    for (int u = 0; u < RPT; ++u) {
        const uint32_t r = (uint32_t)t * RPT + u;
        if (r < n_heads && keepf[r]) out[off + ranks[r]] = sp[heads[r]];
    }
    if (at.rgb || at.intensity || at.timestamps) {
        // optional attributes over the same runs, written at the same output position
        for (uint32_t r = t; r < n_heads; r += VR_THREADS) {
            if (!keepf[r]) continue;
            const size_t o = off + ranks[r];
            const uint32_t l = heads[r];
            const uint32_t i = base + l;
            uint32_t j = i + 1;  // extent and divisor again, in the same order (the head's point is gone)
            float wsum = __ldg(pts + svals[i]).w;
            wsum = __fadd_rn(0.f, wsum);
            const KeyT key = sk[l];
            while (j < n_valid && skeys[j] == key) {
                wsum = __fadd_rn(wsum, __ldg(pts + svals[j]).w);
                ++j;
            }
            if (at.rgb) {
                float rr = 0.f, g = 0.f, b = 0.f, a = 0.f;
                for (uint32_t e = i; e < j; ++e) {
                    const float4 c = __ldg(at.rgb + svals[e]);
                    rr = __fadd_rn(rr, c.x); g = __fadd_rn(g, c.y); b = __fadd_rn(b, c.z); a = __fadd_rn(a, c.w);
                }
                at.rgb_mean[o] = make_float4(__fdiv_rn(rr, wsum), __fdiv_rn(g, wsum), __fdiv_rn(b, wsum), __fdiv_rn(a, wsum));
            }
            if (at.timestamps) {
                float ts = 0.f;
                for (uint32_t e = i; e < j; ++e) ts = __fadd_rn(ts, __ldg(at.timestamps + svals[e]));
                at.ts_mean[o] = __fdiv_rn(ts, wsum);
            }
            if (at.intensity) {
                const uint32_t len = j - i, mid = len / 2;
                const float up = run_select(at.intensity, svals, i, j, mid);
                at.intensity_med[o] = (len & 1u) ? up
                                                 : __fmul_rn(0.5f, __fadd_rn(run_select(at.intensity, svals, i, j, mid - 1), up));
            }
        }
    }
}

__global__ void __launch_bounds__(VX_THREADS) compact_float4_kernel(const float4* __restrict__ in,
                                                                    const uint32_t* __restrict__ flags,
                                                                    const uint32_t* __restrict__ pos, uint32_t n,
                                                                    float4* __restrict__ out) {
    const uint32_t i = blockIdx.x * VX_THREADS + threadIdx.x;
    if (i >= n) return;
    if (flags[i]) out[pos[i]] = in[i];
}

// (compact_index_kernel, the index form of the same compaction, lives in spx_scan.cuh: the outlier filters use it too)
static_assert(VX_THREADS == COMPACT_THREADS, "compact_index_kernel is launched with VX_THREADS threads");

// box_filter — preprocess_operator/box_filter_operator.hpp:36-44 + common.hpp:15-25
__global__ void __launch_bounds__(VX_THREADS) box_flag_kernel(const float4* __restrict__ pts, uint32_t n, float mn,
                                                              float mx, uint32_t* __restrict__ flags) {
    const uint32_t i = blockIdx.x * VX_THREADS + threadIdx.x;
    if (i >= n) return;
    const float4 p = __ldg(pts + i);
    uint32_t keep = 0;
    if (isfinite(p.x) && isfinite(p.y) && isfinite(p.z) && isfinite(p.w)) {
        const float linf = fmaxf(fabsf(p.x), fmaxf(fabsf(p.y), fabsf(p.z)));
        keep = !(linf < mn || linf > mx);
    }
    flags[i] = keep;
}

// angle_incidence_filter — preprocess_operator/angle_incidence_filter_operator.hpp:57-103: keep a point when the
// |cosine| between its direction from the sensor and its surface normal lies in [cos(max_angle), cos(min_angle)];
// the normal is the stored one, or extract_normal of the covariance (covariance.hpp:49-65: eigenvector of the
// smallest eigenvalue; the sign does not matter under the absolute value).  Non-finite points and degenerate
// directions (|p| |n| <= 1e-6) are removed.  The test is the reference's `denom <= 1e-6` negated, not
// `denom > 1e-6`: a NaN normal (a stored one, or the covariance of a list with a non-finite neighbour) makes the
// cosine NaN, and such a point is kept, as in the reference.
__global__ void __launch_bounds__(VX_THREADS) angle_flag_kernel(const float4* __restrict__ pts, const float4* __restrict__ normals,
                                                                const float* __restrict__ covs, uint32_t n, float min_cos,
                                                                float max_cos, uint32_t* __restrict__ flags) {
    const uint32_t i = blockIdx.x * VX_THREADS + threadIdx.x;
    if (i >= n) return;
    const float4 p = __ldg(pts + i);
    uint32_t keep = 0;
    if (isfinite(p.x) && isfinite(p.y) && isfinite(p.z) && isfinite(p.w)) {
        float nx, ny, nz;
        if (normals) {
            const float4 nr = __ldg(normals + i);
            nx = nr.x; ny = nr.y; nz = nr.z;
        } else {
            float ev[3], V[3][3];
            mat3_eigen(load_cov16(covs + (size_t)i * 16), ev, V);
            nx = V[0][0]; ny = V[1][0]; nz = V[2][0];
        }
        const float dot = __fmaf_rn(p.z, nz, __fmaf_rn(p.y, ny, __fmul_rn(p.x, nx)));
        const float pn = __fsqrt_rn(__fmaf_rn(p.z, p.z, __fmaf_rn(p.y, p.y, __fmul_rn(p.x, p.x))));
        const float nn = __fsqrt_rn(__fmaf_rn(nz, nz, __fmaf_rn(ny, ny, __fmul_rn(nx, nx))));
        const float denom = __fmul_rn(pn, nn);
        if (!(denom <= 1e-6f)) {
            const float abs_cos = fabsf(__fdiv_rn(dot, denom));
            keep = !(abs_cos < min_cos || abs_cos > max_cos);
        }
    }
    flags[i] = keep;
}

// farthest_point_sampling — preprocess_operator/farthest_point_sampling_operator.hpp:27-94.  The reference runs one
// kernel (min-distance update) and one host std::max_element per selected point; here the whole selection is ONE
// cooperative launch: per round every block updates its slice against the point selected last, reduces
// (distance, lowest index) to a 64-bit key, the grid meets once and every block reads the blocks' keys to agree on
// the next point.  Same arithmetic (dot<4> fma chain over the xyzw difference, eigen_utils.hpp:245-253,333-335) and
// the same tie rule (std::max_element: the first of equal maxima), so the selected set is the reference's.
constexpr int FPS_THREADS = 256;
__global__ void __launch_bounds__(FPS_THREADS) fps_kernel(const float4* __restrict__ pts, uint32_t n, uint32_t first,
                                                          uint32_t rounds, float* __restrict__ dist_sq,
                                                          uint32_t* __restrict__ flags,
                                                          unsigned long long* __restrict__ block_keys /*[2][gridDim.x]*/) {
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    __shared__ unsigned long long s_key[FPS_THREADS / 32];
    __shared__ uint32_t s_sel;
    const uint32_t stride = gridDim.x * FPS_THREADS;
    for (uint32_t i = blockIdx.x * FPS_THREADS + threadIdx.x; i < n; i += stride) {
        dist_sq[i] = FLT_MAX;
        flags[i] = 0u;
    }
    uint32_t sel = first;
    if (blockIdx.x == 0 && threadIdx.x == 0) flags[sel] = 1u;  // (each thread initialises only its own slots above;
    grid.sync();                                               //  the selected flag is re-asserted after the barrier)
    if (blockIdx.x == 0 && threadIdx.x == 0) flags[sel] = 1u;
    for (uint32_t it = 1; it < rounds; ++it) {
        const float4 c = __ldg(pts + sel);
        unsigned long long best = 0ull;
        for (uint32_t i = blockIdx.x * FPS_THREADS + threadIdx.x; i < n; i += stride) {
            const float4 p = __ldg(pts + i);
            const float dx = __fsub_rn(p.x, c.x), dy = __fsub_rn(p.y, c.y), dz = __fsub_rn(p.z, c.z), dw = __fsub_rn(p.w, c.w);
            const float d = __fmaf_rn(dw, dw, __fmaf_rn(dz, dz, __fmaf_rn(dy, dy, __fmul_rn(dx, dx))));
            const float m = fminf(dist_sq[i], d);
            dist_sq[i] = m;
            // larger distance first, then the LOWER index: key = dist bits (non-negative floats order as integers;
            // a NaN distance — from a non-finite point — never wins, as in std::max_element's operator<) | ~index
            const unsigned long long key = ((unsigned long long)__float_as_uint(m == m ? m : 0.0f) << 32) | (0xffffffffu - i);
            best = key > best ? key : best;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long other = __shfl_xor_sync(0xffffffffu, best, o);
            best = other > best ? other : best;
        }
        if ((threadIdx.x & 31) == 0) s_key[threadIdx.x >> 5] = best;
        __syncthreads();
        unsigned long long* keys = block_keys + (size_t)(it & 1u) * gridDim.x;
        if (threadIdx.x == 0) {
            unsigned long long b = s_key[0];
            for (int w = 1; w < FPS_THREADS / 32; ++w) b = s_key[w] > b ? s_key[w] : b;
            keys[blockIdx.x] = b;
        }
        grid.sync();
        if (threadIdx.x < 32) {
            unsigned long long b = 0ull;
            for (uint32_t j = threadIdx.x; j < gridDim.x; j += 32) {
                const unsigned long long kj = keys[j];
                b = kj > b ? kj : b;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const unsigned long long other = __shfl_xor_sync(0xffffffffu, b, o);
                b = other > b ? other : b;
            }
            if (threadIdx.x == 0) s_sel = 0xffffffffu - (uint32_t)(b & 0xffffffffull);
        }
        __syncthreads();
        sel = s_sel;
        if (blockIdx.x == 0 && threadIdx.x == 0) flags[sel] = 1u;
    }
}

// order given by idx: dst[j] = src[idx[j]], in 4-byte words (points 4 words, covariances 16)
__global__ void __launch_bounds__(VX_THREADS) gather_words_kernel(const uint32_t* __restrict__ src, int words,
                                                                  const int32_t* __restrict__ idx, size_t total,
                                                                  uint32_t* __restrict__ dst) {
    const size_t t = (size_t)blockIdx.x * VX_THREADS + threadIdx.x;
    if (t >= total) return;
    const size_t j = t / words;
    const int w = (int)(t - j * words);
    dst[t] = __ldg(src + (size_t)__ldg(idx + j) * words + w);
}
__global__ void __launch_bounds__(VX_THREADS) gather_vec4_kernel(const uint4* __restrict__ src, int vecs,
                                                                 const int32_t* __restrict__ idx, size_t total,
                                                                 uint4* __restrict__ dst) {
    const size_t t = (size_t)blockIdx.x * VX_THREADS + threadIdx.x;
    if (t >= total) return;
    const size_t j = t / vecs;
    const int w = (int)(t - j * vecs);
    dst[t] = __ldg(src + (size_t)__ldg(idx + j) * vecs + w);
}

struct VoxAttrIO {
    const float4* rgb = nullptr;
    const float* intensity = nullptr;
    const float* timestamps = nullptr;
    float4* out_rgb = nullptr;
    float* out_intensity = nullptr;
    float* out_timestamps = nullptr;
};

template <typename KeyT>
// guessed: the key geometry comes from the previous call (the bounding box of THIS cloud is still on its
// way to the host in `hacc`): the number of valid points is read on the device, and a point outside the
// guessed box raises total_dev[2] — the function then returns false and the caller starts over.
bool sort_and_reduce(spx_queue_t q, const float4* pts, uint32_t n, const CoordMap& cm, const KeyGeom& geom, int key_bits,
                     uint32_t n_valid, float min_count, float4* out, uint32_t* htotal, const VoxAttrIO& io, bool guessed,
                     CoordAcc* acc, CoordAcc* hacc) {
    cudaStream_t st = q->stream;
    KeyT* keys_a = q->take<KeyT>(n);
    KeyT* keys_b = q->take<KeyT>(n);
    uint32_t* vals_a = q->take<uint32_t>(n);
    uint32_t* vals_b = q->take<uint32_t>(n);
    VoxAttrs at{};
    at.rgb = io.rgb;
    at.intensity = io.intensity;
    at.timestamps = io.timestamps;

    const int passes = std::max(1, (key_bits + RADIX_BITS - 1) / RADIX_BITS);
    const bool onesweep = n < OS_LOCAL;
    // one zeroed block for everything the look-backs need:
    // [digit histograms 8 x 256][sort tickets 64][sort status passes x tiles x 256][reduce ticket 2][reduce status 2 x tiles]
    const uint32_t os_tiles = onesweep ? (uint32_t)div_up(n, RS_THREADS * OsItems<KeyT>::value) : 0u;
    const uint32_t vr_tiles = (uint32_t)div_up(guessed ? n : std::max(n_valid, 1u), VrTile<KeyT>::value);
    const size_t os_words = (size_t)OS_MAX_PASSES * RADIX + 64 + (size_t)passes * os_tiles * RADIX;
    const size_t words = os_words + 2 + 2 * (size_t)vr_tiles + 8 + 4;  // ... [box accumulator 8][result counters 4]
    uint32_t* os = q->take<uint32_t>(words);
    uint32_t* lb_ticket = os + os_words;
    unsigned long long* lb_status = reinterpret_cast<unsigned long long*>(os + os_words + 2);
    if (guessed) acc = reinterpret_cast<CoordAcc*>(os + os_words + 2 + 2 * (size_t)vr_tiles);  // zeroed with the rest
    uint32_t* total_dev = os + os_words + 2 + 2 * (size_t)vr_tiles + 8;  // {voxels kept, runs dropped, point outside the box}
    SPX_CUDA(cudaMemsetAsync(os, 0, words * sizeof(uint32_t), st));

    KeyT* kin = keys_a;
    KeyT* kout = keys_b;
    uint32_t* vin = nullptr;  // first pass: value = position
    uint32_t* vout = vals_a;
    if (onesweep) {
        // one kernel per digit: histograms of all passes from the key kernel, look-back instead of scans
        const int kh_grid = std::min((int)div_up(n, VX_THREADS * 4), q->sm_count * 8);
        if (cm.polar)
            voxel_key_hist_kernel<KeyT, true><<<kh_grid, VX_THREADS, 0, st>>>(pts, n, cm, geom, keys_a, passes, os,
                                                                              total_dev + 2, guessed ? acc : nullptr);
        else
            voxel_key_hist_kernel<KeyT, false><<<kh_grid, VX_THREADS, 0, st>>>(pts, n, cm, geom, keys_a, passes, os,
                                                                               total_dev + 2, guessed ? acc : nullptr);
        SPX_LAUNCH_CHECK();
        for (int p = 0; p < passes; ++p) {
            onesweep_kernel<KeyT><<<os_tiles, RS_THREADS, 0, st>>>(
                kin, vin, kout, vout, os + p * RADIX, os + OS_MAX_PASSES * RADIX + 64 + (size_t)p * os_tiles * RADIX,
                os + OS_MAX_PASSES * RADIX + p, n, p * RADIX_BITS);
            SPX_LAUNCH_CHECK();
            std::swap(kin, kout);
            vin = vout;
            vout = (vout == vals_a) ? vals_b : vals_a;
        }
    } else {
        uint32_t* sort_tmp = q->take<uint32_t>(radix_sort_scratch_elems(n));
        if (cm.polar)
            voxel_key_kernel<KeyT, true><<<div_up(n, VX_THREADS), VX_THREADS, 0, st>>>(pts, n, cm, geom, keys_a);
        else
            voxel_key_kernel<KeyT, false><<<div_up(n, VX_THREADS), VX_THREADS, 0, st>>>(pts, n, cm, geom, keys_a);
        SPX_LAUNCH_CHECK();
        KeyT* const keys[2] = {keys_a, keys_b};
        uint32_t* const vals[2] = {vals_a, vals_b};
        radix_sort_pairs<KeyT>(st, n, passes, keys, nullptr, vals, sort_tmp);
        kin = keys[passes & 1];
        vin = vals[(passes - 1) & 1];
    }
    // kin / vin now hold the sorted (key, index) pairs; dropped points (invalid key) sit at the end
    if (!guessed && n_valid == 0) {
        htotal[0] = 0;
        return true;
    }
    at.rgb_mean = io.out_rgb;
    at.intensity_med = io.out_intensity;
    at.ts_mean = io.out_timestamps;
    const uint32_t* n_valid_dev = guessed ? &acc->valid : nullptr;
    const bool early = min_count <= 1.0f;
    if (early)
        voxel_reduce_kernel<KeyT, true><<<vr_tiles, VR_THREADS, 0, st>>>(pts, kin, vin, n_valid, n_valid_dev, min_count,
                                                                        lb_status, lb_ticket, out, total_dev, at);
    else
        voxel_reduce_kernel<KeyT, false><<<vr_tiles, VR_THREADS, 0, st>>>(pts, kin, vin, n_valid, n_valid_dev, min_count,
                                                                         lb_status, lb_ticket, out, total_dev, at);
    SPX_LAUNCH_CHECK();
    SPX_CUDA(cudaMemcpyAsync(htotal, total_dev, 4 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    if (guessed) SPX_CUDA(cudaMemcpyAsync(hacc, acc, sizeof(CoordAcc), cudaMemcpyDeviceToHost, st));
    q->sync();
    if (guessed && htotal[2] != 0) return false;
    if (early && htotal[1] != 0) {
        // some voxel failed the min_voxel_count test (points with w < 1): again, ranking only the kept runs
        SPX_CUDA(cudaMemsetAsync(lb_ticket, 0, (2 + 2 * (size_t)vr_tiles) * sizeof(uint32_t), st));
        SPX_CUDA(cudaMemsetAsync(total_dev, 0, 2 * sizeof(uint32_t), st));
        voxel_reduce_kernel<KeyT, false><<<vr_tiles, VR_THREADS, 0, st>>>(pts, kin, vin, n_valid, n_valid_dev, min_count,
                                                                         lb_status, lb_ticket, out, total_dev, at);
        SPX_LAUNCH_CHECK();
        SPX_CUDA(cudaMemcpyAsync(htotal, total_dev, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        q->sync();
    }
    return true;
}

// The grid filters' common body.  `cm` chooses the grid (voxel or polar); voxel_size is only the tag under which the
// voxel grid's key box is remembered between calls (0 for the polar grid, which never guesses).
void grid_downsample(spx_queue_t q, const CoordMap& cm, float voxel_size, const float* points, size_t n_in,
                     size_t min_voxel_count, const float* rgb, const float* intensity, const float* timestamps,
                     float* out_points, float* out_rgb, float* out_intensity, float* out_timestamps, size_t* m_host) {
    {
        SPX_REQUIRE(q && m_host, "[VoxelGrid::downsampling] null argument");
        SPX_REQUIRE(n_in < (1ull << 31), "[VoxelGrid::downsampling] too many points");
        *m_host = 0;
        q->voxel_last.valid = false;
        if (n_in == 0) return;
        SPX_REQUIRE(points && out_points, "[VoxelGrid::downsampling] null pointer");
        SPX_REQUIRE((!rgb || out_rgb) && (!intensity || out_intensity) && (!timestamps || out_timestamps),
                    "[VoxelGrid::downsampling] attribute given without its output array");
        DeviceGuard dg(q->device);
        cudaStream_t st = q->stream;
        const uint32_t n = (uint32_t)n_in;
        const float4* pts = reinterpret_cast<const float4*>(points);
        const uint32_t nblocks = (uint32_t)div_up(n, RS_TILE);

        q->arena_reset();
        // two key and two index buffers, then either the look-back tables or the histogram + scan scratch
        q->arena_reserve((size_t)n * (8 * 2 + 4 * 2) + ((size_t)RADIX * nblocks + 64) * 4 +
                         scan_scratch_elems((size_t)RADIX * nblocks) * 4 +
                         ((size_t)OS_MAX_PASSES * RADIX + 64 + (size_t)OS_MAX_PASSES * (div_up(n, RS_TILE) + 1) * RADIX) * 4 +
                         (2 + 2 * (div_up(n, 512) + 1) + 12) * 4 + 16 * 256 + 8192);
        const float min_count = (float)min_voxel_count;
        float4* out = reinterpret_cast<float4*>(out_points);
        VoxAttrIO io;
        io.rgb = reinterpret_cast<const float4*>(rgb);
        io.intensity = intensity;
        io.timestamps = timestamps;
        io.out_rgb = reinterpret_cast<float4*>(out_rgb);
        io.out_intensity = out_intensity;
        io.out_timestamps = out_timestamps;
        char* pin = static_cast<char*>(q->pinned_get(256));
        CoordAcc* hacc = reinterpret_cast<CoordAcc*>(pin);
        uint32_t* htotal = reinterpret_cast<uint32_t*>(pin + 128);

        // Key geometry.  The exact one needs this cloud's voxel bounding box on the host — a round trip
        // in the middle of the chain.  When the previous call on this queue used the same voxel size
        // (consecutive scans of one sensor), its box, padded, is used instead and the sort starts at
        // once; the box of THIS cloud is still computed, comes back with the result, and the key kernel
        // checks every point against the guess: one point outside and the call starts over, exactly.
        // The compact key is order-preserving for any box that contains the points, so the output does
        // not depend on which box was used.
        auto& cache = q->voxel_geom;
        bool guessed = !cm.polar && cache.valid && cache.voxel == voxel_size && n < OS_LOCAL &&
                       !std::getenv("SPX_VOXEL_EXACT_BOX");
        bool have_box = false;  // a failed guess leaves this cloud's own box in hacc
        for (;;) {
            CoordAcc* acc = nullptr;  // guessed: lives in sort_and_reduce's zeroed scratch, filled by the key kernel
            if (!have_box && !guessed) {
                acc = q->take<CoordAcc>(1);
                SPX_CUDA(cudaMemsetAsync(acc, 0, sizeof(CoordAcc), st));
                const int bb_grid = std::min((int)div_up(n, VX_THREADS), q->sm_count * 8);
                if (cm.polar) voxel_bbox_kernel<true><<<bb_grid, VX_THREADS, 0, st>>>(pts, n, cm, acc);
                else voxel_bbox_kernel<false><<<bb_grid, VX_THREADS, 0, st>>>(pts, n, cm, acc);
                SPX_LAUNCH_CHECK();
            }
            int box_mn[3], box_mx[3];
            uint32_t n_valid = 0;
            bool has_invalid = true;
            if (!guessed) {
                if (!have_box) {
                    SPX_CUDA(cudaMemcpyAsync(hacc, acc, sizeof(CoordAcc), cudaMemcpyDeviceToHost, st));
                    q->sync();
                    coord_acc_decode(hacc);
                }
                if (hacc->valid == 0) {
                    cache.valid = false;
                    return;
                }
                for (int a = 0; a < 3; ++a) {
                    box_mn[a] = hacc->mn[a];
                    box_mx[a] = hacc->mx[a];
                }
                n_valid = hacc->valid;
                has_invalid = n_valid != n;
            } else {
                // pad by 1/16 of the extent (at least 4 voxels) unless that costs a radix pass
                auto bits_with_pad = [&](int shift, int floor_pad) {
                    unsigned long long cells = 1;
                    for (int a = 0; a < 3; ++a) {
                        const long long d = (long long)cache.mx[a] - cache.mn[a] + 1;
                        const long long pad = shift >= 0 ? std::max<long long>(floor_pad, d >> shift) : 0;
                        const long long lo = std::max<long long>(0, cache.mn[a] - pad);
                        const long long hi = std::min<long long>((1ll << 21) - 1, cache.mx[a] + pad);
                        cells *= (unsigned long long)(hi - lo + 1);
                    }
                    return bits_for(cells);
                };
                const int exact_passes = (bits_with_pad(-1, 0) + RADIX_BITS - 1) / RADIX_BITS;
                int shift = 4, floor_pad = 4;
                if ((bits_with_pad(4, 4) + RADIX_BITS - 1) / RADIX_BITS > exact_passes) {
                    shift = 31;  // d >> 31 == 0
                    floor_pad = (bits_with_pad(31, 2) + RADIX_BITS - 1) / RADIX_BITS > exact_passes ? 0 : 2;
                }
                for (int a = 0; a < 3; ++a) {
                    const long long d = (long long)cache.mx[a] - cache.mn[a] + 1;
                    const long long pad = std::max<long long>(floor_pad, d >> shift);
                    box_mn[a] = (int)std::max<long long>(0, cache.mn[a] - pad);
                    box_mx[a] = (int)std::min<long long>((1ll << 21) - 1, cache.mx[a] + pad);
                }
            }
            KeyGeom geom;
            unsigned long long dim[3];
            for (int a = 0; a < 3; ++a) {
                geom.mn[a] = box_mn[a];
                geom.mx[a] = box_mx[a];
                dim[a] = (unsigned long long)(box_mx[a] - box_mn[a]) + 1ull;
            }
            geom.nx = dim[0];
            geom.nxy = dim[0] * dim[1];
            const unsigned long long max_key = dim[0] * dim[1] * dim[2] - 1ull;  // <= 2^63 - 1
            geom.invalid = max_key + 1ull;
            const int key_bits = bits_for(has_invalid ? geom.invalid : max_key);
            const bool ok = key_bits <= 32 ? sort_and_reduce<uint32_t>(q, pts, n, cm, geom, key_bits, n_valid, min_count, out,
                                                                      htotal, io, guessed, acc, hacc)
                                           : sort_and_reduce<unsigned long long>(q, pts, n, cm, geom, key_bits, n_valid,
                                                                                min_count, out, htotal, io, guessed, acc,
                                                                                hacc);
            if (guessed) coord_acc_decode(hacc);  // this cloud's own box came back with the result
            if (ok) break;
            guessed = false;  // a point fell outside the guessed box: once more with this cloud's own box
            have_box = true;
            q->arena_reset();
        }
        // hacc holds this cloud's box either way: it is the next call's guess — joined with the previous guess
        // when that costs no radix pass (a queue that alternates between two clouds, source and target of a
        // pair, would otherwise miss on every larger one)
        if (cm.polar) {  // polar cells say nothing about a Cartesian box: no hint, no guess for the next call
            cache.valid = false;
            if (hacc->valid == 0) htotal[0] = 0;
            *m_host = htotal[0];
            return;
        }
        q->voxel_last.valid = hacc->valid > 0;
        q->voxel_last.voxel = voxel_size;
        for (int a = 0; a < 3; ++a) {
            q->voxel_last.mn[a] = hacc->mn[a];
            q->voxel_last.mx[a] = hacc->mx[a];
        }
        if (hacc->valid > 0) {
            int mn[3], mx[3];
            bool join = cache.valid && cache.voxel == voxel_size;
            unsigned long long own = 1, both = 1;
            for (int a = 0; a < 3; ++a) {
                mn[a] = join ? std::min(cache.mn[a], hacc->mn[a]) : hacc->mn[a];
                mx[a] = join ? std::max(cache.mx[a], hacc->mx[a]) : hacc->mx[a];
                own *= (unsigned long long)(hacc->mx[a] - hacc->mn[a]) + 1ull;
                both *= (unsigned long long)(mx[a] - mn[a]) + 1ull;
            }
            join = join && (bits_for(both) + RADIX_BITS - 1) / RADIX_BITS == (bits_for(own) + RADIX_BITS - 1) / RADIX_BITS;
            for (int a = 0; a < 3; ++a) {
                cache.mn[a] = join ? mn[a] : hacc->mn[a];
                cache.mx[a] = join ? mx[a] : hacc->mx[a];
            }
            cache.valid = true;
            cache.voxel = voxel_size;
        } else {
            cache.valid = false;
        }
        if (guessed && hacc->valid == 0) htotal[0] = 0;
        *m_host = htotal[0];
    }
}
}  // namespace

extern "C" {

int spx_voxel_downsample_attrs(spx_queue_t q, const float* points, size_t n_in, float voxel_size,
                               size_t min_voxel_count, const float* rgb, const float* intensity,
                               const float* timestamps, float* out_points, float* out_rgb, float* out_intensity,
                               float* out_timestamps, size_t* m_host) {
    return guard([&] {
        if (!(voxel_size > 0.0f)) throw Error(SPX_ERR_INVALID_ARGUMENT, "voxel_size must be positive");
        CoordMap cm;
        cm.inv[0] = cm.inv[1] = cm.inv[2] = 1.0f / voxel_size;  // voxel_downsampling.hpp:27
        cm.polar = 0;
        grid_downsample(q, cm, voxel_size, points, n_in, min_voxel_count, rgb, intensity, timestamps, out_points, out_rgb,
                        out_intensity, out_timestamps, m_host);
    });
}

int spx_polar_downsample_attrs(spx_queue_t q, const float* points, size_t n_in, float distance_voxel_size,
                               float elevation_voxel_size, float azimuth_voxel_size, int coordinate_system,
                               size_t min_voxel_count, const float* rgb, const float* intensity, const float* timestamps,
                               float* out_points, float* out_rgb, float* out_intensity, float* out_timestamps,
                               size_t* m_host) {
    return guard([&] {
        if (!(distance_voxel_size > 0.0f && elevation_voxel_size > 0.0f && azimuth_voxel_size > 0.0f))
            throw Error(SPX_ERR_INVALID_ARGUMENT, "voxel sizes must be positive");  // polar_downsampling.hpp:129-131
        SPX_REQUIRE(coordinate_system == SPX_COORD_LIDAR || coordinate_system == SPX_COORD_CAMERA,
                    "[PolarGrid::downsampling] unknown coordinate system");
        CoordMap cm;
        cm.inv[0] = 1.0f / distance_voxel_size;  // :133-135
        cm.inv[1] = 1.0f / elevation_voxel_size;
        cm.inv[2] = 1.0f / azimuth_voxel_size;
        cm.polar = coordinate_system == SPX_COORD_LIDAR ? 1 : 2;
        grid_downsample(q, cm, 0.0f, points, n_in, min_voxel_count, rgb, intensity, timestamps, out_points, out_rgb,
                        out_intensity, out_timestamps, m_host);
    });
}

int spx_voxel_last_box(spx_queue_t q, float* lo3_host, float* hi3_host, float* voxel_size) {
    return guard([&] {
        SPX_REQUIRE(q && lo3_host && hi3_host, "[VoxelGrid::last_box] null argument");
        SPX_REQUIRE(q->voxel_last.valid, "[VoxelGrid::last_box] no down-sampled cloud on this queue yet");
        // voxel coordinate c (offset by 2^20, voxel_constants.hpp:36-53) covers [c, c + 1) * voxel in floor(p * (1 / voxel));
        // one voxel of slack on both sides absorbs the rounding of p * inv against c * voxel
        const float v = q->voxel_last.voxel;
        for (int a = 0; a < 3; ++a) {
            lo3_host[a] = (float)(q->voxel_last.mn[a] - (1 << 20) - 1) * v;
            hi3_host[a] = (float)(q->voxel_last.mx[a] - (1 << 20) + 2) * v;
        }
        if (voxel_size) *voxel_size = v;
    });
}

int spx_voxel_downsample(spx_queue_t q, const float* points, size_t n_in, float voxel_size, size_t min_voxel_count,
                         float* out_points, size_t* m_host) {
    return spx_voxel_downsample_attrs(q, points, n_in, voxel_size, min_voxel_count, nullptr, nullptr, nullptr,
                                      out_points, nullptr, nullptr, nullptr, m_host);
}

int spx_box_filter(spx_queue_t q, const float* points, size_t n_in, float min_distance, float max_distance,
                   float* out_points, size_t* m_host) {
    return guard([&] {
        SPX_REQUIRE(q && m_host, "[PreprocessFilter::box_filter] null argument");
        SPX_REQUIRE(n_in < (1ull << 31), "[PreprocessFilter::box_filter] too many points");
        *m_host = 0;
        if (n_in == 0) return;
        SPX_REQUIRE(points && out_points, "[PreprocessFilter::box_filter] null pointer");
        DeviceGuard dg(q->device);
        cudaStream_t st = q->stream;
        const uint32_t n = (uint32_t)n_in;
        q->arena_reset();
        q->arena_reserve((size_t)n * 8 + scan_scratch_elems(n) * 4 + 4096);
        uint32_t* flags = q->take<uint32_t>(n);
        uint32_t* pos = q->take<uint32_t>(n);
        uint32_t* scan_tmp = q->take<uint32_t>(scan_scratch_elems(n));
        uint32_t* total_dev = q->take<uint32_t>(16);
        const float4* pts = reinterpret_cast<const float4*>(points);
        box_flag_kernel<<<div_up(n, VX_THREADS), VX_THREADS, 0, st>>>(pts, n, min_distance, max_distance, flags);
        SPX_LAUNCH_CHECK();
        exclusive_scan_u32(st, flags, pos, n, scan_tmp, total_dev);
        compact_float4_kernel<<<div_up(n, VX_THREADS), VX_THREADS, 0, st>>>(pts, flags, pos, n,
                                                                           reinterpret_cast<float4*>(out_points));
        SPX_LAUNCH_CHECK();
        uint32_t* htotal = static_cast<uint32_t*>(q->pinned_get(64));
        SPX_CUDA(cudaMemcpyAsync(htotal, total_dev, 4, cudaMemcpyDeviceToHost, st));
        q->sync();
        *m_host = *htotal;
    });
}

int spx_box_filter_indices(spx_queue_t q, const float* points, size_t n_in, float min_distance, float max_distance,
                           int32_t* idx_out, size_t* m_host) {
    return guard([&] {
        SPX_REQUIRE(q && m_host, "[PreprocessFilter::box_filter] null argument");
        SPX_REQUIRE(n_in < (1ull << 31), "[PreprocessFilter::box_filter] too many points");
        *m_host = 0;
        if (n_in == 0) return;
        SPX_REQUIRE(points && idx_out, "[PreprocessFilter::box_filter] null pointer");
        DeviceGuard dg(q->device);
        cudaStream_t st = q->stream;
        const uint32_t n = (uint32_t)n_in;
        q->arena_reset();
        q->arena_reserve((size_t)n * 8 + scan_scratch_elems(n) * 4 + 4096);
        uint32_t* flags = q->take<uint32_t>(n);
        uint32_t* pos = q->take<uint32_t>(n);
        uint32_t* scan_tmp = q->take<uint32_t>(scan_scratch_elems(n));
        uint32_t* total_dev = q->take<uint32_t>(16);
        box_flag_kernel<<<div_up(n, VX_THREADS), VX_THREADS, 0, st>>>(reinterpret_cast<const float4*>(points), n, min_distance,
                                                                     max_distance, flags);
        SPX_LAUNCH_CHECK();
        exclusive_scan_u32(st, flags, pos, n, scan_tmp, total_dev);
        compact_index_kernel<<<div_up(n, VX_THREADS), VX_THREADS, 0, st>>>(flags, pos, n, idx_out);
        SPX_LAUNCH_CHECK();
        uint32_t* htotal = static_cast<uint32_t*>(q->pinned_get(64));
        SPX_CUDA(cudaMemcpyAsync(htotal, total_dev, 4, cudaMemcpyDeviceToHost, st));
        q->sync();
        *m_host = *htotal;
    });
}

int spx_angle_incidence_indices(spx_queue_t q, const float* points, const float* normals, const float* covs, size_t n_in,
                                float min_angle, float max_angle, int32_t* idx_out, size_t* m_host) {
    return guard([&] {
        SPX_REQUIRE(q && m_host, "[PreprocessFilter::angle_incidence_filter] null argument");
        SPX_REQUIRE(n_in < (1ull << 31), "[PreprocessFilter::angle_incidence_filter] too many points");
        *m_host = 0;
        if (n_in == 0) return;
        if (!normals && !covs)
            throw Error(SPX_ERR_INVALID_ARGUMENT,
                        "[PreprocessFilter::angle_incidence_filter] Normal vector or covariance matrices must be pre-computed.");
        SPX_REQUIRE(!(min_angle < 0.0f || max_angle > 3.14159265358979323846f * 0.5f || min_angle >= max_angle),
                    "[PreprocessFilter::angle_incidence_filter] Invalid angle range");
        SPX_REQUIRE(points && idx_out, "[PreprocessFilter::angle_incidence_filter] null pointer");
        DeviceGuard dg(q->device);
        cudaStream_t st = q->stream;
        const uint32_t n = (uint32_t)n_in;
        q->arena_reset();
        q->arena_reserve((size_t)n * 8 + scan_scratch_elems(n) * 4 + 4096);
        uint32_t* flags = q->take<uint32_t>(n);
        uint32_t* pos = q->take<uint32_t>(n);
        uint32_t* scan_tmp = q->take<uint32_t>(scan_scratch_elems(n));
        uint32_t* total_dev = q->take<uint32_t>(16);
        // std::cos of the host, as the reference evaluates the two bounds before the launch (:68-69)
        const float max_cos = std::cos(min_angle), min_cos = std::cos(max_angle);
        angle_flag_kernel<<<div_up(n, VX_THREADS), VX_THREADS, 0, st>>>(reinterpret_cast<const float4*>(points),
                                                                       reinterpret_cast<const float4*>(normals), covs, n,
                                                                       min_cos, max_cos, flags);
        SPX_LAUNCH_CHECK();
        exclusive_scan_u32(st, flags, pos, n, scan_tmp, total_dev);
        compact_index_kernel<<<div_up(n, VX_THREADS), VX_THREADS, 0, st>>>(flags, pos, n, idx_out);
        SPX_LAUNCH_CHECK();
        uint32_t* htotal = static_cast<uint32_t*>(q->pinned_get(64));
        SPX_CUDA(cudaMemcpyAsync(htotal, total_dev, 4, cudaMemcpyDeviceToHost, st));
        q->sync();
        *m_host = *htotal;
    });
}

int spx_farthest_point_sampling(spx_queue_t q, const float* points, size_t n_in, size_t sampling_num, size_t first_index,
                                int32_t* idx_out, size_t* m_host) {
    return guard([&] {
        SPX_REQUIRE(q && m_host, "[PreprocessFilter::farthest_point_sampling] null argument");
        SPX_REQUIRE(n_in < (1ull << 31), "[PreprocessFilter::farthest_point_sampling] too many points");
        *m_host = 0;
        if (n_in == 0 || sampling_num == 0) return;
        SPX_REQUIRE(points && idx_out, "[PreprocessFilter::farthest_point_sampling] null pointer");
        SPX_REQUIRE(first_index < n_in, "[PreprocessFilter::farthest_point_sampling] first index out of range");
        DeviceGuard dg(q->device);
        cudaStream_t st = q->stream;
        const uint32_t n = (uint32_t)n_in;
        static int per_sm = 0;
        if (!per_sm) SPX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fps_kernel, FPS_THREADS, 0));
        const unsigned blocks = (unsigned)std::min<size_t>(div_up(n, FPS_THREADS), (size_t)std::max(per_sm, 1) * q->sm_count);
        q->arena_reset();
        q->arena_reserve((size_t)n * 12 + scan_scratch_elems(n) * 4 + (size_t)blocks * 16 + 8192);
        float* dist_sq = q->take<float>(n);
        uint32_t* flags = q->take<uint32_t>(n);
        uint32_t* pos = q->take<uint32_t>(n);
        uint32_t* scan_tmp = q->take<uint32_t>(scan_scratch_elems(n));
        unsigned long long* block_keys = q->take<unsigned long long>((size_t)blocks * 2);
        uint32_t* total_dev = q->take<uint32_t>(16);
        const float4* pts = reinterpret_cast<const float4*>(points);
        uint32_t first = (uint32_t)first_index, rounds = (uint32_t)std::min<size_t>(sampling_num, n_in);
        uint32_t nn = n;
        void* args[] = {(void*)&pts, (void*)&nn, (void*)&first, (void*)&rounds, (void*)&dist_sq, (void*)&flags,
                        (void*)&block_keys};
        SPX_CUDA(cudaLaunchCooperativeKernel((const void*)fps_kernel, dim3(blocks), dim3(FPS_THREADS), args, 0, st));
        count_launch();
        exclusive_scan_u32(st, flags, pos, n, scan_tmp, total_dev);
        compact_index_kernel<<<div_up(n, VX_THREADS), VX_THREADS, 0, st>>>(flags, pos, n, idx_out);
        SPX_LAUNCH_CHECK();
        uint32_t* htotal = static_cast<uint32_t*>(q->pinned_get(64));
        SPX_CUDA(cudaMemcpyAsync(htotal, total_dev, 4, cudaMemcpyDeviceToHost, st));
        q->sync();
        *m_host = *htotal;
    });
}

int spx_gather(spx_queue_t q, const void* src, size_t elem_bytes, const int32_t* idx, size_t m, void* dst) {
    return guard([&] {
        SPX_REQUIRE(q, "[spx_gather] null queue");
        SPX_REQUIRE(elem_bytes > 0 && elem_bytes % 4 == 0, "[spx_gather] elem_bytes must be a positive multiple of 4");
        if (m == 0) return;
        SPX_REQUIRE(src && idx && dst, "[spx_gather] null pointer");
        DeviceGuard dg(q->device);
        const bool vec = elem_bytes % 16 == 0 && (reinterpret_cast<uintptr_t>(src) % 16 == 0) &&
                         (reinterpret_cast<uintptr_t>(dst) % 16 == 0);
        if (vec) {
            const size_t total = m * (elem_bytes / 16);
            gather_vec4_kernel<<<div_up(total, VX_THREADS), VX_THREADS, 0, q->stream>>>(
                static_cast<const uint4*>(src), (int)(elem_bytes / 16), idx, total, static_cast<uint4*>(dst));
        } else {
            const size_t total = m * (elem_bytes / 4);
            gather_words_kernel<<<div_up(total, VX_THREADS), VX_THREADS, 0, q->stream>>>(
                static_cast<const uint32_t*>(src), (int)(elem_bytes / 4), idx, total, static_cast<uint32_t*>(dst));
        }
        SPX_LAUNCH_CHECK();
    });
}

}  // extern "C"
