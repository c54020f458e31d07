// FPFH descriptors (Rusu et al. 2009, with the point's own SPFH term) and their nearest-neighbour correspondences,
// pinned in DESIGN.md §3.6.
//
// Descriptors: one thread per point in two passes.  The SPFH pass runs the pair feature of the point with each listed
// neighbour (fp32, every operation written out) and counts its three bins in shared memory; the FPFH pass gathers the
// neighbours' SPFH rows (132 B each) and folds the 1/d^2-weighted sum in registers, in rank order and bins ascending.
// The angle bin of f1 = atan2(Y, X) is decided without a transcendental: (X, Y) against the ten boundary rays by
// cross products that are exact in sign (fp32 x fp32 products are exact in fp64), so the device and the reference bin
// every pair identically.
//
// Correspondences: all pairs, K-bf's problem in 33 dimensions.  Rows are first padded to 36 floats (144 B, so a row
// is one float4-aligned unit in shared memory); target tiles then arrive by TMA bulk copies into two buffers, every
// thread holds two source rows as packed f32x2 pairs and runs the squared distance chain for both with FADD2 / FFMA2
// (IEEE per element: bit-identical to the scalar chain), one broadcast LDS.128 per four dimensions.  The grid spans
// source blocks x target chunks; a thread keeps the lowest (D, t) of its chunk and merges it with one 64-bit atomicMin
// on (bits(D) << 32) | t, which is the same order since D >= 0.  A flag pass (with the reverse search for the mutual
// filter), the device scan and a compaction list the pairs.  One host synchronisation per call.
#include <cmath>

#include "spx_math.cuh"
#include "spx_scan.cuh"
#include "spx_tma.cuh"

using namespace spx;

namespace {

constexpr int FP_THREADS = 128;
constexpr int FP_BINS = 11;
constexpr int FP_DIM = 33;

constexpr int FC_THREADS = 128;
constexpr int FC_ROWS = 2 * FC_THREADS;  // source rows per block: two per thread
constexpr int FC_PAD = 36;               // padded row: 9 float4
constexpr int FC_TILE = 128;             // target rows per shared-memory buffer (18 KB, two buffers)
constexpr unsigned long long FC_NONE = ~0ull;

__device__ __forceinline__ bool finite3(const float4 p) { return isfinite(p.x) && isfinite(p.y) && isfinite(p.z); }

// dot(a, b) = fma(a_z, b_z, fma(a_y, b_y, a_x * b_x))
__device__ __forceinline__ float dotf(float ax, float ay, float az, float bx, float by, float bz) {
    return __fmaf_rn(az, bz, __fmaf_rn(ay, by, __fmul_rn(ax, bx)));
}
// a x b = (fma(a_y, b_z, -(a_z b_y)), fma(a_z, b_x, -(a_x b_z)), fma(a_x, b_y, -(a_y b_x)))
__device__ __forceinline__ void crossf(float ax, float ay, float az, float bx, float by, float bz, float& cx, float& cy,
                                       float& cz) {
    cx = __fmaf_rn(ay, bz, -__fmul_rn(az, by));
    cy = __fmaf_rn(az, bx, -__fmul_rn(ax, bz));
    cz = __fmaf_rn(ax, by, -__fmul_rn(ay, bx));
}

// floor((f + 1) * 5.5) clamped to [0, 10]; NaN -> 0
__device__ __forceinline__ int linear_bin(float f) {
    const float b = floorf(__fmul_rn(__fadd_rn(f, 1.0f), 5.5f));
    return !(b >= 0.0f) ? 0 : (b > 10.0f ? 10 : (int)b);
}

// floor(11 (atan2(Y, X) + pi) / (2 pi)) clamped to [0, 10] = the number of boundary rays -pi + 2 pi k / 11, k = 1..10,
// at or below atan2(Y, X) in (-pi, pi].  Ray k >= 6 is (C[k-6], S[k-6]); ray k <= 5 its mirror (C[5-k], -S[5-k]).  The
// sign of c Y - s X is exact: both products are exact in fp64 and IEEE subtraction is exact in sign.  (0, 0) -> 5;
// Y = +-0 with X < 0 is theta = pi -> 10.
__device__ __forceinline__ int angle_bin(float X, float Y) {
    const float C[5] = {0x1.eb42aap-1f, 0x1.4f49e8p-1f, 0x1.2375f6p-3f, -0x1.a9628ep-2f, -0x1.aeb8c8p-1f};
    const float S[5] = {0x1.207e8p-2f, 0x1.82f19cp-1f, 0x1.fac9ep-1f, 0x1.d1bb48p-1f, 0x1.14ceep-1f};
    if (Y == 0.0f) return X < 0.0f ? 10 : 5;
    const double x = X, y = Y;
    int b = 5;
#pragma unroll
    for (int m = 0; m < 5; ++m) {
        if (Y > 0.0f) {
            b += __dsub_rn(__dmul_rn((double)C[m], y), __dmul_rn((double)S[m], x)) >= 0.0 ? 1 : 0;
        } else {
            b -= __dadd_rn(__dmul_rn((double)C[m], y), __dmul_rn((double)S[m], x)) < 0.0 ? 1 : 0;
        }
    }
    return b;
}

// The three bins of the pair (i, j), false when the pair is skipped (v = e x u is zero).  dp = p_j - p_i.
__device__ __forceinline__ bool pair_bins(const float4 pi, const float4 ni, const float4 pj, const float4 nj, int& b1,
                                          int& b2, int& b3) {
    const float dx = __fsub_rn(pj.x, pi.x), dy = __fsub_rn(pj.y, pi.y), dz = __fsub_rn(pj.z, pi.z);
    const float s2 = dotf(dx, dy, dz, dx, dy, dz);
    const float ai = dotf(ni.x, ni.y, ni.z, dx, dy, dz), aj = dotf(nj.x, nj.y, nj.z, dx, dy, dz);
    const bool sw = fabsf(ai) < fabsf(aj);
    const float4 u = sw ? nj : ni, o = sw ? ni : nj;
    const float ex = sw ? -dx : dx, ey = sw ? -dy : dy, ez = sw ? -dz : dz;
    const float f3 = __fdiv_rn(sw ? -aj : ai, __fsqrt_rn(s2));
    float vx, vy, vz;
    crossf(ex, ey, ez, u.x, u.y, u.z, vx, vy, vz);
    const float vv = dotf(vx, vy, vz, vx, vy, vz);
    if (vv == 0.0f) return false;
    const float l = __fsqrt_rn(vv);
    vx = __fdiv_rn(vx, l);
    vy = __fdiv_rn(vy, l);
    vz = __fdiv_rn(vz, l);
    float wx, wy, wz;
    crossf(u.x, u.y, u.z, vx, vy, vz, wx, wy, wz);
    const float f2 = dotf(vx, vy, vz, o.x, o.y, o.z);
    const float X = dotf(u.x, u.y, u.z, o.x, o.y, o.z), Y = dotf(wx, wy, wz, o.x, o.y, o.z);
    b1 = angle_bin(X, Y);
    b2 = linear_bin(f2);
    b3 = linear_bin(f3);
    return true;
}

__device__ __forceinline__ bool valid_point(const float4* __restrict__ pts, const float4* __restrict__ nrm, int32_t j) {
    return finite3(__ldg(pts + j)) && finite3(__ldg(nrm + j));
}

// spfh[i] = the SPFH of point i (all zeros when it counts no pair or is invalid); valid[i] = 1 iff point and normal are
// finite.  Bin counts live in shared memory, bin-major so that the 128 threads of a block hit distinct banks.
__global__ void __launch_bounds__(FP_THREADS) fp_spfh_kernel(const float4* __restrict__ pts,
                                                             const float4* __restrict__ nrm, uint32_t n,
                                                             const int32_t* __restrict__ idx,
                                                             const float* __restrict__ dist, int k,
                                                             float* __restrict__ spfh, uint8_t* __restrict__ valid) {
    __shared__ uint32_t cnt[FP_DIM][FP_THREADS];
    const uint32_t i = blockIdx.x * FP_THREADS + threadIdx.x;
    if (i >= n) return;
#pragma unroll
    for (int b = 0; b < FP_DIM; ++b) cnt[b][threadIdx.x] = 0u;
    const float4 pi = __ldg(pts + i), ni = __ldg(nrm + i);
    const bool ok = finite3(pi) && finite3(ni);
    valid[i] = ok ? 1 : 0;
    uint32_t m = 0;
    if (ok) {
        const int32_t* row = idx + (size_t)i * k;
        const float* drow = dist + (size_t)i * k;
        for (int r = 0; r < k; ++r) {
            const int32_t j = __ldg(row + r);
            if (j < 0 || j == (int32_t)i || !(__ldg(drow + r) > 0.0f) || !valid_point(pts, nrm, j)) continue;
            int b1, b2, b3;
            if (!pair_bins(pi, ni, __ldg(pts + j), __ldg(nrm + j), b1, b2, b3)) continue;
            ++cnt[b1][threadIdx.x];
            ++cnt[FP_BINS + b2][threadIdx.x];
            ++cnt[2 * FP_BINS + b3][threadIdx.x];
            ++m;
        }
    }
    const float scale = m ? __fdiv_rn(100.0f, (float)m) : 0.0f;
    float* out = spfh + (size_t)i * FP_DIM;
#pragma unroll
    for (int b = 0; b < FP_DIM; ++b) out[b] = __fmul_rn((float)cnt[b][threadIdx.x], scale);
}

// F_i[b] = acc[b] * (100 / sum_g) + SPFH_i[b] with acc[b] = sum over N(i) in rank order of SPFH_j[b] / d^2_ij and
// sum_g = the same sum over b's group (a group with sum_g = 0 contributes 0); an invalid point gets a NaN row.
__global__ void __launch_bounds__(FP_THREADS) fp_fpfh_kernel(const float* __restrict__ spfh,
                                                             const uint8_t* __restrict__ valid, uint32_t n,
                                                             const int32_t* __restrict__ idx,
                                                             const float* __restrict__ dist, int k,
                                                             float* __restrict__ features) {
    const uint32_t i = blockIdx.x * FP_THREADS + threadIdx.x;
    if (i >= n) return;
    float* out = features + (size_t)i * FP_DIM;
    if (!valid[i]) {
        const float q = __int_as_float(0x7fc00000);
#pragma unroll
        for (int b = 0; b < FP_DIM; ++b) out[b] = q;
        return;
    }
    float acc[FP_DIM], sum[3] = {0.0f, 0.0f, 0.0f};
#pragma unroll
    for (int b = 0; b < FP_DIM; ++b) acc[b] = 0.0f;
    const int32_t* row = idx + (size_t)i * k;
    const float* drow = dist + (size_t)i * k;
    for (int r = 0; r < k; ++r) {
        const int32_t j = __ldg(row + r);
        const float d2 = __ldg(drow + r);
        if (j < 0 || j == (int32_t)i || !(d2 > 0.0f) || !valid[j]) continue;
        const float w = __fdiv_rn(1.0f, d2);
        const float* sj = spfh + (size_t)j * FP_DIM;
#pragma unroll
        for (int b = 0; b < FP_DIM; ++b) {
            const float v = __fmul_rn(__ldg(sj + b), w);
            acc[b] = __fadd_rn(acc[b], v);
            sum[b / FP_BINS] = __fadd_rn(sum[b / FP_BINS], v);
        }
    }
    float f[3];
#pragma unroll
    for (int g = 0; g < 3; ++g) f[g] = sum[g] != 0.0f ? __fdiv_rn(100.0f, sum[g]) : 0.0f;
    const float* si = spfh + (size_t)i * FP_DIM;
#pragma unroll
    for (int b = 0; b < FP_DIM; ++b) {
        const float c = sum[b / FP_BINS] != 0.0f ? __fmul_rn(acc[b], f[b / FP_BINS]) : 0.0f;
        out[b] = __fadd_rn(c, si[b]);
    }
}

// out[r] = row r padded to 36 floats with zeros (the pad is never read into a distance)
__global__ void __launch_bounds__(256) fc_pad_kernel(const float* __restrict__ rows, uint32_t n, float* __restrict__ out) {
    const size_t e = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (e >= (size_t)n * FC_PAD) return;
    const size_t r = e / FC_PAD;
    const int c = (int)(e - r * FC_PAD);
    out[e] = c < FP_DIM ? __ldg(rows + r * FP_DIM + c) : 0.0f;
}

// best[i] = min over the targets of chunk blockIdx.y with D(i, t) not NaN of (bits(D) << 32) | t, merged by atomicMin
// (FC_NONE: none).  D = fma(d_32, d_32, ... fma(d_1, d_1, d_0 d_0)), d_b = s_b - t_b.  Thread x holds source rows
// blockIdx.x * FC_ROWS + x and + FC_THREADS as packed pairs; every thread walks every target of the tile.
__global__ void __launch_bounds__(FC_THREADS) fc_nn_kernel(const float* __restrict__ src, uint32_t ns,
                                                           const float* __restrict__ tgt, uint32_t nt, uint32_t chunk,
                                                           unsigned long long* __restrict__ best) {
    __shared__ __align__(128) float tiles[2][FC_TILE * FC_PAD];
    __shared__ __align__(8) unsigned long long bars[2];
    const uint32_t ia = blockIdx.x * FC_ROWS + threadIdx.x, ib = ia + FC_THREADS;
    const uint32_t begin = blockIdx.y * chunk, end = min(nt, begin + chunk);
    unsigned long long S[FP_DIM];
    {
        const float* ra = src + (size_t)min(ia, ns - 1) * FC_PAD;
        const float* rb = src + (size_t)min(ib, ns - 1) * FC_PAD;
#pragma unroll
        for (int b = 0; b < FP_DIM; ++b) S[b] = pack2(__ldg(ra + b), __ldg(rb + b));
    }
    uint32_t best_a = 0xFFFFFFFFu, best_b = 0xFFFFFFFFu, ta = 0xFFFFFFFFu, tb = 0xFFFFFFFFu;
    if (threadIdx.x == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t bytes = min((uint32_t)FC_TILE, end - begin) * (uint32_t)(FC_PAD * sizeof(float));
        mbar_expect_tx(&bars[0], bytes);
        bulk_g2s(&tiles[0][0], tgt + (size_t)begin * FC_PAD, bytes, &bars[0]);
    }
    uint32_t it = 0;
    for (uint32_t base = begin; base < end; base += FC_TILE, ++it) {
        const uint32_t buf = it & 1u;
        const int lim = (int)min((uint32_t)FC_TILE, end - base);
        // the other buffer was read in the previous iteration, which ended in a block barrier: refill it now
        if (threadIdx.x == 0 && base + FC_TILE < end) {
            const uint32_t bytes = min((uint32_t)FC_TILE, end - base - FC_TILE) * (uint32_t)(FC_PAD * sizeof(float));
            mbar_expect_tx(&bars[buf ^ 1u], bytes);
            bulk_g2s(&tiles[buf ^ 1u][0], tgt + (size_t)(base + FC_TILE) * FC_PAD, bytes, &bars[buf ^ 1u]);
        }
        mbar_wait(&bars[buf], (it >> 1) & 1u);
        const float4* tp = reinterpret_cast<const float4*>(tiles[buf]);
#pragma unroll 1
        for (int r = 0; r < lim; ++r) {
            const float4* row = tp + r * (FC_PAD / 4);  // (the same address in every lane: broadcast LDS.128)
            unsigned long long acc = 0ull;
#pragma unroll
            for (int q = 0; q < FC_PAD / 4; ++q) {
                const float4 t4 = row[q];
                const float tv[4] = {t4.x, t4.y, t4.z, t4.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int b = 4 * q + e;
                    if (b >= FP_DIM) break;
                    unsigned long long d;
                    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(S[b]), "l"(pack2(tv[e], tv[e])));
                    if (b == 0) {
                        asm("mul.rn.f32x2 %0, %1, %1;" : "=l"(acc) : "l"(d));
                    } else {
                        asm("fma.rn.f32x2 %0, %1, %1, %2;" : "=l"(acc) : "l"(d), "l"(acc));
                    }
                }
            }
            float da, db;
            unpack2(acc, da, db);
            // D >= 0 or NaN: as unsigned bits the order of D, with every NaN (0x7fffffff on the device) above +inf
            const uint32_t ua = __float_as_uint(da), ub = __float_as_uint(db);
            if (ua < best_a) { best_a = ua; ta = base + r; }
            if (ub < best_b) { best_b = ub; tb = base + r; }
        }
        __syncthreads();  // every thread is done with this buffer before the next iteration refills it
    }
    if (ia < ns && best_a <= 0x7f800000u) atomicMin(best + ia, ((unsigned long long)best_a << 32) | ta);
    if (ib < ns && best_b <= 0x7f800000u) atomicMin(best + ib, ((unsigned long long)best_b << 32) | tb);
}

// flags[i] = 1 iff source row i has a nearest target (and, with mutual, that target's nearest source is i)
__global__ void __launch_bounds__(256) fc_flag_kernel(const unsigned long long* __restrict__ st, uint32_t ns,
                                                      const unsigned long long* __restrict__ ts, int mutual,
                                                      uint32_t* __restrict__ flags) {
    const uint32_t i = blockIdx.x * 256 + threadIdx.x;
    if (i >= ns) return;
    const unsigned long long b = st[i];
    bool keep = b != FC_NONE;
    if (keep && mutual) {
        const unsigned long long r = ts[(uint32_t)b];
        keep = r != FC_NONE && (uint32_t)r == i;
    }
    flags[i] = keep ? 1u : 0u;
}

__global__ void __launch_bounds__(256) fc_pairs_kernel(const uint32_t* __restrict__ flags,
                                                       const uint32_t* __restrict__ pos,
                                                       const unsigned long long* __restrict__ st, uint32_t ns,
                                                       int32_t* __restrict__ src_out, int32_t* __restrict__ tgt_out) {
    const uint32_t i = blockIdx.x * 256 + threadIdx.x;
    if (i >= ns || !flags[i]) return;
    src_out[pos[i]] = (int32_t)i;
    tgt_out[pos[i]] = (int32_t)(uint32_t)st[i];
}

// best[0..ns) <- the nearest target of every source row (padded rows)
void nearest_rows(cudaStream_t st, int sms, const float* src, uint32_t ns, const float* tgt, uint32_t nt,
                  unsigned long long* best) {
    SPX_CUDA(cudaMemsetAsync(best, 0xFF, (size_t)ns * sizeof(unsigned long long), st));
    // enough target chunks for ~4 blocks per SM, chunks whole tiles
    const uint32_t sblocks = div_up(ns, FC_ROWS), ttiles = div_up(nt, FC_TILE);
    const uint32_t want = std::max<uint32_t>(1u, (uint32_t)div_up((size_t)sms * 4, sblocks));
    const uint32_t chunk = div_up(ttiles, std::min(ttiles, want)) * FC_TILE;
    fc_nn_kernel<<<dim3(sblocks, div_up(nt, chunk)), FC_THREADS, 0, st>>>(src, ns, tgt, nt, chunk, best);
    SPX_LAUNCH_CHECK();
}

}  // namespace

extern "C" {

int spx_fpfh(spx_queue_t q, const float* points, const float* normals, size_t n_in, const int32_t* nn_idx,
             const float* nn_dist, int k, float* features) {
    return guard([&] {
        SPX_REQUIRE(q, "[FPFHEstimation] null queue");
        SPX_REQUIRE(n_in < (1ull << 31), "[FPFHEstimation] at most 2^31 - 1 points");
        SPX_REQUIRE(k >= 1 && k <= 128, "[FPFHEstimation] `k` must be in [1, 128]");
        if (n_in == 0) return;
        SPX_REQUIRE(points && normals && nn_idx && nn_dist && features, "[FPFHEstimation] null pointer");
        SPX_REQUIRE(((reinterpret_cast<uintptr_t>(points) | reinterpret_cast<uintptr_t>(normals) |
                      reinterpret_cast<uintptr_t>(features)) & 15) == 0,
                    "[FPFHEstimation] points, normals and features must be 16-byte aligned");
        DeviceGuard dg(q->device);
        cudaStream_t st = q->stream;
        const uint32_t n = (uint32_t)n_in;
        q->arena_reset();
        q->arena_reserve(4 * (size_t)n * FP_DIM + n + 1024);
        float* spfh = q->take<float>((size_t)n * FP_DIM);
        uint8_t* valid = q->take<uint8_t>(n);
        const float4* pts = reinterpret_cast<const float4*>(points);
        const float4* nrm = reinterpret_cast<const float4*>(normals);
        fp_spfh_kernel<<<div_up(n, FP_THREADS), FP_THREADS, 0, st>>>(pts, nrm, n, nn_idx, nn_dist, k, spfh, valid);
        SPX_LAUNCH_CHECK();
        fp_fpfh_kernel<<<div_up(n, FP_THREADS), FP_THREADS, 0, st>>>(spfh, valid, n, nn_idx, nn_dist, k, features);
        SPX_LAUNCH_CHECK();
    });
}

int spx_feature_correspondences(spx_queue_t q, const float* source_features, size_t ns_in, const float* target_features,
                                size_t nt_in, int mutual, int32_t* src_idx_out, int32_t* tgt_idx_out, size_t* m_host) {
    return guard([&] {
        SPX_REQUIRE(q && m_host, "[match_features] null argument");
        SPX_REQUIRE(ns_in < (1ull << 31) && nt_in < (1ull << 31), "[match_features] at most 2^31 - 1 rows");
        *m_host = 0;
        if (ns_in == 0 || nt_in == 0) return;
        SPX_REQUIRE(source_features && target_features && src_idx_out && tgt_idx_out, "[match_features] null pointer");
        DeviceGuard dg(q->device);
        cudaStream_t st = q->stream;
        const uint32_t ns = (uint32_t)ns_in, nt = (uint32_t)nt_in;
        q->arena_reset();
        q->arena_reserve(4 * (size_t)FC_PAD * (ns + nt) + 8 * ((size_t)ns + nt) +
                         4 * (2 * align_up(ns, 64) + scan_scratch_elems(ns)) + 8192);
        float* S = q->take<float>((size_t)ns * FC_PAD);
        float* T = q->take<float>((size_t)nt * FC_PAD);
        unsigned long long* st_best = q->take<unsigned long long>(ns);
        unsigned long long* ts_best = mutual ? q->take<unsigned long long>(nt) : nullptr;
        uint32_t* flags = q->take<uint32_t>(ns);
        uint32_t* pos = q->take<uint32_t>(ns);
        uint32_t* scan_tmp = q->take<uint32_t>(scan_scratch_elems(ns));
        uint32_t* count = q->take<uint32_t>(1);
        fc_pad_kernel<<<div_up((size_t)ns * FC_PAD, 256), 256, 0, st>>>(source_features, ns, S);
        SPX_LAUNCH_CHECK();
        fc_pad_kernel<<<div_up((size_t)nt * FC_PAD, 256), 256, 0, st>>>(target_features, nt, T);
        SPX_LAUNCH_CHECK();
        int sms = 0;
        SPX_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, q->device));
        nearest_rows(st, sms, S, ns, T, nt, st_best);
        if (mutual) nearest_rows(st, sms, T, nt, S, ns, ts_best);
        fc_flag_kernel<<<div_up(ns, 256), 256, 0, st>>>(st_best, ns, ts_best, mutual, flags);
        SPX_LAUNCH_CHECK();
        exclusive_scan_u32(st, flags, pos, ns, scan_tmp, count);
        fc_pairs_kernel<<<div_up(ns, 256), 256, 0, st>>>(flags, pos, st_best, ns, src_idx_out, tgt_idx_out);
        SPX_LAUNCH_CHECK();
        uint32_t* h = static_cast<uint32_t*>(q->pinned_get(sizeof(uint32_t)));
        SPX_CUDA(cudaMemcpyAsync(h, count, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        q->sync();
        *m_host = *h;
    });
}

}  // extern "C"
