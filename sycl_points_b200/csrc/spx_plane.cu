// RANSAC plane segmentation (semantics of PCL's SACSegmentation with SACMODEL_PLANE / SACMODEL_PERPENDICULAR_PLANE and
// SAC_RANSAC, pinned in DESIGN.md §3.5).
//
// The finite points are listed by a flag pass, the device scan and compact_index_kernel (F; n_f stays on the device).
// One thread per hypothesis draws its three positions in F from a counter-based SplitMix64 stream, builds the plane in
// fp64 and writes fp32 coefficients (NaN for an invalid hypothesis, which then counts nothing).  The scoring kernel is
// the hot path: hypotheses x points distance tests, as the brute-force k-NN streams its targets — point tiles arrive in
// shared memory by TMA bulk copies into two buffers, every lane holds four hypotheses in registers and tests two at a
// time with packed FFMA2, one broadcast LDS.128 per point feeds all four; the grid spans hypothesis tiles x point
// chunks and the per-block counts are added with integer atomics (order-free, so deterministic).  The best hypothesis
// is one 64-bit atomicMax on (count << 32) | ~h.  The refinement sums the inliers' moments in fp64 per block; the last
// block folds the partials in block order and solves the 3x3 eigenproblem (jacobi3).  A flag pass with the final
// plane, the scan and one compaction write the inliers and the remainder.  One host synchronisation per call.
#include <cmath>

#include "spx_math.cuh"
#include "spx_scan.cuh"
#include "spx_tma.cuh"

using namespace spx;

namespace {

constexpr int PL_THREADS = 256;
constexpr int PL_WARPS = PL_THREADS / 32;
constexpr int PL_HPT = 4;                   // hypotheses per lane, tested in packed pairs
constexpr int PL_HTILE = 32 * PL_HPT;       // hypotheses per block: every warp scores the same 128 on its own points
constexpr int PL_TILE = 1024;               // points per shared-memory buffer (16 KB, two buffers)
constexpr int PL_UNROLL = 4;                // points per step of a warp
constexpr int PL_MOMENT_BLOCKS = 296;       // fixed, so the fold order of the refinement sums depends on n only
constexpr int PL_MOMENTS = 10;              // count, sum q (3), sum q q^T (6), q = p - p0

// Device state of one call, copied to the host in one piece at its end.
struct __align__(16) PlaneState {
    float coef[4];            // the plane the inliers are selected with; NaN without a model
    unsigned long long best;  // max over valid hypotheses of (count << 32) | ~h; 0: none
    uint32_t n_inliers;
    uint32_t n_finite;
    uint32_t ticket;          // refinement blocks done
    uint32_t pad;
};

__device__ __forceinline__ bool finite3(const float4 p) { return isfinite(p.x) && isfinite(p.y) && isfinite(p.z); }

// fma(a_z, b_z, fma(a_y, b_y, a_x * b_x)) in fp64, nothing fused or split beyond what is written
__device__ __forceinline__ double dot3d(double ax, double ay, double az, double bx, double by, double bz) {
    return __fma_rn(az, bz, __fma_rn(ay, by, __dmul_rn(ax, bx)));
}

// the inlier test of DESIGN.md §3.5 (false for every non-finite point and for NaN coefficients)
__device__ __forceinline__ bool inlier(const float4 c, const float4 p, float t) {
    return fabsf(__fmaf_rn(c.z, p.z, __fmaf_rn(c.y, p.y, __fmaf_rn(c.x, p.x, c.w)))) < t;
}

__device__ __forceinline__ float4 nan4() {
    const float q = __int_as_float(0x7fc00000);  // (the quiet NaN of nanf(""), as the host side writes)
    return make_float4(q, q, q, q);
}

__global__ void __launch_bounds__(PL_THREADS) pl_finite_kernel(const float4* __restrict__ pts, uint32_t n,
                                                               uint32_t* __restrict__ flags) {
    const uint32_t i = blockIdx.x * PL_THREADS + threadIdx.x;
    if (i < n) flags[i] = finite3(__ldg(pts + i)) ? 1u : 0u;
}

// One thread per hypothesis: its sample, its fp64 plane, its validity and its fp32 coefficients; sample0[h] = the
// point index of p0 (the refinement's shift), -1 for an invalid hypothesis.
__global__ void __launch_bounds__(PL_THREADS) pl_hypothesis_kernel(const float4* __restrict__ pts,
                                                                   const int32_t* __restrict__ F,
                                                                   const PlaneState* __restrict__ st, uint32_t H,
                                                                   unsigned long long seed, int has_axis, double ax,
                                                                   double ay, double az, double cos_eps,
                                                                   float4* __restrict__ coef,
                                                                   int32_t* __restrict__ sample0) {
    const uint32_t h = blockIdx.x * PL_THREADS + threadIdx.x;
    if (h >= H) return;
    const unsigned long long nf = st->n_finite;
    float4 c = nan4();
    int32_t s0 = -1;
    uint32_t j[3];
#pragma unroll
    for (int s = 0; s < 3; ++s) j[s] = ransac_draw(seed, h, (unsigned long long)s, nf);
    if (nf >= 3 && j[0] != j[1] && j[0] != j[2] && j[1] != j[2]) {
        const int32_t i0 = F[j[0]];
        const float4 p0 = __ldg(pts + i0), p1 = __ldg(pts + F[j[1]]), p2 = __ldg(pts + F[j[2]]);
        const double x0 = p0.x, y0 = p0.y, z0 = p0.z;
        const double ux = __dsub_rn((double)p1.x, x0), uy = __dsub_rn((double)p1.y, y0), uz = __dsub_rn((double)p1.z, z0);
        const double vx = __dsub_rn((double)p2.x, x0), vy = __dsub_rn((double)p2.y, y0), vz = __dsub_rn((double)p2.z, z0);
        double nx = __fma_rn(uy, vz, -__dmul_rn(uz, vy));
        double ny = __fma_rn(uz, vx, -__dmul_rn(ux, vz));
        double nz = __fma_rn(ux, vy, -__dmul_rn(uy, vx));
        const double l2 = dot3d(nx, ny, nz, nx, ny, nz);
        const double uu = dot3d(ux, uy, uz, ux, uy, uz), vv = dot3d(vx, vy, vz, vx, vy, vz);
        if (l2 > __dmul_rn(__dmul_rn(1e-12, uu), vv)) {  // (false for NaN: collinear triples, duplicates)
            const double l = __dsqrt_rn(l2);
            nx = __ddiv_rn(nx, l);
            ny = __ddiv_rn(ny, l);
            nz = __ddiv_rn(nz, l);
            const double d = -dot3d(nx, ny, nz, x0, y0, z0);
            if (!(has_axis && fabs(dot3d(nx, ny, nz, ax, ay, az)) < cos_eps)) {
                c = make_float4(__double2float_rn(nx), __double2float_rn(ny), __double2float_rn(nz), __double2float_rn(d));
                s0 = i0;
            }
        }
    }
    coef[h] = c;
    sample0[h] = s0;
}

// counts[h] += the points of this block's chunk within t of plane h.  Block (x, y) scores hypotheses
// [y * PL_HTILE, (y + 1) * PL_HTILE) over points [x * chunk, (x + 1) * chunk): lane l holds hypotheses
// y * PL_HTILE + 4 l .. + 3, and warp w takes the w-th eighth of every tile.  Hypotheses past H are NaN (count nothing).
__global__ void __launch_bounds__(PL_THREADS) pl_score_kernel(const float4* __restrict__ pts, uint32_t n, uint32_t chunk,
                                                              const float4* __restrict__ coef, uint32_t H, float t,
                                                              uint32_t* __restrict__ counts) {
    __shared__ __align__(128) float4 tiles[2][PL_TILE];
    __shared__ __align__(8) unsigned long long bars[2];
    __shared__ uint32_t s_cnt[PL_HTILE];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t h0 = blockIdx.y * PL_HTILE + lane * PL_HPT;
    const uint32_t begin = blockIdx.x * chunk, end = min(n, begin + chunk);

    unsigned long long NX[PL_HPT / 2], NY[PL_HPT / 2], NZ[PL_HPT / 2], D[PL_HPT / 2];
#pragma unroll
    for (int u = 0; u < PL_HPT / 2; ++u) {
        const uint32_t ha = h0 + 2 * u, hb = ha + 1;
        const float4 a = ha < H ? __ldg(coef + ha) : nan4();
        const float4 b = hb < H ? __ldg(coef + hb) : nan4();
        NX[u] = pack2(a.x, b.x);
        NY[u] = pack2(a.y, b.y);
        NZ[u] = pack2(a.z, b.z);
        D[u] = pack2(a.w, b.w);
    }
    uint32_t cnt[PL_HPT];
#pragma unroll
    for (int u = 0; u < PL_HPT; ++u) cnt[u] = 0u;

    if (threadIdx.x < PL_HTILE) s_cnt[threadIdx.x] = 0u;
    if (threadIdx.x == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t bytes = min((uint32_t)PL_TILE, end - begin) * (uint32_t)sizeof(float4);
        mbar_expect_tx(&bars[0], bytes);
        bulk_g2s(&tiles[0][0], pts + begin, bytes, &bars[0]);
    }
    uint32_t it = 0;
    for (uint32_t base = begin; base < end; base += PL_TILE, ++it) {
        const uint32_t buf = it & 1u;
        const int lim = (int)min((uint32_t)PL_TILE, end - base);
        constexpr int STEP = PL_WARPS * PL_UNROLL;
        const int limb = (lim + STEP - 1) / STEP * STEP;
        // the other buffer was read in the previous iteration, which ended in a block barrier: refill it now
        if (threadIdx.x == 0 && base + PL_TILE < end) {
            const uint32_t bytes = min((uint32_t)PL_TILE, end - base - PL_TILE) * (uint32_t)sizeof(float4);
            mbar_expect_tx(&bars[buf ^ 1u], bytes);
            bulk_g2s(&tiles[buf ^ 1u][0], pts + base + PL_TILE, bytes, &bars[buf ^ 1u]);
        }
        mbar_wait(&bars[buf], (it >> 1) & 1u);
        if (lim < limb) {  // (last tile of a chunk only) NaN points beyond the end count for no plane
            if (threadIdx.x < (unsigned)(limb - lim)) tiles[buf][lim + threadIdx.x] = nan4();
            __syncthreads();
        }
        const int seg = limb / PL_WARPS;
        const float4* tp = tiles[buf] + warp * seg;
#pragma unroll 2
        for (int j = 0; j < seg; j += PL_UNROLL) {
#pragma unroll
            for (int v = 0; v < PL_UNROLL; ++v) {
                const float4 p = tp[j + v];  // (the same address in every lane: one broadcast LDS.128)
                const unsigned long long X = pack2(p.x, p.x), Y = pack2(p.y, p.y), Z = pack2(p.z, p.z);
#pragma unroll
                for (int u = 0; u < PL_HPT / 2; ++u) {
                    // fmaf(n_z, z, fmaf(n_y, y, fmaf(n_x, x, d))) for two planes at once
                    unsigned long long r;
                    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(NX[u]), "l"(X), "l"(D[u]));
                    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(NY[u]), "l"(Y), "l"(r));
                    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(NZ[u]), "l"(Z), "l"(r));
                    float lo, hi;
                    unpack2(r, lo, hi);
                    // |r| < t  <=>  the sign bit of fl(|r| - t): IEEE subtraction is exact in sign (a - b rounds to +0
                    // only when a == b), and |NaN| - t is a NaN with a clear sign bit.  FADD + LEA.HI: two instructions
                    // per test, where the compiler's FSETP + SEL + add took two and a half
                    cnt[2 * u] += __float_as_uint(__fsub_rn(fabsf(lo), t)) >> 31;
                    cnt[2 * u + 1] += __float_as_uint(__fsub_rn(fabsf(hi), t)) >> 31;
                }
            }
        }
        __syncthreads();  // every thread is done with this buffer before the next iteration refills it
    }
#pragma unroll
    for (int u = 0; u < PL_HPT; ++u)
        if (cnt[u]) atomicAdd(&s_cnt[lane * PL_HPT + u], cnt[u]);
    __syncthreads();
    if (threadIdx.x < PL_HTILE) {
        const uint32_t h = blockIdx.y * PL_HTILE + threadIdx.x;
        if (h < H && s_cnt[threadIdx.x]) atomicAdd(counts + h, s_cnt[threadIdx.x]);
    }
}

// counts[h] = 0xFFFFFFFF for the invalid hypotheses; st->best = max over the valid ones of (count << 32) | ~h, so the
// most inliers win and ties go to the lowest h
__global__ void __launch_bounds__(PL_THREADS) pl_select_kernel(const float4* __restrict__ coef, uint32_t H,
                                                               uint32_t* __restrict__ counts, PlaneState* st) {
    const uint32_t h = blockIdx.x * PL_THREADS + threadIdx.x;
    unsigned long long key = 0ull;
    if (h < H) {
        if (isnan(coef[h].x)) {
            counts[h] = 0xFFFFFFFFu;
        } else {
            key = ((unsigned long long)counts[h] << 32) | (unsigned long long)(~h);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) key = max(key, __shfl_xor_sync(0xffffffffu, key, o));
    if ((threadIdx.x & 31) == 0 && key) atomicMax(&st->best, key);
}

// v[k] of every thread summed in a fixed order (warp trees, then the warps in order): the total is in thread 0.
// s_red is reused by the next call only after a barrier.
__device__ __forceinline__ void block_sum(double (&v)[PL_MOMENTS], double (*s_red)[PL_MOMENTS]) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < PL_MOMENTS; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_down_sync(0xffffffffu, v[k], o);
        if (lane == 0) s_red[warp][k] = v[k];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < PL_MOMENTS; ++k) {
            double s = s_red[0][k];
            for (int w = 1; w < PL_WARPS; ++w) s += s_red[w][k];
            v[k] = s;
        }
    }
}

// st->coef = the plane the inliers are selected with: the best hypothesis's, refined from the moments S of its inliers
// when S is given and counts at least 3 points and the refined plane is finite; NaN without a model.  One thread.
__device__ void plane_finish(PlaneState* st, const float4* __restrict__ coef, const int32_t* __restrict__ sample0,
                             const float4* __restrict__ pts, const double* S) {
    float4 out = nan4();
    if (st->best) {
        const uint32_t h = ~(uint32_t)st->best;
        out = coef[h];
        if (S && S[0] >= 3.0) {
            const double N = S[0];
            const double m[3] = {S[1] / N, S[2] / N, S[3] / N};
            const double C[3][3] = {{S[4] / N - m[0] * m[0], S[5] / N - m[0] * m[1], S[6] / N - m[0] * m[2]},
                                    {S[5] / N - m[1] * m[0], S[7] / N - m[1] * m[1], S[8] / N - m[1] * m[2]},
                                    {S[6] / N - m[2] * m[0], S[8] / N - m[2] * m[1], S[9] / N - m[2] * m[2]}};
            double ev[3], V[3][3];
            jacobi3(C, ev, V);
            int k = 0;
            for (int e = 1; e < 3; ++e)
                if (ev[e] < ev[k]) k = e;
            double nx = V[0][k], ny = V[1][k], nz = V[2][k];
            if (nx * (double)out.x + ny * (double)out.y + nz * (double)out.z < 0.0) {
                nx = -nx;
                ny = -ny;
                nz = -nz;
            }
            const float4 p0 = pts[sample0[h]];
            const double cx = (double)p0.x + m[0], cy = (double)p0.y + m[1], cz = (double)p0.z + m[2];
            const float4 r = make_float4((float)nx, (float)ny, (float)nz, (float)-(nx * cx + ny * cy + nz * cz));
            if (isfinite(r.x) && isfinite(r.y) && isfinite(r.z) && isfinite(r.w)) out = r;
        }
    }
    *reinterpret_cast<float4*>(st->coef) = out;
}

// The refinement: the fp64 moments of the best hypothesis's inliers, shifted by its p0, per block into partials[]; the
// last block folds them in block order (each thread the blocks b, b + PL_THREADS, ...; then block_sum) and finishes.
__global__ void __launch_bounds__(PL_THREADS) pl_moments_kernel(const float4* __restrict__ pts, uint32_t n,
                                                                const float4* __restrict__ coef,
                                                                const int32_t* __restrict__ sample0, float t,
                                                                PlaneState* st, double* partials) {
    __shared__ double s_red[PL_WARPS][PL_MOMENTS];
    __shared__ bool s_last;
    double acc[PL_MOMENTS];
#pragma unroll
    for (int k = 0; k < PL_MOMENTS; ++k) acc[k] = 0.0;
    const unsigned long long best = st->best;
    if (best) {
        const uint32_t h = ~(uint32_t)best;
        const float4 c = coef[h], p0 = pts[sample0[h]];
        for (uint32_t i = blockIdx.x * PL_THREADS + threadIdx.x; i < n; i += gridDim.x * PL_THREADS) {
            const float4 p = __ldg(pts + i);
            if (!inlier(c, p, t)) continue;
            const double qx = (double)p.x - (double)p0.x, qy = (double)p.y - (double)p0.y, qz = (double)p.z - (double)p0.z;
            acc[0] += 1.0;
            acc[1] += qx;
            acc[2] += qy;
            acc[3] += qz;
            acc[4] += qx * qx;
            acc[5] += qx * qy;
            acc[6] += qx * qz;
            acc[7] += qy * qy;
            acc[8] += qy * qz;
            acc[9] += qz * qz;
        }
    }
    block_sum(acc, s_red);
    if (threadIdx.x == 0) {
        for (int k = 0; k < PL_MOMENTS; ++k) partials[blockIdx.x * PL_MOMENTS + k] = acc[k];
        __threadfence();
        s_last = atomicAdd(&st->ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
#pragma unroll
    for (int k = 0; k < PL_MOMENTS; ++k) acc[k] = 0.0;
    for (uint32_t b = threadIdx.x; b < gridDim.x; b += PL_THREADS)
#pragma unroll
        for (int k = 0; k < PL_MOMENTS; ++k) acc[k] += __ldcg(partials + b * PL_MOMENTS + k);
    __syncthreads();  // (s_red is reused)
    block_sum(acc, s_red);
    if (threadIdx.x == 0) plane_finish(st, coef, sample0, pts, acc);
}

// without refinement
__global__ void pl_finish_kernel(PlaneState* st, const float4* __restrict__ coef, const int32_t* __restrict__ sample0,
                                 const float4* __restrict__ pts) {
    plane_finish(st, coef, sample0, pts, nullptr);
}

__global__ void __launch_bounds__(PL_THREADS) pl_inlier_flag_kernel(const float4* __restrict__ pts, uint32_t n,
                                                                    const PlaneState* __restrict__ st, float t,
                                                                    uint32_t* __restrict__ flags) {
    const uint32_t i = blockIdx.x * PL_THREADS + threadIdx.x;
    if (i >= n) return;
    const float4 c = *reinterpret_cast<const float4*>(st->coef);
    flags[i] = inlier(c, __ldg(pts + i), t) ? 1u : 0u;
}

// inliers[pos[i]] = i for the flagged points, remainder[i - pos[i]] = i for the others (both ascending)
__global__ void __launch_bounds__(PL_THREADS) pl_split_kernel(const uint32_t* __restrict__ flags,
                                                              const uint32_t* __restrict__ pos, uint32_t n,
                                                              int32_t* __restrict__ inliers,
                                                              int32_t* __restrict__ remainder) {
    const uint32_t i = blockIdx.x * PL_THREADS + threadIdx.x;
    if (i >= n) return;
    if (flags[i]) {
        inliers[pos[i]] = (int32_t)i;
    } else if (remainder) {
        remainder[i - pos[i]] = (int32_t)i;
    }
}

}  // namespace

extern "C" {

int spx_plane_segment(spx_queue_t q, const float* points, size_t n_in, float threshold, uint32_t max_iterations,
                      uint64_t seed, const float* axis3_host, double eps_angle, int optimize, float* coeffs4_host,
                      int32_t* hypothesis_host, int32_t* inliers_out, size_t* n_inliers_host, int32_t* remainder_out,
                      uint32_t* counts_out) {
    return guard([&] {
        SPX_REQUIRE(q && coeffs4_host && hypothesis_host && n_inliers_host, "[PlaneSegmentation] null argument");
        SPX_REQUIRE(n_in < (1ull << 31), "[PlaneSegmentation] at most 2^31 - 1 points");
        SPX_REQUIRE(std::isfinite(threshold) && threshold > 0.0f,
                    "[PlaneSegmentation] `distance_threshold` must be finite and > 0");
        SPX_REQUIRE(max_iterations >= 1u && max_iterations <= (1u << 20),
                    "[PlaneSegmentation] `max_iterations` must be in [1, 2^20]");
        SPX_REQUIRE(eps_angle >= 0.0 && eps_angle <= M_PI / 2, "[PlaneSegmentation] `eps_angle` must be in [0, pi/2]");
        int has_axis = 0;
        double a[3] = {0.0, 0.0, 0.0}, cos_eps = 0.0;
        if (axis3_host) {
            const double x = axis3_host[0], y = axis3_host[1], z = axis3_host[2];
            SPX_REQUIRE(std::isfinite(x) && std::isfinite(y) && std::isfinite(z),
                        "[PlaneSegmentation] `axis` must be finite");
            const double l2 = std::fma(z, z, std::fma(y, y, x * x));
            SPX_REQUIRE(l2 > 0.0, "[PlaneSegmentation] `axis` must be nonzero");
            const double l = std::sqrt(l2);
            a[0] = x / l;
            a[1] = y / l;
            a[2] = z / l;
            cos_eps = std::cos(eps_angle);
            has_axis = 1;
        }
        const float qnan = std::nanf("");
        for (int k = 0; k < 4; ++k) coeffs4_host[k] = qnan;
        *hypothesis_host = -1;
        *n_inliers_host = 0;
        if (n_in == 0) return;
        SPX_REQUIRE(points && inliers_out, "[PlaneSegmentation] null pointer");
        SPX_REQUIRE((reinterpret_cast<uintptr_t>(points) & 15) == 0, "[PlaneSegmentation] points must be 16-byte aligned");
        DeviceGuard dg(q->device);
        cudaStream_t st = q->stream;
        const uint32_t n = (uint32_t)n_in, H = max_iterations;
        q->arena_reset();
        q->arena_reserve(4 * (3 * align_up(n, 64) + scan_scratch_elems(n) + 6 * align_up(H, 64)) +
                         8 * PL_MOMENT_BLOCKS * PL_MOMENTS + 4096);
        uint32_t* flags = q->take<uint32_t>(n);
        uint32_t* pos = q->take<uint32_t>(n);
        int32_t* F = q->take<int32_t>(n);
        uint32_t* scan_tmp = q->take<uint32_t>(scan_scratch_elems(n));
        float4* coef = q->take<float4>(H);
        int32_t* sample0 = q->take<int32_t>(H);
        uint32_t* counts = counts_out ? counts_out : q->take<uint32_t>(H);
        double* partials = q->take<double>(PL_MOMENT_BLOCKS * PL_MOMENTS);
        PlaneState* state = q->take<PlaneState>(1);
        const float4* pts = reinterpret_cast<const float4*>(points);
        const int blocks = div_up(n, PL_THREADS);

        SPX_CUDA(cudaMemsetAsync(state, 0, sizeof(PlaneState), st));
        SPX_CUDA(cudaMemsetAsync(counts, 0, (size_t)H * 4, st));
        // F: the finite points in ascending order, n_f on the device
        pl_finite_kernel<<<blocks, PL_THREADS, 0, st>>>(pts, n, flags);
        SPX_LAUNCH_CHECK();
        exclusive_scan_u32(st, flags, pos, n, scan_tmp, &state->n_finite);
        compact_index_kernel<<<div_up(n, COMPACT_THREADS), COMPACT_THREADS, 0, st>>>(flags, pos, n, F);
        SPX_LAUNCH_CHECK();
        pl_hypothesis_kernel<<<div_up(H, PL_THREADS), PL_THREADS, 0, st>>>(pts, F, state, H, seed, has_axis, a[0], a[1],
                                                                            a[2], cos_eps, coef, sample0);
        SPX_LAUNCH_CHECK();
        // the hot path: enough point chunks per hypothesis tile for ~8 blocks per SM, chunks whole tiles
        int sms = 0;
        SPX_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, q->device));
        const uint32_t htiles = div_up(H, PL_HTILE), ptiles = div_up(n, PL_TILE);
        const uint32_t want = std::max<uint32_t>(1u, (uint32_t)div_up((size_t)sms * 8, htiles));
        const uint32_t chunk = div_up(ptiles, std::min(ptiles, want)) * PL_TILE;
        pl_score_kernel<<<dim3(div_up(n, chunk), htiles), PL_THREADS, 0, st>>>(pts, n, chunk, coef, H, threshold, counts);
        SPX_LAUNCH_CHECK();
        pl_select_kernel<<<div_up(H, PL_THREADS), PL_THREADS, 0, st>>>(coef, H, counts, state);
        SPX_LAUNCH_CHECK();
        if (optimize) {
            pl_moments_kernel<<<std::min(blocks, PL_MOMENT_BLOCKS), PL_THREADS, 0, st>>>(pts, n, coef, sample0, threshold,
                                                                                         state, partials);
        } else {
            pl_finish_kernel<<<1, 1, 0, st>>>(state, coef, sample0, pts);
        }
        SPX_LAUNCH_CHECK();
        pl_inlier_flag_kernel<<<blocks, PL_THREADS, 0, st>>>(pts, n, state, threshold, flags);
        SPX_LAUNCH_CHECK();
        exclusive_scan_u32(st, flags, pos, n, scan_tmp, &state->n_inliers);
        pl_split_kernel<<<blocks, PL_THREADS, 0, st>>>(flags, pos, n, inliers_out, remainder_out);
        SPX_LAUNCH_CHECK();
        PlaneState* hs = static_cast<PlaneState*>(q->pinned_get(sizeof(PlaneState)));
        SPX_CUDA(cudaMemcpyAsync(hs, state, sizeof(PlaneState), cudaMemcpyDeviceToHost, st));
        q->sync();
        for (int k = 0; k < 4; ++k) coeffs4_host[k] = hs->coef[k];
        *hypothesis_host = hs->best ? (int32_t)(~(uint32_t)hs->best) : -1;
        *n_inliers_host = hs->n_inliers;
    });
}

}  // extern "C"
