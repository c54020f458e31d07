// RANSAC registration over feature correspondences (the usual feature-matching RANSAC with an edge-length check, as in
// Open3D's registration_ransac_based_on_feature_matching), pinned in DESIGN.md §3.6.
//
// The correspondences' points are gathered once into a packed list of (p, q) float4 pairs; a pair with a non-finite
// coordinate or an index out of range is stored as p = 0, q = +inf, which no pose counts.  One thread per hypothesis
// draws three positions from the plane RANSAC's counter-based stream (spx_math.cuh), checks distinctness, edge lengths
// and both triangles in fp64, and builds the closed-form triad pose in fp64, rounded to fp32 (NaN for an invalid one).
// The scoring kernel is the hot path, laid out like pl_score_kernel: pair tiles arrive in shared memory by TMA bulk
// copies into two buffers, every lane holds four hypotheses' 12 coefficients as packed pairs and tests two at a time
// with FFMA2, and the strict test d^2 < eps^2 is the sign bit of fl(d^2 - eps^2), added with one LEA.HI.  Counts are
// added with integer atomics (order-free), the best hypothesis is one 64-bit atomicMax on (count << 32) | ~h.  The
// refinement sums the inliers' fp64 moments per block over a fixed grid; the last block folds them in block order and
// solves the least-squares rotation (Kabsch through the eigenvectors of H^T H: rank 2 is enough).  A flag pass, the
// scan and one compaction list the final inliers.  One host synchronisation per call.
#include <cmath>

#include "spx_math.cuh"
#include "spx_scan.cuh"
#include "spx_tma.cuh"

using namespace spx;

namespace {

constexpr int RS_THREADS = 256;
constexpr int RS_WARPS = RS_THREADS / 32;
constexpr int RS_HPT = 4;                // hypotheses per lane, tested in packed pairs
constexpr int RS_HTILE = 32 * RS_HPT;    // hypotheses per block: every warp scores the same 128 on its own pairs
constexpr int RS_TILE = 512;             // correspondences per shared-memory buffer (16 KB, two buffers)
constexpr int RS_UNROLL = 2;             // correspondences per step of a warp
constexpr int RS_MOMENT_BLOCKS = 148;    // fixed, so the fold order of the refinement sums depends on M only
constexpr int RS_MOMENTS = 16;           // count, sum a (3), sum b (3), sum a b^T (9); a = p - p0, b = q - q0

struct __align__(16) RansacState {
    float pose[12];           // rows (R_r0, R_r1, R_r2, t_r) the inliers are selected with; NaN without a model
    unsigned long long best;  // max over valid hypotheses of (count << 32) | ~h; 0: none
    uint32_t n_inliers;
    uint32_t ticket;          // refinement blocks done
};

__device__ __forceinline__ float qnan() { return __int_as_float(0x7fc00000); }

// fma(a_z, b_z, fma(a_y, b_y, a_x * b_x)) in fp64
__device__ __forceinline__ double dot3d(double ax, double ay, double az, double bx, double by, double bz) {
    return __fma_rn(az, bz, __fma_rn(ay, by, __dmul_rn(ax, bx)));
}
__device__ __forceinline__ void cross3d(const double a[3], const double b[3], double c[3]) {
    c[0] = __fma_rn(a[1], b[2], -__dmul_rn(a[2], b[1]));
    c[1] = __fma_rn(a[2], b[0], -__dmul_rn(a[0], b[2]));
    c[2] = __fma_rn(a[0], b[1], -__dmul_rn(a[1], b[0]));
}

// the inlier test: y_r = fma(R_r2, p_z, fma(R_r1, p_y, fma(R_r0, p_x, t_r))), d = y - q, dot(d, d) < eps2
__device__ __forceinline__ bool inlier(const float* P, const float4 p, const float4 q, float eps2) {
    float d[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const float y = __fmaf_rn(P[4 * r + 2], p.z, __fmaf_rn(P[4 * r + 1], p.y, __fmaf_rn(P[4 * r], p.x, P[4 * r + 3])));
        d[r] = __fsub_rn(y, r == 0 ? q.x : (r == 1 ? q.y : q.z));
    }
    return (__float_as_uint(__fsub_rn(__fmaf_rn(d[2], d[2], __fmaf_rn(d[1], d[1], __fmul_rn(d[0], d[0]))), eps2)) >> 31) != 0u;
}

__global__ void __launch_bounds__(RS_THREADS) rs_gather_kernel(const float4* __restrict__ src, size_t ns,
                                                               const float4* __restrict__ tgt, size_t nt,
                                                               const int32_t* __restrict__ si,
                                                               const int32_t* __restrict__ ti, uint32_t M,
                                                               float4* __restrict__ pairs) {
    const uint32_t k = blockIdx.x * RS_THREADS + threadIdx.x;
    if (k >= M) return;
    const int32_t a = si[k], b = ti[k];
    float4 p = make_float4(0.f, 0.f, 0.f, 0.f), q = make_float4(INFINITY, INFINITY, INFINITY, 0.f);
    if (a >= 0 && (size_t)a < ns && b >= 0 && (size_t)b < nt) {
        const float4 pa = __ldg(src + a), qb = __ldg(tgt + b);
        if (isfinite(pa.x) && isfinite(pa.y) && isfinite(pa.z) && isfinite(qb.x) && isfinite(qb.y) && isfinite(qb.z)) {
            p = make_float4(pa.x, pa.y, pa.z, 1.f);
            q = make_float4(qb.x, qb.y, qb.z, 1.f);
        }
    }
    pairs[2 * k] = p;
    pairs[2 * k + 1] = q;
}

// the triad frame F = [e1 e2 e3] of the triangle (x0, x1, x2): e1 = u / |u|, e3 = n / |n|, e2 = e3 x e1 with u = x1 - x0,
// v = x2 - x0, n = u x v; c = ((x0 + x1) + x2) / 3.  False when degenerate: l^2 <= 1e-12 |u|^2 |v|^2 (or NaN).
__device__ __forceinline__ bool triad_frame(const float4 x0, const float4 x1, const float4 x2, double F[3][3],
                                            double c[3]) {
    const double a0[3] = {x0.x, x0.y, x0.z}, a1[3] = {x1.x, x1.y, x1.z}, a2[3] = {x2.x, x2.y, x2.z};
    double u[3], v[3], n[3], e2[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        u[r] = __dsub_rn(a1[r], a0[r]);
        v[r] = __dsub_rn(a2[r], a0[r]);
        c[r] = __ddiv_rn(__dadd_rn(__dadd_rn(a0[r], a1[r]), a2[r]), 3.0);
    }
    cross3d(u, v, n);
    const double l2 = dot3d(n[0], n[1], n[2], n[0], n[1], n[2]);
    const double uu = dot3d(u[0], u[1], u[2], u[0], u[1], u[2]), vv = dot3d(v[0], v[1], v[2], v[0], v[1], v[2]);
    if (!(l2 > __dmul_rn(__dmul_rn(1e-12, uu), vv))) return false;
    const double lu = __dsqrt_rn(uu), ln = __dsqrt_rn(l2);
    double e1[3], e3[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        e1[r] = __ddiv_rn(u[r], lu);
        e3[r] = __ddiv_rn(n[r], ln);
    }
    cross3d(e3, e1, e2);
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        F[r][0] = e1[r];
        F[r][1] = e2[r];
        F[r][2] = e3[r];
    }
    return true;
}

// squared length of x_a - x_b in fp64
__device__ __forceinline__ double edge2(const float4 a, const float4 b) {
    const double dx = __dsub_rn((double)a.x, (double)b.x), dy = __dsub_rn((double)a.y, (double)b.y),
                 dz = __dsub_rn((double)a.z, (double)b.z);
    return dot3d(dx, dy, dz, dx, dy, dz);
}

// One thread per hypothesis: its three draws, its validity and its fp32 pose (rows (R_r0, R_r1, R_r2, t_r); NaN when
// invalid); sample0[h] = the position of its first correspondence (the refinement's shift), -1 when invalid.
__global__ void __launch_bounds__(RS_THREADS) rs_hypothesis_kernel(const float4* __restrict__ pairs, uint32_t M,
                                                                   uint32_t H, unsigned long long seed, double tau2,
                                                                   float4* __restrict__ pose,
                                                                   int32_t* __restrict__ sample0) {
    const uint32_t h = blockIdx.x * RS_THREADS + threadIdx.x;
    if (h >= H) return;
    float out[12];
#pragma unroll
    for (int e = 0; e < 12; ++e) out[e] = qnan();
    int32_t s0 = -1;
    uint32_t c[3];
#pragma unroll
    for (int s = 0; s < 3; ++s) c[s] = ransac_draw(seed, h, (unsigned long long)s, M);
    if (M >= 3 && c[0] != c[1] && c[0] != c[2] && c[1] != c[2]) {
        float4 p[3], q[3];
#pragma unroll
        for (int s = 0; s < 3; ++s) {
            p[s] = __ldg(pairs + 2 * c[s]);
            q[s] = __ldg(pairs + 2 * c[s] + 1);
        }
        bool ok = true;
        const int A[3] = {0, 0, 1}, B[3] = {1, 2, 2};
#pragma unroll
        for (int e = 0; e < 3; ++e) {
            const double ds = edge2(p[A[e]], p[B[e]]), dt = edge2(q[A[e]], q[B[e]]);
            ok = ok && ds >= __dmul_rn(tau2, dt) && dt >= __dmul_rn(tau2, ds);
        }
        double Fp[3][3], Fq[3][3], cp[3], cq[3];
        if (ok && triad_frame(p[0], p[1], p[2], Fp, cp) && triad_frame(q[0], q[1], q[2], Fq, cq)) {
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                double R[3];
#pragma unroll
                for (int col = 0; col < 3; ++col)
                    R[col] = __fma_rn(Fq[r][2], Fp[col][2], __fma_rn(Fq[r][1], Fp[col][1], __dmul_rn(Fq[r][0], Fp[col][0])));
                const double t = __dsub_rn(cq[r], __fma_rn(R[2], cp[2], __fma_rn(R[1], cp[1], __dmul_rn(R[0], cp[0]))));
                out[4 * r] = __double2float_rn(R[0]);
                out[4 * r + 1] = __double2float_rn(R[1]);
                out[4 * r + 2] = __double2float_rn(R[2]);
                out[4 * r + 3] = __double2float_rn(t);
            }
            s0 = (int32_t)c[0];
        }
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) pose[3 * h + r] = make_float4(out[4 * r], out[4 * r + 1], out[4 * r + 2], out[4 * r + 3]);
    sample0[h] = s0;
}

// counts[h] += the correspondences of this block's chunk that pose h counts.  Block (x, y) scores hypotheses
// [y * RS_HTILE, (y + 1) * RS_HTILE) over correspondences [x * chunk, (x + 1) * chunk): lane l holds hypotheses
// y * RS_HTILE + 4 l .. + 3, and warp w takes the w-th eighth of every tile.  Hypotheses past H are NaN (count nothing).
__global__ void __launch_bounds__(RS_THREADS) rs_score_kernel(const float4* __restrict__ pairs, uint32_t M,
                                                              uint32_t chunk, const float4* __restrict__ pose,
                                                              uint32_t H, float eps2, uint32_t* __restrict__ counts) {
    __shared__ __align__(128) float4 tiles[2][2 * RS_TILE];
    __shared__ __align__(8) unsigned long long bars[2];
    __shared__ uint32_t s_cnt[RS_HTILE];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t h0 = blockIdx.y * RS_HTILE + lane * RS_HPT;
    const uint32_t begin = blockIdx.x * chunk, end = min(M, begin + chunk);

    // C[u][4 r + c]: row r, column c (3 = t) of hypotheses h0 + 2u and h0 + 2u + 1
    unsigned long long Cf[RS_HPT / 2][12];
#pragma unroll
    for (int u = 0; u < RS_HPT / 2; ++u) {
        const uint32_t ha = h0 + 2 * u, hb = ha + 1;
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const float4 a = ha < H ? __ldg(pose + 3 * ha + r) : make_float4(qnan(), qnan(), qnan(), qnan());
            const float4 b = hb < H ? __ldg(pose + 3 * hb + r) : make_float4(qnan(), qnan(), qnan(), qnan());
            Cf[u][4 * r] = pack2(a.x, b.x);
            Cf[u][4 * r + 1] = pack2(a.y, b.y);
            Cf[u][4 * r + 2] = pack2(a.z, b.z);
            Cf[u][4 * r + 3] = pack2(a.w, b.w);
        }
    }
    const unsigned long long E2 = pack2(eps2, eps2);
    uint32_t cnt[RS_HPT];
#pragma unroll
    for (int u = 0; u < RS_HPT; ++u) cnt[u] = 0u;

    if (threadIdx.x < RS_HTILE) s_cnt[threadIdx.x] = 0u;
    if (threadIdx.x == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t bytes = min((uint32_t)RS_TILE, end - begin) * (uint32_t)(2 * sizeof(float4));
        mbar_expect_tx(&bars[0], bytes);
        bulk_g2s(&tiles[0][0], pairs + 2 * (size_t)begin, bytes, &bars[0]);
    }
    uint32_t it = 0;
    for (uint32_t base = begin; base < end; base += RS_TILE, ++it) {
        const uint32_t buf = it & 1u;
        const int lim = (int)min((uint32_t)RS_TILE, end - base);
        constexpr int STEP = RS_WARPS * RS_UNROLL;
        const int limb = (lim + STEP - 1) / STEP * STEP;
        // the other buffer was read in the previous iteration, which ended in a block barrier: refill it now
        if (threadIdx.x == 0 && base + RS_TILE < end) {
            const uint32_t bytes = min((uint32_t)RS_TILE, end - base - RS_TILE) * (uint32_t)(2 * sizeof(float4));
            mbar_expect_tx(&bars[buf ^ 1u], bytes);
            bulk_g2s(&tiles[buf ^ 1u][0], pairs + 2 * (size_t)(base + RS_TILE), bytes, &bars[buf ^ 1u]);
        }
        mbar_wait(&bars[buf], (it >> 1) & 1u);
        if (lim < limb) {  // (last tile of a chunk only) pairs beyond the end count for no pose
            if (threadIdx.x < (unsigned)(limb - lim)) {
                tiles[buf][2 * (lim + threadIdx.x)] = make_float4(0.f, 0.f, 0.f, 0.f);
                tiles[buf][2 * (lim + threadIdx.x) + 1] = make_float4(INFINITY, INFINITY, INFINITY, 0.f);
            }
            __syncthreads();
        }
        const int seg = limb / RS_WARPS;
        const float4* tp = tiles[buf] + 2 * warp * seg;
#pragma unroll 2
        for (int j = 0; j < seg; j += RS_UNROLL) {
#pragma unroll
            for (int v = 0; v < RS_UNROLL; ++v) {
                const float4 p = tp[2 * (j + v)], q = tp[2 * (j + v) + 1];  // (broadcast LDS.128)
                const unsigned long long PX = pack2(p.x, p.x), PY = pack2(p.y, p.y), PZ = pack2(p.z, p.z);
                const unsigned long long Q[3] = {pack2(q.x, q.x), pack2(q.y, q.y), pack2(q.z, q.z)};
#pragma unroll
                for (int u = 0; u < RS_HPT / 2; ++u) {
                    unsigned long long d[3];
#pragma unroll
                    for (int r = 0; r < 3; ++r) {
                        unsigned long long y;
                        asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(y) : "l"(Cf[u][4 * r]), "l"(PX), "l"(Cf[u][4 * r + 3]));
                        asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(y) : "l"(Cf[u][4 * r + 1]), "l"(PY), "l"(y));
                        asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(y) : "l"(Cf[u][4 * r + 2]), "l"(PZ), "l"(y));
                        asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d[r]) : "l"(y), "l"(Q[r]));
                    }
                    unsigned long long s;
                    asm("mul.rn.f32x2 %0, %1, %1;" : "=l"(s) : "l"(d[0]));
                    asm("fma.rn.f32x2 %0, %1, %1, %2;" : "=l"(s) : "l"(d[1]), "l"(s));
                    asm("fma.rn.f32x2 %0, %1, %1, %2;" : "=l"(s) : "l"(d[2]), "l"(s));
                    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(s) : "l"(s), "l"(E2));
                    float lo, hi;
                    unpack2(s, lo, hi);
                    // d^2 < eps^2  <=>  the sign bit of fl(d^2 - eps^2): IEEE subtraction is exact in sign, and the
                    // device's NaN (a NaN pose, a q = +inf pair) has a clear sign bit
                    cnt[2 * u] += __float_as_uint(lo) >> 31;
                    cnt[2 * u + 1] += __float_as_uint(hi) >> 31;
                }
            }
        }
        __syncthreads();  // every thread is done with this buffer before the next iteration refills it
    }
#pragma unroll
    for (int u = 0; u < RS_HPT; ++u)
        if (cnt[u]) atomicAdd(&s_cnt[lane * RS_HPT + u], cnt[u]);
    __syncthreads();
    if (threadIdx.x < RS_HTILE) {
        const uint32_t h = blockIdx.y * RS_HTILE + threadIdx.x;
        if (h < H && s_cnt[threadIdx.x]) atomicAdd(counts + h, s_cnt[threadIdx.x]);
    }
}

// counts[h] = 0xFFFFFFFF for the invalid hypotheses; st->best = max over the valid ones of (count << 32) | ~h
__global__ void __launch_bounds__(RS_THREADS) rs_select_kernel(const float4* __restrict__ pose, uint32_t H,
                                                               uint32_t* __restrict__ counts, RansacState* st) {
    const uint32_t h = blockIdx.x * RS_THREADS + threadIdx.x;
    unsigned long long key = 0ull;
    if (h < H) {
        if (isnan(pose[3 * h].x)) {
            counts[h] = 0xFFFFFFFFu;
        } else {
            key = ((unsigned long long)counts[h] << 32) | (unsigned long long)(~h);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) key = max(key, __shfl_xor_sync(0xffffffffu, key, o));
    if ((threadIdx.x & 31) == 0 && key) atomicMax(&st->best, key);
}

// v[k] of every thread summed in a fixed order (warp trees, then the warps in order): the total is in thread 0
__device__ __forceinline__ void block_sum(double (&v)[RS_MOMENTS], double (*s_red)[RS_MOMENTS]) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < RS_MOMENTS; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_down_sync(0xffffffffu, v[k], o);
        if (lane == 0) s_red[warp][k] = v[k];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < RS_MOMENTS; ++k) {
            double s = s_red[0][k];
            for (int w = 1; w < RS_WARPS; ++w) s += s_red[w][k];
            v[k] = s;
        }
    }
}

// the least-squares pose of the moments S (shifted by p0, q0) into P; false when it is not defined (rank < 2) or not
// finite.  H = sum a b^T / N - mean(a) mean(b)^T = U S V^T; R = V U^T with v_i the eigenvectors of H^T H (largest
// two), u_i = H v_i / sigma_i, and the third columns v0 x v1, u0 x u1, so that R is a rotation even for a coplanar
// (rank-2) set.
__device__ bool kabsch(const double* S, const float4 p0, const float4 q0, float* P) {
    const double N = S[0];
    const double ma[3] = {S[1] / N, S[2] / N, S[3] / N}, mb[3] = {S[4] / N, S[5] / N, S[6] / N};
    double Hm[3][3], HtH[3][3];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) Hm[i][j] = S[7 + 3 * i + j] / N - ma[i] * mb[j];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) HtH[i][j] = Hm[0][i] * Hm[0][j] + Hm[1][i] * Hm[1][j] + Hm[2][i] * Hm[2][j];
    double ev[3], V[3][3];
    jacobi3(HtH, ev, V);
    int o[3] = {0, 1, 2};  // eigenvalues descending
    for (int a = 0; a < 2; ++a)
        for (int b = a + 1; b < 3; ++b)
            if (ev[o[b]] > ev[o[a]]) {
                const int t = o[a];
                o[a] = o[b];
                o[b] = t;
            }
    if (!(ev[o[0]] > 0.0) || !(ev[o[1]] > 1e-18 * ev[o[0]])) return false;
    double v[3][3], u[3][3];
    for (int i = 0; i < 2; ++i)
        for (int r = 0; r < 3; ++r) v[i][r] = V[r][o[i]];
    for (int i = 0; i < 2; ++i)
        for (int r = 0; r < 3; ++r) u[i][r] = Hm[r][0] * v[i][0] + Hm[r][1] * v[i][1] + Hm[r][2] * v[i][2];
    // Gram-Schmidt: u1 orthogonal to u0, both unit
    double l0 = sqrt(u[0][0] * u[0][0] + u[0][1] * u[0][1] + u[0][2] * u[0][2]);
    for (int r = 0; r < 3; ++r) u[0][r] /= l0;
    const double d01 = u[0][0] * u[1][0] + u[0][1] * u[1][1] + u[0][2] * u[1][2];
    for (int r = 0; r < 3; ++r) u[1][r] -= d01 * u[0][r];
    const double l1 = sqrt(u[1][0] * u[1][0] + u[1][1] * u[1][1] + u[1][2] * u[1][2]);
    for (int r = 0; r < 3; ++r) u[1][r] /= l1;
    cross3d(u[0], u[1], u[2]);
    cross3d(v[0], v[1], v[2]);
    double R[3][3];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) R[r][c] = v[0][r] * u[0][c] + v[1][r] * u[1][c] + v[2][r] * u[2][c];
    const double cp[3] = {(double)p0.x + ma[0], (double)p0.y + ma[1], (double)p0.z + ma[2]};
    const double cq[3] = {(double)q0.x + mb[0], (double)q0.y + mb[1], (double)q0.z + mb[2]};
    float out[12];
    bool fin = true;
    for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 3; ++c) out[4 * r + c] = (float)R[r][c];
        out[4 * r + 3] = (float)(cq[r] - (R[r][0] * cp[0] + R[r][1] * cp[1] + R[r][2] * cp[2]));
    }
    for (int e = 0; e < 12; ++e) fin = fin && isfinite(out[e]);
    if (!fin) return false;
    for (int e = 0; e < 12; ++e) P[e] = out[e];
    return true;
}

// st->pose = the pose the inliers are selected with: the best hypothesis's, refined from the moments S of its inliers
// when S is given, counts at least 3 of them and the refined pose is finite; NaN without a model.  One thread.
__device__ void ransac_finish(RansacState* st, const float4* __restrict__ pose, const int32_t* __restrict__ sample0,
                              const float4* __restrict__ pairs, const double* S) {
    float P[12];
    for (int e = 0; e < 12; ++e) P[e] = qnan();
    if (st->best) {
        const uint32_t h = ~(uint32_t)st->best;
        for (int r = 0; r < 3; ++r) {
            const float4 v = pose[3 * h + r];
            P[4 * r] = v.x;
            P[4 * r + 1] = v.y;
            P[4 * r + 2] = v.z;
            P[4 * r + 3] = v.w;
        }
        if (S && S[0] >= 3.0) kabsch(S, pairs[2 * sample0[h]], pairs[2 * sample0[h] + 1], P);
    }
    for (int e = 0; e < 12; ++e) st->pose[e] = P[e];
}

// The refinement: the fp64 moments of the best hypothesis's inliers, shifted by its first pair (p0, q0), per block into
// partials[]; the last block folds them in block order (each thread the blocks b, b + RS_THREADS, ...; then
// block_sum) and finishes.
__global__ void __launch_bounds__(RS_THREADS) rs_moments_kernel(const float4* __restrict__ pairs, uint32_t M,
                                                                const float4* __restrict__ pose,
                                                                const int32_t* __restrict__ sample0, float eps2,
                                                                RansacState* st, double* partials) {
    __shared__ double s_red[RS_WARPS][RS_MOMENTS];
    __shared__ bool s_last;
    double acc[RS_MOMENTS];
#pragma unroll
    for (int k = 0; k < RS_MOMENTS; ++k) acc[k] = 0.0;
    const unsigned long long best = st->best;
    if (best) {
        const uint32_t h = ~(uint32_t)best;
        float P[12];
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const float4 v = pose[3 * h + r];
            P[4 * r] = v.x;
            P[4 * r + 1] = v.y;
            P[4 * r + 2] = v.z;
            P[4 * r + 3] = v.w;
        }
        const float4 p0 = pairs[2 * sample0[h]], q0 = pairs[2 * sample0[h] + 1];
        for (uint32_t k = blockIdx.x * RS_THREADS + threadIdx.x; k < M; k += gridDim.x * RS_THREADS) {
            const float4 p = __ldg(pairs + 2 * k), q = __ldg(pairs + 2 * k + 1);
            if (!inlier(P, p, q, eps2)) continue;
            const double a[3] = {(double)p.x - (double)p0.x, (double)p.y - (double)p0.y, (double)p.z - (double)p0.z};
            const double b[3] = {(double)q.x - (double)q0.x, (double)q.y - (double)q0.y, (double)q.z - (double)q0.z};
            acc[0] += 1.0;
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                acc[1 + r] += a[r];
                acc[4 + r] += b[r];
            }
#pragma unroll
            for (int i = 0; i < 3; ++i)
#pragma unroll
                for (int j = 0; j < 3; ++j) acc[7 + 3 * i + j] += a[i] * b[j];
        }
    }
    block_sum(acc, s_red);
    if (threadIdx.x == 0) {
        for (int k = 0; k < RS_MOMENTS; ++k) partials[blockIdx.x * RS_MOMENTS + k] = acc[k];
        __threadfence();
        s_last = atomicAdd(&st->ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
#pragma unroll
    for (int k = 0; k < RS_MOMENTS; ++k) acc[k] = 0.0;
    for (uint32_t b = threadIdx.x; b < gridDim.x; b += RS_THREADS)
#pragma unroll
        for (int k = 0; k < RS_MOMENTS; ++k) acc[k] += __ldcg(partials + b * RS_MOMENTS + k);
    __syncthreads();  // (s_red is reused)
    block_sum(acc, s_red);
    if (threadIdx.x == 0) ransac_finish(st, pose, sample0, pairs, acc);
}

// without refinement
__global__ void rs_finish_kernel(RansacState* st, const float4* __restrict__ pose, const int32_t* __restrict__ sample0,
                                 const float4* __restrict__ pairs) {
    ransac_finish(st, pose, sample0, pairs, nullptr);
}

__global__ void __launch_bounds__(RS_THREADS) rs_inlier_flag_kernel(const float4* __restrict__ pairs, uint32_t M,
                                                                    const RansacState* __restrict__ st, float eps2,
                                                                    uint32_t* __restrict__ flags) {
    const uint32_t k = blockIdx.x * RS_THREADS + threadIdx.x;
    if (k >= M) return;
    float P[12];
#pragma unroll
    for (int e = 0; e < 12; ++e) P[e] = st->pose[e];
    flags[k] = inlier(P, __ldg(pairs + 2 * k), __ldg(pairs + 2 * k + 1), eps2) ? 1u : 0u;
}

}  // namespace

extern "C" {

int spx_ransac_registration(spx_queue_t q, const float* source_points, size_t n_source, const float* target_points,
                            size_t n_target, const int32_t* src_idx, const int32_t* tgt_idx, size_t m_in,
                            float max_correspondence_distance, uint32_t max_iterations, uint64_t seed,
                            float edge_length_similarity, int optimize, float* T4x4_host, int32_t* hypothesis_host,
                            int32_t* inliers_out, size_t* n_inliers_host, uint32_t* counts_out) {
    return guard([&] {
        SPX_REQUIRE(q && T4x4_host && hypothesis_host && n_inliers_host, "[RANSACRegistration] null argument");
        SPX_REQUIRE(m_in < (1ull << 31), "[RANSACRegistration] at most 2^31 - 1 correspondences");
        const float eps = max_correspondence_distance;
        SPX_REQUIRE(std::isfinite(eps) && eps > 0.0f,
                    "[RANSACRegistration] `max_correspondence_distance` must be finite and > 0");
        SPX_REQUIRE(max_iterations >= 1u && max_iterations <= (1u << 20),
                    "[RANSACRegistration] `max_iterations` must be in [1, 2^20]");
        SPX_REQUIRE(edge_length_similarity > 0.0f && edge_length_similarity <= 1.0f,
                    "[RANSACRegistration] `edge_length_similarity` must be in (0, 1]");
        const float qn = std::nanf("");
        for (int e = 0; e < 16; ++e) T4x4_host[e] = qn;
        *hypothesis_host = -1;
        *n_inliers_host = 0;
        if (m_in == 0) {  // every hypothesis is invalid; a memset launches no kernel
            if (counts_out) {
                DeviceGuard dg(q->device);
                SPX_CUDA(cudaMemsetAsync(counts_out, 0xFF, (size_t)max_iterations * 4, q->stream));
                q->sync();
            }
            return;
        }
        SPX_REQUIRE(source_points && target_points && src_idx && tgt_idx && inliers_out, "[RANSACRegistration] null pointer");
        SPX_REQUIRE(((reinterpret_cast<uintptr_t>(source_points) | reinterpret_cast<uintptr_t>(target_points)) & 15) == 0,
                    "[RANSACRegistration] points must be 16-byte aligned");
        DeviceGuard dg(q->device);
        cudaStream_t st = q->stream;
        const uint32_t M = (uint32_t)m_in, H = max_iterations;
        const float eps2 = eps * eps;
        const double tau2 = (double)edge_length_similarity * (double)edge_length_similarity;
        q->arena_reset();
        q->arena_reserve(32 * (size_t)M + 4 * (2 * align_up(M, 64) + scan_scratch_elems(M)) +
                         4 * 15 * align_up(H, 64) + 8 * RS_MOMENT_BLOCKS * RS_MOMENTS + 4096);
        float4* pairs = q->take<float4>(2 * (size_t)M);
        uint32_t* flags = q->take<uint32_t>(M);
        uint32_t* pos = q->take<uint32_t>(M);
        uint32_t* scan_tmp = q->take<uint32_t>(scan_scratch_elems(M));
        float4* pose = q->take<float4>(3 * (size_t)H);
        int32_t* sample0 = q->take<int32_t>(H);
        uint32_t* counts = counts_out ? counts_out : q->take<uint32_t>(H);
        double* partials = q->take<double>(RS_MOMENT_BLOCKS * RS_MOMENTS);
        RansacState* state = q->take<RansacState>(1);

        SPX_CUDA(cudaMemsetAsync(state, 0, sizeof(RansacState), st));
        SPX_CUDA(cudaMemsetAsync(counts, 0, (size_t)H * 4, st));
        rs_gather_kernel<<<div_up(M, RS_THREADS), RS_THREADS, 0, st>>>(
            reinterpret_cast<const float4*>(source_points), n_source, reinterpret_cast<const float4*>(target_points),
            n_target, src_idx, tgt_idx, M, pairs);
        SPX_LAUNCH_CHECK();
        rs_hypothesis_kernel<<<div_up(H, RS_THREADS), RS_THREADS, 0, st>>>(pairs, M, H, seed, tau2, pose, sample0);
        SPX_LAUNCH_CHECK();
        // the hot path: enough correspondence chunks per hypothesis tile for ~8 blocks per SM, chunks whole tiles
        int sms = 0;
        SPX_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, q->device));
        const uint32_t htiles = div_up(H, RS_HTILE), ptiles = div_up(M, RS_TILE);
        const uint32_t want = std::max<uint32_t>(1u, (uint32_t)div_up((size_t)sms * 8, htiles));
        const uint32_t chunk = div_up(ptiles, std::min(ptiles, want)) * RS_TILE;
        rs_score_kernel<<<dim3(div_up(M, chunk), htiles), RS_THREADS, 0, st>>>(pairs, M, chunk, pose, H, eps2, counts);
        SPX_LAUNCH_CHECK();
        rs_select_kernel<<<div_up(H, RS_THREADS), RS_THREADS, 0, st>>>(pose, H, counts, state);
        SPX_LAUNCH_CHECK();
        if (optimize) {
            rs_moments_kernel<<<std::min(div_up(M, RS_THREADS), RS_MOMENT_BLOCKS), RS_THREADS, 0, st>>>(
                pairs, M, pose, sample0, eps2, state, partials);
        } else {
            rs_finish_kernel<<<1, 1, 0, st>>>(state, pose, sample0, pairs);
        }
        SPX_LAUNCH_CHECK();
        rs_inlier_flag_kernel<<<div_up(M, RS_THREADS), RS_THREADS, 0, st>>>(pairs, M, state, eps2, flags);
        SPX_LAUNCH_CHECK();
        exclusive_scan_u32(st, flags, pos, M, scan_tmp, &state->n_inliers);
        compact_index_kernel<<<div_up(M, COMPACT_THREADS), COMPACT_THREADS, 0, st>>>(flags, pos, M, inliers_out);
        SPX_LAUNCH_CHECK();
        RansacState* hs = static_cast<RansacState*>(q->pinned_get(sizeof(RansacState)));
        SPX_CUDA(cudaMemcpyAsync(hs, state, sizeof(RansacState), cudaMemcpyDeviceToHost, st));
        q->sync();
        for (int r = 0; r < 3; ++r) {
            for (int c = 0; c < 3; ++c) T4x4_host[4 * c + r] = hs->pose[4 * r + c];
            T4x4_host[12 + r] = hs->pose[4 * r + 3];
        }
        if (hs->best) {
            T4x4_host[3] = T4x4_host[7] = T4x4_host[11] = 0.0f;
            T4x4_host[15] = 1.0f;
        } else {
            for (int e = 0; e < 16; ++e) T4x4_host[e] = qn;
        }
        *hypothesis_host = hs->best ? (int32_t)(~(uint32_t)hs->best) : -1;
        *n_inliers_host = hs->n_inliers;
    });
}

}  // extern "C"
