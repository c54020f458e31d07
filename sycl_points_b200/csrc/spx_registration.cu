// Registration hot loop on the device: nearest neighbour -> per-point factor -> robust weight ->
// block reduction to the 21 unique H terms, 6 b terms, error and inlier count -> 6x6 solve and
// pose update.  Reference: I/algorithms/registration/registration.hpp:201-276 (align loop),
// :513-676 (linearise + sycl::reduction), :678-789 (error pass), :803-964 (GN / LM / dog-leg),
// factors I/algorithms/registration/factor.hpp:63-278, robust kernels I/algorithms/robust/robust.hpp.
//
// What is different from the reference by design (results stay within the stated tolerances):
//  * GICP's plane regularisation of both covariances (2 eigen-decompositions per point per
//    iteration inside linearize_gicp, factor.hpp:250-255) is pose-independent, so align() hoists
//    it into one pass per cloud and the iteration kernel reads 6 floats per covariance.
//  * H is symmetric: 21 terms are reduced instead of 36 (registration.hpp:565-571 sums all 36).
//  * sums: fp32 per thread, fp32 warp shuffles, fp64 from the block level up, folded in a fixed
//    order by the last block to finish -> deterministic, and closer to the exact sum than any
//    fp32 sycl::reduction order.
//  * Gauss-Newton never returns to the host inside the loop: the last block also solves the 6x6
//    system (fp64 LDL^T) and advances the pose that the next launch reads.
#include <cooperative_groups.h>

#include <cmath>
#include <cstdlib>
#include <cstring>
#include <type_traits>

#include "spx_grid.cuh"
#include "spx_math.cuh"

using namespace spx;

namespace {

constexpr int LIN_THREADS = 256;
constexpr int LIN_WARPS = LIN_THREADS / 32;
constexpr int S_B = 21, S_ERR = 27, S_INL = 28;
constexpr int N_ACC = 28;  // float accumulators per thread (21 H + 6 b + error)

// device-resident optimiser state (one per spx_registration)
struct RegState {
    float T[4][4];  // row-major current pose
    int iterations;
    int converged;
    int stop;  // set once converged: later launches of the same align() return immediately
    int solve_ok;
    float H[36];
    float b[6];
    float error;
    uint32_t inlier;
    float delta[6];
    float pad[2];
    float Tp[4][4];  // pose of the previous iteration (keep test of the split search kernels, icp_keep)
};

// view of the NVLink mailboxes handed to the sharded align kernel (spx_comm_s, DESIGN.md §6)
struct PeerX {
    int world, rank;
    double* rows[SPX_MAX_RANKS];               // rows[p]: rank p's mailbox rows [2][SPX_MAX_RANKS][32]
    unsigned long long* flags[SPX_MAX_RANKS];  // flags[p]: rank p's arrival flags [2][SPX_MAX_RANKS]
    double* gsum;                              // local [2][32]
    unsigned long long* ready;                 // local [2]
    unsigned int* error;                       // local
    unsigned long long seq0;                   // sequence number of iteration 0 of this align
};

struct LinArgs {
    // source
    const float4* src_pts;
    const float4* src_cm;  // prepared (plane-regularised) covariance, 3 rows of the full 3x3 per point
    const float* src_cov16;  // raw reference layout (generic entry points)
    uint32_t ns;
    // target (original index order)
    const float4* tgt_pts;
    const float4* tgt_cm;
    const float* tgt_cov16;
    const float4* tgt_normals;
    // correspondences
    const int32_t* idx_in;
    const float* dist_in;
    int32_t* idx_out;
    float* dist_out;
    float* slack_out;    // keep test (icp_keep): metres each query may still move before it is searched again
    float keep_infl;     // most metres a margin-tracking search adds to a candidate's distance when it prunes / certifies
    int keep_last;       // the previous iteration's search tracked margins: slack_out is valid
    uint32_t* redo;      // [ns] queries the keep pass could not keep (count: wl_counters[WL_REDO + parity])
    int warm_start;      // idx_out holds a previous iteration's result (per-launch kernels)
    uint32_t* worklist;          // [ns] source indices whose search the first pass could not finish
    unsigned int* wl_counters;   // [2 parities][count, cursor]
    GridLevels grid;
    // pose
    RegState* state;
    Xform T;
    int use_state;
    // gating / robust kernel
    float max_corr;
    float max_corr_sq;
    float scale;
    int loss;
    // reduction
    double* partials;  // [gridDim.x][32]
    unsigned int* ticket;
    double* sums_out;  // [32]
    // fused Gauss-Newton step
    float lambda, crit_rot, crit_trans;
    int iter_index;
    float* trace;  // [max_iterations][16] column-major poses, nullable
    float* weights_out;  // compute_icp_robust_weights
    // GenZ (factor.hpp:378-449): planarity threshold and the {planar inliers, inliers} counters alpha comes from
    float genz_threshold;
    unsigned int* genz_counts;
    // rotation constraint (rotation_constraint.hpp:15-121), an extra term per correspondence on the RAW covariances
    int rot_enable;
    float rot_weight, rot_scale;
    PeerX px;            // sharded align only
    // optional phase timestamps (tuning aid, spx_registration_phase_times): [iteration][PH_N] ns,
    // entry p = latest time any block reached phase p of that iteration
    unsigned long long* phase;
};
constexpr int PH_START = 0, PH_NN = 1, PH_COOP = 2, PH_ACC = 3, PH_PART = 4, PH_SYNC = 5, PH_FOLD = 6, PH_SOLVE = 7, PH_N = 8;
constexpr int WL_REDO = 4;   // wl_counters[WL_REDO + parity]: length of the keep pass's redo list
constexpr int WL_KEPT = 12;  // wl_counters[WL_KEPT]: correspondences kept without a search, summed over the align's iterations
constexpr int PH_MAX_ITERS = 64;
constexpr int PH_MAX_WARPS = 8192;
constexpr size_t PH_WORDS = (size_t)PH_MAX_ITERS * PH_N + (size_t)PH_MAX_WARPS * 5;

__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_gpu(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
constexpr unsigned long long PEER_TIMEOUT_NS = 5000000000ull;

// ------------------------------------------------------------------ factors
struct Jac {
    float j[3][6];  // rows 0..2 of the 4x6 SE(3) Jacobian [R skew(p) | -R]; row 3 is zero
};

// compute_se3_jacobian — factor.hpp:69-84; the zero terms of skew() drop out of the fma chains
__device__ __forceinline__ Jac se3_jacobian(const Xform& T, const float4 p) {
    Jac J;
    const float R[3][3] = {{T.r0.x, T.r0.y, T.r0.z}, {T.r1.x, T.r1.y, T.r1.z}, {T.r2.x, T.r2.y, T.r2.z}};
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        J.j[i][0] = __fmaf_rn(R[i][2], -p.y, __fmul_rn(R[i][1], p.z));
        J.j[i][1] = __fmaf_rn(R[i][2], p.x, __fmul_rn(R[i][0], -p.z));
        J.j[i][2] = __fmaf_rn(R[i][1], -p.x, __fmul_rn(R[i][0], p.y));
        J.j[i][3] = -R[i][0];
        J.j[i][4] = -R[i][1];
        J.j[i][5] = -R[i][2];
    }
    return J;
}

__device__ __forceinline__ float chain3(float a0, float b0, float a1, float b1, float a2, float b2) {
    return __fmaf_rn(a2, b2, __fmaf_rn(a1, b1, __fmul_rn(a0, b0)));
}

// compute_mahalanobis_covariance + inverse — factor.hpp:111-123, transform.hpp:14-22 (T (C T^T), the
// 4x4 products' zero terms are exact no-ops), covariance.hpp:136-141, eigen_utils.hpp:403-423;
// cs / ct already plane-regularised.  All nine entries, as the reference: R C R^T is symmetric only
// up to rounding and the inverse amplifies the difference.
__device__ __forceinline__ Mat3 gicp_minv(const Xform& T, const Mat3& cs, const Mat3& ct) {
    const float R[3][3] = {{T.r0.x, T.r0.y, T.r0.z}, {T.r1.x, T.r1.y, T.r1.z}, {T.r2.x, T.r2.y, T.r2.z}};
    float X[3][3];  // C R^T
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
        for (int j = 0; j < 3; ++j)
            X[k][j] = chain3(cs.m[k][0], R[j][0], cs.m[k][1], R[j][1], cs.m[k][2], R[j][2]);
    Mat3 M;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j)
            M.m[i][j] = __fadd_rn(chain3(R[i][0], X[0][j], R[i][1], X[1][j], R[i][2], X[2][j]), ct.m[i][j]);
    return mat3_inverse(M);
}

// One correspondence: factor terms (factor.hpp:130-278), robust weight (robust.hpp:56-90), and
// the weighted accumulation of registration.hpp:613-626,653-659.  The residual norm and weight are
// formed first, then every H / b entry is computed and added straight into its accumulator, so no
// 27-entry temporary is ever live (register pressure, not arithmetic, limits this kernel).
// point-to-point terms (factor.hpp:130-149).  GW: every H / b entry is first scaled by the GenZ weight gw
// (linearize_geometry<GENZ>, factor.hpp:436-440: H * w, b * w elementwise) — the other factors never multiply.
template <bool GW>
__device__ __forceinline__ void acc_p2p(const Jac& J, float r0, float r1, float r2, int loss, float scale, float gw, float* acc) {
    const float e2 = chain3(r0, r0, r1, r1, r2, r2);
    const float rn = __fsqrt_rn(e2);
    const float w = robust_weight(loss, rn, scale);
    int t = 0;
#pragma unroll
    for (int a = 0; a < 6; ++a) {
#pragma unroll
        for (int c = a; c < 6; ++c, ++t) {
            float h = chain3(J.j[0][a], J.j[0][c], J.j[1][a], J.j[1][c], J.j[2][a], J.j[2][c]);
            if (GW) h = __fmul_rn(h, gw);
            acc[t] = __fadd_rn(acc[t], __fmul_rn(w, h));
        }
        float bb = chain3(J.j[0][a], r0, J.j[1][a], r1, J.j[2][a], r2);
        if (GW) bb = __fmul_rn(bb, gw);
        acc[S_B + a] = __fadd_rn(acc[S_B + a], __fmul_rn(w, bb));
    }
    const float rho = robust_error(loss, rn, scale);
    acc[S_ERR] = __fadd_rn(acc[S_ERR], GW ? __fmul_rn(gw, rho) : rho);
}

// point-to-plane terms (factor.hpp:172-210)
template <bool GW>
__device__ __forceinline__ void acc_p2plane(const Jac& J, float r0, float r1, float r2, const float4 nrm, int loss, float scale,
                                            float gw, float* acc) {
    const float d = chain3(nrm.x, r0, nrm.y, r1, nrm.z, r2);
    const float rn = fabsf(d);
    const float w = robust_weight(loss, rn, scale);
    const float n[3] = {nrm.x, nrm.y, nrm.z};
    float row[6];
#pragma unroll
    for (int c = 0; c < 6; ++c) row[c] = chain3(n[0], J.j[0][c], n[1], J.j[1][c], n[2], J.j[2][c]);
    const float pe0 = __fmul_rn(n[0], d), pe1 = __fmul_rn(n[1], d), pe2 = __fmul_rn(n[2], d);
    int t = 0;
#pragma unroll
    for (int a = 0; a < 6; ++a) {
        const float ja0 = __fmul_rn(n[0], row[a]), ja1 = __fmul_rn(n[1], row[a]), ja2 = __fmul_rn(n[2], row[a]);
#pragma unroll
        for (int c = a; c < 6; ++c, ++t) {
            float h = chain3(ja0, __fmul_rn(n[0], row[c]), ja1, __fmul_rn(n[1], row[c]), ja2, __fmul_rn(n[2], row[c]));
            if (GW) h = __fmul_rn(h, gw);
            acc[t] = __fadd_rn(acc[t], __fmul_rn(w, h));
        }
        float bb = chain3(ja0, pe0, ja1, pe1, ja2, pe2);
        if (GW) bb = __fmul_rn(bb, gw);
        acc[S_B + a] = __fadd_rn(acc[S_B + a], __fmul_rn(w, bb));
    }
    const float rho = robust_error(loss, rn, scale);
    acc[S_ERR] = __fadd_rn(acc[S_ERR], GW ? __fmul_rn(gw, rho) : rho);
}

// is_genz_planar_correspondence — factor.hpp:378-393: PCA normalised curvature l0 / (l0 + l1 + l2) of the TARGET
// covariance below the threshold
__device__ __forceinline__ bool genz_planar(const Mat3& ct, float threshold) {
    float ev[3], V[3][3];
    mat3_eigen(ct, ev, V);
    const float sum = __fadd_rn(__fadd_rn(ev[0], ev[1]), ev[2]);
    const float curv = sum > 1e-12f ? __fdiv_rn(ev[0], sum) : 1.0f;
    return curv < threshold;
}

template <int REG>
__device__ __forceinline__ void accumulate_point(const Xform& T, const float4 ps, const Mat3& cs, const float4 pt,
                                                 const Mat3& ct, const float4 nrm, int loss, float scale,
                                                 float* acc, bool planar = false, float gw = 1.0f) {
    const float4 tp = transform_point(T, ps);
    const float r0 = __fsub_rn(pt.x, tp.x), r1 = __fsub_rn(pt.y, tp.y), r2 = __fsub_rn(pt.z, tp.z);
    const Jac J = se3_jacobian(T, ps);
    if (REG == SPX_REG_POINT_TO_POINT) {
        acc_p2p<false>(J, r0, r1, r2, loss, scale, 1.0f, acc);
    } else if (REG == SPX_REG_POINT_TO_PLANE) {
        acc_p2plane<false>(J, r0, r1, r2, nrm, loss, scale, 1.0f, acc);
    } else if (REG == SPX_REG_GENZ) {  // factor.hpp:425-443: plane factor x alpha or point factor x (1 - alpha)
        if (planar) acc_p2plane<true>(J, r0, r1, r2, nrm, loss, scale, gw, acc);
        else acc_p2p<true>(J, r0, r1, r2, loss, scale, gw, acc);
    } else {  // GICP, factor.hpp:239-278; point-to-distribution, :326-354 (ct already holds inverse(C_t))
        const Mat3 Mi = (REG == SPX_REG_POINT_TO_DISTRIBUTION) ? ct : gicp_minv(T, cs, ct);
        const float m0 = chain3(Mi.m[0][0], r0, Mi.m[0][1], r1, Mi.m[0][2], r2);  // M^-1 r, rows of the full inverse
        const float m1 = chain3(Mi.m[1][0], r0, Mi.m[1][1], r1, Mi.m[1][2], r2);
        const float m2 = chain3(Mi.m[2][0], r0, Mi.m[2][1], r1, Mi.m[2][2], r2);
        const float e2 = chain3(r0, m0, r1, m1, r2, m2);
        const float rn = __fsqrt_rn(e2);
        const float w = robust_weight(loss, rn, scale);
        float q[6][3];  // J^T M^-1 : q[a][j] = sum_k J(k,a) Minv(k,j)
#pragma unroll
        for (int a = 0; a < 6; ++a)
#pragma unroll
            for (int j = 0; j < 3; ++j)
                q[a][j] = chain3(J.j[0][a], Mi.m[0][j], J.j[1][a], Mi.m[1][j], J.j[2][a], Mi.m[2][j]);
        int t = 0;
#pragma unroll
        for (int a = 0; a < 6; ++a) {
#pragma unroll
            for (int c = a; c < 6; ++c, ++t) {
                // ensure_symmetric(J^T M^-1 J) — eigen_utils.hpp:208-219: (H(a,c) + H(c,a)) * 0.5 off the diagonal
                const float hac = chain3(q[a][0], J.j[0][c], q[a][1], J.j[1][c], q[a][2], J.j[2][c]);
                float h = hac;
                if (c != a) {
                    const float hca = chain3(q[c][0], J.j[0][a], q[c][1], J.j[1][a], q[c][2], J.j[2][a]);
                    h = __fmul_rn(__fadd_rn(hac, hca), 0.5f);
                }
                acc[t] = __fadd_rn(acc[t], __fmul_rn(w, h));
            }
            acc[S_B + a] = __fadd_rn(acc[S_B + a], __fmul_rn(w, chain3(q[a][0], r0, q[a][1], r1, q[a][2], r2)));
        }
        acc[S_ERR] = __fadd_rn(acc[S_ERR], robust_error(loss, rn, scale));
    }
}

template <int REG>
__device__ __forceinline__ float point_error(const Xform& T, const float4 ps, const Mat3& cs, const float4 pt,
                                             const Mat3& ct, const float4 nrm, bool planar = false) {
    const float4 tp = transform_point(T, ps);
    const float r0 = __fsub_rn(pt.x, tp.x), r1 = __fsub_rn(pt.y, tp.y), r2 = __fsub_rn(pt.z, tp.z);
    if (REG == SPX_REG_POINT_TO_POINT || (REG == SPX_REG_GENZ && !planar)) return chain3(r0, r0, r1, r1, r2, r2);  // factor.hpp:156-164
    if (REG == SPX_REG_POINT_TO_PLANE || REG == SPX_REG_GENZ) {                // factor.hpp:218-230, :474-478
        const float d = chain3(nrm.x, r0, nrm.y, r1, nrm.z, r2);
        return __fmul_rn(d, d);
    }
    const Mat3 Mi = (REG == SPX_REG_POINT_TO_DISTRIBUTION) ? ct : gicp_minv(T, cs, ct);  // factor.hpp:287-306, 362-373
    const float m0 = chain3(Mi.m[0][0], r0, Mi.m[0][1], r1, Mi.m[0][2], r2);
    const float m1 = chain3(Mi.m[1][0], r0, Mi.m[1][1], r1, Mi.m[1][2], r2);
    const float m2 = chain3(Mi.m[2][0], r0, Mi.m[2][1], r1, Mi.m[2][2], r2);
    return chain3(r0, m0, r1, m1, r2, m2);
}

// prepared matrices: three float4 rows per point (w unused), 48 B
__device__ __forceinline__ Mat3 load_mat(const float4* cm, size_t i) {
    const float4 a = __ldg(cm + 3 * i), b = __ldg(cm + 3 * i + 1), c = __ldg(cm + 3 * i + 2);
    Mat3 s;
    s.m[0][0] = a.x; s.m[0][1] = a.y; s.m[0][2] = a.z;
    s.m[1][0] = b.x; s.m[1][1] = b.y; s.m[1][2] = b.z;
    s.m[2][0] = c.x; s.m[2][1] = c.y; s.m[2][2] = c.z;
    return s;
}
__device__ __forceinline__ void store_mat(float4* cm, size_t i, const Mat3& s) {
    cm[3 * i] = make_float4(s.m[0][0], s.m[0][1], s.m[0][2], 0.f);
    cm[3 * i + 1] = make_float4(s.m[1][0], s.m[1][1], s.m[1][2], 0.f);
    cm[3 * i + 2] = make_float4(s.m[2][0], s.m[2][1], s.m[2][2], 0.f);
}

// covariances for one correspondence.  Prepared (already regularised) arrays win; raw 16-float
// reference covariances are regularised on the fly (what the reference does every iteration);
// missing covariances are identity (registration.hpp:589-590) — and identity goes through
// update_covariance_plane like any other matrix.
template <int REG>
__device__ __forceinline__ void load_covs(const LinArgs& a, uint32_t i, int ti, Mat3& cs, Mat3& ct) {
    if (REG == SPX_REG_POINT_TO_DISTRIBUTION) {
        // only the target covariance matters: prepared = inverse(C_t) (compute_target_mahalanobis,
        // factor.hpp:311-317 — the RAW covariance, no plane regularisation); missing -> identity
        if (a.tgt_cm) ct = load_mat(a.tgt_cm, (size_t)ti);
        else ct = mat3_inverse(a.tgt_cov16 ? load_cov16(a.tgt_cov16 + (size_t)ti * 16) : mat3_identity());
        return;
    }
    if (REG == SPX_REG_GENZ) {  // the RAW target covariance decides planar / non-planar; missing -> identity
        ct = a.tgt_cov16 ? load_cov16(a.tgt_cov16 + (size_t)ti * 16) : mat3_identity();
        return;
    }
    if (REG != SPX_REG_GICP) return;
    if (a.src_cm) cs = load_mat(a.src_cm, i);
    else cs = plane_regularize(a.src_cov16 ? load_cov16(a.src_cov16 + (size_t)i * 16) : mat3_identity());
    if (a.tgt_cm) ct = load_mat(a.tgt_cm, (size_t)ti);
    else ct = plane_regularize(a.tgt_cov16 ? load_cov16(a.tgt_cov16 + (size_t)ti * 16) : mat3_identity());
}

}  // namespace

// SPX_KEEP_FRAC (tuning aid): inflation of the search bound in finest cells, default 0.2; negative = search every
// query in every iteration.  Results do not depend on it.
static float keep_fraction() {
    const char* e = std::getenv("SPX_KEEP_FRAC");
    return e ? (float)std::atof(e) : 0.2f;
}

namespace {

__device__ __forceinline__ Xform state_xform_prev(const RegState* s) {
    Xform T;
    T.r0 = make_float4(s->Tp[0][0], s->Tp[0][1], s->Tp[0][2], s->Tp[0][3]);
    T.r1 = make_float4(s->Tp[1][0], s->Tp[1][1], s->Tp[1][2], s->Tp[1][3]);
    T.r2 = make_float4(s->Tp[2][0], s->Tp[2][1], s->Tp[2][2], s->Tp[2][3]);
    T.r3 = make_float4(s->Tp[3][0], s->Tp[3][1], s->Tp[3][2], s->Tp[3][3]);
    return T;
}

// Keep test of the ICP loop (DESIGN.md §3 K-align): a finished search leaves, per query, how far the query may still
// move before another target point can become the nearest (icp_keep_slack, spx_grid.cuh).  An iteration moves query
// i by delta_i = |T p_i - T_prev p_i|; while the allowance lasts the correspondence is kept and only its distance
// is recomputed — the same index and the same fp32 distance a new search would return.  A kept correspondence that
// leaves max_correspondence_distance is searched again, so that rejected entries match a search's as well.
// Returns true when the query needs a search.
__device__ __forceinline__ bool icp_keep(const Xform& T, const Xform& Tp, const float4 ps, const float4 q, int prev_i,
                                         float slack, const float4* __restrict__ tgt_pts, float max_corr_sq,
                                         float* dist_i, float* slack_i) {
    if (prev_i < 0 || !(slack > 0.0f)) return true;
    const float4 qp = transform_point(Tp, ps);
    const float moved = sqrtf(dist_sq(q.x, q.y, q.z, qp.x, qp.y, qp.z));
    const float left = __fmaf_rn(-2.0002f, moved, slack);
    if (!(left > 0.0f)) return true;
    const float4 pt = __ldg(tgt_pts + prev_i);
    const float dn = dist_sq(q.x, q.y, q.z, pt.x, pt.y, pt.z);
    if (!(dn <= max_corr_sq)) return true;
    *dist_i = dn;
    *slack_i = left;
    return false;
}

// How far a search inflates its bound for a query that moved `moved` metres in the last step: three such steps (the
// iteration contracts) plus the rounding allowance of icp_keep_slack; nothing when that exceeds infl_max — the
// query would be searched again anyway, and an inflated bound costs candidates.
__device__ __forceinline__ float icp_keep_infl(const Xform& T, const Xform& Tp, const float4 ps, float qinf, float infl_max) {
    const float4 q = transform_point(T, ps), qp = transform_point(Tp, ps);
    const float want = __fmaf_rn(3.0f, sqrtf(dist_sq(q.x, q.y, q.z, qp.x, qp.y, qp.z)), 2.0e-3f + 2.0e-5f * qinf);
    return want <= infl_max ? want : 0.0f;
}

__device__ __forceinline__ Xform state_xform(const RegState* s) {
    Xform T;
    T.r0 = make_float4(s->T[0][0], s->T[0][1], s->T[0][2], s->T[0][3]);
    T.r1 = make_float4(s->T[1][0], s->T[1][1], s->T[1][2], s->T[1][3]);
    T.r2 = make_float4(s->T[2][0], s->T[2][1], s->T[2][2], s->T[2][3]);
    T.r3 = make_float4(s->T[3][0], s->T[3][1], s->T[3][2], s->T[3][3]);
    return T;
}

// Gauss-Newton step on the reduced sums — registration.hpp:803-828 (+ :407-410, :791-801)
__device__ void gn_update(RegState* st, const double* sums, float lambda, float crit_rot, float crit_trans,
                          int iter_index, float* trace) {
    float H[36], b[6];
    int t = 0;
    for (int a = 0; a < 6; ++a)
        for (int c = a; c < 6; ++c) {
            const float v = (float)sums[t++];
            H[a * 6 + c] = v;
            H[c * 6 + a] = v;
        }
    for (int a = 0; a < 6; ++a) b[a] = (float)sums[S_B + a];
    float delta[6];
    const bool ok = solve_damped6_device(H, b, lambda, delta);
    const bool conv = ok && norm3f(delta) < crit_rot && norm3f(delta + 3) < crit_trans;
    float E[4][4], Tn[4][4];
    se3_exp_rm(delta, E);
    isometry_mul_rm(st->T, E, Tn);
    for (int i = 0; i < 4; ++i)
        for (int j = 0; j < 4; ++j) {
            st->Tp[i][j] = st->T[i][j];
            st->T[i][j] = Tn[i][j];
        }
    st->iterations = iter_index;
    st->converged = conv ? 1 : 0;
    st->stop = conv ? 1 : 0;
    st->solve_ok = ok ? 1 : 0;
    for (int i = 0; i < 36; ++i) st->H[i] = H[i];
    for (int i = 0; i < 6; ++i) {
        st->b[i] = b[i];
        st->delta[i] = delta[i];
    }
    st->error = (float)sums[S_ERR];
    st->inlier = (uint32_t)(sums[S_INL] + 0.5);
    if (trace)
        for (int j = 0; j < 4; ++j)
            for (int i = 0; i < 4; ++i) trace[(size_t)iter_index * 16 + j * 4 + i] = Tn[i][j];
}

// block reduction of `nv` (<= 29) per-thread values -> partials -> ordered fold by the last block.
// Returns true in the last block, with the folded sums in `fold` (shared memory, 32 doubles).
__device__ bool reduce_to_sums(const float* acc, int nacc, uint32_t inl, double* partials, unsigned int* ticket,
                               double* sums_out, double (*fold)[32], float (*red)[32]) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int v = 0; v < nacc; ++v) {
        const float s = warp_sum(acc[v]);
        if (lane == 0) red[warp][v] = s;
    }
    {
        uint32_t c = inl;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        if (lane == 0) red[warp][31] = __uint_as_float(c);
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        double s = 0.0;
        if ((int)threadIdx.x < nacc) {
            for (int w = 0; w < LIN_WARPS; ++w) s += (double)red[w][threadIdx.x];
        } else if (threadIdx.x == S_INL) {
            for (int w = 0; w < LIN_WARPS; ++w) s += (double)__float_as_uint(red[w][31]);
        }
        // error-only passes keep the layout: error at S_ERR, inliers at S_INL
        int slot = threadIdx.x;
        if (nacc == 1 && threadIdx.x == 0) slot = S_ERR;
        if (nacc == 1 && threadIdx.x == S_ERR) slot = 0;
        __stcg(partials + (size_t)blockIdx.x * 32 + slot, s);
    }
    __shared__ bool is_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int t = atomicAdd(ticket, 1u);
        is_last = (t == gridDim.x - 1);
    }
    __syncthreads();
    if (!is_last) return false;
    __threadfence();
    {
        const int v = threadIdx.x & 31, slice = threadIdx.x >> 5;
        double s = 0.0;
        for (unsigned b = slice; b < gridDim.x; b += LIN_WARPS) s += __ldcg(partials + (size_t)b * 32 + v);
        fold[slice][v] = s;
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        double s = 0.0;
        for (int w = 0; w < LIN_WARPS; ++w) s += fold[w][threadIdx.x];
        fold[0][threadIdx.x] = s;
        if (sums_out) sums_out[threadIdx.x] = s;
    }
    if (threadIdx.x == 0) *ticket = 0;  // ready for the next launch on this stream
    __syncthreads();
    return true;
}

// Per-thread accumulation over a grid-stride slice of the source points.
// MODE 0: correspondences given.  MODE 1: nearest neighbour through the index fused in front
// (bounded by max_correspondence_distance; writes idx/dist for the frozen-neighbour error passes).
__device__ __forceinline__ void phase_mark(unsigned long long* phase, int it, int p) {
    if (phase && threadIdx.x == 0 && it < PH_MAX_ITERS) atomicMax(phase + it * PH_N + p, global_ns());
}

// Correspondence search of one iteration over the whole grid (MODE 1).  Three steps separated by
// grid barriers (the kernels that call this are cooperative launches):
//   1. every lane: warm start + pruned first pass for its own source points; finished queries write
//      their result, unfinished ones write the bound reached and are appended to the work list;
//   2. every warp of the grid pulls unfinished queries off the list (one atomic per grab) and
//      completes them cooperatively — the expensive queries cluster in space, i.e. in a few warps,
//      and this is what spreads them over all SMs;
//   3. (caller) factor evaluation reads the finished idx / dist arrays.
// Work-list counters are double-buffered by `par` and the other pair is cleared in step 2, so no
// extra barrier or host memset is needed between iterations.
__device__ __forceinline__ void nn_search_grid(const LinArgs& a, const Xform& T, int it, cooperative_groups::grid_group& grid) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const bool warm = it > 0 || a.warm_start;
    const int par = it & 1;
    unsigned int* wl_count = a.wl_counters + par * 2;
    unsigned int* wl_cursor = a.wl_counters + par * 2 + 1;
    for (uint32_t base = blockIdx.x * LIN_THREADS; base < a.ns; base += gridDim.x * LIN_THREADS) {
        const uint32_t i = base + threadIdx.x;
        bool pending = false;
        if (i < a.ns) {
            Best1 best;
            best.init();
            // the two loads are independent: issued together, one round trip instead of two
            const float4 ps = __ldg(a.src_pts + i);
            const int prev_i = warm ? __ldcg(a.idx_out + i) : -1;
            const float4 q = transform_point(T, ps);
            if (a.grid.lv[0].n > 0 && isfinite(q.x) && isfinite(q.y) && isfinite(q.z))
                pending = !icp_fast(a.grid, q.x, q.y, q.z, prev_i, a.tgt_pts, a.max_corr, best);
            a.idx_out[i] = best.i;
            a.dist_out[i] = best.d;
        }
        // warp-aggregated append
        const unsigned m = __ballot_sync(FULL, pending);
        if (m) {
            unsigned int slot = 0;
            if (lane == __ffs(m) - 1) slot = atomicAdd(wl_count, (unsigned int)__popc(m));
            slot = __shfl_sync(FULL, slot, __ffs(m) - 1);
            if (pending) a.worklist[slot + __popc(m & ((1u << lane) - 1u))] = i;
        }
    }
    phase_mark(a.phase, it, PH_NN);
    __threadfence();
    grid.sync();
    if (blockIdx.x == 0 && threadIdx.x == 0) {  // the other parity's counters: idle until the next iteration
        a.wl_counters[(par ^ 1) * 2] = 0;
        a.wl_counters[(par ^ 1) * 2 + 1] = 0;
    }
    const unsigned int n_slow = __ldcg(wl_count);
    // tuning aid (phase buffer attached, iteration 2): per-warp {ns in this loop, queries, slowest query ns, list size}
    const bool rec = a.phase != nullptr && it == 2;
    const unsigned long long t_loop = rec ? global_ns() : 0ull;
    unsigned long long t_worst = 0;
    unsigned int n_done = 0;
    for (;;) {
        unsigned int k = 0;
        if (lane == 0) k = atomicAdd(wl_cursor, 1u);
        k = __shfl_sync(FULL, k, 0);
        if (k >= n_slow) break;
        const unsigned long long t_q = rec ? global_ns() : 0ull;
        const uint32_t i = __ldcg(a.worklist + k);
        const float4 q = transform_point(T, __ldg(a.src_pts + i));
        Best1 best;
        best.i = __ldcg(a.idx_out + i);
        best.d = __ldcg(a.dist_out + i);
        icp_coop_search(a.grid, q.x, q.y, q.z, best, a.max_corr);
        if (lane == 0) {
            a.idx_out[i] = best.i;
            a.dist_out[i] = best.d;
        }
        if (rec) {
            t_worst = max(t_worst, global_ns() - t_q);
            ++n_done;
        }
    }
    if (rec && lane == 0) {
        unsigned long long* w = a.phase + PH_MAX_ITERS * PH_N + (size_t)(blockIdx.x * LIN_WARPS + (threadIdx.x >> 5)) * 5;
        w[0] = global_ns() - t_loop;
        w[1] = n_done;
        w[2] = t_worst;
        w[3] = n_slow;
        w[4] = 1;
    }
    __threadfence();
    grid.sync();
}

// nn_search_grid with the keep test (icp_keep) for the sharded one-launch align, whose shards of a dense cloud run many
// iterations: from the third iteration on a streaming keep pass carries over every correspondence whose allowance
// outlasts the query's step and lists the others (block-aggregated append); one more grid barrier, then the first
// pass runs densely over that redo list.  Searches track margins (Best1M) from the first iteration on.  a.keep_infl
// < 0: every query is searched in every iteration (results are the same either way).
__device__ __forceinline__ void nn_search_grid_keep(const LinArgs& a, const Xform& T, const Xform& Tp, int it,
                                                    cooperative_groups::grid_group& grid) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool warm = it > 0;
    const bool keep_it = it >= 2 && a.keep_infl >= 0.0f;
    const float infl_max = fmaxf(a.keep_infl, 0.0f);
    const int par = it & 1;
    unsigned int* wl_count = a.wl_counters + par * 2;
    unsigned int* wl_cursor = a.wl_counters + par * 2 + 1;
    unsigned int* redo_count = a.wl_counters + WL_REDO + par;
    __shared__ unsigned int warp_redo[LIN_WARPS];
    __shared__ unsigned int block_slot;
    if (keep_it) {
        for (uint32_t base = blockIdx.x * LIN_THREADS; base < a.ns; base += gridDim.x * LIN_THREADS) {
            const uint32_t i = base + threadIdx.x;
            bool search = i < a.ns;
            if (search) {
                const float4 ps = __ldg(a.src_pts + i);
                search = icp_keep(T, Tp, ps, transform_point(T, ps), __ldcg(a.idx_out + i), __ldcg(a.slack_out + i), a.tgt_pts,
                                  a.max_corr_sq, a.dist_out + i, a.slack_out + i);
            }
            const unsigned m = __ballot_sync(FULL, search);
            if (lane == 0) warp_redo[warp] = __popc(m);
            __syncthreads();
            if (threadIdx.x == 0) {
                unsigned int total = 0;
                for (int w = 0; w < LIN_WARPS; ++w) {
                    const unsigned int c = warp_redo[w];
                    warp_redo[w] = total;
                    total += c;
                }
                const unsigned int live = min((unsigned int)LIN_THREADS, a.ns - base);
                if (live > total) atomicAdd(a.wl_counters + WL_KEPT, live - total);
                block_slot = total ? atomicAdd(redo_count, total) : 0u;
            }
            __syncthreads();
            if (search) a.redo[block_slot + warp_redo[warp] + __popc(m & ((1u << lane) - 1u))] = i;
            __syncthreads();
        }
        __threadfence();
        grid.sync();
    }
    const uint32_t n_first = keep_it ? __ldcg(redo_count) : a.ns;
    for (uint32_t base = blockIdx.x * LIN_THREADS; base < n_first; base += gridDim.x * LIN_THREADS) {
        const uint32_t k = base + threadIdx.x;
        bool pending = false;
        uint32_t i = k;
        if (k < n_first) {
            if (keep_it) i = __ldcg(a.redo + k);
            Best1M best;
            best.init();
            const float4 ps = __ldg(a.src_pts + i);
            const int prev_i = warm ? __ldcg(a.idx_out + i) : -1;
            const float4 q = transform_point(T, ps);
            const float qinf = fmaxf(fmaxf(fabsf(q.x), fabsf(q.y)), fabsf(q.z));
            if (a.grid.lv[0].n > 0 && isfinite(q.x) && isfinite(q.y) && isfinite(q.z)) {
                const float infl = warm && a.keep_infl >= 0.0f ? icp_keep_infl(T, Tp, ps, qinf, infl_max) : 0.0f;
                pending = !icp_fast(a.grid, q.x, q.y, q.z, prev_i, a.tgt_pts, a.max_corr, best, infl);
            }
            a.idx_out[i] = best.i;
            a.dist_out[i] = best.d;
            // unfinished: the runner-up bound travels to the cooperative phase in the allowance's slot
            a.slack_out[i] = pending ? best.d2 : icp_keep_slack(best, qinf, a.max_corr_sq);
        }
        const unsigned m = __ballot_sync(FULL, pending);
        if (m) {
            unsigned int slot = 0;
            if (lane == __ffs(m) - 1) slot = atomicAdd(wl_count, (unsigned int)__popc(m));
            slot = __shfl_sync(FULL, slot, __ffs(m) - 1);
            if (pending) a.worklist[slot + __popc(m & ((1u << lane) - 1u))] = i;
        }
    }
    phase_mark(a.phase, it, PH_NN);
    __threadfence();
    grid.sync();
    if (blockIdx.x == 0 && threadIdx.x == 0) {  // the other parity's counters: idle until the next iteration
        a.wl_counters[(par ^ 1) * 2] = 0;
        a.wl_counters[(par ^ 1) * 2 + 1] = 0;
        a.wl_counters[WL_REDO + (par ^ 1)] = 0;
    }
    const unsigned int n_slow = __ldcg(wl_count);
    for (;;) {
        unsigned int k = 0;
        if (lane == 0) k = atomicAdd(wl_cursor, 1u);
        k = __shfl_sync(FULL, k, 0);
        if (k >= n_slow) break;
        const uint32_t i = __ldcg(a.worklist + k);
        const float4 ps = __ldg(a.src_pts + i);
        const float4 q = transform_point(T, ps);
        const float qinf = fmaxf(fmaxf(fabsf(q.x), fabsf(q.y)), fabsf(q.z));
        Best1M best;
        best.init();
        best.i = __ldcg(a.idx_out + i);
        best.d = __ldcg(a.dist_out + i);
        best.d2 = __ldcg(a.slack_out + i);
        const float infl = warm && a.keep_infl >= 0.0f ? icp_keep_infl(T, Tp, ps, qinf, infl_max) : 0.0f;
        icp_coop_search(a.grid, q.x, q.y, q.z, best, a.max_corr, nullptr, infl);
        if (lane == 0) {
            a.idx_out[i] = best.i;
            a.dist_out[i] = best.d;
            a.slack_out[i] = icp_keep_slack(best, qinf, a.max_corr_sq);
        }
    }
    __threadfence();
    grid.sync();
}

// ---- the same search as three ordinary launches per iteration (large clouds)
// The cooperative kernels carry the factor arithmetic's register budget (128/thread -> 16 warps per
// SM) through the search, which is latency-bound and wants warps in flight.  Above a few hundred
// thousand source points launch overhead no longer matters, so the search gets kernels of its own
// (64 registers -> 4x the resident warps) and the factor pass runs as linearize_kernel<REG, 0, SOLVE>.
constexpr int NN_THREADS = 128;

// Keep pass (icp_keep) of an iteration whose predecessor tracked margins: one lane per source point, streaming.  A
// kept correspondence gets its new distance and the rest of its allowance; the others go to the redo list that
// icp_fast_kernel<true> searches densely (left in place they would keep every warp on the search path).
constexpr int KEEP_THREADS = 512;
__global__ void __launch_bounds__(KEEP_THREADS) icp_keep_kernel(const LinArgs a) {
    if (a.state->stop) return;
    __shared__ unsigned int warp_redo[KEEP_THREADS / 32];
    __shared__ unsigned int block_slot;
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t i = blockIdx.x * KEEP_THREADS + threadIdx.x;
    bool search = i < a.ns;
    if (search) {
        const Xform T = state_xform(a.state), Tp = state_xform_prev(a.state);
        const float4 ps = __ldg(a.src_pts + i);
        search = icp_keep(T, Tp, ps, transform_point(T, ps), a.idx_out[i], a.slack_out[i], a.tgt_pts, a.max_corr_sq,
                          a.dist_out + i, a.slack_out + i);
    }
    // block-aggregated append: same-address atomics serialise, one per warp would cost more than the pass itself
    const unsigned m = __ballot_sync(FULL, search);
    if (lane == 0) warp_redo[warp] = __popc(m);
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int total = 0;
        for (int w = 0; w < KEEP_THREADS / 32; ++w) {
            const unsigned int c = warp_redo[w];
            warp_redo[w] = total;
            total += c;
        }
        const unsigned int live = min((unsigned int)KEEP_THREADS, a.ns - blockIdx.x * KEEP_THREADS);
        if (live > total) atomicAdd(a.wl_counters + WL_KEPT, live - total);
        block_slot = total ? atomicAdd(a.wl_counters + WL_REDO + (a.iter_index & 1), total) : 0u;
    }
    __syncthreads();
    if (search) a.redo[block_slot + warp_redo[warp] + __popc(m & ((1u << lane) - 1u))] = i;
}

// M: the search tracks margins (Best1M); with a.keep_last it searches the keep pass's redo list only.
template <bool M>
__global__ void __launch_bounds__(NN_THREADS, 8) icp_fast_kernel(const LinArgs a) {
    if (a.state->stop) return;
    using BestT = typename std::conditional<M, Best1M, Best1>::type;
    const Xform T = state_xform(a.state);
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const bool warm = a.iter_index > 0 || a.warm_start;
    const int par = a.iter_index & 1;
    unsigned int* wl_count = a.wl_counters + par * 2;
    uint32_t i = blockIdx.x * NN_THREADS + threadIdx.x;
    bool search = i < a.ns;
    if (M && a.keep_last) {
        const unsigned int n_redo = a.wl_counters[WL_REDO + par];
        if (blockIdx.x * NN_THREADS >= n_redo) return;
        search = i < n_redo;
        if (search) i = a.redo[i];
    }
    bool pending = false;
    if (search) {
        BestT best;
        best.init();
        const float4 ps = __ldg(a.src_pts + i);
        const int prev_i = warm ? a.idx_out[i] : -1;
        const float4 q = transform_point(T, ps);
        const float qinf = fmaxf(fmaxf(fabsf(q.x), fabsf(q.y)), fabsf(q.z));
        if (a.grid.lv[0].n > 0 && isfinite(q.x) && isfinite(q.y) && isfinite(q.z)) {
            const float infl = M ? icp_keep_infl(T, state_xform_prev(a.state), ps, qinf, a.keep_infl) : 0.0f;
            pending = !icp_fast(a.grid, q.x, q.y, q.z, prev_i, a.tgt_pts, a.max_corr, best, infl);
        }
        a.idx_out[i] = best.i;
        a.dist_out[i] = best.d;
        // unfinished: the runner-up bound travels to the cooperative kernel in the allowance's slot
        if constexpr (M) a.slack_out[i] = pending ? best.d2 : icp_keep_slack(best, qinf, a.max_corr_sq);
    }
    const unsigned m = __ballot_sync(FULL, pending);
    if (m) {
        unsigned int slot = 0;
        if (lane == __ffs(m) - 1) slot = atomicAdd(wl_count, (unsigned int)__popc(m));
        slot = __shfl_sync(FULL, slot, __ffs(m) - 1);
        if (pending) a.worklist[slot + __popc(m & ((1u << lane) - 1u))] = i;
    }
}

template <bool M>
__global__ void __launch_bounds__(NN_THREADS, 8) icp_coop_kernel(const LinArgs a) {
    if (a.state->stop) return;
    using BestT = typename std::conditional<M, Best1M, Best1>::type;
    const Xform T = state_xform(a.state);
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int par = a.iter_index & 1;
    const unsigned int n_slow = a.wl_counters[par * 2];
    unsigned int* wl_cursor = a.wl_counters + par * 2 + 1;
    if (blockIdx.x == 0 && threadIdx.x == 0) {  // next iteration's counters (idle during this launch)
        a.wl_counters[(par ^ 1) * 2] = 0;
        a.wl_counters[(par ^ 1) * 2 + 1] = 0;
        a.wl_counters[WL_REDO + (par ^ 1)] = 0;
    }
    for (;;) {
        unsigned int k = 0;
        if (lane == 0) k = atomicAdd(wl_cursor, 1u);
        k = __shfl_sync(FULL, k, 0);
        if (k >= n_slow) break;
        const uint32_t i = a.worklist[k];
        const float4 ps = __ldg(a.src_pts + i);
        const float4 q = transform_point(T, ps);
        const float qinf = fmaxf(fmaxf(fabsf(q.x), fabsf(q.y)), fabsf(q.z));
        BestT best;
        best.init();
        best.i = a.idx_out[i];
        best.d = a.dist_out[i];
        float infl = 0.0f;
        if constexpr (M) {
            best.d2 = a.slack_out[i];
            infl = icp_keep_infl(T, state_xform_prev(a.state), ps, qinf, a.keep_infl);
        }
        icp_coop_search(a.grid, q.x, q.y, q.z, best, a.max_corr, nullptr, infl);
        if (lane == 0) {
            a.idx_out[i] = best.i;
            a.dist_out[i] = best.d;
            if constexpr (M) a.slack_out[i] = icp_keep_slack(best, qinf, a.max_corr_sq);
        }
    }
}

// ---- rotation constraint — rotation_constraint.hpp:15-121: Jensen-Bregman LogDet divergence between the rotated
// source covariance Cs' = R Cs R^T and the target covariance, D = log det(0.5 (Cs' + Ct)) - 0.5 (log det Cs + log det Ct),
// residual max(D, 0), Jacobian (rotation block only) g = -R^T vex([Cs', M^-1]).  Full 3x3 arithmetic in the
// reference's fma order; log correctly rounded (spx_math.cuh cr_logf).
__device__ __forceinline__ float rot_logdet(const Mat3& m) { return cr_logf(fmaxf(mat3_det(m), 1e-10f)); }

__device__ inline float rot_divergence(const Xform& T, const Mat3& Cs, const Mat3& Ct, float grad[3], bool want_grad) {
    const float R[3][3] = {{T.r0.x, T.r0.y, T.r0.z}, {T.r1.x, T.r1.y, T.r1.z}, {T.r2.x, T.r2.y, T.r2.z}};
    float X[3][3];  // Cs R^T
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) X[i][j] = chain3(Cs.m[i][0], R[j][0], Cs.m[i][1], R[j][1], Cs.m[i][2], R[j][2]);
    Mat3 Csp, M;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            Csp.m[i][j] = chain3(R[i][0], X[0][j], R[i][1], X[1][j], R[i][2], X[2][j]);
            M.m[i][j] = __fmul_rn(__fadd_rn(Csp.m[i][j], Ct.m[i][j]), 0.5f);
        }
    const float log_det_M = rot_logdet(M);
    const float log_det_ref = __fmul_rn(0.5f, __fadd_rn(rot_logdet(Cs), rot_logdet(Ct)));
    const float D = fmaxf(__fsub_rn(log_det_M, log_det_ref), 0.0f);
    if (!want_grad) return D;
    const Mat3 Mi = mat3_inverse(M);
    float comm[3][3];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j)
            comm[i][j] = __fsub_rn(chain3(Csp.m[i][0], Mi.m[0][j], Csp.m[i][1], Mi.m[1][j], Csp.m[i][2], Mi.m[2][j]),
                                   chain3(Mi.m[i][0], Csp.m[0][j], Mi.m[i][1], Csp.m[1][j], Mi.m[i][2], Csp.m[2][j]));
    const float g0 = __fmul_rn(-0.5f, __fsub_rn(comm[2][1], comm[1][2]));
    const float g1 = __fmul_rn(-0.5f, __fsub_rn(comm[0][2], comm[2][0]));
    const float g2 = __fmul_rn(-0.5f, __fsub_rn(comm[1][0], comm[0][1]));
#pragma unroll
    for (int i = 0; i < 3; ++i) grad[i] = chain3(R[0][i], g0, R[1][i], g1, R[2][i], g2);  // R^T g
    return D;
}

// the term's share of H / b / error, added on top of the factor's (registration.hpp:629-649)
__device__ __forceinline__ void accumulate_rotation(const Xform& T, const Mat3& Cs, const Mat3& Ct, int loss, float weight,
                                                    float scale, float* acc) {
    float g[3];
    const float D = rot_divergence(T, Cs, Ct, g, true);
    const float sq = __fmul_rn(__fmul_rn(0.5f, D), D);
    const float rn = __fsqrt_rn(sq);
    const float ww = __fmul_rn(weight, robust_weight(loss, rn, scale));
    constexpr int TIDX[3][3] = {{0, 1, 2}, {1, 6, 7}, {2, 7, 11}};  // packed upper-triangle slot of H(a, c), a, c < 3
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int c = a; c < 3; ++c) acc[TIDX[a][c]] = __fadd_rn(acc[TIDX[a][c]], __fmul_rn(ww, __fmul_rn(g[a], g[c])));
        acc[S_B + a] = __fadd_rn(acc[S_B + a], __fmul_rn(ww, __fmul_rn(D, g[a])));
    }
    acc[S_ERR] = __fadd_rn(acc[S_ERR], __fmul_rn(weight, robust_error(loss, rn, scale)));
}

// Registration::compute_genz_alpha — registration.hpp:464-511: {planar inliers, inliers} of the current
// correspondences, added to a.genz_counts (zeroed by the host before the launch)
template <int MODE>
__device__ __forceinline__ void genz_count(const LinArgs& a) {
    const int32_t* idx = MODE == 1 ? a.idx_out : a.idx_in;
    const float* dist = MODE == 1 ? a.dist_out : a.dist_in;
    unsigned int plane = 0, inl = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < a.ns; i += gridDim.x * blockDim.x) {
        const float d = MODE == 1 ? __ldcg(dist + i) : __ldg(dist + i);
        const int ti = MODE == 1 ? __ldcg(idx + i) : __ldg(idx + i);
        if (d > a.max_corr_sq || ti < 0) continue;
        const Mat3 ct = a.tgt_cov16 ? load_cov16(a.tgt_cov16 + (size_t)ti * 16) : mat3_identity();
        plane += genz_planar(ct, a.genz_threshold) ? 1u : 0u;
        ++inl;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        plane += __shfl_xor_sync(0xffffffffu, plane, o);
        inl += __shfl_xor_sync(0xffffffffu, inl, o);
    }
    if ((threadIdx.x & 31) == 0 && inl) {
        atomicAdd(a.genz_counts, plane);
        atomicAdd(a.genz_counts + 1, inl);
    }
}
__global__ void __launch_bounds__(LIN_THREADS) genz_count_kernel(const LinArgs a) { genz_count<0>(a); }

__device__ __forceinline__ float genz_alpha(const LinArgs& a) {
    const unsigned int plane = __ldcg(a.genz_counts), inl = __ldcg(a.genz_counts + 1);
    return inl == 0u ? 1.0f : __fdiv_rn((float)plane, (float)inl);
}

template <int REG, int MODE>
__device__ __forceinline__ void lin_accumulate(const LinArgs& a, const Xform& T, float* acc, uint32_t& inl) {
    const int32_t* idx = MODE == 1 ? a.idx_out : a.idx_in;
    const float* dist = MODE == 1 ? a.dist_out : a.dist_in;
    const float genz_alpha_v = REG == SPX_REG_GENZ ? genz_alpha(a) : 1.0f;
    for (uint32_t i = blockIdx.x * LIN_THREADS + threadIdx.x; i < a.ns; i += gridDim.x * LIN_THREADS) {
        const float d = MODE == 1 ? __ldcg(dist + i) : __ldg(dist + i);
        const int ti = MODE == 1 ? __ldcg(idx + i) : __ldg(idx + i);
        if (d > a.max_corr_sq || ti < 0) continue;  // registration.hpp:584 (+ guard for the -1 fill)
        const float4 ps = __ldg(a.src_pts + i);
        const float4 pt = __ldg(a.tgt_pts + ti);
        const float4 nrm = ((REG == SPX_REG_POINT_TO_PLANE || REG == SPX_REG_GENZ) && a.tgt_normals)
                               ? __ldg(a.tgt_normals + ti)
                               : make_float4(0.f, 0.f, 0.f, 0.f);
        Mat3 cs, ct;
        load_covs<REG>(a, i, ti, cs, ct);
        if (REG == SPX_REG_GENZ) {
            const bool planar = genz_planar(ct, a.genz_threshold);
            accumulate_point<REG>(T, ps, cs, pt, ct, nrm, a.loss, a.scale, acc, planar,
                                  planar ? genz_alpha_v : __fsub_rn(1.0f, genz_alpha_v));
        } else {
            accumulate_point<REG>(T, ps, cs, pt, ct, nrm, a.loss, a.scale, acc);
        }
        if (a.rot_enable)  // on the raw covariances; missing -> identity (registration.hpp:589-590)
            accumulate_rotation(T, a.src_cov16 ? load_cov16(a.src_cov16 + (size_t)i * 16) : mat3_identity(),
                                a.tgt_cov16 ? load_cov16(a.tgt_cov16 + (size_t)ti * 16) : mat3_identity(), a.loss, a.rot_weight,
                                a.rot_scale, acc);
        ++inl;
    }
}

// One launch = one linearisation.  SOLVE: the last block also performs the Gauss-Newton update of
// the device-resident pose (used by callers that interleave their own work between iterations).
template <int REG, int MODE, bool SOLVE>
__global__ void __launch_bounds__(LIN_THREADS, 2) linearize_kernel(const LinArgs a) {
    __shared__ double fold[LIN_WARPS][32];
    __shared__ float red[LIN_WARPS][32];
    Xform T = a.T;
    if (a.use_state) {
        if (a.state->stop) return;  // converged earlier in this align(): nothing left to do (whole grid)
        T = state_xform(a.state);
    }
    if (MODE == 1) {  // cooperative launch: the correspondence search has grid barriers inside
        cooperative_groups::grid_group grid = cooperative_groups::this_grid();
        nn_search_grid(a, T, a.iter_index, grid);
        if (REG == SPX_REG_GENZ) {  // alpha of the fresh correspondences, before any factor is evaluated
            genz_count<1>(a);
            __threadfence();
            grid.sync();
        }
    }
    float acc[N_ACC];
#pragma unroll
    for (int v = 0; v < N_ACC; ++v) acc[v] = 0.0f;
    uint32_t inl = 0;
    lin_accumulate<REG, MODE>(a, T, acc, inl);
    if (!reduce_to_sums(acc, N_ACC, inl, a.partials, a.ticket, a.sums_out, fold, red)) return;
    if (SOLVE && threadIdx.x == 0)
        gn_update(a.state, &fold[0][0], a.lambda, a.crit_rot, a.crit_trans, a.iter_index, a.trace);
}

// The whole Gauss-Newton align() as ONE cooperative launch (registration.hpp:227-272 + :803-828):
// every iteration is nearest neighbour + linearise + block reduce, one grid-wide barrier, then
// every block folds the per-block partials in the same fixed order and solves the same 6x6 system
// (bitwise identical results, so no second barrier and no broadcast), advances its copy of the
// pose and goes on.  Block 0 records the state for the host.  Partials are double-buffered by
// iteration parity so a block that races ahead never overwrites what a slower block still reads.
//
// SHARDED: this GPU holds one shard of the source.  After the barrier block 0 folds the local
// partial rows, stores the result into every rank's mailbox over NVLink (its own included), raises
// the per-rank arrival flag (release, system scope), waits for every peer's flag (acquire), folds
// the rows in rank order and publishes the global sums to the other blocks of this grid through a
// local flag.  Every rank folds the same rows in the same order, so all poses stay bitwise equal
// and converge at the same iteration.  Mailbox rows and flags are double-buffered by iteration
// parity: a rank can be at most one exchange ahead of the slowest peer.
template <int REG, bool SHARDED>
__global__ void __launch_bounds__(LIN_THREADS, 3) align_gn_kernel(const LinArgs a, int max_iterations) {
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    __shared__ double fold[LIN_WARPS][32];
    __shared__ float red[LIN_WARPS][32];
    __shared__ RegState st;
    if (threadIdx.x == 0) st = *a.state;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int it = 0; it < max_iterations; ++it) {
        const Xform T = state_xform(&st);
        float acc[N_ACC];
#pragma unroll
        for (int v = 0; v < N_ACC; ++v) acc[v] = 0.0f;
        uint32_t inl = 0;
        phase_mark(a.phase, it, PH_START);
        if constexpr (SHARDED) nn_search_grid_keep(a, T, state_xform_prev(&st), it, grid);
        else nn_search_grid(a, T, it, grid);
        phase_mark(a.phase, it, PH_COOP);
        lin_accumulate<REG, 1>(a, T, acc, inl);
        if (a.phase) {
            __syncthreads();
            phase_mark(a.phase, it, PH_ACC);
        }
        // block reduce -> this block's partial row
        for (int v = 0; v < N_ACC; ++v) {
            const float s = warp_sum(acc[v]);
            if (lane == 0) red[warp][v] = s;
        }
        {
            uint32_t c = inl;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
            if (lane == 0) red[warp][31] = __uint_as_float(c);
        }
        __syncthreads();
        double* part = a.partials + (size_t)(it & 1) * gridDim.x * 32;
        if (threadIdx.x < 32) {
            double s = 0.0;
            if (threadIdx.x < N_ACC) {
                for (int w = 0; w < LIN_WARPS; ++w) s += (double)red[w][threadIdx.x];
            } else if (threadIdx.x == S_INL) {
                for (int w = 0; w < LIN_WARPS; ++w) s += (double)__float_as_uint(red[w][31]);
            }
            __stcg(part + (size_t)blockIdx.x * 32 + threadIdx.x, s);
        }
        __threadfence();
        phase_mark(a.phase, it, PH_PART);
        grid.sync();
        phase_mark(a.phase, it, PH_SYNC);
        if (!SHARDED || blockIdx.x == 0) {
            const int v = threadIdx.x & 31, slice = threadIdx.x >> 5;
            double s = 0.0;
            for (unsigned b = slice; b < gridDim.x; b += LIN_WARPS) s += __ldcg(part + (size_t)b * 32 + v);
            fold[slice][v] = s;
            __syncthreads();
            if (threadIdx.x < 32) {
                double t = 0.0;
                for (int w = 0; w < LIN_WARPS; ++w) t += fold[w][threadIdx.x];
                fold[0][threadIdx.x] = t;
            }
            __syncthreads();
        }
        if (SHARDED) {
            const PeerX& x = a.px;
            // mailbox rows and flags are double-buffered by the parity of the GLOBAL row sequence number, which
            // runs on contiguously from one align to the next (the host advances it by the iterations actually
            // executed): a rank is never more than one exchange ahead of a peer, across aligns too
            const unsigned long long seq = x.seq0 + (unsigned long long)it;
            const int par = (int)(seq & 1ull);
            if (blockIdx.x == 0) {
                if (threadIdx.x < 32) {
                    const double v = fold[0][threadIdx.x];
                    for (int p = 0; p < x.world; ++p)
                        __stcg(x.rows[p] + ((size_t)par * SPX_MAX_RANKS + x.rank) * 32 + threadIdx.x, v);
                }
                __threadfence_system();
                __syncthreads();
                if ((int)threadIdx.x < x.world) {
                    st_release_sys(x.flags[threadIdx.x] + par * SPX_MAX_RANKS + x.rank, seq);
                    const unsigned long long* f = x.flags[x.rank] + par * SPX_MAX_RANKS + threadIdx.x;
                    const unsigned long long t0 = global_ns();
                    while (ld_acquire_sys(f) < seq) {
                        if (global_ns() - t0 > PEER_TIMEOUT_NS) {
                            atomicExch(x.error, 1u);
                            break;
                        }
                    }
                    __threadfence_system();
                }
                __syncthreads();
                if (threadIdx.x < 32) {
                    double t = 0.0;
                    for (int r = 0; r < x.world; ++r)
                        t += __ldcg(x.rows[x.rank] + ((size_t)par * SPX_MAX_RANKS + r) * 32 + threadIdx.x);
                    fold[0][threadIdx.x] = t;
                    __stcg(x.gsum + par * 32 + threadIdx.x, t);
                }
                __threadfence();
                __syncthreads();
                if (threadIdx.x == 0) st_release_gpu(x.ready + par, seq);
            } else {
                if (threadIdx.x == 0)
                    while (ld_acquire_gpu(x.ready + par) < seq) {
                    }
                __syncthreads();
                if (threadIdx.x < 32) fold[0][threadIdx.x] = __ldcg(x.gsum + par * 32 + threadIdx.x);
                __syncthreads();
            }
            if (__ldcg(x.error)) break;  // a peer went silent: every block leaves, the host reports it
        }
        phase_mark(a.phase, it, PH_FOLD);
        if (threadIdx.x == 0)
            gn_update(&st, &fold[0][0], a.lambda, a.crit_rot, a.crit_trans, it, blockIdx.x == 0 ? a.trace : nullptr);
        __syncthreads();
        phase_mark(a.phase, it, PH_SOLVE);
        if (st.stop) break;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *a.state = st;
}

// ------------------------------------------------------------------ batched Gauss-Newton align
// ONE cooperative launch aligns P independent scan pairs (P = 1: Registration::align, registration.hpp:201-276;
// P > 1: BASELINE config 5, SURVEY.md §8(e) "all pairs share launches via a pair-id segment key").
// The source points of all pairs are cut into CHUNKs of LIN_THREADS consecutive points of ONE pair; chunk c
// belongs to block c mod gridDim.x in every phase of every iteration.  A chunk's 28 sums are reduced by its
// block (fp32 per lane and warp, fp64 across the warps) into the chunk's own partial row, and a pair's rows are
// folded in chunk order: the sums of a pair — and therefore its poses, iteration counts and results — are a
// function of that pair's data alone, bit for bit the same whether it is aligned alone or inside any batch
// on any grid size.  Per-pair state (pose, flags) lives in global memory (RegState[P]); a pair that has
// converged is skipped by every phase.  Per iteration: first-pass search -> barrier -> work-list drain ->
// barrier -> factor pass + chunk rows -> barrier -> fold + 6x6 solve (P = 1: every block, redundantly, no
// further barrier; P > 1: pair p by block p mod gridDim.x, then a barrier).
constexpr int CHUNK = LIN_THREADS;
// resident CTAs per SM the persistent kernel is compiled for: the search phases are latency-bound and want warps,
// the factor pass wants registers.  Measured (B200): one pair of 120 k points 74 / 71 / 69 us per iteration at
// 2 / 3 / 4 CTAs, a batch of 64 pairs of 66 k points 2.56 / 2.19 / 2.31 ms.
constexpr int ALIGN_CTAS_SINGLE = 4, ALIGN_CTAS_BATCH = 3;

struct PairDesc {
    const float4* src_pts;
    const float4* src_cm;  // prepared matrices (GICP), 3 float4 per point
    const float4* tgt_pts;
    const float4* tgt_cm;  // GICP: regularised covariance; point-to-distribution: inverse(C_t)
    const float4* tgt_normals;
    int32_t* idx;          // [ns] correspondences of the current iteration (and the next one's warm start)
    float* dist;
    RegState* state;
    float* trace;          // [max_iterations][16] column-major poses, nullable
    uint32_t ns;
    uint32_t chunk0;       // first chunk of this pair
    uint32_t nchunks;
    float scale;           // robust scale of this pair (registration.hpp:217-218)
    GridLevels grid;       // the target's index
};

struct BatchArgs {
    const PairDesc* pairs;      // [n_pairs]
    const uint32_t* chunk_end;  // [n_pairs] chunk0 + nchunks, ascending: chunk -> pair lookup
    uint32_t n_pairs, total_chunks;
    float4* wl_q;               // work list: transformed query xyz, w = bits of the source index
    float4* wl_b;               //            best so far {dist, idx bits, -}, w = bits of the pair id
    unsigned int* wl_counters;  // [2 parities][count, cursor]
    double* partials;           // [2 parities][total_chunks][32]
    float max_corr, max_corr_sq;
    int loss;
    float lambda, crit_rot, crit_trans;
    unsigned long long* phase;
};

__device__ __forceinline__ uint32_t pair_of_chunk(const BatchArgs& a, uint32_t c) {
    uint32_t lo = 0, hi = a.n_pairs - 1;  // first pair whose chunk_end > c
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(a.chunk_end + mid) > c) hi = mid;
        else lo = mid + 1;
    }
    return lo;
}

// pose of a pair: P = 1 keeps it in shared memory; P > 1 reads what the pair's owner block wrote before the
// last grid barrier (L2: another SM's L1 may hold a stale line)
__device__ __forceinline__ Xform pose_ldcg(const RegState* st) {
    const float4* t = reinterpret_cast<const float4*>(&st->T[0][0]);
    Xform T;
    T.r0 = __ldcg(t);
    T.r1 = __ldcg(t + 1);
    T.r2 = __ldcg(t + 2);
    T.r3 = __ldcg(t + 3);
    return T;
}

template <int REG, int CTAS>
__global__ void __launch_bounds__(LIN_THREADS, CTAS) align_batch_kernel(const BatchArgs a, int max_iterations) {
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    __shared__ double fold[LIN_WARPS][32];
    __shared__ float red[LIN_WARPS][32];
    __shared__ RegState st1;  // P = 1: this block's copy of the optimiser state
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool single = a.n_pairs == 1;
    if (single) {
        if (threadIdx.x == 0) st1 = *a.pairs[0].state;
        __syncthreads();
    }
    for (int it = 0; it < max_iterations; ++it) {
        const int par = it & 1;
        const bool warm = it > 0;
        unsigned int* wl_count = a.wl_counters + par * 2;
        unsigned int* wl_cursor = a.wl_counters + par * 2 + 1;
        phase_mark(a.phase, it, PH_START);
        // ---- 1. first-pass search: one lane per source point
        for (uint32_t c = blockIdx.x; c < a.total_chunks; c += gridDim.x) {
            const uint32_t p = single ? 0u : pair_of_chunk(a, c);
            const PairDesc* d = a.pairs + p;
            const RegState* st = d->state;
            if (!single && __ldcg(&st->stop)) continue;  // block-uniform
            const Xform T = single ? state_xform(&st1) : pose_ldcg(st);
            const uint32_t ns = __ldg(&d->ns);
            const uint32_t i = (c - __ldg(&d->chunk0)) * CHUNK + threadIdx.x;
            bool pending = false;
            Best1 best;
            best.init();
            float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i < ns) {
                int32_t* idx = d->idx;
                float* dist = d->dist;
                // the two loads are independent: issued together, one round trip instead of two
                const float4 ps = __ldg(d->src_pts + i);
                const int prev_i = warm ? __ldcg(idx + i) : -1;
                q = transform_point(T, ps);
                if (__ldg(&d->grid.lv[0].n) > 0 && isfinite(q.x) && isfinite(q.y) && isfinite(q.z))
                    pending = !icp_fast(d->grid, q.x, q.y, q.z, prev_i, d->tgt_pts, a.max_corr, best);
                idx[i] = best.i;
                dist[i] = best.d;
            }
            const unsigned m = __ballot_sync(FULL, pending);  // warp-aggregated append
            if (m) {
                unsigned int slot = 0;
                if (lane == __ffs(m) - 1) slot = atomicAdd(wl_count, (unsigned int)__popc(m));
                slot = __shfl_sync(FULL, slot, __ffs(m) - 1);
                if (pending) {
                    const unsigned int w = slot + __popc(m & ((1u << lane) - 1u));
                    a.wl_q[w] = make_float4(q.x, q.y, q.z, __uint_as_float(i));
                    a.wl_b[w] = make_float4(best.d, __int_as_float(best.i), 0.0f, __uint_as_float(p));
                }
            }
        }
        phase_mark(a.phase, it, PH_NN);
        __threadfence();
        grid.sync();
        if (blockIdx.x == 0 && threadIdx.x == 0) {  // the other parity's counters: idle until the next iteration
            a.wl_counters[(par ^ 1) * 2] = 0;
            a.wl_counters[(par ^ 1) * 2 + 1] = 0;
        }
        // ---- 2. the queries the first pass could not certify: one per warp, drained by the whole grid
        {
            const unsigned int n_slow = __ldcg(wl_count);
            for (;;) {
                unsigned int k = 0;
                if (lane == 0) k = atomicAdd(wl_cursor, 1u);
                k = __shfl_sync(FULL, k, 0);
                if (k >= n_slow) break;
                const float4 qv = __ldcg(a.wl_q + k);
                const float4 bv = __ldcg(a.wl_b + k);
                const PairDesc* d = a.pairs + __float_as_uint(bv.w);
                const uint32_t i = __float_as_uint(qv.w);
                Best1 best;
                best.d = bv.x;
                best.i = __float_as_int(bv.y);
                icp_coop_search(d->grid, qv.x, qv.y, qv.z, best, a.max_corr);
                if (lane == 0) {
                    d->idx[i] = best.i;
                    d->dist[i] = best.d;
                    // tuning aid: {list size, list queries that end without a neighbour inside max_corr} per iteration
                    if (a.phase && it < PH_MAX_ITERS) {
                        unsigned long long* w = a.phase + PH_MAX_ITERS * PH_N + it * 2;
                        if (k == 0) w[0] = n_slow;
                        if (!(best.d <= a.max_corr * a.max_corr)) atomicAdd(w + 1, 1ull);
                    }
                }
            }
        }
        __threadfence();
        grid.sync();
        phase_mark(a.phase, it, PH_COOP);
        // ---- 3. factor pass: one correspondence per lane, one partial row per chunk
        double* part = a.partials + (size_t)par * a.total_chunks * 32;
        for (uint32_t c = blockIdx.x; c < a.total_chunks; c += gridDim.x) {
            const uint32_t p = single ? 0u : pair_of_chunk(a, c);
            const PairDesc* d = a.pairs + p;
            const RegState* st = d->state;
            if (!single && __ldcg(&st->stop)) continue;
            const Xform T = single ? state_xform(&st1) : pose_ldcg(st);
            const uint32_t i = (c - __ldg(&d->chunk0)) * CHUNK + threadIdx.x;
            float acc[N_ACC];
#pragma unroll
            for (int v = 0; v < N_ACC; ++v) acc[v] = 0.0f;
            uint32_t inl = 0;
            if (i < __ldg(&d->ns)) {
                const float dd = __ldcg(d->dist + i);
                const int ti = __ldcg(d->idx + i);
                if (!(dd > a.max_corr_sq || ti < 0)) {  // registration.hpp:584 (+ guard for the -1 fill)
                    const float4 ps = __ldg(d->src_pts + i);
                    const float4 pt = __ldg(d->tgt_pts + ti);
                    const float4* nrm_p = d->tgt_normals;
                    const float4 nrm = (REG == SPX_REG_POINT_TO_PLANE && nrm_p) ? __ldg(nrm_p + ti) : make_float4(0.f, 0.f, 0.f, 0.f);
                    Mat3 cs, ct;
                    if (REG == SPX_REG_GICP) cs = load_mat(d->src_cm, i);
                    if (REG == SPX_REG_GICP || REG == SPX_REG_POINT_TO_DISTRIBUTION) ct = load_mat(d->tgt_cm, (size_t)ti);
                    accumulate_point<REG>(T, ps, cs, pt, ct, nrm, a.loss, __ldg(&d->scale), acc);
                    inl = 1;
                }
            }
            for (int v = 0; v < N_ACC; ++v) {
                const float s = warp_sum(acc[v]);
                if (lane == 0) red[warp][v] = s;
            }
            {
                const unsigned c1 = __popc(__ballot_sync(FULL, inl != 0));
                if (lane == 0) red[warp][31] = __uint_as_float(c1);
            }
            __syncthreads();
            if (threadIdx.x < 32) {
                double s = 0.0;
                if (threadIdx.x < N_ACC) {
                    for (int w = 0; w < LIN_WARPS; ++w) s += (double)red[w][threadIdx.x];
                } else if (threadIdx.x == S_INL) {
                    for (int w = 0; w < LIN_WARPS; ++w) s += (double)__float_as_uint(red[w][31]);
                }
                __stcg(part + (size_t)c * 32 + threadIdx.x, s);
            }
            __syncthreads();
        }
        __threadfence();
        phase_mark(a.phase, it, PH_PART);
        grid.sync();
        phase_mark(a.phase, it, PH_SYNC);
        // ---- 4. fold a pair's rows in chunk order, solve, advance its pose
        if (single) {
            const PairDesc* d = a.pairs;
            {
                const int v = threadIdx.x & 31, slice = threadIdx.x >> 5;
                double s = 0.0;
                for (uint32_t b = slice; b < a.total_chunks; b += LIN_WARPS) s += __ldcg(part + (size_t)b * 32 + v);
                fold[slice][v] = s;
            }
            __syncthreads();
            if (threadIdx.x < 32) {
                double t = 0.0;
                for (int w = 0; w < LIN_WARPS; ++w) t += fold[w][threadIdx.x];
                fold[0][threadIdx.x] = t;
            }
            __syncthreads();
            phase_mark(a.phase, it, PH_FOLD);
            if (threadIdx.x == 0)
                gn_update(&st1, &fold[0][0], a.lambda, a.crit_rot, a.crit_trans, it, blockIdx.x == 0 ? d->trace : nullptr);
            __syncthreads();
            phase_mark(a.phase, it, PH_SOLVE);
            if (st1.stop) break;
        } else {
            for (uint32_t p = blockIdx.x; p < a.n_pairs; p += gridDim.x) {
                const PairDesc* d = a.pairs + p;
                RegState* st = d->state;
                if (st->stop) continue;  // written by this block only
                const uint32_t c0 = __ldg(&d->chunk0), nc = __ldg(&d->nchunks);
                {
                    const int v = threadIdx.x & 31, slice = threadIdx.x >> 5;
                    double s = 0.0;
                    for (uint32_t b = slice; b < nc; b += LIN_WARPS) s += __ldcg(part + (size_t)(c0 + b) * 32 + v);
                    fold[slice][v] = s;
                }
                __syncthreads();
                if (threadIdx.x < 32) {
                    double t = 0.0;
                    for (int w = 0; w < LIN_WARPS; ++w) t += fold[w][threadIdx.x];
                    fold[0][threadIdx.x] = t;
                }
                __syncthreads();
                if (threadIdx.x == 0) gn_update(st, &fold[0][0], a.lambda, a.crit_rot, a.crit_trans, it, d->trace);
                __syncthreads();
            }
            __threadfence();
            phase_mark(a.phase, it, PH_FOLD);
            grid.sync();
            phase_mark(a.phase, it, PH_SOLVE);
            int active = 0;
            for (uint32_t p = threadIdx.x; p < a.n_pairs; p += LIN_THREADS)
                active |= !__ldcg(&a.pairs[p].state->stop);
            if (!__syncthreads_or(active)) break;
        }
    }
    if (single && blockIdx.x == 0 && threadIdx.x == 0) *a.pairs[0].state = st1;
}

// error-only pass with frozen neighbours — registration.hpp:678-777; WEIGHTS: per-point robust
// weights instead of the sum (registration.hpp:412-462)
template <int REG, bool WEIGHTS>
__global__ void __launch_bounds__(LIN_THREADS, 2) error_kernel(const LinArgs a) {
    __shared__ double fold[LIN_WARPS][32];
    __shared__ float red[LIN_WARPS][32];
    const Xform T = a.T;
    float acc[1] = {0.0f};
    uint32_t inl = 0;
    // GenZ: the error sum weights every term by alpha / 1 - alpha (registration.hpp:749-753); the weights export does not (:449)
    const float alpha = (REG == SPX_REG_GENZ && !WEIGHTS) ? genz_alpha(a) : 1.0f;
    for (uint32_t i = blockIdx.x * LIN_THREADS + threadIdx.x; i < a.ns; i += gridDim.x * LIN_THREADS) {
        const float d = __ldg(a.dist_in + i);
        const int ti = __ldg(a.idx_in + i);
        float w = 0.0f;
        if (!(d > a.max_corr_sq || ti < 0)) {
            const float4 ps = __ldg(a.src_pts + i);
            const float4 pt = __ldg(a.tgt_pts + ti);
            const float4 nrm = ((REG == SPX_REG_POINT_TO_PLANE || REG == SPX_REG_GENZ) && a.tgt_normals)
                                   ? __ldg(a.tgt_normals + ti)
                                   : make_float4(0.f, 0.f, 0.f, 0.f);
            Mat3 cs, ct;
            load_covs<REG>(a, i, ti, cs, ct);
            const bool planar = REG == SPX_REG_GENZ ? genz_planar(ct, a.genz_threshold) : false;
            const float rn = __fsqrt_rn(point_error<REG>(T, ps, cs, pt, ct, nrm, planar));
            if (WEIGHTS) {
                w = robust_weight(a.loss, rn, a.scale);
            } else {
                const float rho = robust_error(a.loss, rn, a.scale);
                acc[0] = __fadd_rn(acc[0], REG == SPX_REG_GENZ ? __fmul_rn(planar ? alpha : __fsub_rn(1.0f, alpha), rho) : rho);
                if (a.rot_enable) {  // registration.hpp:757-764
                    float g[3];
                    const float D = rot_divergence(T, a.src_cov16 ? load_cov16(a.src_cov16 + (size_t)i * 16) : mat3_identity(),
                                                   a.tgt_cov16 ? load_cov16(a.tgt_cov16 + (size_t)ti * 16) : mat3_identity(), g, false);
                    const float rr = __fsqrt_rn(__fmul_rn(__fmul_rn(0.5f, D), D));
                    acc[0] = __fadd_rn(acc[0], __fmul_rn(a.rot_weight, robust_error(a.loss, rr, a.rot_scale)));
                }
                ++inl;
            }
        }
        if (WEIGHTS) a.weights_out[i] = w;
    }
    if (WEIGHTS) return;
    reduce_to_sums(acc, 1, inl, a.partials, a.ticket, a.sums_out, fold, red);
}

// stand-alone update for the sharded path: sums were all-reduced across ranks by the caller
__global__ void gn_update_kernel(RegState* st, const double* sums, float lambda, float crit_rot, float crit_trans,
                                 int iter_index, float* trace) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    if (st->stop) return;
    gn_update(st, sums, lambda, crit_rot, crit_trans, iter_index, trace);
}

// Everything an align needs before its first iteration, in ONE launch: the pose-independent
// per-point matrices of both clouds (16-float reference covariance -> plane-regularised 6 floats, or
// the inverse for point-to-distribution), the optimiser state, and the zeroed work-list counters and
// ticket.  Written on the device — a small H2D copy would queue behind another queue's bulk upload on
// the copy engine, and five separate stream operations cost ~20 us of launch gaps per align.
struct PrepArgs {
    const float* src_cov16;
    uint32_t ns;  // 0: the source needs no matrices
    float4* src_cm;
    const float* tgt_cov16;
    uint32_t nt;  // 0: the target needs no matrices
    float4* tgt_cm;
    int invert_tgt;
    RegState* state;
    Xform T;
    unsigned int* wl_counters;
    unsigned int* ticket;
};
__global__ void __launch_bounds__(128) align_prepare_kernel(PrepArgs p) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        RegState s;
        memset(&s, 0, sizeof(s));
        const float4 r[4] = {p.T.r0, p.T.r1, p.T.r2, p.T.r3};
        for (int i = 0; i < 4; ++i) {
            s.T[i][0] = r[i].x; s.T[i][1] = r[i].y; s.T[i][2] = r[i].z; s.T[i][3] = r[i].w;
        }
        s.error = FLT_MAX;
        *p.state = s;
        for (int i = 0; i < 6; ++i) p.wl_counters[i] = 0u;
        p.wl_counters[WL_KEPT] = 0u;
        *p.ticket = 0u;
    }
    uint32_t i = blockIdx.x * 128 + threadIdx.x;
    const float* cov16 = p.src_cov16;
    float4* cm = p.src_cm;
    bool invert = false;
    if (i >= p.ns) {
        i -= p.ns;
        if (i >= p.nt) return;
        cov16 = p.tgt_cov16;
        cm = p.tgt_cm;
        invert = p.invert_tgt != 0;
    }
    const Mat3 raw = cov16 ? load_cov16(cov16 + (size_t)i * 16) : mat3_identity();
    store_mat(cm, i, invert ? mat3_inverse(raw) : plane_regularize(raw));  // invert: point-to-distribution
}

// set-up of the batched align: per pair, the pose-independent matrices of both clouds, the optimiser state and
// the pair's row of the descriptor table; block (0, 0) also zeroes the work-list counters.  P = 1 receives its
// PairPrep as a kernel parameter (no H2D copy in front of the align: DESIGN.md §3 K-prep), P > 1 reads a table.
struct PairPrep {
    const float* src_cov16;
    const float* tgt_cov16;
    uint32_t n_src_m;  // source matrices to prepare (0: none)
    uint32_t n_tgt_m;  // target matrices to prepare
    float4* src_cm;
    float4* tgt_cm;
    int invert_tgt;
    int pad;
    Xform T;
    PairDesc desc;
};
__global__ void __launch_bounds__(128) align_prepare_batch_kernel(const PairPrep* __restrict__ table, const PairPrep one,
                                                                  PairDesc* descs, uint32_t* chunk_end,
                                                                  unsigned int* wl_counters) {
    const PairPrep& pp = table ? table[blockIdx.y] : one;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        RegState s;
        memset(&s, 0, sizeof(s));
        const float4 r[4] = {pp.T.r0, pp.T.r1, pp.T.r2, pp.T.r3};
        for (int i = 0; i < 4; ++i) {
            s.T[i][0] = r[i].x; s.T[i][1] = r[i].y; s.T[i][2] = r[i].z; s.T[i][3] = r[i].w;
        }
        s.error = FLT_MAX;
        *pp.desc.state = s;
        descs[blockIdx.y] = pp.desc;
        chunk_end[blockIdx.y] = pp.desc.chunk0 + pp.desc.nchunks;
        if (blockIdx.y == 0)
            for (int i = 0; i < 4; ++i) wl_counters[i] = 0u;
    }
    uint32_t i = blockIdx.x * 128 + threadIdx.x;
    const float* cov16 = pp.src_cov16;
    float4* cm = pp.src_cm;
    bool invert = false;
    if (i >= pp.n_src_m) {
        i -= pp.n_src_m;
        if (i >= pp.n_tgt_m) return;
        cov16 = pp.tgt_cov16;
        cm = pp.tgt_cm;
        invert = pp.invert_tgt != 0;
    }
    const Mat3 raw = cov16 ? load_cov16(cov16 + (size_t)i * 16) : mat3_identity();
    store_mat(cm, i, invert ? mat3_inverse(raw) : plane_regularize(raw));
}

template <int REG, int MODE, bool SOLVE>
void launch_linearize_one(const LinArgs& a, unsigned blocks, cudaStream_t st, int sm_count) {
    if (MODE == 1) {
        // the fused correspondence search synchronises the grid: cooperative launch, one resident wave
        static int per_sm = 0;  // queried once per variant
        if (per_sm == 0)
            SPX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, linearize_kernel<REG, MODE, SOLVE>, LIN_THREADS, 0));
        blocks = std::max(1u, std::min(blocks, (unsigned)std::max(per_sm, 1) * (unsigned)sm_count));
        void* args[] = {(void*)&a};
        SPX_CUDA(cudaLaunchCooperativeKernel((const void*)linearize_kernel<REG, MODE, SOLVE>, dim3(blocks), dim3(LIN_THREADS),
                                             args, 0, st));
    } else {
        linearize_kernel<REG, MODE, SOLVE><<<blocks, LIN_THREADS, 0, st>>>(a);
    }
}

template <int MODE, bool SOLVE>
void launch_linearize(int reg, const LinArgs& a, unsigned blocks, cudaStream_t st, int sm_count = 148) {
    switch (reg) {
        case SPX_REG_POINT_TO_POINT: launch_linearize_one<SPX_REG_POINT_TO_POINT, MODE, SOLVE>(a, blocks, st, sm_count); break;
        case SPX_REG_POINT_TO_PLANE: launch_linearize_one<SPX_REG_POINT_TO_PLANE, MODE, SOLVE>(a, blocks, st, sm_count); break;
        case SPX_REG_POINT_TO_DISTRIBUTION:
            launch_linearize_one<SPX_REG_POINT_TO_DISTRIBUTION, MODE, SOLVE>(a, blocks, st, sm_count);
            break;
        case SPX_REG_GENZ:
            // alpha needs the counts of the correspondences: MODE 1 counts inside the kernel (after its search), MODE 0
            // (correspondences given) by a launch in front
            SPX_CUDA(cudaMemsetAsync(a.genz_counts, 0, 2 * sizeof(unsigned int), st));
            if (MODE == 0) {
                genz_count_kernel<<<blocks, LIN_THREADS, 0, st>>>(a);
                SPX_LAUNCH_CHECK();
            }
            launch_linearize_one<SPX_REG_GENZ, MODE, SOLVE>(a, blocks, st, sm_count);
            break;
        default: launch_linearize_one<SPX_REG_GICP, MODE, SOLVE>(a, blocks, st, sm_count); break;
    }
    SPX_LAUNCH_CHECK();
}

template <bool WEIGHTS>
void launch_error(int reg, const LinArgs& a, unsigned blocks, cudaStream_t st) {
    switch (reg) {
        case SPX_REG_POINT_TO_POINT: error_kernel<SPX_REG_POINT_TO_POINT, WEIGHTS><<<blocks, LIN_THREADS, 0, st>>>(a); break;
        case SPX_REG_POINT_TO_PLANE: error_kernel<SPX_REG_POINT_TO_PLANE, WEIGHTS><<<blocks, LIN_THREADS, 0, st>>>(a); break;
        case SPX_REG_POINT_TO_DISTRIBUTION:
            error_kernel<SPX_REG_POINT_TO_DISTRIBUTION, WEIGHTS><<<blocks, LIN_THREADS, 0, st>>>(a);
            break;
        case SPX_REG_GENZ:
            if (!WEIGHTS) {  // alpha of the frozen correspondences (what the linearisation on them stored, registration.hpp:370)
                SPX_CUDA(cudaMemsetAsync(a.genz_counts, 0, 2 * sizeof(unsigned int), st));
                genz_count_kernel<<<std::min(blocks, 1024u), LIN_THREADS, 0, st>>>(a);
                SPX_LAUNCH_CHECK();
            }
            error_kernel<SPX_REG_GENZ, WEIGHTS><<<blocks, LIN_THREADS, 0, st>>>(a);
            break;
        default: error_kernel<SPX_REG_GICP, WEIGHTS><<<blocks, LIN_THREADS, 0, st>>>(a); break;
    }
    SPX_LAUNCH_CHECK();
}

template <int REG, bool SHARDED>
unsigned coop_blocks(int device_sm_count) {
    static int per_sm = 0;  // same on every device this library targets (sm_100a); queried once per variant
    if (per_sm == 0)
        SPX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, align_gn_kernel<REG, SHARDED>, LIN_THREADS, 0));
    return (unsigned)std::max(per_sm, 1) * (unsigned)device_sm_count;
}

void check_reg_loss(int reg, int loss, const char* where) {
    (void)where;
    if (!(reg == SPX_REG_POINT_TO_POINT || reg == SPX_REG_POINT_TO_PLANE || reg == SPX_REG_GICP ||
          reg == SPX_REG_POINT_TO_DISTRIBUTION || reg == SPX_REG_GENZ))
        throw Error(SPX_ERR_INVALID_ARGUMENT, "[Registration::dispatch] Combination not found in tags!");
    if (loss < SPX_LOSS_NONE || loss > SPX_LOSS_GEMAN_MCCLURE)
        throw Error(SPX_ERR_INVALID_ARGUMENT, "[Registration::dispatch] Combination not found in tags!");
}

unsigned lin_blocks(spx_queue_t q, size_t ns) {
    const unsigned need = (unsigned)div_up(ns, LIN_THREADS);
    const unsigned cap = (unsigned)q->sm_count * 2;  // one resident wave (2 CTAs per SM), grid-stride beyond
    return std::max(1u, std::min(need, cap));
}

void sums_to_host(const double* s, float* H, float* b, float* err, uint32_t* inl) {
    int t = 0;
    for (int a = 0; a < 6; ++a)
        for (int c = a; c < 6; ++c) {
            const float v = (float)s[t++];
            H[a * 6 + c] = v;
            H[c * 6 + a] = v;
        }
    for (int a = 0; a < 6; ++a) b[a] = (float)s[S_B + a];
    *err = (float)s[S_ERR];
    *inl = (uint32_t)(s[S_INL] + 0.5);
}

}  // namespace

// ------------------------------------------------------------------ handle
struct spx_registration_s {
    spx_queue_t q = nullptr;
    spx_registration_params P{};
    RegState* state = nullptr;       // device
    double* partials = nullptr;      // device [max_blocks][32]
    unsigned max_blocks = 0;
    unsigned int* ticket = nullptr;  // device
    double* sums = nullptr;          // device [32]
    int32_t* nn_idx = nullptr;
    float* nn_dist = nullptr;
    uint32_t* worklist = nullptr;
    uint32_t* keep_buf = nullptr;  // split-kernel loop: [ns] allowances (float) + [ns] redo list
    size_t keep_cap = 0;
    unsigned int* wl_counters = nullptr;
    size_t nn_cap = 0;
    float4* src_cm = nullptr;  // [3 * src_cap]
    size_t src_cap = 0;
    float4* tgt_cm = nullptr;
    size_t tgt_cap = 0;
    // batched Gauss-Newton align (P = 1: the single-pair path)
    RegState* states = nullptr;   // [pairs_cap] (P > 1; P = 1 uses `state`)
    PairDesc* descs = nullptr;    // [pairs_cap]
    uint32_t* chunk_end = nullptr;
    PairPrep* preps = nullptr;    // [pairs_cap] device copy of the set-up table
    size_t pairs_cap = 0;
    float4* wl_q = nullptr;       // [wl_cap]
    float4* wl_b = nullptr;
    size_t wl_cap = 0;
    double* cpartials = nullptr;  // [2][cpart_cap][32]
    size_t cpart_cap = 0;
    float* trace = nullptr;
    size_t trace_cap = 0;
    size_t nn_n = 0;
    // sharded / staged context
    LinArgs shard{};
    int shard_reg = 0;
    int shard_iter = 0;
    bool shard_active = false;
    unsigned long long* phase = nullptr;  // [PH_MAX_ITERS][PH_N], allocated by spx_registration_phase_times(enable)
    spx_comm_t shard_comm = nullptr;  // fused (mailbox) sharded align in flight
    float4* shard_derived_normals = nullptr;
    int shard_max_it = 0;
    // solver add-ons (host side): nl-reg parameters and the MAP prior of the next align
    spx_registration_addons addons{0, 10.0f, 1.0f, 1.0f, 0, 1.0f, 1.0f, 3.16e-2f, 1e-2f};
    bool prior_active = false;
    float prior_omega[36] = {};
    float prior_T_pred_inv[4][4] = {};
    // live timing of the iteration kernels (bench.py roofline)
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    int last_launches = 0;
    int last_iterations = 0;
    bool timed = false;
};

namespace {

void reg_free(spx_registration_t r) {
    auto f = [](auto*& p) {
        if (p) cudaFree(p);
        p = nullptr;
    };
    f(r->state); f(r->partials); f(r->ticket); f(r->sums); f(r->nn_idx); f(r->nn_dist); f(r->worklist); f(r->keep_buf); f(r->wl_counters);
    f(r->src_cm); f(r->tgt_cm); f(r->states); f(r->descs); f(r->chunk_end); f(r->preps); f(r->wl_q); f(r->wl_b); f(r->cpartials); f(r->trace); f(r->phase);
    if (r->ev0) cudaEventDestroy(r->ev0);
    if (r->ev1) cudaEventDestroy(r->ev1);
    r->ev0 = r->ev1 = nullptr;
}

template <typename T>
void ensure(T*& p, size_t& cap, size_t need, cudaStream_t st) {
    if (need <= cap && p) return;
    if (p) {
        SPX_CUDA(cudaStreamSynchronize(st));
        SPX_CUDA(cudaFree(p));
        p = nullptr;
    }
    const size_t c = std::max<size_t>(need, 1024);
    SPX_CUDA(cudaMalloc(&p, c * sizeof(T)));
    cap = c;
}

// prepared matrices: 3 float4 per point
void ensure3(float4*& p, size_t& cap, size_t need, cudaStream_t st) {
    if (need <= cap && p) return;
    if (p) {
        SPX_CUDA(cudaStreamSynchronize(st));
        SPX_CUDA(cudaFree(p));
        p = nullptr;
    }
    const size_t c = std::max<size_t>(need, 1024);
    SPX_CUDA(cudaMalloc(&p, c * 3 * sizeof(float4)));
    cap = c;
}

// reference validate_params — registration.hpp:129-193
void validate(const spx_registration_params& P, const float* src_covs, const float* tgt_covs,
              const float* tgt_normals) {
    if (P.reg_type == SPX_REG_POINT_TO_PLANE && !tgt_normals && !tgt_covs)
        throw Error(SPX_ERR_INVALID_ARGUMENT,
                    "[Registration::validate_params] Normal vector or covariance matrices of target must be "
                    "pre-computed before performing Point-to-Plane ICP matching.");
    if (P.reg_type == SPX_REG_GICP && (!src_covs || !tgt_covs))
        throw Error(SPX_ERR_INVALID_ARGUMENT,
                    "[Registration::validate_params] Covariance matrices of source and target must be pre-computed "
                    "before performing GICP matching.");
    if (P.reg_type == SPX_REG_GENZ && !tgt_covs)
        throw Error(SPX_ERR_INVALID_ARGUMENT,
                    "[Registration::validate_params] Covariance matrices of target must be pre-computed before "
                    "performing GenZ-ICP matching.");
    if (P.rotation_constraint_enable && !src_covs)
        throw Error(SPX_ERR_INVALID_ARGUMENT,
                    "[Registration::validate_params] Covariance matrices of source are required for performing rotation "
                    "constraint matching.");
    if (P.rotation_constraint_enable && !tgt_covs)
        throw Error(SPX_ERR_INVALID_ARGUMENT,
                    "[Registration::validate_params] Covariance matrices of target are required for performing rotation "
                    "constraint matching.");
    if (P.reg_type == SPX_REG_POINT_TO_DISTRIBUTION && !tgt_covs)
        throw Error(SPX_ERR_INVALID_ARGUMENT,
                    "[Registration::validate_params] Covariance matrices of target must be pre-computed before "
                    "performing Point-to-Distribution ICP matching.");
}

struct AlignCtx {
    LinArgs a;
    int reg;
    unsigned blocks;
};

// shared set-up of align / shard_begin: scratch, covariance preparation, initial state upload
AlignCtx align_setup(spx_registration_t r, const float* src_points, const float* src_covs, size_t ns,
                     const float* tgt_points, const float* tgt_covs, const float* tgt_normals, size_t nt,
                     spx_index_t index, const float* T_init_host, float robust_scale, float4** derived_normals) {
    spx_queue_t q = r->q;
    cudaStream_t st = q->stream;
    spx_registration_params& P = r->P;
    SPX_REQUIRE(index, "[Registration::align] target_knn (spx_index) is null");
    SPX_REQUIRE(index->q->device == q->device, "[Registration::align] index lives on another device");
    SPX_REQUIRE(index->n_total == nt, "[Registration::align] target_knn was built on a different cloud size");
    if (index->q != q && index->ready) SPX_CUDA(cudaStreamWaitEvent(st, index->ready, 0));  // built on another queue
    SPX_REQUIRE(ns < (1ull << 31) && nt < (1ull << 31), "[Registration::align] too many points");
    check_reg_loss(P.reg_type, P.robust_loss, "[Registration::align]");
    validate(P, src_covs, tgt_covs, tgt_normals);
    int loss = P.robust_loss;
    if (loss != SPX_LOSS_NONE && P.robust_default_scale <= 0.0f) loss = SPX_LOSS_NONE;  // registration.hpp:186-192

    size_t cap_dummy = r->nn_cap;
    ensure(r->nn_idx, cap_dummy, ns, st);
    cap_dummy = r->nn_cap;
    ensure(r->worklist, cap_dummy, ns, st);
    ensure(r->nn_dist, r->nn_cap, ns, st);
    r->nn_n = ns;
    size_t tcap = r->trace_cap;
    ensure(r->trace, tcap, (size_t)std::max(P.max_iterations, 1) * 16, st);
    r->trace_cap = tcap;

    AlignCtx c;
    c.reg = P.reg_type;
    c.blocks = lin_blocks(q, ns);
    if (c.blocks > r->max_blocks) {
        if (r->partials) {
            SPX_CUDA(cudaStreamSynchronize(st));
            SPX_CUDA(cudaFree(r->partials));
        }
        r->max_blocks = std::max(c.blocks, (unsigned)q->sm_count * 4);
        SPX_CUDA(cudaMalloc(&r->partials, (size_t)r->max_blocks * 32 * sizeof(double)));
    }
    LinArgs& a = c.a;
    std::memset(&a, 0, sizeof(a));
    PrepArgs prep;
    std::memset(&prep, 0, sizeof(prep));
    a.src_pts = reinterpret_cast<const float4*>(src_points);
    a.ns = (uint32_t)ns;
    a.tgt_pts = reinterpret_cast<const float4*>(tgt_points);
    a.tgt_normals = reinterpret_cast<const float4*>(tgt_normals);
    if (P.reg_type == SPX_REG_GICP || P.reg_type == SPX_REG_POINT_TO_DISTRIBUTION) {
        // pose-independent per-point matrices, prepared once per align: GICP = plane-regularised
        // covariances of both clouds; point-to-distribution = inverse of the raw target covariance
        const bool gicp = P.reg_type == SPX_REG_GICP;
        if (gicp) ensure3(r->src_cm, r->src_cap, ns, st);
        ensure3(r->tgt_cm, r->tgt_cap, nt, st);
        prep.src_cov16 = src_covs;
        prep.ns = gicp ? (uint32_t)ns : 0u;
        prep.src_cm = r->src_cm;
        prep.tgt_cov16 = tgt_covs;
        prep.nt = (uint32_t)nt;
        prep.tgt_cm = r->tgt_cm;
        prep.invert_tgt = gicp ? 0 : 1;
        if (gicp) a.src_cm = r->src_cm;
        a.tgt_cm = r->tgt_cm;
    }
    if ((P.reg_type == SPX_REG_POINT_TO_PLANE || P.reg_type == SPX_REG_GENZ) && !tgt_normals) {
        // registration.hpp:139-141,157-164: normals derived from the pre-computed covariances
        fprintf(stdout, "[Caution] Normal vectors for %s are not provided. \n"
                        "          Attempting to derive them from pre-computed covariance matrices.\n",
                P.reg_type == SPX_REG_GENZ ? "GenZ-ICP" : "Point-to-Plane ICP");
        float4* nrm = nullptr;
        SPX_CUDA(cudaMalloc(&nrm, std::max<size_t>(nt, 1) * sizeof(float4)));
        *derived_normals = nrm;
        if (spx_normals_from_covs(q, tgt_points, tgt_covs, nt, reinterpret_cast<float*>(nrm)) != SPX_OK)
            throw Error(SPX_ERR_INTERNAL, spx_last_error());
        a.tgt_normals = nrm;
    }
    if (P.reg_type == SPX_REG_GENZ) a.tgt_cov16 = tgt_covs;  // the raw target covariance classifies planar / non-planar
    if (P.rotation_constraint_enable) {  // the rotation-constraint term reads the RAW covariances of both clouds
        a.src_cov16 = src_covs;
        a.tgt_cov16 = tgt_covs;
        a.rot_enable = 1;
        a.rot_weight = P.rotation_constraint_weight;
        a.rot_scale = P.rotation_constraint_robust_scale > 0.0f ? P.rotation_constraint_robust_scale : 10.0f;
    }
    a.genz_threshold = P.genz_planarity_threshold > 0.0f ? P.genz_planarity_threshold : 0.2f;
    a.genz_counts = r->wl_counters + 8;
    a.idx_in = r->nn_idx; a.dist_in = r->nn_dist;
    a.idx_out = r->nn_idx; a.dist_out = r->nn_dist;
    a.slack_out = nullptr;
    a.redo = nullptr;
    a.keep_infl = 0.0f;
    a.keep_last = 0;
    a.warm_start = 0;
    a.worklist = r->worklist;
    a.wl_counters = r->wl_counters;
    a.grid = index->levels;
    a.state = r->state;
    a.use_state = 1;
    a.T = xform_identity();
    a.max_corr = P.max_correspondence_distance;
    a.max_corr_sq = P.max_correspondence_distance * P.max_correspondence_distance;
    a.scale = robust_scale > 0.0f ? robust_scale : P.robust_default_scale;  // registration.hpp:217-218
    a.loss = loss;
    a.partials = r->partials;
    a.ticket = r->ticket;
    a.sums_out = r->sums;
    a.lambda = P.gn_lambda;
    a.crit_rot = P.criteria_rotation;
    a.crit_trans = P.criteria_translation;
    a.trace = r->trace;
    a.phase = r->phase;
    if (r->phase) SPX_CUDA(cudaMemsetAsync(r->phase, 0, PH_WORDS * sizeof(unsigned long long), st));

    {
        const float I16[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
        prep.state = r->state;
        prep.T = xform_from_colmajor(T_init_host ? T_init_host : I16);
        prep.wl_counters = r->wl_counters;
        prep.ticket = r->ticket;
        align_prepare_kernel<<<std::max<unsigned>(1u, (unsigned)div_up((size_t)prep.ns + prep.nt, 128)), 128, 0, st>>>(prep);
        SPX_LAUNCH_CHECK();
    }
    return c;
}

void fill_result(const RegState& s, spx_registration_result* R) {
    for (int j = 0; j < 4; ++j)
        for (int i = 0; i < 4; ++i) R->T[j * 4 + i] = s.T[i][j];
    R->converged = s.converged;
    R->iterations = s.iterations;
    std::memcpy(R->H, s.H, sizeof(R->H));
    std::memcpy(R->b, s.b, sizeof(R->b));
    R->error = s.error;
    std::memcpy(R->H_raw, s.H, sizeof(R->H));
    std::memcpy(R->b_raw, s.b, sizeof(R->b));
    R->error_raw = s.error;
    R->inlier = s.inlier;
}

void host_T_to_xform(const float T[4][4], Xform& x) {
    x.r0 = make_float4(T[0][0], T[0][1], T[0][2], T[0][3]);
    x.r1 = make_float4(T[1][0], T[1][1], T[1][2], T[1][3]);
    x.r2 = make_float4(T[2][0], T[2][1], T[2][2], T[2][3]);
    x.r3 = make_float4(T[3][0], T[3][1], T[3][2], T[3][3]);
}

// dogleg_step.hpp:34-102 on the host (N = 6)
void dogleg_host(const float* H, const float* g, float radius, float* p, float* step_norm, float* pred) {
    float p_gn[6] = {0}, n_gn = 0.0f;
    bool valid_gn = false;
    {
        double A[6][6], rhs[6], x[6];
        for (int i = 0; i < 6; ++i) {
            for (int j = 0; j < 6; ++j) A[i][j] = (double)H[i * 6 + j];
            rhs[i] = -(double)g[i];
        }
        Ldlt6 f;
        ldlt6_compute(A, f);
        double mind = f.D[0];
        for (int i = 1; i < 6; ++i) mind = std::min(mind, f.D[i]);
        if (f.ok && mind > 0.0) {
            ldlt6_solve(f, rhs, x);
            float s = 0.0f;
            for (int i = 0; i < 6; ++i) {
                p_gn[i] = (float)x[i];
                s += p_gn[i] * p_gn[i];
            }
            n_gn = std::sqrt(s);
            valid_gn = std::isfinite(n_gn);
        }
    }
    float g2 = 0.0f, Hg[6], gHg = 0.0f;
    for (int i = 0; i < 6; ++i) g2 += g[i] * g[i];
    for (int i = 0; i < 6; ++i) {
        float s = 0.0f;
        for (int j = 0; j < 6; ++j) s += H[i * 6 + j] * g[j];
        Hg[i] = s;
    }
    for (int i = 0; i < 6; ++i) gHg += g[i] * Hg[i];
    float p_sd[6];
    for (int i = 0; i < 6; ++i) p_sd[i] = -g[i];
    if (gHg > FLT_EPSILON) {
        const float alpha = g2 / gHg;
        if (std::isfinite(alpha))
            for (int i = 0; i < 6; ++i) p_sd[i] = -alpha * g[i];
    }
    float n_sd2 = 0.0f;
    for (int i = 0; i < 6; ++i) n_sd2 += p_sd[i] * p_sd[i];
    const float n_sd = std::sqrt(n_sd2);
    for (int i = 0; i < 6; ++i) p[i] = 0.0f;
    if (valid_gn && n_gn <= radius) {
        std::memcpy(p, p_gn, sizeof(p_gn));
        *step_norm = n_gn;
    } else if (n_sd >= radius) {
        if (n_sd > FLT_EPSILON)
            for (int i = 0; i < 6; ++i) p[i] = (radius / n_sd) * p_sd[i];
        *step_norm = radius;
    } else if (valid_gn) {
        float diff[6], aq = 0.0f, bq = 0.0f;
        for (int i = 0; i < 6; ++i) {
            diff[i] = p_gn[i] - p_sd[i];
            aq += diff[i] * diff[i];
            bq += p_sd[i] * diff[i];
        }
        bq *= 2.0f;
        const float cq = n_sd2 - radius * radius;
        const float disc = std::max(bq * bq - 4.0f * aq * cq, 0.0f);
        float tau = 0.0f;
        if (aq > FLT_EPSILON) tau = (-bq + std::sqrt(disc)) / (2.0f * aq);
        tau = std::min(std::max(tau, 0.0f), 1.0f);
        float s = 0.0f;
        for (int i = 0; i < 6; ++i) {
            p[i] = p_sd[i] + tau * diff[i];
            s += p[i] * p[i];
        }
        *step_norm = std::sqrt(s);
    } else {
        std::memcpy(p, p_sd, sizeof(p_sd));
        if (n_sd > radius && n_sd > FLT_EPSILON) {
            for (int i = 0; i < 6; ++i) p[i] *= radius / n_sd;
            *step_norm = radius;
        } else {
            *step_norm = n_sd;
        }
    }
    float gp = 0.0f, pHp = 0.0f;
    for (int i = 0; i < 6; ++i) {
        gp += g[i] * p[i];
        float s = 0.0f;
        for (int j = 0; j < 6; ++j) s += H[i * 6 + j] * p[j];
        pHp += p[i] * s;
    }
    *pred = -(gp + 0.5f * pHp);
}

template <bool SHARDED>
void launch_align_gn(int reg_type, LinArgs& a, int max_it, spx_queue_t q, spx_registration_t reg) {
    unsigned resident;
    const void* fn;
    switch (reg_type) {
        case SPX_REG_POINT_TO_POINT:
            resident = coop_blocks<SPX_REG_POINT_TO_POINT, SHARDED>(q->sm_count);
            fn = (const void*)align_gn_kernel<SPX_REG_POINT_TO_POINT, SHARDED>;
            break;
        case SPX_REG_POINT_TO_PLANE:
            resident = coop_blocks<SPX_REG_POINT_TO_PLANE, SHARDED>(q->sm_count);
            fn = (const void*)align_gn_kernel<SPX_REG_POINT_TO_PLANE, SHARDED>;
            break;
        case SPX_REG_POINT_TO_DISTRIBUTION:
            resident = coop_blocks<SPX_REG_POINT_TO_DISTRIBUTION, SHARDED>(q->sm_count);
            fn = (const void*)align_gn_kernel<SPX_REG_POINT_TO_DISTRIBUTION, SHARDED>;
            break;
        default:
            resident = coop_blocks<SPX_REG_GICP, SHARDED>(q->sm_count);
            fn = (const void*)align_gn_kernel<SPX_REG_GICP, SHARDED>;
            break;
    }
    unsigned blocks = std::max(1u, std::min((unsigned)div_up(a.ns, LIN_THREADS), resident));
    // max_grid_blocks = cap on the persistent grid (0 = one full wave).  Lets several aligns share one
    // GPU (concurrent queues; two ranks of the exchange protocol on one device in the tests).
    if (reg->P.max_grid_blocks > 0) blocks = std::min(blocks, (unsigned)reg->P.max_grid_blocks);
    if (2 * blocks > reg->max_blocks) {
        SPX_CUDA(cudaStreamSynchronize(q->stream));
        if (reg->partials) SPX_CUDA(cudaFree(reg->partials));
        reg->max_blocks = 2 * blocks;
        SPX_CUDA(cudaMalloc(&reg->partials, (size_t)reg->max_blocks * 32 * sizeof(double)));
        a.partials = reg->partials;
    }
    void* args[] = {(void*)&a, (void*)&max_it};
    SPX_CUDA(cudaLaunchCooperativeKernel(fn, dim3(blocks), dim3(LIN_THREADS), args, 0, q->stream));
    SPX_LAUNCH_CHECK();
}

template <int REG, int CTAS>
unsigned batch_coop_blocks(int device_sm_count, const void** fn) {
    static int per_sm = 0;
    if (per_sm == 0)
        SPX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, align_batch_kernel<REG, CTAS>, LIN_THREADS, 0));
    *fn = (const void*)align_batch_kernel<REG, CTAS>;
    return (unsigned)std::max(per_sm, 1) * (unsigned)device_sm_count;
}
template <int REG>
unsigned batch_coop_pick(bool single, int device_sm_count, const void** fn) {
    return single ? batch_coop_blocks<REG, ALIGN_CTAS_SINGLE>(device_sm_count, fn)
                  : batch_coop_blocks<REG, ALIGN_CTAS_BATCH>(device_sm_count, fn);
}

template <typename T>
void ensure_n(T*& p, size_t& cap, size_t need, size_t elems_per, cudaStream_t st) {
    if (need <= cap && p) return;
    if (p) {
        SPX_CUDA(cudaStreamSynchronize(st));
        SPX_CUDA(cudaFree(p));
        p = nullptr;
    }
    const size_t c = std::max<size_t>(need + need / 8, 1024);
    SPX_CUDA(cudaMalloc(&p, c * elems_per * sizeof(T)));
    cap = c;
}

// Gauss-Newton align of P pairs in one cooperative launch (align_batch_kernel).  `pairs` are host structs;
// results[p] receives pair p's RegistrationResult.  T_trace_host: P == 1 only.  Synchronises once.
void gn_align_batch(spx_registration_t r, size_t P, const spx_align_pair* pairs, spx_registration_result* results,
                    float* T_trace_host) {
    spx_queue_t q = r->q;
    cudaStream_t st = q->stream;
    const spx_registration_params& Pm = r->P;
    check_reg_loss(Pm.reg_type, Pm.robust_loss, "[Registration::align]");
    int loss = Pm.robust_loss;
    if (loss != SPX_LOSS_NONE && Pm.robust_default_scale <= 0.0f) loss = SPX_LOSS_NONE;  // registration.hpp:186-192
    const bool gicp = Pm.reg_type == SPX_REG_GICP, p2d = Pm.reg_type == SPX_REG_POINT_TO_DISTRIBUTION;
    const int max_it = Pm.max_iterations;
    static const float I16[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};

    // RegistrationResult defaults — result.hpp:16-25; pairs with an empty source stay at them (registration.hpp:209-211)
    size_t total_ns = 0, total_nt = 0, total_chunks = 0, n_active = 0;
    for (size_t p = 0; p < P; ++p) {
        const spx_align_pair& A = pairs[p];
        spx_registration_result* R = results + p;
        std::memset(R, 0, sizeof(*R));
        const float* T0 = A.T_init_host ? A.T_init_host : I16;
        std::memcpy(R->T, T0, 64);
        R->error = FLT_MAX;
        R->error_raw = FLT_MAX;
        if (A.ns == 0) continue;
        SPX_REQUIRE(A.src_points && (A.tgt_points || A.nt == 0), "[Registration::align] null points");
        SPX_REQUIRE(A.target_index, "[Registration::align] target_knn (spx_index) is null");
        SPX_REQUIRE(A.target_index->q->device == q->device, "[Registration::align] index lives on another device");
        if (A.target_index->q != q && A.target_index->ready)  // built on another queue: ordered behind its build
            SPX_CUDA(cudaStreamWaitEvent(q->stream, A.target_index->ready, 0));
        SPX_REQUIRE(A.target_index->n_total == A.nt, "[Registration::align] target_knn was built on a different cloud size");
        SPX_REQUIRE(A.ns < (1ull << 31) && A.nt < (1ull << 31), "[Registration::align] too many points");
        validate(Pm, A.src_covs, A.tgt_covs, A.tgt_normals);
        SPX_REQUIRE(!(Pm.reg_type == SPX_REG_POINT_TO_PLANE && !A.tgt_normals) || P == 1,
                    "[Registration::align_batch] Point-to-Plane needs target normals");
        total_ns += A.ns;
        total_nt += A.nt;
        total_chunks += (size_t)div_up(A.ns, CHUNK);
        ++n_active;
    }
    r->timed = false;
    r->nn_n = P == 1 ? pairs[0].ns : 0;
    if (n_active == 0 || max_it <= 0) return;
    SPX_REQUIRE(total_chunks < (1ull << 31), "[Registration::align_batch] too many points in one batch");

    // scratch
    {
        size_t cap = r->nn_cap;
        ensure(r->nn_idx, cap, total_ns, st);
        cap = r->nn_cap;
        ensure(r->worklist, cap, total_ns, st);
        ensure(r->nn_dist, r->nn_cap, total_ns, st);
        cap = r->wl_cap;
        ensure_n(r->wl_q, cap, total_ns, 1, st);
        ensure_n(r->wl_b, r->wl_cap, total_ns, 1, st);
        ensure_n(r->cpartials, r->cpart_cap, total_chunks, 64, st);
        if (gicp) ensure3(r->src_cm, r->src_cap, total_ns, st);
        if (gicp || p2d) ensure3(r->tgt_cm, r->tgt_cap, total_nt, st);
        if (n_active > r->pairs_cap) {
            SPX_CUDA(cudaStreamSynchronize(st));
            if (r->states) SPX_CUDA(cudaFree(r->states));
            if (r->descs) SPX_CUDA(cudaFree(r->descs));
            if (r->chunk_end) SPX_CUDA(cudaFree(r->chunk_end));
            if (r->preps) SPX_CUDA(cudaFree(r->preps));
            r->states = nullptr; r->descs = nullptr; r->chunk_end = nullptr; r->preps = nullptr;
            const size_t c = std::max<size_t>(n_active, 8);
            SPX_CUDA(cudaMalloc(&r->states, c * sizeof(RegState)));
            SPX_CUDA(cudaMalloc(&r->descs, c * sizeof(PairDesc)));
            SPX_CUDA(cudaMalloc(&r->chunk_end, c * sizeof(uint32_t)));
            SPX_CUDA(cudaMalloc(&r->preps, c * sizeof(PairPrep)));
            r->pairs_cap = c;
        }
        if (T_trace_host && P == 1) {
            size_t tcap = r->trace_cap;
            ensure(r->trace, tcap, (size_t)std::max(max_it, 1) * 16, st);
            r->trace_cap = tcap;
        }
    }
    float4* derived_normals = nullptr;
    // the set-up table (pinned staging for P > 1)
    std::vector<PairPrep> table(n_active);
    std::vector<size_t> slot_of(n_active);
    size_t so = 0, to = 0, co = 0, k = 0;
    unsigned prep_blocks = 1;
    for (size_t p = 0; p < P; ++p) {
        const spx_align_pair& A = pairs[p];
        if (A.ns == 0) continue;
        PairPrep& pp = table[k];
        std::memset(&pp, 0, sizeof(pp));
        slot_of[k] = p;
        pp.src_cov16 = A.src_covs;
        pp.tgt_cov16 = A.tgt_covs;
        pp.n_src_m = gicp ? (uint32_t)A.ns : 0u;
        pp.n_tgt_m = (gicp || p2d) ? (uint32_t)A.nt : 0u;
        pp.src_cm = gicp ? r->src_cm + 3 * so : nullptr;
        pp.tgt_cm = (gicp || p2d) ? r->tgt_cm + 3 * to : nullptr;
        pp.invert_tgt = p2d ? 1 : 0;
        pp.T = xform_from_colmajor(A.T_init_host ? A.T_init_host : I16);
        PairDesc& d = pp.desc;
        d.src_pts = reinterpret_cast<const float4*>(A.src_points);
        d.src_cm = pp.src_cm;
        d.tgt_pts = reinterpret_cast<const float4*>(A.tgt_points);
        d.tgt_cm = pp.tgt_cm;
        d.tgt_normals = reinterpret_cast<const float4*>(A.tgt_normals);
        if (Pm.reg_type == SPX_REG_POINT_TO_PLANE && !A.tgt_normals) {
            // registration.hpp:139-141: normals derived from the pre-computed covariances (P == 1 only, checked above)
            fprintf(stdout, "[Caution] Normal vectors for Point-to-Plane ICP are not provided. \n"
                            "          Attempting to derive them from pre-computed covariance matrices.\n");
            SPX_CUDA(cudaMalloc(&derived_normals, std::max<size_t>(A.nt, 1) * sizeof(float4)));
            if (spx_normals_from_covs(q, A.tgt_points, A.tgt_covs, A.nt, reinterpret_cast<float*>(derived_normals)) != SPX_OK) {
                cudaFree(derived_normals);
                throw Error(SPX_ERR_INTERNAL, spx_last_error());
            }
            d.tgt_normals = derived_normals;
        }
        d.idx = r->nn_idx + so;
        d.dist = r->nn_dist + so;
        d.state = (P == 1) ? r->state : r->states + k;
        d.trace = (P == 1 && T_trace_host) ? r->trace : nullptr;
        d.ns = (uint32_t)A.ns;
        d.chunk0 = (uint32_t)co;
        d.nchunks = (uint32_t)div_up(A.ns, CHUNK);
        d.scale = A.robust_scale > 0.0f ? A.robust_scale : Pm.robust_default_scale;  // registration.hpp:217-218
        d.grid = A.target_index->levels;
        prep_blocks = std::max(prep_blocks, (unsigned)div_up((size_t)pp.n_src_m + pp.n_tgt_m, 128));
        so += A.ns;
        to += A.nt;
        co += d.nchunks;
        ++k;
    }
    auto free_normals = [&] {
        if (derived_normals) {
            cudaStreamSynchronize(st);
            cudaFree(derived_normals);
        }
    };
    try {
        if (r->phase) SPX_CUDA(cudaMemsetAsync(r->phase, 0, PH_WORDS * sizeof(unsigned long long), st));
        if (n_active == 1) {
            align_prepare_batch_kernel<<<dim3(prep_blocks, 1), 128, 0, st>>>(nullptr, table[0], r->descs, r->chunk_end,
                                                                            r->wl_counters);
        } else {
            PairPrep* pin = static_cast<PairPrep*>(q->pinned_get(n_active * sizeof(PairPrep) + n_active * sizeof(RegState)));
            std::memcpy(pin, table.data(), n_active * sizeof(PairPrep));
            SPX_CUDA(cudaMemcpyAsync(r->preps, pin, n_active * sizeof(PairPrep), cudaMemcpyHostToDevice, st));
            align_prepare_batch_kernel<<<dim3(prep_blocks, (unsigned)n_active), 128, 0, st>>>(r->preps, table[0], r->descs,
                                                                                             r->chunk_end, r->wl_counters);
        }
        SPX_LAUNCH_CHECK();

        BatchArgs a;
        std::memset(&a, 0, sizeof(a));
        a.pairs = r->descs;
        a.chunk_end = r->chunk_end;
        a.n_pairs = (uint32_t)n_active;
        a.total_chunks = (uint32_t)total_chunks;
        a.wl_q = r->wl_q;
        a.wl_b = r->wl_b;
        a.wl_counters = r->wl_counters;
        a.partials = r->cpartials;
        a.max_corr = Pm.max_correspondence_distance;
        a.max_corr_sq = Pm.max_correspondence_distance * Pm.max_correspondence_distance;
        a.loss = loss;
        a.lambda = Pm.gn_lambda;
        a.crit_rot = Pm.criteria_rotation;
        a.crit_trans = Pm.criteria_translation;
        a.phase = r->phase;
        unsigned resident;
        const void* fn = nullptr;
        const bool one = n_active == 1;
        switch (Pm.reg_type) {
            case SPX_REG_POINT_TO_POINT: resident = batch_coop_pick<SPX_REG_POINT_TO_POINT>(one, q->sm_count, &fn); break;
            case SPX_REG_POINT_TO_PLANE: resident = batch_coop_pick<SPX_REG_POINT_TO_PLANE>(one, q->sm_count, &fn); break;
            case SPX_REG_POINT_TO_DISTRIBUTION: resident = batch_coop_pick<SPX_REG_POINT_TO_DISTRIBUTION>(one, q->sm_count, &fn); break;
            default: resident = batch_coop_pick<SPX_REG_GICP>(one, q->sm_count, &fn); break;
        }
        unsigned blocks = std::max(1u, std::min((unsigned)total_chunks, resident));
        // max_grid_blocks = cap on the persistent grid (0 = one full wave): lets several aligns share one GPU
        if (Pm.max_grid_blocks > 0) blocks = std::min(blocks, (unsigned)Pm.max_grid_blocks);
        int mi = max_it;
        void* args[] = {(void*)&a, (void*)&mi};
        SPX_CUDA(cudaEventRecord(r->ev0, st));
        SPX_CUDA(cudaLaunchCooperativeKernel(fn, dim3(blocks), dim3(LIN_THREADS), args, 0, st));
        SPX_LAUNCH_CHECK();
        SPX_CUDA(cudaEventRecord(r->ev1, st));

        RegState* hs = static_cast<RegState*>(q->pinned_get(n_active * sizeof(PairPrep) + n_active * sizeof(RegState)));
        if (n_active > 1) hs = reinterpret_cast<RegState*>(reinterpret_cast<char*>(hs) + n_active * sizeof(PairPrep));
        SPX_CUDA(cudaMemcpyAsync(hs, P == 1 ? r->state : r->states, n_active * sizeof(RegState), cudaMemcpyDeviceToHost, st));
        q->sync();
        int most = 0;
        for (size_t j = 0; j < n_active; ++j) {
            fill_result(hs[j], results + slot_of[j]);
            most = std::max(most, hs[j].iterations + 1);
        }
        r->timed = true;
        r->last_launches = 1;
        r->last_iterations = most;
        if (T_trace_host && P == 1) {
            // iterations never run (converged earlier) repeat the final pose
            SPX_CUDA(cudaMemcpyAsync(T_trace_host, r->trace, (size_t)(hs[0].iterations + 1) * 16 * sizeof(float),
                                     cudaMemcpyDeviceToHost, st));
            q->sync();
            for (int it = hs[0].iterations + 1; it < max_it; ++it)
                std::memcpy(T_trace_host + (size_t)it * 16, T_trace_host + (size_t)hs[0].iterations * 16, 64);
        }
    } catch (...) {
        free_normals();
        throw;
    }
    free_normals();
}

// GenZ planarity threshold of the stateless entry points (spx_linearize / spx_error / spx_robust_weights), which take no
// parameter struct: RegistrationParams::genz.planarity_threshold's default unless spx_set_genz_planarity_threshold changed it
thread_local float t_genz_planarity_threshold = 0.2f;
// the same for RegistrationParams::rotation_constraint (spx_set_rotation_constraint)
thread_local int t_rot_enable = 0;
thread_local float t_rot_weight = 1.0f, t_rot_scale = 10.0f;

// generic (caller-supplied correspondences) argument block for spx_linearize / spx_error / weights
LinArgs generic_args(spx_queue_t q, int loss, const float* src_points, const float* src_covs, size_t ns,
                     const float* tgt_points, const float* tgt_covs, const float* tgt_normals, const int32_t* nn_idx,
                     const float* nn_dist, const float* T_host, float max_corr_sq, float robust_scale, unsigned blocks) {
    LinArgs a;
    std::memset(&a, 0, sizeof(a));
    a.src_pts = reinterpret_cast<const float4*>(src_points);
    a.src_cov16 = src_covs;
    a.ns = (uint32_t)ns;
    a.tgt_pts = reinterpret_cast<const float4*>(tgt_points);
    a.tgt_cov16 = tgt_covs;
    a.tgt_normals = reinterpret_cast<const float4*>(tgt_normals);
    a.idx_in = nn_idx;
    a.dist_in = nn_dist;
    a.T = T_host ? xform_from_colmajor(T_host) : xform_identity();
    a.max_corr_sq = max_corr_sq;
    a.max_corr = std::sqrt(std::max(max_corr_sq, 0.0f));
    a.scale = robust_scale;
    a.loss = loss;
    q->arena_reset();
    q->arena_reserve((size_t)blocks * 32 * sizeof(double) + 32 * sizeof(double) + 4096);
    a.partials = q->take<double>((size_t)blocks * 32);
    a.sums_out = q->take<double>(32);
    a.ticket = q->take<unsigned int>(16);
    a.genz_counts = a.ticket + 8;
    a.genz_threshold = t_genz_planarity_threshold;
    a.rot_enable = t_rot_enable;
    a.rot_weight = t_rot_weight;
    a.rot_scale = t_rot_scale;
    SPX_CUDA(cudaMemsetAsync(a.ticket, 0, sizeof(unsigned int), q->stream));
    return a;
}

}  // namespace

extern "C" {

void spx_default_registration_params(spx_registration_params* p) {
    if (!p) return;
    std::memset(p, 0, sizeof(*p));
    p->reg_type = SPX_REG_GICP;
    p->robust_loss = SPX_LOSS_NONE;
    p->optimization_method = SPX_OPT_GAUSS_NEWTON;
    p->max_iterations = 20;
    p->max_correspondence_distance = 2.0f;
    p->robust_default_scale = 10.0f;
    p->criteria_translation = 1e-3f;
    p->criteria_rotation = 1e-3f;
    p->gn_lambda = 1.0f;
    p->lm_max_inner_iterations = 10;
    p->lm_lambda_factor = 2.0f;
    p->lm_init_lambda = 1.0f;
    p->lm_max_lambda = 1e3f;
    p->lm_min_lambda = 1e-6f;
    p->dogleg_initial_trust_region_radius = 1.0f;
    p->dogleg_min_trust_region_radius = 1e-4f;
    p->dogleg_max_trust_region_radius = 10.0f;
    p->dogleg_eta1 = 0.25f;
    p->dogleg_eta2 = 0.75f;
    p->dogleg_gamma_decrease = 0.25f;
    p->dogleg_gamma_increase = 2.0f;
    p->genz_planarity_threshold = 0.2f;
    p->rotation_constraint_enable = 0;
    p->rotation_constraint_weight = 1.0f;
    p->rotation_constraint_robust_scale = 10.0f;
}

int spx_set_rotation_constraint(int enable, float weight, float robust_scale) {
    return guard([&] {
        SPX_REQUIRE(!enable || robust_scale > 0.0f, "[spx_set_rotation_constraint] robust_scale must be positive");
        t_rot_enable = enable ? 1 : 0;
        t_rot_weight = weight;
        t_rot_scale = robust_scale;
    });
}

int spx_set_genz_planarity_threshold(float threshold) {
    return guard([&] {
        SPX_REQUIRE(threshold > 0.0f, "[spx_set_genz_planarity_threshold] threshold must be positive");
        t_genz_planarity_threshold = threshold;
    });
}

int spx_solve_6x6(const float* H_host, const float* b_host, float lambda, float* delta_host, int* success) {
    return guard([&] {
        SPX_REQUIRE(H_host && b_host && delta_host, "[spx_solve_6x6] null pointer");
        const bool ok = solve_damped6(H_host, b_host, lambda, delta_host);
        if (success) *success = ok ? 1 : 0;
    });
}

int spx_se3_exp(const float* twist6_host, float* T_host) {
    return guard([&] {
        SPX_REQUIRE(twist6_host && T_host, "[spx_se3_exp] null pointer");
        float E[4][4];
        se3_exp_rm(twist6_host, E);
        for (int j = 0; j < 4; ++j)
            for (int i = 0; i < 4; ++i) T_host[j * 4 + i] = E[i][j];
    });
}

int spx_dogleg_step(const float* H_host, const float* g_host, float radius, float* p_host, float* step_norm,
                    float* predicted_reduction) {
    return guard([&] {
        SPX_REQUIRE(H_host && g_host && p_host && step_norm && predicted_reduction, "[spx_dogleg_step] null pointer");
        dogleg_host(H_host, g_host, radius, p_host, step_norm, predicted_reduction);
    });
}

int spx_linearize(spx_queue_t q, int reg_type, int robust_loss, const float* src_points, const float* src_covs,
                  size_t ns, const float* tgt_points, const float* tgt_covs, const float* tgt_normals,
                  const int32_t* nn_idx, const float* nn_dist, const float* T_host, float max_corr_sq,
                  float robust_scale, float* H_host, float* b_host, float* error_host, uint32_t* inlier_host) {
    return guard([&] {
        SPX_REQUIRE(q && H_host && b_host && error_host && inlier_host, "[Registration::linearize] null argument");
        check_reg_loss(reg_type, robust_loss, "[Registration::linearize]");
        SPX_REQUIRE(ns < (1ull << 31), "[Registration::linearize] too many points");
        std::memset(H_host, 0, 36 * sizeof(float));
        std::memset(b_host, 0, 6 * sizeof(float));
        *error_host = 0.0f;
        *inlier_host = 0;
        if (ns == 0) return;
        SPX_REQUIRE(src_points && tgt_points && nn_idx && nn_dist, "[Registration::linearize] null pointer");
        DeviceGuard g(q->device);
        const unsigned blocks = lin_blocks(q, ns);
        LinArgs a = generic_args(q, robust_loss, src_points, src_covs, ns, tgt_points, tgt_covs, tgt_normals, nn_idx,
                                 nn_dist, T_host, max_corr_sq, robust_scale, blocks);
        launch_linearize<0, false>(reg_type, a, blocks, q->stream);
        double* hs = static_cast<double*>(q->pinned_get(32 * sizeof(double)));
        SPX_CUDA(cudaMemcpyAsync(hs, a.sums_out, 32 * sizeof(double), cudaMemcpyDeviceToHost, q->stream));
        q->sync();
        sums_to_host(hs, H_host, b_host, error_host, inlier_host);
    });
}

int spx_error(spx_queue_t q, int reg_type, int robust_loss, const float* src_points, const float* src_covs, size_t ns,
              const float* tgt_points, const float* tgt_covs, const float* tgt_normals, const int32_t* nn_idx,
              const float* nn_dist, const float* T_host, float max_corr_sq, float robust_scale, float* error_host,
              uint32_t* inlier_host) {
    return guard([&] {
        SPX_REQUIRE(q && error_host && inlier_host, "[Registration::compute_error] null argument");
        check_reg_loss(reg_type, robust_loss, "[Registration::compute_error]");
        SPX_REQUIRE(ns < (1ull << 31), "[Registration::compute_error] too many points");
        *error_host = 0.0f;
        *inlier_host = 0;
        if (ns == 0) return;
        SPX_REQUIRE(src_points && tgt_points && nn_idx && nn_dist, "[Registration::compute_error] null pointer");
        DeviceGuard g(q->device);
        const unsigned blocks = lin_blocks(q, ns);
        LinArgs a = generic_args(q, robust_loss, src_points, src_covs, ns, tgt_points, tgt_covs, tgt_normals, nn_idx,
                                 nn_dist, T_host, max_corr_sq, robust_scale, blocks);
        launch_error<false>(reg_type, a, blocks, q->stream);
        double* hs = static_cast<double*>(q->pinned_get(32 * sizeof(double)));
        SPX_CUDA(cudaMemcpyAsync(hs, a.sums_out, 32 * sizeof(double), cudaMemcpyDeviceToHost, q->stream));
        q->sync();
        *error_host = (float)hs[S_ERR];
        *inlier_host = (uint32_t)(hs[S_INL] + 0.5);
    });
}

int spx_robust_weights(spx_queue_t q, int reg_type, int robust_loss, const float* src_points, const float* src_covs,
                       size_t ns, const float* tgt_points, const float* tgt_covs, const float* tgt_normals,
                       const int32_t* nn_idx, const float* nn_dist, const float* T_host, float max_corr_sq,
                       float robust_scale, float* weights) {
    return guard([&] {
        SPX_REQUIRE(q, "[Registration::compute_icp_robust_weights] null queue");
        check_reg_loss(reg_type, robust_loss, "[Registration::compute_icp_robust_weights]");
        SPX_REQUIRE(ns < (1ull << 31), "[Registration::compute_icp_robust_weights] too many points");
        if (ns == 0) return;
        SPX_REQUIRE(src_points && tgt_points && nn_idx && nn_dist && weights,
                    "[Registration::compute_icp_robust_weights] null pointer");
        DeviceGuard g(q->device);
        const unsigned blocks = (unsigned)div_up(ns, LIN_THREADS);
        LinArgs a = generic_args(q, robust_loss, src_points, src_covs, ns, tgt_points, tgt_covs, tgt_normals, nn_idx,
                                 nn_dist, T_host, max_corr_sq, robust_scale, 1);
        a.weights_out = weights;
        launch_error<true>(reg_type, a, blocks, q->stream);
    });
}

int spx_registration_create(spx_queue_t q, const spx_registration_params* params, spx_registration_t* out) {
    return guard([&] {
        SPX_REQUIRE(q && out, "[Registration::Registration] null argument");
        DeviceGuard g(q->device);
        auto* r = new spx_registration_s();
        r->q = q;
        if (params) r->P = *params;
        else spx_default_registration_params(&r->P);
        try {
            SPX_CUDA(cudaMalloc(&r->state, sizeof(RegState)));
            SPX_CUDA(cudaMalloc(&r->ticket, 64));
            SPX_CUDA(cudaMalloc(&r->wl_counters, 64));
            SPX_CUDA(cudaMalloc(&r->sums, 32 * sizeof(double)));
            SPX_CUDA(cudaMemsetAsync(r->ticket, 0, 64, q->stream));
            r->max_blocks = (unsigned)q->sm_count * 4;
            SPX_CUDA(cudaMalloc(&r->partials, (size_t)r->max_blocks * 32 * sizeof(double)));
            SPX_CUDA(cudaEventCreate(&r->ev0));
            SPX_CUDA(cudaEventCreate(&r->ev1));
        } catch (...) {
            reg_free(r);
            delete r;
            throw;
        }
        *out = r;
    });
}

int spx_registration_destroy(spx_registration_t reg) {
    return guard([&] {
        if (!reg) return;
        if (queue_is_live(reg->q)) {
            DeviceGuard g(reg->q->device);
            cudaStreamSynchronize(reg->q->stream);
            reg_free(reg);
        } else {
            cudaDeviceSynchronize();
            reg_free(reg);
        }
        delete reg;
    });
}

}  // extern "C"

namespace {

void colmajor_to_rm(const float* T16, float T[4][4]) {
    for (int i = 0; i < 4; ++i)
        for (int j = 0; j < 4; ++j) T[i][j] = T16[j * 4 + i];
}
void isometry_inverse_rm(const float T[4][4], float out[4][4]) {
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) out[i][j] = T[j][i];
        out[i][3] = -(T[0][i] * T[0][3] + T[1][i] * T[1][3] + T[2][i] * T[2][3]);
        out[3][i] = 0.0f;
    }
    out[3][3] = 1.0f;
}

// DegenerateRegularization::regularize_impl — degenerate_regularization.hpp:58-112.  H row-major 6x6 (symmetric).
void nl_reg_apply(const spx_registration_addons& A, float* H, float* b, uint32_t inlier, const float T_cur[4][4],
                  const float T_init[4][4]) {
    if (inlier == 0 || A.degenerate_type != 1) return;
    const float lambda = A.base_factor * (float)inlier;
    float Hp[36] = {};
    for (int blk = 0; blk < 2; ++blk) {
        const float thr = blk == 0 ? A.rot_eigenvalue_threshold : A.trans_eigenvalue_threshold;
        if (!(thr > 0.0f)) continue;
        float B[3][3];
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) B[i][j] = H[(3 * blk + i) * 6 + 3 * blk + j];
        double ev[3], V[3][3];
        jacobi3(B, ev, V);
        for (int k = 0; k < 3; ++k) {
            const float val = (float)ev[k] / (float)inlier;
            if (!(val < thr)) continue;
            for (int i = 0; i < 3; ++i)
                for (int j = 0; j < 3; ++j)
                    Hp[(3 * blk + i) * 6 + 3 * blk + j] += lambda * ((float)V[i][k] * (float)V[j][k]);
        }
    }
    float Ti[4][4], D[4][4], tw[6];
    isometry_inverse_rm(T_init, Ti);
    isometry_mul_rm(Ti, T_cur, D);
    se3_log_rm(D, tw);
    for (int i = 0; i < 6; ++i) {
        float acc = 0.0f;
        for (int j = 0; j < 6; ++j) acc += Hp[i * 6 + j] * tw[j];
        b[i] += acc;
    }
    for (int i = 0; i < 36; ++i) H[i] += Hp[i];
}

// MapPrior::update — map_prior.hpp:30-117
void map_prior_update(spx_registration_t reg, const spx_registration_result& prev, const float* T_pred16) {
    reg->prior_active = false;
    const spx_registration_addons& A = reg->addons;
    if (!A.map_prior_enabled) return;
    const float dof = 3.0f * (float)prev.inlier - 6.0f;
    if (dof <= 0.0f) return;
    if (!std::isfinite(prev.error_raw) || prev.error_raw < 0.0f) return;
    const float s_sq = std::max(1.0f, 2.0f * prev.error_raw / dof);
    float Tp[4][4], To[4][4];
    colmajor_to_rm(T_pred16, Tp);
    colmajor_to_rm(prev.T, To);
    float Rrel[4][4] = {};
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) Rrel[i][j] = To[0][i] * Tp[0][j] + To[1][i] * Tp[1][j] + To[2][i] * Tp[2][j];
    Rrel[3][3] = 1.0f;
    float tw[6];
    se3_log_rm(Rrel, tw);  // rotation vector = axis * angle (translation part zero)
    const float dt[3] = {Tp[0][3] - To[0][3], Tp[1][3] - To[1][3], Tp[2][3] - To[2][3]};
    float dtb[3];
    for (int i = 0; i < 3; ++i) dtb[i] = Tp[0][i] * dt[0] + Tp[1][i] * dt[1] + Tp[2][i] * dt[2];
    double q[6];
    for (int i = 0; i < 3; ++i) {
        q[i] = std::fabs(tw[i]) * A.rot_vel_sigma * A.rot_vel_sigma + A.rot_base_sigma * A.rot_base_sigma;
        q[3 + i] = std::fabs(dtb[i]) * A.trans_vel_sigma * A.trans_vel_sigma + A.trans_base_sigma * A.trans_base_sigma;
    }
    // H_curr = Ad^T (H_raw / s^2) Ad, Ad = blockdiag(R_rel, R_rel)
    double Hc[6][6], tmp[6][6];
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j < 6; ++j) {
            double acc = 0.0;
            for (int k = 0; k < 3; ++k) acc += (double)prev.H_raw[i * 6 + (j / 3) * 3 + k] / s_sq * Rrel[k][j % 3];
            tmp[i][j] = acc;  // (H Ad)
        }
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j < 6; ++j) {
            double acc = 0.0;
            for (int k = 0; k < 3; ++k) acc += (double)Rrel[k][i % 3] * tmp[(i / 3) * 3 + k][j];
            Hc[i][j] = acc;  // Ad^T (H Ad)
        }
    // Omega = R - R (H + R)^-1 R with R = diag(1 / q): Gauss-Jordan with partial pivoting in fp64 (H + R is PD)
    double M[6][12];
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j < 6; ++j) {
            M[i][j] = Hc[i][j] + (i == j ? 1.0 / q[i] : 0.0);
            M[i][6 + j] = i == j ? 1.0 / q[i] : 0.0;  // right-hand sides: R
        }
    for (int c = 0; c < 6; ++c) {
        int piv = c;
        for (int r = c + 1; r < 6; ++r)
            if (std::fabs(M[r][c]) > std::fabs(M[piv][c])) piv = r;
        if (!(std::fabs(M[piv][c]) > 1e-300) || !std::isfinite(M[piv][c])) return;
        if (piv != c)
            for (int k = 0; k < 12; ++k) std::swap(M[c][k], M[piv][k]);
        const double inv = 1.0 / M[c][c];
        for (int k = 0; k < 12; ++k) M[c][k] *= inv;
        for (int r = 0; r < 6; ++r) {
            if (r == c) continue;
            const double f = M[r][c];
            if (f != 0.0)
                for (int k = 0; k < 12; ++k) M[r][k] -= f * M[c][k];
        }
    }
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j < 6; ++j) {
            const double v = (i == j ? 1.0 / q[i] : 0.0) - (1.0 / q[i]) * M[i][6 + j];
            if (!std::isfinite(v)) return;
            reg->prior_omega[i * 6 + j] = (float)v;
        }
    isometry_inverse_rm(Tp, reg->prior_T_pred_inv);
    reg->prior_active = true;
}

// e = Log(T_pred^-1 T), Omega e, 1/2 e^T Omega e — map_prior.hpp:119-146
float map_prior_terms(const spx_registration_t reg, const float T[4][4], float* omega_e) {
    float D[4][4], e[6];
    isometry_mul_rm(reg->prior_T_pred_inv, T, D);
    se3_log_rm(D, e);
    float oe[6], dot = 0.0f;
    for (int i = 0; i < 6; ++i) {
        float acc = 0.0f;
        for (int j = 0; j < 6; ++j) acc += reg->prior_omega[i * 6 + j] * e[j];
        oe[i] = acc;
        dot += e[i] * acc;
    }
    if (omega_e) std::memcpy(omega_e, oe, sizeof(oe));
    return 0.5f * dot;
}

}  // namespace

extern "C" {

void spx_default_registration_addons(spx_registration_addons* a) {
    if (!a) return;
    *a = spx_registration_addons{0, 10.0f, 1.0f, 1.0f, 0, 1.0f, 1.0f, 3.16e-2f, 1e-2f};
}

int spx_registration_set_addons(spx_registration_t reg, const spx_registration_addons* a) {
    return guard([&] {
        SPX_REQUIRE(reg && a, "[Registration::set_params] null argument");
        SPX_REQUIRE(a->degenerate_type == 0 || a->degenerate_type == 1, "[Registration::set_params] unknown degenerate regularization type");
        reg->addons = *a;
        reg->prior_active = false;
    });
}

int spx_registration_set_map_prior_state(spx_registration_t reg, const spx_registration_result* prev_result,
                                         const float* T_pred16, int* active_out, float* omega36_out) {
    return guard([&] {
        SPX_REQUIRE(reg && prev_result && T_pred16, "[Registration::set_map_prior_state] null argument");
        map_prior_update(reg, *prev_result, T_pred16);
        if (active_out) *active_out = reg->prior_active ? 1 : 0;
        if (omega36_out && reg->prior_active) std::memcpy(omega36_out, reg->prior_omega, sizeof(reg->prior_omega));
    });
}

int spx_degenerate_regularize(const spx_registration_addons* a, float* H36, float* b6, uint32_t inlier,
                              const float* T_current16, const float* T_initial16) {
    return guard([&] {
        SPX_REQUIRE(a && H36 && b6 && T_current16 && T_initial16, "[DegenerateRegularization::regularize] null argument");
        float Tc[4][4], Ti[4][4];
        colmajor_to_rm(T_current16, Tc);
        colmajor_to_rm(T_initial16, Ti);
        nl_reg_apply(*a, H36, b6, inlier, Tc, Ti);
    });
}

int spx_registration_set_params(spx_registration_t reg, const spx_registration_params* params) {
    return guard([&] {
        SPX_REQUIRE(reg && params, "[Registration::set_params] null argument");
        reg->P = *params;
    });
}

int spx_registration_kept_correspondences(spx_registration_t reg, uint64_t* kept) {
    return guard([&] {
        SPX_REQUIRE(reg && kept, "[Registration::kept_correspondences] null argument");
        DeviceGuard g(reg->q->device);
        *kept = 0;
        if (!reg->wl_counters) return;
        unsigned int v = 0;
        SPX_CUDA(cudaMemcpyAsync(&v, reg->wl_counters + WL_KEPT, sizeof(v), cudaMemcpyDeviceToHost, reg->q->stream));
        reg->q->sync();
        *kept = v;
    });
}

int spx_registration_last_timing(spx_registration_t reg, float* loop_ms, int32_t* launches, int32_t* iterations) {
    return guard([&] {
        SPX_REQUIRE(reg, "[Registration::last_timing] null handle");
        SPX_REQUIRE(reg->timed, "[Registration::last_timing] no timed Gauss-Newton align on this handle yet");
        DeviceGuard g(reg->q->device);
        float ms = 0.0f;
        SPX_CUDA(cudaEventElapsedTime(&ms, reg->ev0, reg->ev1));
        if (loop_ms) *loop_ms = ms;
        if (launches) *launches = reg->last_launches;
        if (iterations) *iterations = reg->last_iterations;
    });
}

int spx_registration_phase_times(spx_registration_t reg, int enable, uint64_t* times_host, int max_iterations) {
    return guard([&] {
        SPX_REQUIRE(reg, "[Registration::phase_times] null handle");
        DeviceGuard g(reg->q->device);
        if (enable && !reg->phase) {
            SPX_CUDA(cudaMalloc(&reg->phase, PH_WORDS * sizeof(unsigned long long)));
            SPX_CUDA(cudaMemsetAsync(reg->phase, 0, PH_WORDS * sizeof(unsigned long long), reg->q->stream));
        }
        if (!enable && reg->phase) {
            SPX_CUDA(cudaStreamSynchronize(reg->q->stream));
            SPX_CUDA(cudaFree(reg->phase));
            reg->phase = nullptr;
        }
        if (times_host && reg->phase) {
            // max_iterations < 0: the whole buffer (phase table + per-warp records of iteration 1)
            const size_t words = max_iterations < 0 ? PH_WORDS
                                                    : (size_t)std::min(max_iterations, PH_MAX_ITERS) * PH_N;
            SPX_CUDA(cudaMemcpyAsync(times_host, reg->phase, words * sizeof(unsigned long long),
                                     cudaMemcpyDeviceToHost, reg->q->stream));
            reg->q->sync();
        }
    });
}

int spx_registration_neighbors(spx_registration_t reg, const int32_t** nn_idx, const float** nn_dist, size_t* n) {
    return guard([&] {
        SPX_REQUIRE(reg, "[Registration::neighbors] null handle");
        if (nn_idx) *nn_idx = reg->nn_idx;
        if (nn_dist) *nn_dist = reg->nn_dist;
        if (n) *n = reg->nn_n;
    });
}

int spx_registration_align(spx_registration_t reg, const float* src_points, const float* src_covs, size_t ns,
                           const float* tgt_points, const float* tgt_covs, const float* tgt_normals, size_t nt,
                           spx_index_t target_index, const float* T_init_host, float robust_scale,
                           spx_registration_result* R, float* T_trace_host) {
    float4* derived_normals = nullptr;
    const int rc = guard([&] {
        SPX_REQUIRE(reg && R, "[Registration::align] null argument");
        spx_queue_t q = reg->q;
        DeviceGuard g(q->device);
        cudaStream_t st = q->stream;
        const spx_registration_params P = reg->P;
        // RegistrationResult defaults — result.hpp:16-25
        std::memset(R, 0, sizeof(*R));
        for (int j = 0; j < 4; ++j)
            for (int i = 0; i < 4; ++i) R->T[j * 4 + i] = T_init_host ? T_init_host[j * 4 + i] : (i == j ? 1.0f : 0.0f);
        R->error = FLT_MAX;
        R->error_raw = FLT_MAX;
        if (ns == 0) return;  // registration.hpp:209-211
        SPX_REQUIRE(src_points && (tgt_points || nt == 0), "[Registration::align] null points");
        // nl-reg / MAP prior sit between the linearisation and the step (registration.hpp:248-253): with either in
        // force every method runs as the host-decided loop below (one 32-double read-back per iteration)
        const bool addons_active = reg->addons.degenerate_type == 1 || reg->prior_active;
        {
            size_t split_min = 400000;
            if (const char* e = std::getenv("SPX_SPLIT_MIN")) split_min = (size_t)std::atoll(e);  // tuning aid
            if (P.optimization_method == SPX_OPT_GAUSS_NEWTON && ns < split_min && P.reg_type != SPX_REG_GENZ &&
                !P.rotation_constraint_enable && !addons_active) {
                // the cooperative one-launch path: the batched kernel with one pair
                spx_align_pair one{};
                one.src_points = src_points; one.src_covs = src_covs; one.ns = ns;
                one.tgt_points = tgt_points; one.tgt_covs = tgt_covs; one.tgt_normals = tgt_normals; one.nt = nt;
                one.target_index = target_index;
                one.T_init_host = T_init_host;
                one.robust_scale = robust_scale;
                gn_align_batch(reg, 1, &one, R, T_trace_host);
                return;
            }
        }
        AlignCtx c = align_setup(reg, src_points, src_covs, ns, tgt_points, tgt_covs, tgt_normals, nt, target_index,
                                 T_init_host, robust_scale, &derived_normals);
        LinArgs& a = c.a;
        RegState* hs = static_cast<RegState*>(q->pinned_get(sizeof(RegState) + 64 + 32 * sizeof(double)));
        double* hsums = reinterpret_cast<double*>(reinterpret_cast<char*>(hs) + sizeof(RegState) + 64);
        const int max_it = P.max_iterations;

        reg->timed = false;
        if (P.optimization_method == SPX_OPT_GAUSS_NEWTON && !addons_active) {
            // small clouds: one cooperative launch for the whole loop.  Large clouds: three ordinary
            // launches per iteration (search kernels with their own register budget), converged-state
            // polled every SPLIT_POLL iterations; launches after convergence return immediately.
            size_t split_min = 400000;
            if (const char* e = std::getenv("SPX_SPLIT_MIN")) split_min = (size_t)std::atoll(e);  // tuning aid
            const bool split = ns >= split_min;
            int launches = 0;
            SPX_CUDA(cudaEventRecord(reg->ev0, st));
            if (max_it > 0) {  // split kernels (large clouds); smaller ones took the batched kernel above
                (void)split;
                constexpr int SPLIT_POLL = 4;
                // the first search has no previous pose to measure a query's step against: plain; from then on the
                // searches track margins, and from the third iteration on correspondences can be kept (icp_keep)
                const float keep_frac = keep_fraction();
                const bool keep = keep_frac >= 0.0f;
                a.keep_infl = keep ? keep_frac * a.grid.lv[0].cell : 0.0f;
                if (keep) {  // allowances + redo list
                    ensure(reg->keep_buf, reg->keep_cap, 2 * ns, st);
                    a.slack_out = reinterpret_cast<float*>(reg->keep_buf);
                    a.redo = reg->keep_buf + ns;
                }
                LinArgs f = a;  // factor pass: correspondences given, fused solve
                f.idx_in = reg->nn_idx;
                f.dist_in = reg->nn_dist;
                for (int it = 0; it < max_it; ++it) {
                    a.iter_index = f.iter_index = it;
                    a.keep_last = keep && it >= 2;
                    if (a.keep_last) {
                        icp_keep_kernel<<<div_up(ns, KEEP_THREADS), KEEP_THREADS, 0, st>>>(a);
                        SPX_LAUNCH_CHECK();
                        ++launches;
                    }
                    if (keep && it >= 1) {
                        icp_fast_kernel<true><<<div_up(ns, NN_THREADS), NN_THREADS, 0, st>>>(a);
                        SPX_LAUNCH_CHECK();
                        icp_coop_kernel<true><<<q->sm_count * 16, NN_THREADS, 0, st>>>(a);
                    } else {
                        icp_fast_kernel<false><<<div_up(ns, NN_THREADS), NN_THREADS, 0, st>>>(a);
                        SPX_LAUNCH_CHECK();
                        icp_coop_kernel<false><<<q->sm_count * 16, NN_THREADS, 0, st>>>(a);
                    }
                    SPX_LAUNCH_CHECK();
                    launch_linearize<0, true>(c.reg, f, c.blocks, st, q->sm_count);
                    launches += 3;
                    if ((it + 1) % SPLIT_POLL == 0 && it + 1 < max_it) {
                        SPX_CUDA(cudaMemcpyAsync(hs, reg->state, sizeof(RegState), cudaMemcpyDeviceToHost, st));
                        q->sync();
                        if (hs->stop) break;
                    }
                }
            }
            SPX_CUDA(cudaEventRecord(reg->ev1, st));
            SPX_CUDA(cudaMemcpyAsync(hs, reg->state, sizeof(RegState), cudaMemcpyDeviceToHost, st));
            q->sync();
            if (max_it > 0) fill_result(*hs, R);
            reg->timed = max_it > 0;
            reg->last_launches = launches;
            reg->last_iterations = max_it > 0 ? hs->iterations + 1 : 0;
            if (T_trace_host && max_it > 0) {
                // iterations never run (converged earlier) repeat the final pose
                SPX_CUDA(cudaMemcpyAsync(T_trace_host, reg->trace, (size_t)(hs->iterations + 1) * 16 * sizeof(float),
                                         cudaMemcpyDeviceToHost, st));
                q->sync();
                for (int it = hs->iterations + 1; it < max_it; ++it)
                    std::memcpy(T_trace_host + (size_t)it * 16, T_trace_host + (size_t)hs->iterations * 16, 64);
            }
            return;
        }

        // LM / dog-leg: one host decision per trial step (registration.hpp:830-964)
        float T[4][4], T_initial[4][4];
        for (int i = 0; i < 4; ++i)
            for (int j = 0; j < 4; ++j) T[i][j] = T_initial[i][j] = R->T[j * 4 + i];
        float lambda = P.lm_init_lambda;
        float radius = P.dogleg_initial_trust_region_radius;
        a.use_state = 0;
        a.state = nullptr;
        auto converged = [&](const float* d) {
            return norm3f(d) < P.criteria_rotation && norm3f(d + 3) < P.criteria_translation;
        };
        auto trial_error = [&](const float Tn[4][4], float* err, uint32_t* inl) {
            LinArgs e = a;
            host_T_to_xform(Tn, e.T);
            launch_error<false>(c.reg, e, c.blocks, st);
            SPX_CUDA(cudaMemcpyAsync(hsums, reg->sums, 32 * sizeof(double), cudaMemcpyDeviceToHost, st));
            q->sync();
            *err = (float)hsums[S_ERR];
            *inl = (uint32_t)(hsums[S_INL] + 0.5);
            if (reg->prior_active) *err += map_prior_terms(reg, Tn, nullptr);  // registration.hpp:854,933
        };
        auto clampf = [](float v, float lo, float hi) { return std::min(std::max(v, lo), hi); };
        for (int it = 0; it < max_it; ++it) {
            host_T_to_xform(T, a.T);
            a.warm_start = it > 0;
            a.iter_index = it;
            launch_linearize<1, false>(c.reg, a, c.blocks, st, q->sm_count);
            SPX_CUDA(cudaMemcpyAsync(hsums, reg->sums, 32 * sizeof(double), cudaMemcpyDeviceToHost, st));
            q->sync();
            float H[36], b[6], err;
            uint32_t inl;
            sums_to_host(hsums, H, b, &err, &inl);
            std::memcpy(R->H_raw, H, sizeof(H));
            std::memcpy(R->b_raw, b, sizeof(b));
            R->error_raw = err;
            nl_reg_apply(reg->addons, H, b, inl, T, T_initial);  // registration.hpp:249-250
            if (reg->prior_active) {                             // :253, map_prior.hpp:119-132
                float oe[6];
                err += map_prior_terms(reg, T, oe);
                for (int i = 0; i < 36; ++i) H[i] += reg->prior_omega[i];
                for (int i = 0; i < 6; ++i) b[i] += oe[i];
            }
            if (P.optimization_method == SPX_OPT_GAUSS_NEWTON) {  // optimize_gauss_newton, registration.hpp:803-828
                float d[6];
                const bool ok = solve_damped6(H, b, P.gn_lambda, d);
                R->converged = ok ? converged(d) : 0;
                float E[4][4], Tn[4][4];
                se3_exp_rm(d, E);
                isometry_mul_rm(T, E, Tn);
                std::memcpy(T, Tn, sizeof(T));
                R->iterations = it;
                std::memcpy(R->H, H, sizeof(H));
                std::memcpy(R->b, b, sizeof(b));
                R->error = err;
                R->inlier = inl;
            } else if (P.optimization_method == SPX_OPT_LEVENBERG_MARQUARDT) {
                float last = FLT_MAX, d[6];
                for (int in = 0; in < P.lm_max_inner_iterations; ++in) {
                    const bool ok = solve_damped6(H, b, lambda, d);
                    R->converged = ok ? converged(d) : 0;
                    float E[4][4], Tn[4][4];
                    se3_exp_rm(d, E);
                    isometry_mul_rm(T, E, Tn);
                    float ne;
                    uint32_t ni;
                    trial_error(Tn, &ne, &ni);
                    if (ne <= err) {
                        R->converged = converged(d);
                        std::memcpy(T, Tn, sizeof(T));
                        R->error = ne;
                        R->inlier = ni;
                        lambda = clampf(lambda / P.lm_lambda_factor, P.lm_min_lambda, P.lm_max_lambda);
                        break;
                    } else if (std::fabs(ne - last) <= 1e-6f) {
                        R->converged = converged(d);
                        std::memcpy(T, Tn, sizeof(T));
                        R->error = ne;
                        R->inlier = ni;
                        break;
                    } else {
                        lambda = clampf(lambda * P.lm_lambda_factor, P.lm_min_lambda, P.lm_max_lambda);
                    }
                    last = ne;
                }
                R->iterations = it;
                std::memcpy(R->H, H, sizeof(H));
                std::memcpy(R->b, b, sizeof(b));
            } else {
                std::memcpy(R->H, H, sizeof(H));
                std::memcpy(R->b, b, sizeof(b));
                R->error = err;
                R->inlier = inl;
                R->iterations = it;
                radius = clampf(radius, P.dogleg_min_trust_region_radius, P.dogleg_max_trust_region_radius);
                float p[6], step_norm, pred;
                dogleg_host(H, b, radius, p, &step_norm, &pred);
                if (pred <= 0.0f) {
                    radius = clampf(radius * P.dogleg_gamma_decrease, P.dogleg_min_trust_region_radius,
                                    P.dogleg_max_trust_region_radius);
                } else {
                    float E[4][4], Tn[4][4];
                    se3_exp_rm(p, E);
                    isometry_mul_rm(T, E, Tn);
                    float ne;
                    uint32_t ni;
                    trial_error(Tn, &ne, &ni);
                    const float rho = (err - ne) / pred;
                    if (rho < P.dogleg_eta1) {
                        radius = clampf(radius * P.dogleg_gamma_decrease, P.dogleg_min_trust_region_radius,
                                        P.dogleg_max_trust_region_radius);
                    } else {
                        R->converged = converged(p);
                        std::memcpy(T, Tn, sizeof(T));
                        R->error = ne;
                        R->inlier = ni;
                        if (rho > P.dogleg_eta2 && step_norm >= radius * 0.99f)
                            radius = clampf(radius * P.dogleg_gamma_increase, P.dogleg_min_trust_region_radius,
                                            P.dogleg_max_trust_region_radius);
                    }
                }
            }
            for (int j = 0; j < 4; ++j)
                for (int i = 0; i < 4; ++i) R->T[j * 4 + i] = T[i][j];
            if (T_trace_host) std::memcpy(T_trace_host + (size_t)it * 16, R->T, 64);
            if (R->converged) {
                if (T_trace_host)
                    for (int k2 = it + 1; k2 < max_it; ++k2) std::memcpy(T_trace_host + (size_t)k2 * 16, R->T, 64);
                break;
            }
        }
    });
    if (derived_normals) {
        cudaStreamSynchronize(reg->q->stream);
        cudaFree(derived_normals);
    }
    return rc;
}

int spx_registration_align_batch(spx_registration_t reg, size_t n_pairs, const spx_align_pair* pairs_host,
                                 spx_registration_result* results_host) {
    return guard([&] {
        SPX_REQUIRE(reg && (n_pairs == 0 || (pairs_host && results_host)), "[Registration::align_batch] null argument");
        if (n_pairs == 0) return;
        DeviceGuard g(reg->q->device);
        if (reg->P.optimization_method == SPX_OPT_GAUSS_NEWTON && reg->P.reg_type != SPX_REG_GENZ &&
            !reg->P.rotation_constraint_enable) {
            gn_align_batch(reg, n_pairs, pairs_host, results_host, nullptr);
            return;
        }
        // LM / dog-leg take host decisions per trial step, GenZ needs a count reduction in front of every
        // linearisation: one pair after the other
        for (size_t p = 0; p < n_pairs; ++p) {
            const spx_align_pair& A = pairs_host[p];
            const int rc = spx_registration_align(reg, A.src_points, A.src_covs, A.ns, A.tgt_points, A.tgt_covs, A.tgt_normals,
                                                  A.nt, A.target_index, A.T_init_host, A.robust_scale, results_host + p, nullptr);
            if (rc != SPX_OK) throw Error(rc, spx_last_error());
        }
    });
}

// ------------------------------------------------------------------ sharded building blocks
int spx_registration_shard_begin(spx_registration_t reg, const float* src_points, const float* src_covs, size_t ns,
                                 const float* tgt_points, const float* tgt_covs, const float* tgt_normals, size_t nt,
                                 spx_index_t target_index, const float* T_init_host, float robust_scale) {
    return guard([&] {
        SPX_REQUIRE(reg, "[Registration::shard_begin] null handle");
        SPX_REQUIRE(reg->P.optimization_method == SPX_OPT_GAUSS_NEWTON,
                    "[Registration::shard_begin] the sharded path is Gauss-Newton only");
        if (reg->P.reg_type == SPX_REG_POINT_TO_PLANE)
            SPX_REQUIRE(tgt_normals, "[Registration::shard_begin] Point-to-Plane needs target normals");
        DeviceGuard g(reg->q->device);
        float4* dn = nullptr;
        AlignCtx c = align_setup(reg, src_points, src_covs, ns, tgt_points, tgt_covs, tgt_normals, nt, target_index,
                                 T_init_host, robust_scale, &dn);
        reg->shard = c.a;
        reg->shard_reg = c.reg;
        reg->shard_iter = 0;
        reg->shard_active = true;
    });
}

int spx_registration_shard_linearize(spx_registration_t reg, double* sums_dev) {
    return guard([&] {
        SPX_REQUIRE(reg && reg->shard_active && sums_dev, "[Registration::shard_linearize] no active shard");
        DeviceGuard g(reg->q->device);
        LinArgs a = reg->shard;
        a.sums_out = sums_dev;
        a.warm_start = reg->shard_iter > 0;
        a.iter_index = reg->shard_iter;
        const unsigned blocks = lin_blocks(reg->q, a.ns);
        if (a.ns == 0) {
            // an empty shard still contributes zeros (and must not leave stale sums behind)
            SPX_CUDA(cudaMemsetAsync(sums_dev, 0, 32 * sizeof(double), reg->q->stream));
            return;
        }
        launch_linearize<1, false>(reg->shard_reg, a, blocks, reg->q->stream, reg->q->sm_count);
    });
}

int spx_registration_shard_update(spx_registration_t reg, const double* sums_dev) {
    return guard([&] {
        SPX_REQUIRE(reg && reg->shard_active && sums_dev, "[Registration::shard_update] no active shard");
        DeviceGuard g(reg->q->device);
        const LinArgs& a = reg->shard;
        gn_update_kernel<<<1, 32, 0, reg->q->stream>>>(reg->state, sums_dev, a.lambda, a.crit_rot, a.crit_trans,
                                                      reg->shard_iter, reg->trace);
        SPX_LAUNCH_CHECK();
        ++reg->shard_iter;
    });
}

int spx_registration_shard_finish(spx_registration_t reg, spx_registration_result* R) {
    return guard([&] {
        SPX_REQUIRE(reg && reg->shard_active && R, "[Registration::shard_finish] no active shard");
        spx_queue_t q = reg->q;
        DeviceGuard g(q->device);
        RegState* hs = static_cast<RegState*>(q->pinned_get(sizeof(RegState) + 64 + 32 * sizeof(double)));
        SPX_CUDA(cudaMemcpyAsync(hs, reg->state, sizeof(RegState), cudaMemcpyDeviceToHost, q->stream));
        q->sync();
        std::memset(R, 0, sizeof(*R));
        fill_result(*hs, R);
        reg->shard_active = false;
    });
}

// ------------------------------------------------------------------ fused linearise + NVLink exchange
int spx_registration_align_sharded_launch(spx_registration_t reg, spx_comm_t comm, const float* src_points,
                                          const float* src_covs, size_t ns, const float* tgt_points,
                                          const float* tgt_covs, const float* tgt_normals, size_t nt,
                                          spx_index_t target_index, const float* T_init_host, float robust_scale) {
    return guard([&] {
        SPX_REQUIRE(reg && comm, "[Registration::align_sharded] null argument");
        SPX_REQUIRE(comm->connected, "[Registration::align_sharded] communicator is not connected");
        SPX_REQUIRE(comm->q->device == reg->q->device, "[Registration::align_sharded] communicator lives on another device");
        SPX_REQUIRE(reg->P.optimization_method == SPX_OPT_GAUSS_NEWTON,
                    "[Registration::align_sharded] the sharded path is Gauss-Newton only");
        SPX_REQUIRE(!reg->shard_comm, "[Registration::align_sharded] previous sharded align not finished");
        SPX_REQUIRE(tgt_points || nt == 0, "[Registration::align_sharded] null target");
        SPX_REQUIRE(src_points || ns == 0, "[Registration::align_sharded] null source");
        spx_queue_t q = reg->q;
        DeviceGuard g(q->device);
        cudaStream_t st = q->stream;
        // an empty shard still takes part in every exchange: one block, no points
        float4* dn = nullptr;
        AlignCtx c = align_setup(reg, ns ? src_points : tgt_points, ns ? src_covs : tgt_covs, ns, tgt_points, tgt_covs,
                                 tgt_normals, nt, target_index, T_init_host, robust_scale, &dn);
        reg->shard_derived_normals = dn;
        LinArgs& a = c.a;
        PeerX& x = a.px;
        x.world = comm->world;
        x.rank = comm->rank;
        for (int r = 0; r < comm->world; ++r) {
            SPX_REQUIRE(comm->peer[r], "[Registration::align_sharded] peer mailbox not mapped");
            x.rows[r] = reinterpret_cast<double*>(comm->peer[r] + SPX_MBOX_ROWS);
            x.flags[r] = reinterpret_cast<unsigned long long*>(comm->peer[r] + SPX_MBOX_FLAGS);
        }
        x.gsum = reinterpret_cast<double*>(comm->local + SPX_MBOX_GSUM);
        x.ready = reinterpret_cast<unsigned long long*>(comm->local + SPX_MBOX_READY);
        x.error = reinterpret_cast<unsigned int*>(comm->local + SPX_MBOX_ERROR);
        const int max_it = std::max(reg->P.max_iterations, 0);
        {  // keep test of the search (nn_search_grid_keep): allowances + redo list
            const float keep_frac = keep_fraction();
            ensure(reg->keep_buf, reg->keep_cap, 2 * std::max<size_t>(ns, 1), st);
            a.slack_out = reinterpret_cast<float*>(reg->keep_buf);
            a.redo = reg->keep_buf + std::max<size_t>(ns, 1);
            a.keep_infl = keep_frac >= 0.0f ? keep_frac * a.grid.lv[0].cell : -1.0f;
        }
        x.seq0 = comm->seq;  // advanced by spx_registration_align_sharded_finish, by the iterations that ran
        SPX_CUDA(cudaMemsetAsync(x.error, 0, sizeof(unsigned int), st));
        reg->timed = false;
        SPX_CUDA(cudaEventRecord(reg->ev0, st));
        if (max_it > 0) launch_align_gn<true>(c.reg, a, max_it, q, reg);
        SPX_CUDA(cudaEventRecord(reg->ev1, st));
        reg->shard_comm = comm;
        reg->shard_max_it = max_it;
    });
}

int spx_registration_align_sharded_finish(spx_registration_t reg, spx_registration_result* R) {
    float4* dn = nullptr;
    const int rc = guard([&] {
        SPX_REQUIRE(reg && R, "[Registration::align_sharded] null argument");
        SPX_REQUIRE(reg->shard_comm, "[Registration::align_sharded] no sharded align in flight");
        spx_queue_t q = reg->q;
        DeviceGuard g(q->device);
        spx_comm_t comm = reg->shard_comm;
        reg->shard_comm = nullptr;
        dn = reg->shard_derived_normals;
        reg->shard_derived_normals = nullptr;
        char* pin = static_cast<char*>(q->pinned_get(sizeof(RegState) + 64 + 32 * sizeof(double)));
        RegState* hs = reinterpret_cast<RegState*>(pin);
        unsigned int* herr = reinterpret_cast<unsigned int*>(pin + sizeof(RegState));
        SPX_CUDA(cudaMemcpyAsync(hs, reg->state, sizeof(RegState), cudaMemcpyDeviceToHost, q->stream));
        SPX_CUDA(cudaMemcpyAsync(herr, comm->local + SPX_MBOX_ERROR, sizeof(unsigned int), cudaMemcpyDeviceToHost,
                                 q->stream));
        q->sync();
        if (*herr) throw Error(SPX_ERR_INTERNAL, "[Registration::align_sharded] a peer rank did not answer (timeout)");
        if (reg->shard_max_it > 0) {
            // every rank ran the same number of exchanges (identical poses -> identical stop): the next align's
            // first row follows this align's last one in sequence
            comm->seq += (unsigned long long)(hs->iterations + 1);
            fill_result(*hs, R);
            reg->timed = true;
            reg->last_launches = 1;
            reg->last_iterations = hs->iterations + 1;
        } else {
            std::memset(R, 0, sizeof(*R));
            for (int j = 0; j < 4; ++j)
                for (int i = 0; i < 4; ++i) R->T[j * 4 + i] = hs->T[i][j];
            R->error = FLT_MAX;
            R->error_raw = FLT_MAX;
        }
    });
    if (dn) {
        cudaStreamSynchronize(reg->q->stream);
        cudaFree(dn);
    }
    return rc;
}

}  // extern "C"
