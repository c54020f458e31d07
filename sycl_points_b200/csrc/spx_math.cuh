// Small fixed-size math used inside the kernels and by the host-side optimiser pieces.
// Rounding contract: where the reference spells an fma chain (I/utils/eigen_utils.hpp), the same
// chain is spelled here with __fmaf_rn/__fmul_rn (device) so nvcc neither fuses nor splits
// anything; symmetric 3x3 matrices are carried as their 6 upper-triangle entries.
#pragma once

#include <cmath>

#include "spx_common.cuh"

#ifdef __CUDA_ARCH__
#define SPX_FMA(a, b, c) __fmaf_rn((a), (b), (c))
#define SPX_MUL(a, b) __fmul_rn((a), (b))
#define SPX_ADD(a, b) __fadd_rn((a), (b))
#define SPX_SUB(a, b) __fsub_rn((a), (b))
#define SPX_DIV(a, b) __fdiv_rn((a), (b))
#else
#define SPX_FMA(a, b, c) fmaf((a), (b), (c))
#define SPX_MUL(a, b) ((a) * (b))
#define SPX_ADD(a, b) ((a) + (b))
#define SPX_SUB(a, b) ((a) - (b))
#define SPX_DIV(a, b) ((a) / (b))
#endif

#define SPX_HD __host__ __device__ __forceinline__

namespace spx {

// Transcendentals.  The reference calls sycl::cos / acos / cbrt / sin / log / pow, whose rounding is
// implementation-defined (SURVEY.md §8(c): unpinned).  The contract here and in the oracle is the
// CORRECTLY ROUNDED fp32 value, obtained by evaluating in fp64 and rounding once: CUDA's and glibc's
// fp64 routines are both < 2 ulp(fp64), so the two sides round to the same float except when the
// exact value lies within ~1e-16 relative of a rounding boundary (probability ~1e-8 per call).
// None of these sit on a per-iteration hot loop (plane regularisation and normals run once per
// point per align; se3_exp once per iteration on one thread).
SPX_HD float cr_cosf(float x) { return (float)cos((double)x); }
SPX_HD float cr_sinf(float x) { return (float)sin((double)x); }
SPX_HD float cr_acosf(float x) { return (float)acos((double)x); }
SPX_HD float cr_cbrtf(float x) { return (float)cbrt((double)x); }
SPX_HD float cr_logf(float x) { return (float)log((double)x); }
SPX_HD float cr_cubef(float x) {  // pow(x, 3.0f)
    const double d = (double)x;
    return (float)(d * d * d);
}

// symmetric 3x3: xx xy xz yy yz zz (what covariance::estimate produces: exactly symmetric)
struct Sym3 {
    float xx, xy, xz, yy, yz, zz;
};

// general 3x3, row-major m[i][j].  The reference's covariance arithmetic (update_covariance_plane,
// transform_covs, inverse) runs on FULL matrices: V diag V^T, R C R^T and the adjugate are symmetric
// only up to rounding, and with GICP's 1e-3 regularisation (condition ~1e3) an ulp of asymmetry is
// 1e-4 relative in H.  Every consumer therefore carries all nine entries, like the reference.
struct Mat3 {
    float m[3][3];
};

SPX_HD Mat3 mat3_from_sym(const Sym3& s) {
    Mat3 r;
    r.m[0][0] = s.xx; r.m[0][1] = s.xy; r.m[0][2] = s.xz;
    r.m[1][0] = s.xy; r.m[1][1] = s.yy; r.m[1][2] = s.yz;
    r.m[2][0] = s.xz; r.m[2][1] = s.yz; r.m[2][2] = s.zz;
    return r;
}
SPX_HD Mat3 mat3_identity() {
    Mat3 r;
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) r.m[i][j] = (i == j) ? 1.0f : 0.0f;
    return r;
}

// a*b - c*d the way eigen_utils.hpp writes its 2x2 minors: fma(a, b, -(c*d))
SPX_HD float minor2(float a, float b, float c, float d) { return SPX_FMA(a, b, -SPX_MUL(c, d)); }

// determinant(A) — eigen_utils.hpp:303-307
SPX_HD float mat3_det(const Mat3& A) {
    return SPX_FMA(A.m[0][0], minor2(A.m[1][1], A.m[2][2], A.m[1][2], A.m[2][1]),
                   SPX_FMA(-A.m[0][1], minor2(A.m[1][0], A.m[2][2], A.m[1][2], A.m[2][0]),
                           SPX_MUL(A.m[0][2], minor2(A.m[1][0], A.m[2][1], A.m[1][1], A.m[2][0]))));
}

// inverse(A) — eigen_utils.hpp:403-423: adjugate / det, the ZERO matrix when |det| < 1e-6
SPX_HD Mat3 mat3_inverse(const Mat3& s) {
    const float det = mat3_det(s);
    Mat3 r;
    if (fabsf(det) < 1e-6f) {
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) r.m[i][j] = 0.0f;
        return r;
    }
    const float id = SPX_DIV(1.0f, det);
    r.m[0][0] = SPX_MUL(minor2(s.m[1][1], s.m[2][2], s.m[1][2], s.m[2][1]), id);
    r.m[1][0] = SPX_MUL(minor2(s.m[1][2], s.m[2][0], s.m[1][0], s.m[2][2]), id);
    r.m[2][0] = SPX_MUL(minor2(s.m[1][0], s.m[2][1], s.m[1][1], s.m[2][0]), id);
    r.m[0][1] = SPX_MUL(minor2(s.m[0][2], s.m[2][1], s.m[0][1], s.m[2][2]), id);
    r.m[1][1] = SPX_MUL(minor2(s.m[0][0], s.m[2][2], s.m[0][2], s.m[2][0]), id);
    r.m[2][1] = SPX_MUL(minor2(s.m[0][1], s.m[2][0], s.m[0][0], s.m[2][1]), id);
    r.m[0][2] = SPX_MUL(minor2(s.m[0][1], s.m[1][2], s.m[0][2], s.m[1][1]), id);
    r.m[1][2] = SPX_MUL(minor2(s.m[0][2], s.m[1][0], s.m[0][0], s.m[1][2]), id);
    r.m[2][2] = SPX_MUL(minor2(s.m[0][0], s.m[1][1], s.m[0][1], s.m[1][0]), id);
    return r;
}

#ifdef __CUDACC__
// symmetric_eigen_decomposition_3x3 — eigen_utils.hpp:443-562 (scaled trigonometric Cardano,
// eigenvalues ascending, eigenvector k = largest-norm column of adj(A - l_k I)), on the full
// matrix exactly as the reference indexes it (both triangles are read).  V holds the eigenvectors in
// its columns; eigenvalues are rescaled at the end.
__device__ inline void mat3_eigen(const Mat3& A, float ev[3], float V[3][3]) {
    constexpr float EPS = 1.1920929e-07f;
    constexpr float FMIN = 1.17549435e-38f;
    constexpr float PI = 3.14159265358979323846f;
    float mx = 0.0f;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) mx = fmaxf(mx, fabsf(A.m[i][j]));
    if (mx < FMIN) {
        ev[0] = ev[1] = ev[2] = 0.0f;
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) V[i][j] = (i == j) ? 1.0f : 0.0f;
        return;
    }
    const float si = __fdiv_rn(1.0f, mx);
    Mat3 S;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) S.m[i][j] = __fmul_rn(A.m[i][j], si);

    const float c2 = -__fadd_rn(__fadd_rn(__fadd_rn(0.0f, S.m[0][0]), S.m[1][1]), S.m[2][2]);
    const float c1 = __fsub_rn(
        __fmaf_rn(S.m[0][0], S.m[1][1], __fmaf_rn(S.m[0][0], S.m[2][2], __fmul_rn(S.m[1][1], S.m[2][2]))),
        __fmaf_rn(S.m[0][1], S.m[1][0], __fmaf_rn(S.m[0][2], S.m[2][0], __fmul_rn(S.m[1][2], S.m[2][1]))));
    const float c0 = -mat3_det(S);

    const float p = __fsub_rn(c1, __fdiv_rn(__fmul_rn(c2, c2), 3.0f));
    const float q = __fadd_rn(__fsub_rn(__fdiv_rn(__fmul_rn(__fmul_rn(__fmul_rn(2.0f, c2), c2), c2), 27.0f),
                                        __fdiv_rn(__fmul_rn(c2, c1), 3.0f)),
                              c0);
    const float disc = __fadd_rn(__fmul_rn(__fmul_rn(__fmul_rn(4.0f, p), p), p), __fmul_rn(__fmul_rn(27.0f, q), q));
    const float c2_3 = __fdiv_rn(c2, 3.0f);
    if (fabsf(disc) <= EPS) {
        const float u = q >= 0 ? -cr_cbrtf(__fdiv_rn(q, 2.0f)) : cr_cbrtf(__fdiv_rn(-q, 2.0f));
        ev[0] = __fsub_rn(__fmul_rn(2.0f, u), c2_3);
        ev[1] = ev[2] = __fsub_rn(-u, c2_3);
    } else {
        const float sp = __fsqrt_rn(__fdiv_rn(-p, 3.0f));
        const float den = __fmul_rn(__fmul_rn(__fmul_rn(2.0f, sp), sp), sp);
        const float cs = fmaxf(-1.0f, fminf(1.0f, __fdiv_rn(-q, den)));
        const float phi = fabsf(p) < EPS ? 0.0f : cr_acosf(cs);
        const float two_sp = __fmul_rn(2.0f, sp);
        ev[0] = __fmaf_rn(two_sp, cr_cosf(__fdiv_rn(phi, 3.0f)), -c2_3);
        ev[2] = __fmaf_rn(two_sp, cr_cosf(__fdiv_rn(__fadd_rn(phi, __fmul_rn(4.0f, PI)), 3.0f)), -c2_3);
        ev[1] = __fmaf_rn(two_sp, cr_cosf(__fdiv_rn(__fadd_rn(phi, __fmul_rn(2.0f, PI)), 3.0f)), -c2_3);
    }
    float t;
    if (ev[0] > ev[1]) { t = ev[0]; ev[0] = ev[1]; ev[1] = t; }
    if (ev[1] > ev[2]) { t = ev[1]; ev[1] = ev[2]; ev[2] = t; }
    if (ev[0] > ev[1]) { t = ev[0]; ev[0] = ev[1]; ev[1] = t; }

#pragma unroll
    for (int k = 0; k < 3; ++k) {
        Mat3 M = S;
        M.m[0][0] = __fsub_rn(S.m[0][0], ev[k]);
        M.m[1][1] = __fsub_rn(S.m[1][1], ev[k]);
        M.m[2][2] = __fsub_rn(S.m[2][2], ev[k]);
        const float m00 = minor2(M.m[1][1], M.m[2][2], M.m[1][2], M.m[2][1]);
        const float m01 = minor2(M.m[1][2], M.m[2][0], M.m[1][0], M.m[2][2]);
        const float m02 = minor2(M.m[1][0], M.m[2][1], M.m[1][1], M.m[2][0]);
        const float m10 = minor2(M.m[0][2], M.m[2][1], M.m[0][1], M.m[2][2]);
        const float m11 = minor2(M.m[0][0], M.m[2][2], M.m[0][2], M.m[2][0]);
        const float m12 = minor2(M.m[0][1], M.m[2][0], M.m[0][0], M.m[2][1]);
        const float m20 = minor2(M.m[0][1], M.m[1][2], M.m[0][2], M.m[1][1]);
        const float m21 = minor2(M.m[0][2], M.m[1][0], M.m[0][0], M.m[1][2]);
        const float m22 = minor2(M.m[0][0], M.m[1][1], M.m[0][1], M.m[1][0]);
        const float s0 = __fmaf_rn(m00, m00, __fmaf_rn(m10, m10, __fmul_rn(m20, m20)));
        const float s1 = __fmaf_rn(m01, m01, __fmaf_rn(m11, m11, __fmul_rn(m21, m21)));
        const float s2 = __fmaf_rn(m02, m02, __fmaf_rn(m12, m12, __fmul_rn(m22, m22)));
        float vx, vy, vz;
        if (s0 >= s1 && s0 >= s2) {
            vx = m00; vy = m10; vz = m20;
        } else if (s1 >= s0 && s1 >= s2) {
            vx = m01; vy = m11; vz = m21;
        } else {
            vx = m02; vy = m12; vz = m22;
        }
        float n2 = __fadd_rn(__fadd_rn(__fmul_rn(vx, vx), __fmul_rn(vy, vy)), __fmul_rn(vz, vz));
        if (n2 < FMIN) {
            vx = 1.0f; vy = 0.0f; vz = 0.0f;
            n2 = 1.0f;
        }
        const float il = __fdiv_rn(1.0f, __fsqrt_rn(n2));
        V[0][k] = __fmul_rn(vx, il);
        V[1][k] = __fmul_rn(vy, il);
        V[2][k] = __fmul_rn(vz, il);
    }
    ev[0] = __fmul_rn(ev[0], mx);
    ev[1] = __fmul_rn(ev[1], mx);
    ev[2] = __fmul_rn(ev[2], mx);
}

// update_covariance_plane — I/algorithms/feature/covariance.hpp:67-74: C <- (V diag(1e-3,1,1)) V^T
// (eigenvalues discarded), all nine entries of the reference's fma chains: entry (i,j) and (j,i)
// differ in the rounding of (V_i0 * 1e-3) * V_j0.
__device__ inline Mat3 plane_regularize(const Mat3& C) {
    float ev[3], V[3][3];
    mat3_eigen(C, ev, V);
    float VD[3][3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        VD[i][0] = __fmul_rn(V[i][0], 1e-3f);
        VD[i][1] = V[i][1];
        VD[i][2] = V[i][2];
    }
    Mat3 r;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j)
            r.m[i][j] = __fmaf_rn(VD[i][2], V[j][2], __fmaf_rn(VD[i][1], V[j][1], __fmul_rn(VD[i][0], V[j][0])));
    return r;
}

// covariance stored by the reference: float[16] column-major 4x4 — all nine entries of the upper 3x3
__device__ __forceinline__ Mat3 load_cov16(const float* __restrict__ c) {
    const float4 c0 = __ldg(reinterpret_cast<const float4*>(c));
    const float4 c1 = __ldg(reinterpret_cast<const float4*>(c) + 1);
    const float4 c2 = __ldg(reinterpret_cast<const float4*>(c) + 2);
    Mat3 s;
    s.m[0][0] = c0.x; s.m[1][0] = c0.y; s.m[2][0] = c0.z;
    s.m[0][1] = c1.x; s.m[1][1] = c1.y; s.m[2][1] = c1.z;
    s.m[0][2] = c2.x; s.m[1][2] = c2.y; s.m[2][2] = c2.z;
    return s;
}
__device__ __forceinline__ void store_cov16(float* __restrict__ out, const Mat3& C) {
    float4* o = reinterpret_cast<float4*>(out);
    o[0] = make_float4(C.m[0][0], C.m[1][0], C.m[2][0], 0.f);
    o[1] = make_float4(C.m[0][1], C.m[1][1], C.m[2][1], 0.f);
    o[2] = make_float4(C.m[0][2], C.m[1][2], C.m[2][2], 0.f);
    o[3] = make_float4(0.f, 0.f, 0.f, 0.f);
}
#endif  // __CUDACC__

#ifdef __CUDACC__
// ------------------------------------------------------------------ robust kernels (robust.hpp:56-114)
__device__ __forceinline__ float robust_weight(int loss, float r, float s) {
    if (loss == SPX_LOSS_NONE) return 1.0f;
    if (r <= 1e-8f) return 1.0f;
    const float x = __fdiv_rn(r, s);
    switch (loss) {
        case SPX_LOSS_HUBER: return fminf(1.0f, __fdiv_rn(1.0f, x));
        case SPX_LOSS_TUKEY: {
            if (x >= 1.0f) return 0.0f;
            const float f = __fsub_rn(1.0f, __fmul_rn(x, x));
            return __fmul_rn(f, f);
        }
        case SPX_LOSS_CAUCHY: return __fdiv_rn(1.0f, __fadd_rn(1.0f, __fmul_rn(x, x)));
        default: {
            const float d = __fadd_rn(1.0f, __fmul_rn(x, x));
            return __fdiv_rn(1.0f, __fmul_rn(d, d));
        }
    }
}

__device__ __forceinline__ float robust_error(int loss, float r, float s) {
    const float r2 = __fmul_rn(r, r), s2 = __fmul_rn(s, s);
    switch (loss) {
        case SPX_LOSS_HUBER:
            return r <= s ? __fmul_rn(__fmul_rn(0.5f, r), r) : __fmul_rn(s, __fsub_rn(r, __fmul_rn(0.5f, s)));
        case SPX_LOSS_TUKEY:
            return r <= s ? __fmul_rn(__fdiv_rn(s2, 6.0f), __fsub_rn(1.0f, cr_cubef(__fsub_rn(1.0f, __fdiv_rn(r2, s2)))))
                          : __fdiv_rn(s2, 6.0f);
        case SPX_LOSS_CAUCHY:
            return __fmul_rn(__fmul_rn(__fmul_rn(0.5f, s), s), cr_logf(__fadd_rn(1.0f, __fdiv_rn(r2, s2))));
        case SPX_LOSS_GEMAN_MCCLURE:
            return __fdiv_rn(__fmul_rn(0.5f, __fmul_rn(__fmul_rn(s2, r), r)), __fadd_rn(s2, r2));
        default: return __fmul_rn(__fmul_rn(0.5f, r), r);
    }
}

#endif  // __CUDACC__

// ---------------------------------------------------------------- SE(3) pieces (host + device)
// lie::se3_exp — eigen_utils.hpp:886-943 (so3_exp -> quaternion -> rotation; V matrix).  Row-major out.
SPX_HD void se3_exp_rm(const float a[6], float T[4][4]) {
    const float ox = a[0], oy = a[1], oz = a[2];
    const float th2 = SPX_FMA(oz, oz, SPX_FMA(oy, oy, SPX_MUL(ox, ox)));
    float imag, real;
    if (th2 < 1e-6f) {
        const float th4 = SPX_MUL(th2, th2);
        imag = SPX_ADD(SPX_SUB(0.5f, SPX_MUL(SPX_DIV(1.0f, 48.0f), th2)), SPX_MUL(SPX_DIV(1.0f, 3840.0f), th4));
        real = SPX_ADD(SPX_SUB(1.0f, SPX_MUL(SPX_DIV(1.0f, 8.0f), th2)), SPX_MUL(SPX_DIV(1.0f, 384.0f), th4));
    } else {
        const float th = sqrtf(th2);
        const float h = SPX_MUL(0.5f, th);
        imag = SPX_DIV(cr_sinf(h), th);
        real = cr_cosf(h);
    }
    const float x = SPX_MUL(imag, ox), y = SPX_MUL(imag, oy), z = SPX_MUL(imag, oz), w = real;
    const float x2 = SPX_MUL(x, x), y2 = SPX_MUL(y, y), z2 = SPX_MUL(z, z);
    const float xy = SPX_MUL(x, y), xz = SPX_MUL(x, z), yz = SPX_MUL(y, z);
    const float wx = SPX_MUL(w, x), wy = SPX_MUL(w, y), wz = SPX_MUL(w, z);
    float R[3][3];
    R[0][0] = SPX_SUB(1.0f, SPX_MUL(2.0f, SPX_ADD(y2, z2)));
    R[0][1] = SPX_MUL(2.0f, SPX_SUB(xy, wz));
    R[0][2] = SPX_MUL(2.0f, SPX_ADD(xz, wy));
    R[1][0] = SPX_MUL(2.0f, SPX_ADD(xy, wz));
    R[1][1] = SPX_SUB(1.0f, SPX_MUL(2.0f, SPX_ADD(x2, z2)));
    R[1][2] = SPX_MUL(2.0f, SPX_SUB(yz, wx));
    R[2][0] = SPX_MUL(2.0f, SPX_SUB(xz, wy));
    R[2][1] = SPX_MUL(2.0f, SPX_ADD(yz, wx));
    R[2][2] = SPX_SUB(1.0f, SPX_MUL(2.0f, SPX_ADD(x2, y2)));
    for (int i = 0; i < 4; ++i)
        for (int j = 0; j < 4; ++j) T[i][j] = (i == j) ? 1.0f : 0.0f;
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) T[i][j] = R[i][j];
    const float tv[3] = {a[3], a[4], a[5]};
    const float th = sqrtf(th2);
    float Vm[3][3];
    if (th < 1e-6f) {
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) Vm[i][j] = R[i][j];
    } else {
        const float Om[3][3] = {{0.0f, -oz, oy}, {oz, 0.0f, -ox}, {-oy, ox, 0.0f}};
        float Om2[3][3];
        for (int j = 0; j < 3; ++j)
            for (int i = 0; i < 3; ++i) {
                float s = 0.0f;
                for (int k = 0; k < 3; ++k) s = SPX_FMA(Om[i][k], Om[k][j], s);
                Om2[i][j] = s;
            }
        const float A = SPX_DIV(SPX_SUB(1.0f, cr_cosf(th)), th2);
        const float B = SPX_DIV(SPX_SUB(th, cr_sinf(th)), SPX_MUL(th2, th));
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j)
                Vm[i][j] = SPX_ADD((i == j) ? 1.0f : 0.0f, SPX_ADD(SPX_MUL(Om[i][j], A), SPX_MUL(Om2[i][j], B)));
    }
    for (int i = 0; i < 3; ++i) {
        float s = 0.0f;
        for (int j = 0; j < 3; ++j) s = SPX_FMA(Vm[i][j], tv[j], s);
        T[i][3] = s;
    }
}

// lie::se3_log — eigen_utils.hpp:774-803 (rotation -> quaternion), :948-986 (so3_log), :991-1034.  Host code in
// the reference too (velocity_update.hpp:71, relative_pose_deskew.hpp:108); atan2 / sin / cos are evaluated in
// fp64 and cast, like every transcendental of this library.  Row-major 4x4 in, [rx ry rz tx ty tz] out.
SPX_HD void se3_log_rm(const float T[4][4], float a[6]) {
    float q[4];
    const float tr = SPX_ADD(SPX_ADD(T[0][0], T[1][1]), T[2][2]);
    if (tr > 0.0f) {
        const float S = SPX_MUL(sqrtf(SPX_ADD(tr, 1.0f)), 2.0f);
        q[0] = SPX_DIV(SPX_SUB(T[2][1], T[1][2]), S);
        q[1] = SPX_DIV(SPX_SUB(T[0][2], T[2][0]), S);
        q[2] = SPX_DIV(SPX_SUB(T[1][0], T[0][1]), S);
        q[3] = SPX_MUL(0.25f, S);
    } else if (T[0][0] > T[1][1] && T[0][0] > T[2][2]) {
        const float S = SPX_MUL(sqrtf(SPX_SUB(SPX_SUB(SPX_ADD(1.0f, T[0][0]), T[1][1]), T[2][2])), 2.0f);
        q[0] = SPX_MUL(0.25f, S);
        q[1] = SPX_DIV(SPX_ADD(T[0][1], T[1][0]), S);
        q[2] = SPX_DIV(SPX_ADD(T[0][2], T[2][0]), S);
        q[3] = SPX_DIV(SPX_SUB(T[2][1], T[1][2]), S);
    } else if (T[1][1] > T[2][2]) {
        const float S = SPX_MUL(sqrtf(SPX_SUB(SPX_SUB(SPX_ADD(1.0f, T[1][1]), T[0][0]), T[2][2])), 2.0f);
        q[0] = SPX_DIV(SPX_ADD(T[0][1], T[1][0]), S);
        q[1] = SPX_MUL(0.25f, S);
        q[2] = SPX_DIV(SPX_ADD(T[1][2], T[2][1]), S);
        q[3] = SPX_DIV(SPX_SUB(T[0][2], T[2][0]), S);
    } else {
        const float S = SPX_MUL(sqrtf(SPX_SUB(SPX_SUB(SPX_ADD(1.0f, T[2][2]), T[0][0]), T[1][1])), 2.0f);
        q[2] = SPX_MUL(0.25f, S);
        q[3] = SPX_DIV(SPX_SUB(T[1][0], T[0][1]), S);
        q[0] = SPX_DIV(SPX_ADD(T[0][2], T[2][0]), S);
        q[1] = SPX_DIV(SPX_ADD(T[1][2], T[2][1]), S);
    }
    // so3_log: normalise, w >= 0, three angle regimes
    const float nrm = sqrtf(SPX_FMA(q[3], q[3], SPX_FMA(q[2], q[2], SPX_FMA(q[1], q[1], SPX_FMA(q[0], q[0], 0.0f)))));
    if (nrm < 1e-6f) {
        q[0] = q[1] = q[2] = q[3] = 0.0f;
    } else {
        const float inv = SPX_DIV(1.0f, nrm);
        for (int i = 0; i < 4; ++i) q[i] = SPX_MUL(q[i], inv);
    }
    if (q[3] < 0.0f)
        for (int i = 0; i < 4; ++i) q[i] = SPX_MUL(q[i], -1.0f);
    const float w = q[3];
    const float n = sqrtf(SPX_FMA(q[2], q[2], SPX_FMA(q[1], q[1], SPX_FMA(q[0], q[0], 0.0f))));
    float sc;
    if (n < 1e-6f) {
        sc = SPX_MUL(SPX_DIV(2.0f, w), SPX_ADD(1.0f, SPX_DIV(SPX_MUL(n, n), SPX_MUL(SPX_MUL(6.0f, w), w))));
    } else if (fabsf(w) < 1e-6f) {
        sc = SPX_DIV(3.14159265358979323846f, n);
    } else {
        sc = SPX_DIV(SPX_MUL(2.0f, (float)atan2((double)n, (double)fabsf(w))), n);
    }
    const float om[3] = {SPX_MUL(q[0], sc), SPX_MUL(q[1], sc), SPX_MUL(q[2], sc)};
    a[0] = om[0];
    a[1] = om[1];
    a[2] = om[2];
    const float th = sqrtf(SPX_FMA(om[2], om[2], SPX_FMA(om[1], om[1], SPX_FMA(om[0], om[0], 0.0f))));
    const float Om[3][3] = {{0.0f, -om[2], om[1]}, {om[2], 0.0f, -om[0]}, {-om[1], om[0], 0.0f}};
    float Vinv[3][3];
    if (th < 1e-6f) {
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) Vinv[i][j] = SPX_SUB((i == j) ? 1.0f : 0.0f, SPX_MUL(0.5f, Om[i][j]));
    } else {
        const float h = SPX_MUL(0.5f, th);
        const float sh = cr_sinf(h), ch = cr_cosf(h);
        const float coeff = SPX_DIV(SPX_SUB(1.0f, SPX_DIV(SPX_MUL(th, ch), SPX_MUL(2.0f, sh))), SPX_MUL(th, th));
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) {
                float s2 = 0.0f;
                for (int k = 0; k < 3; ++k) s2 = SPX_ADD(s2, SPX_MUL(Om[i][k], Om[k][j]));
                Vinv[i][j] = SPX_ADD(SPX_SUB((i == j) ? 1.0f : 0.0f, SPX_MUL(0.5f, Om[i][j])), SPX_MUL(coeff, s2));
            }
    }
    for (int i = 0; i < 3; ++i) {
        float s = 0.0f;
        for (int k = 0; k < 3; ++k) s = SPX_ADD(s, SPX_MUL(Vinv[i][k], T[k][3]));
        a[3 + i] = s;
    }
}

// result.T * Isometry3f(se3_exp(delta)) — registration.hpp:814 (Eigen isometry product:
// linear = L1*L2, translation = L1*t2 + t1).  Row-major 4x4.
SPX_HD void isometry_mul_rm(const float A[4][4], const float B[4][4], float out[4][4]) {
    float r[4][4];
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) {
            float s = 0.0f;
            for (int k = 0; k < 3; ++k) s = SPX_ADD(s, SPX_MUL(A[i][k], B[k][j]));
            r[i][j] = s;
        }
        float s = 0.0f;
        for (int k = 0; k < 3; ++k) s = SPX_ADD(s, SPX_MUL(A[i][k], B[k][3]));
        r[i][3] = SPX_ADD(s, A[i][3]);
    }
    r[3][0] = r[3][1] = r[3][2] = 0.0f;
    r[3][3] = 1.0f;
    for (int i = 0; i < 4; ++i)
        for (int j = 0; j < 4; ++j) out[i][j] = r[i][j];
}

// ---------------------------------------------------------------- 6x6 LDL^T (fp64, diagonal pivoting)
// Stands in for Eigen::LDLT<Matrix<float,6,6>> at registration.hpp:791-801 / dogleg_step.hpp:43-50
// (Eigen is an unpinned third-party dependency of the reference; the factorisation is evaluated
// in fp64 and the solution cast to fp32, which agrees with any backward-stable fp32 LDLT to far
// below the 1e-5 pose tolerance).
struct Ldlt6 {
    double L[6][6];
    double D[6];
    int perm[6];
    bool ok;
};

SPX_HD void ldlt6_compute(const double Ain[6][6], Ldlt6& f) {
    double A[6][6];
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j < 6; ++j) A[i][j] = Ain[i][j];
    for (int i = 0; i < 6; ++i) f.perm[i] = i;
    f.ok = true;
    for (int k = 0; k < 6; ++k) {
        int piv = k;
        double best = fabs(A[k][k]);
        for (int i = k + 1; i < 6; ++i)
            if (fabs(A[i][i]) > best) {
                best = fabs(A[i][i]);
                piv = i;
            }
        if (piv != k) {
            for (int j = 0; j < 6; ++j) {
                const double t = A[k][j];
                A[k][j] = A[piv][j];
                A[piv][j] = t;
            }
            for (int j = 0; j < 6; ++j) {
                const double t = A[j][k];
                A[j][k] = A[j][piv];
                A[j][piv] = t;
            }
            const int t = f.perm[k];
            f.perm[k] = f.perm[piv];
            f.perm[piv] = t;
        }
        const double d = A[k][k];
        if (d == 0.0) {
            for (int i = k + 1; i < 6; ++i) {
                if (A[i][k] != 0.0) f.ok = false;
                A[i][k] = 0.0;
            }
            continue;
        }
        for (int i = k + 1; i < 6; ++i) A[i][k] /= d;
        for (int i = k + 1; i < 6; ++i)
            for (int j = k + 1; j <= i; ++j) {
                A[i][j] -= A[i][k] * d * A[j][k];
                A[j][i] = A[i][j];
            }
    }
    for (int i = 0; i < 6; ++i) {
        f.D[i] = A[i][i];
        for (int j = 0; j < 6; ++j) f.L[i][j] = (j < i) ? A[i][j] : (i == j ? 1.0 : 0.0);
    }
}

SPX_HD void ldlt6_solve(const Ldlt6& f, const double rhs[6], double x[6]) {
    double y[6];
    for (int i = 0; i < 6; ++i) y[i] = rhs[f.perm[i]];
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j < i; ++j) y[i] -= f.L[i][j] * y[j];
    for (int i = 0; i < 6; ++i) y[i] = (fabs(f.D[i]) > 2.2250738585072014e-308) ? y[i] / f.D[i] : 0.0;
    for (int i = 5; i >= 0; --i)
        for (int j = i + 1; j < 6; ++j) y[i] -= f.L[j][i] * y[j];
    for (int i = 0; i < 6; ++i) x[f.perm[i]] = y[i];
}

// solve (H + lambda I) delta = -b; H row-major 36 floats.  registration.hpp:791-801,806-808.
SPX_HD bool solve_damped6(const float* H, const float* b, float lambda, float* delta) {
    double A[6][6], rhs[6], x[6];
    for (int i = 0; i < 6; ++i) {
        for (int j = 0; j < 6; ++j) A[i][j] = (double)H[i * 6 + j];
        A[i][i] = (double)SPX_ADD(H[i * 6 + i], lambda);
        rhs[i] = -(double)b[i];
    }
    Ldlt6 f;
    ldlt6_compute(A, f);
    if (!f.ok) {
        for (int i = 0; i < 6; ++i) delta[i] = 0.0f;
        return false;
    }
    ldlt6_solve(f, rhs, x);
    for (int i = 0; i < 6; ++i) delta[i] = (float)x[i];
    return true;
}

#ifdef __CUDACC__
// Device fast path of solve_damped6 for the in-kernel Gauss-Newton step: H + lambda I is symmetric
// positive definite in every healthy iteration, so the factorisation needs no pivoting and, fully
// unrolled, lives in registers (the pivoted version indexes its arrays dynamically, i.e. local
// memory: ~9 us on one thread, which every block of the cooperative kernel waited for).  Any
// non-positive or tiny pivot falls back to the pivoted routine, so degenerate systems behave as
// before.  Same fp64 arithmetic, different elimination order: solutions agree to ~1e-15 relative.
__device__ __forceinline__ bool solve_damped6_device(const float* H, const float* b, float lambda, float* delta) {
    double A[6][6];
    double maxd = 0.0;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
#pragma unroll
        for (int j = 0; j < i; ++j) A[i][j] = (double)H[i * 6 + j];
        A[i][i] = (double)SPX_ADD(H[i * 6 + i], lambda);
        maxd = fmax(maxd, A[i][i]);
    }
    bool ok = maxd > 0.0;
    double y[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) y[i] = -(double)b[i];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        const double d = A[k][k];
        ok = ok && d > 1e-10 * maxd && isfinite(d);
        const double inv = 1.0 / d;
        double l[6];
#pragma unroll
        for (int i = k + 1; i < 6; ++i) l[i] = A[i][k] * inv;
#pragma unroll
        for (int i = k + 1; i < 6; ++i) {
#pragma unroll
            for (int j = k + 1; j <= i; ++j) A[i][j] -= l[i] * A[j][k];
        }
#pragma unroll
        for (int i = k + 1; i < 6; ++i) {
            A[i][k] = l[i];
            y[i] -= l[i] * y[k];  // forward substitution rides along
        }
    }
    if (!ok) return solve_damped6(H, b, lambda, delta);
#pragma unroll
    for (int i = 0; i < 6; ++i) y[i] /= A[i][i];
#pragma unroll
    for (int i = 5; i >= 0; --i) {
#pragma unroll
        for (int j = i + 1; j < 6; ++j) y[i] -= A[j][i] * y[j];
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) delta[i] = (float)y[i];
    return true;
}
#endif

SPX_HD float norm3f(const float* v) {
    return sqrtf(SPX_ADD(SPX_ADD(SPX_MUL(v[0], v[0]), SPX_MUL(v[1], v[1])), SPX_MUL(v[2], v[2])));
}

// ---------------------------------------------------------------- RANSAC sampling (DESIGN.md §3.5, §3.6)
// the SplitMix64 finalizer
SPX_HD unsigned long long splitmix64(unsigned long long z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// the position in [0, count) that hypothesis h draws for its sample s: a counter-based stream keyed by the seed, the
// same for the plane RANSAC and the correspondence RANSAC (uint64 wrap-around throughout)
SPX_HD uint32_t ransac_draw(unsigned long long seed, unsigned long long h, unsigned long long s,
                            unsigned long long count) {
    const unsigned long long r = splitmix64(seed + (3ull * h + s + 1ull) * 0x9E3779B97F4A7C15ull);
    return (uint32_t)(((r >> 32) * count) >> 32);
}

// eigen-decomposition of a symmetric 3x3 by cyclic Jacobi rotations in fp64 (the reference calls
// Eigen::SelfAdjointEigenSolver<Matrix3f>, third-party and unpinned: any backward-stable solver agrees with it to
// fp32 rounding).  evec columns = eigenvectors.  Called host-side by the nl-reg regularisation (fp32 input) and
// device-side by the RANSAC plane refinement (fp64 input).
template <class T>
SPX_HD void jacobi3(const T A[3][3], double ev[3], double V[3][3]) {
    double a[3][3];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            a[i][j] = 0.5 * ((double)A[i][j] + (double)A[j][i]);
            V[i][j] = i == j ? 1.0 : 0.0;
        }
    for (int sweep = 0; sweep < 32; ++sweep) {
        const double off = a[0][1] * a[0][1] + a[0][2] * a[0][2] + a[1][2] * a[1][2];
        if (off < 1e-300) break;
        for (int p = 0; p < 2; ++p)
            for (int q = p + 1; q < 3; ++q) {
                if (a[p][q] == 0.0) continue;
                const double theta = (a[q][q] - a[p][p]) / (2.0 * a[p][q]);
                const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                const double c = 1.0 / sqrt(t * t + 1.0), s_ = t * c;
                for (int k = 0; k < 3; ++k) {
                    const double akp = a[k][p], akq = a[k][q];
                    a[k][p] = c * akp - s_ * akq;
                    a[k][q] = s_ * akp + c * akq;
                }
                for (int k = 0; k < 3; ++k) {
                    const double apk = a[p][k], aqk = a[q][k];
                    a[p][k] = c * apk - s_ * aqk;
                    a[q][k] = s_ * apk + c * aqk;
                }
                for (int k = 0; k < 3; ++k) {
                    const double vkp = V[k][p], vkq = V[k][q];
                    V[k][p] = c * vkp - s_ * vkq;
                    V[k][q] = s_ * vkp + c * vkq;
                }
            }
    }
    for (int i = 0; i < 3; ++i) ev[i] = a[i][i];
}

}  // namespace spx
