// CPU reference of correspondence RANSAC (DESIGN.md §3.6), for the tests only: the counter-based sampler, the edge and
// degeneracy checks, the fp64 closed-form triad pose rounded to fp32 and the strict fp32 inlier count.  Built by
// tests/global_reference.py with -ffp-contract=off, so every operation is the one written here.
#include <cmath>
#include <cstddef>
#include <cstdint>

static inline uint64_t splitmix64(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

static inline uint32_t draw(uint64_t seed, uint64_t h, uint64_t s, uint64_t m) {
    const uint64_t r = splitmix64(seed + (3 * h + s + 1) * 0x9E3779B97F4A7C15ull);
    return (uint32_t)(((r >> 32) * m) >> 32);
}

static inline double dot3(const double* a, const double* b) { return std::fma(a[2], b[2], std::fma(a[1], b[1], a[0] * b[0])); }
static inline void cross3(const double* a, const double* b, double* c) {
    c[0] = std::fma(a[1], b[2], -(a[2] * b[1]));
    c[1] = std::fma(a[2], b[0], -(a[0] * b[2]));
    c[2] = std::fma(a[0], b[1], -(a[1] * b[0]));
}

static bool frame(const float* x0, const float* x1, const float* x2, double F[3][3], double c[3]) {
    double u[3], v[3], n[3], e1[3], e2[3], e3[3];
    for (int r = 0; r < 3; ++r) {
        u[r] = (double)x1[r] - (double)x0[r];
        v[r] = (double)x2[r] - (double)x0[r];
        c[r] = (((double)x0[r] + (double)x1[r]) + (double)x2[r]) / 3.0;
    }
    cross3(u, v, n);
    const double l2 = dot3(n, n), uu = dot3(u, u), vv = dot3(v, v);
    if (!(l2 > 1e-12 * uu * vv)) return false;
    const double lu = std::sqrt(uu), ln = std::sqrt(l2);
    for (int r = 0; r < 3; ++r) {
        e1[r] = u[r] / lu;
        e3[r] = n[r] / ln;
    }
    cross3(e3, e1, e2);
    for (int r = 0; r < 3; ++r) {
        F[r][0] = e1[r];
        F[r][1] = e2[r];
        F[r][2] = e3[r];
    }
    return true;
}

static inline double edge2(const float* a, const float* b) {
    const double d[3] = {(double)a[0] - (double)b[0], (double)a[1] - (double)b[1], (double)a[2] - (double)b[2]};
    return dot3(d, d);
}

// P: rows (R_r0, R_r1, R_r2, t_r); p, q: xyz
static inline bool inlier(const float* P, const float* p, const float* q, float eps2) {
    float d[3];
    for (int r = 0; r < 3; ++r) {
        const float y = std::fma(P[4 * r + 2], p[2], std::fma(P[4 * r + 1], p[1], std::fma(P[4 * r], p[0], P[4 * r + 3])));
        d[r] = y - q[r];
    }
    return std::fma(d[2], d[2], std::fma(d[1], d[1], d[0] * d[0])) < eps2;
}

// c[3h + s] = the correspondence hypothesis h draws for sample s
extern "C" void ref_ransac_draws(uint32_t H, uint64_t seed, uint64_t m, uint32_t* c) {
    for (uint64_t h = 0; h < H; ++h)
        for (uint64_t s = 0; s < 3; ++s) c[3 * h + s] = draw(seed, h, s, m);
}

// the triad pose of p[0..2] -> q[0..2] (xyz rows of 3 floats) into P[12] (fp32) and P64[12] (nullable: the fp64 pose
// before rounding); 0 when a triangle is degenerate
extern "C" int ref_triad(const float* p, const float* q, float* P, double* P64) {
    double Fp[3][3], Fq[3][3], cp[3], cq[3];
    if (!frame(p, p + 3, p + 6, Fp, cp) || !frame(q, q + 3, q + 6, Fq, cq)) return 0;
    for (int r = 0; r < 3; ++r) {
        double R[3];
        for (int c = 0; c < 3; ++c) R[c] = std::fma(Fq[r][2], Fp[c][2], std::fma(Fq[r][1], Fp[c][1], Fq[r][0] * Fp[c][0]));
        const double t = cq[r] - std::fma(R[2], cp[2], std::fma(R[1], cp[1], R[0] * cp[0]));
        P[4 * r] = (float)R[0];
        P[4 * r + 1] = (float)R[1];
        P[4 * r + 2] = (float)R[2];
        P[4 * r + 3] = (float)t;
        if (P64) {
            for (int c = 0; c < 3; ++c) P64[4 * r + c] = R[c];
            P64[4 * r + 3] = t;
        }
    }
    return 1;
}

// 1 iff the three edges pass ds^2 >= tau^2 dt^2 and dt^2 >= tau^2 ds^2 (fp64, tau^2 from the fp32 tau)
extern "C" int ref_edges_ok(const float* p, const float* q, float tau) {
    const double t2 = (double)tau * (double)tau;
    const int A[3] = {0, 0, 1}, B[3] = {1, 2, 2};
    for (int e = 0; e < 3; ++e) {
        const double ds = edge2(p + 3 * A[e], p + 3 * B[e]), dt = edge2(q + 3 * A[e], q + 3 * B[e]);
        if (!(ds >= t2 * dt && dt >= t2 * ds)) return 0;
    }
    return 1;
}

// Every hypothesis over the M correspondences (ps[k], qs[k]: xyz float rows of 3, the pairs already gathered; a
// non-finite pair makes the hypotheses sampling it invalid and is never an inlier): pose[12h..] (NaN when invalid),
// sample0[h] (-1 when invalid), counts[h] (0xFFFFFFFF when invalid).
extern "C" void ref_ransac_hypotheses(const float* ps, const float* qs, size_t M, uint32_t H, uint64_t seed, float tau,
                                      float eps, float* pose, int64_t* sample0, uint32_t* counts) {
    const float eps2 = eps * eps;
#pragma omp parallel for schedule(dynamic, 16)
    for (int64_t h = 0; h < (int64_t)H; ++h) {
        float* P = pose + 12 * h;
        for (int e = 0; e < 12; ++e) P[e] = std::nanf("");
        sample0[h] = -1;
        counts[h] = 0xFFFFFFFFu;
        const uint32_t c[3] = {draw(seed, h, 0, M), draw(seed, h, 1, M), draw(seed, h, 2, M)};
        if (M < 3 || c[0] == c[1] || c[0] == c[2] || c[1] == c[2]) continue;
        float p[9], q[9];
        bool fin = true;
        for (int s = 0; s < 3; ++s)
            for (int r = 0; r < 3; ++r) {
                p[3 * s + r] = ps[3 * c[s] + r];
                q[3 * s + r] = qs[3 * c[s] + r];
                fin = fin && std::isfinite(p[3 * s + r]) && std::isfinite(q[3 * s + r]);
            }
        if (!fin || !ref_edges_ok(p, q, tau)) continue;
        float T[12];
        if (!ref_triad(p, q, T, nullptr)) continue;
        for (int e = 0; e < 12; ++e) P[e] = T[e];
        sample0[h] = c[0];
        uint32_t cnt = 0;
        for (size_t k = 0; k < M; ++k) cnt += inlier(T, ps + 3 * k, qs + 3 * k, eps2) ? 1u : 0u;
        counts[h] = cnt;
    }
}

// flags[k] = 1 iff correspondence k is an inlier of the pose P[12]
extern "C" void ref_ransac_inliers(const float* ps, const float* qs, size_t M, const float* P, float eps, uint8_t* flags) {
    const float eps2 = eps * eps;
    for (size_t k = 0; k < M; ++k) flags[k] = inlier(P, ps + 3 * k, qs + 3 * k, eps2) ? 1 : 0;
}
