// CPU reference of RANSAC plane segmentation (DESIGN.md §3.5), for the tests only: the counter-based sampler, the fp64
// plane of a hypothesis with every fma written out, its validity, its fp32 coefficients and its strict fp32 inlier
// count.  Built by tests/plane_reference.py with -ffp-contract=off, so every operation is the one written here.
#include <cmath>
#include <cstddef>
#include <cstdint>

static inline uint64_t splitmix64(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

static inline bool finite3(const float* p) { return std::isfinite(p[0]) && std::isfinite(p[1]) && std::isfinite(p[2]); }

static inline double dot3(double ax, double ay, double az, double bx, double by, double bz) {
    return std::fma(az, bz, std::fma(ay, by, ax * bx));
}

static inline bool inlier(const float* c, const float* p, float t) {
    return finite3(p) && std::fabs(std::fma(c[2], p[2], std::fma(c[1], p[1], std::fma(c[0], p[0], c[3])))) < t;
}

// the position in F that hypothesis h draws for sample s (uint64 wrap-around throughout)
static inline uint32_t draw(uint64_t seed, uint64_t h, uint64_t s, uint64_t nf) {
    const uint64_t r = splitmix64(seed + (3 * h + s + 1) * 0x9E3779B97F4A7C15ull);
    return (uint32_t)(((r >> 32) * nf) >> 32);
}

// j[3h + s] = draw(seed, h, s, nf)
extern "C" void ref_plane_draws(uint32_t H, uint64_t seed, uint64_t nf, uint32_t* j) {
    for (uint64_t h = 0; h < H; ++h)
        for (uint64_t s = 0; s < 3; ++s) j[3 * h + s] = draw(seed, h, s, nf);
}

// Every hypothesis: coef[4h..4h+3] (NaN when invalid), sample0[h] (the point index of p0, -1 when invalid) and
// counts[h] (its inliers over all finite points, 0xFFFFFFFF when invalid).  F: the finite indices ascending.
// axis: nullable, 3 floats.
extern "C" void ref_plane_hypotheses(const float* pts, size_t n, const int64_t* F, uint64_t nf, uint32_t H,
                                     uint64_t seed, const float* axis, double eps_angle, float t, float* coef,
                                     int64_t* sample0, uint32_t* counts) {
    double a[3] = {0.0, 0.0, 0.0}, cos_eps = 0.0;
    if (axis) {
        const double x = axis[0], y = axis[1], z = axis[2];
        const double l = std::sqrt(std::fma(z, z, std::fma(y, y, x * x)));
        a[0] = x / l;
        a[1] = y / l;
        a[2] = z / l;
        cos_eps = std::cos(eps_angle);
    }
#pragma omp parallel for schedule(dynamic, 1)
    for (int64_t h = 0; h < (int64_t)H; ++h) {
        float* c = coef + 4 * h;
        c[0] = c[1] = c[2] = c[3] = std::nanf("");
        sample0[h] = -1;
        counts[h] = 0xFFFFFFFFu;
        const uint32_t j[3] = {draw(seed, h, 0, nf), draw(seed, h, 1, nf), draw(seed, h, 2, nf)};
        if (nf < 3 || j[0] == j[1] || j[0] == j[2] || j[1] == j[2]) continue;
        const float* p0 = pts + 4 * F[j[0]];
        const float* p1 = pts + 4 * F[j[1]];
        const float* p2 = pts + 4 * F[j[2]];
        const double x0 = p0[0], y0 = p0[1], z0 = p0[2];
        const double ux = (double)p1[0] - x0, uy = (double)p1[1] - y0, uz = (double)p1[2] - z0;
        const double vx = (double)p2[0] - x0, vy = (double)p2[1] - y0, vz = (double)p2[2] - z0;
        double nx = std::fma(uy, vz, -(uz * vy));
        double ny = std::fma(uz, vx, -(ux * vz));
        double nz = std::fma(ux, vy, -(uy * vx));
        const double l2 = dot3(nx, ny, nz, nx, ny, nz);
        const double uu = dot3(ux, uy, uz, ux, uy, uz), vv = dot3(vx, vy, vz, vx, vy, vz);
        if (!(l2 > 1e-12 * uu * vv)) continue;
        const double l = std::sqrt(l2);
        nx /= l;
        ny /= l;
        nz /= l;
        const double d = -dot3(nx, ny, nz, x0, y0, z0);
        if (axis && std::fabs(dot3(nx, ny, nz, a[0], a[1], a[2])) < cos_eps) continue;
        c[0] = (float)nx;
        c[1] = (float)ny;
        c[2] = (float)nz;
        c[3] = (float)d;
        sample0[h] = F[j[0]];
        uint32_t cnt = 0;
        for (size_t i = 0; i < n; ++i) cnt += inlier(c, pts + 4 * i, t) ? 1u : 0u;
        counts[h] = cnt;
    }
}

// flags[i] = 1 iff point i is an inlier of the plane coef (4 floats)
extern "C" void ref_plane_inliers(const float* pts, size_t n, const float* coef, float t, uint8_t* flags) {
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < (int64_t)n; ++i) flags[i] = inlier(coef, pts + 4 * i, t) ? 1 : 0;
}
