// CPU reference of FPFH descriptors and their nearest-feature correspondences (DESIGN.md §3.6), for the tests only:
// the pair feature, its bins (the angle bin by exact-in-sign tests against the ten boundary rays), SPFH and FPFH, and
// the brute-force feature search.  Built by tests/global_reference.py with -ffp-contract=off, so every operation is
// the one written here.
#include <cmath>
#include <cstddef>
#include <cstdint>
#include <vector>

static const int DIM = 33, BINS = 11;

static inline bool finite3(const float* p) { return std::isfinite(p[0]) && std::isfinite(p[1]) && std::isfinite(p[2]); }

static inline float dotf(float ax, float ay, float az, float bx, float by, float bz) {
    return std::fma(az, bz, std::fma(ay, by, ax * bx));
}
static inline void crossf(float ax, float ay, float az, float bx, float by, float bz, float& cx, float& cy, float& cz) {
    cx = std::fma(ay, bz, -(az * by));
    cy = std::fma(az, bx, -(ax * bz));
    cz = std::fma(ax, by, -(ay * bx));
}

static inline int linear_bin(float f) {
    const float b = std::floor((f + 1.0f) * 5.5f);
    return !(b >= 0.0f) ? 0 : (b > 10.0f ? 10 : (int)b);
}

// the boundary rays -pi + 2 pi k / 11 for k = 6..10, rounded to fp32; ray k <= 5 is the mirror of ray 11 - k
static const float RAY_C[5] = {0x1.eb42aap-1f, 0x1.4f49e8p-1f, 0x1.2375f6p-3f, -0x1.a9628ep-2f, -0x1.aeb8c8p-1f};
static const float RAY_S[5] = {0x1.207e8p-2f, 0x1.82f19cp-1f, 0x1.fac9ep-1f, 0x1.d1bb48p-1f, 0x1.14ceep-1f};

extern "C" int ref_angle_bin(float X, float Y) {
    if (Y == 0.0f) return X < 0.0f ? 10 : 5;
    const double x = X, y = Y;
    int b = 5;
    for (int m = 0; m < 5; ++m) {
        if (Y > 0.0f) {
            b += ((double)RAY_C[m] * y - (double)RAY_S[m] * x >= 0.0) ? 1 : 0;
        } else {
            b -= ((double)RAY_C[m] * y + (double)RAY_S[m] * x < 0.0) ? 1 : 0;
        }
    }
    return b;
}

// out[0..5] = f2, f3, X, Y (the atan2 arguments), swapped; bins[0..2]; returns 0 when the pair is skipped
extern "C" int ref_pair_feature(const float* pi, const float* ni, const float* pj, const float* nj, float* out,
                                int32_t* bins) {
    const float dx = pj[0] - pi[0], dy = pj[1] - pi[1], dz = pj[2] - pi[2];
    const float s2 = dotf(dx, dy, dz, dx, dy, dz);
    const float ai = dotf(ni[0], ni[1], ni[2], dx, dy, dz), aj = dotf(nj[0], nj[1], nj[2], dx, dy, dz);
    const bool sw = std::fabs(ai) < std::fabs(aj);
    const float* u = sw ? nj : ni;
    const float* o = sw ? ni : nj;
    const float ex = sw ? -dx : dx, ey = sw ? -dy : dy, ez = sw ? -dz : dz;
    const float f3 = (sw ? -aj : ai) / std::sqrt(s2);
    float vx, vy, vz;
    crossf(ex, ey, ez, u[0], u[1], u[2], vx, vy, vz);
    const float vv = dotf(vx, vy, vz, vx, vy, vz);
    if (vv == 0.0f) return 0;
    const float l = std::sqrt(vv);
    vx = vx / l;
    vy = vy / l;
    vz = vz / l;
    float wx, wy, wz;
    crossf(u[0], u[1], u[2], vx, vy, vz, wx, wy, wz);
    const float f2 = dotf(vx, vy, vz, o[0], o[1], o[2]);
    const float X = dotf(u[0], u[1], u[2], o[0], o[1], o[2]), Y = dotf(wx, wy, wz, o[0], o[1], o[2]);
    if (out) {
        out[0] = f2;
        out[1] = f3;
        out[2] = X;
        out[3] = Y;
        out[4] = sw ? 1.0f : 0.0f;
    }
    bins[0] = ref_angle_bin(X, Y);
    bins[1] = linear_bin(f2);
    bins[2] = linear_bin(f3);
    return 1;
}

// features[n][33] from points / normals (float4 rows) and the radius neighbours idx / dist [n][k]; spfh_out nullable
extern "C" void ref_fpfh(const float* pts, const float* nrm, size_t n, const int32_t* idx, const float* dist, int k,
                         float* features, float* spfh_out) {
    std::vector<float> S((size_t)n * DIM, 0.0f);
    std::vector<uint8_t> valid(n);
    for (size_t i = 0; i < n; ++i) valid[i] = finite3(pts + 4 * i) && finite3(nrm + 4 * i);
#pragma omp parallel for schedule(dynamic, 64)
    for (int64_t i = 0; i < (int64_t)n; ++i) {
        if (!valid[i]) continue;
        uint32_t cnt[DIM] = {0};
        uint32_t m = 0;
        for (int r = 0; r < k; ++r) {
            const int32_t j = idx[i * k + r];
            if (j < 0 || j == (int32_t)i || !(dist[i * k + r] > 0.0f) || !valid[j]) continue;
            int32_t b[3];
            if (!ref_pair_feature(pts + 4 * i, nrm + 4 * i, pts + 4 * (size_t)j, nrm + 4 * (size_t)j, nullptr, b)) continue;
            ++cnt[b[0]];
            ++cnt[BINS + b[1]];
            ++cnt[2 * BINS + b[2]];
            ++m;
        }
        const float scale = m ? 100.0f / (float)m : 0.0f;
        for (int b = 0; b < DIM; ++b) S[i * DIM + b] = (float)cnt[b] * scale;
    }
#pragma omp parallel for schedule(dynamic, 64)
    for (int64_t i = 0; i < (int64_t)n; ++i) {
        float* out = features + i * DIM;
        if (!valid[i]) {
            for (int b = 0; b < DIM; ++b) out[b] = std::nanf("");
            continue;
        }
        float acc[DIM] = {0.0f}, sum[3] = {0.0f, 0.0f, 0.0f};
        for (int r = 0; r < k; ++r) {
            const int32_t j = idx[i * k + r];
            const float d2 = dist[i * k + r];
            if (j < 0 || j == (int32_t)i || !(d2 > 0.0f) || !valid[j]) continue;
            const float w = 1.0f / d2;
            for (int b = 0; b < DIM; ++b) {
                const float v = S[(size_t)j * DIM + b] * w;
                acc[b] = acc[b] + v;
                sum[b / BINS] = sum[b / BINS] + v;
            }
        }
        for (int b = 0; b < DIM; ++b) {
            const float g = sum[b / BINS];
            const float c = g != 0.0f ? acc[b] * (100.0f / g) : 0.0f;
            out[b] = c + S[i * DIM + b];
        }
    }
    if (spfh_out)
        for (size_t e = 0; e < S.size(); ++e) spfh_out[e] = S[e];
}

// nn[i] = the target row with the lowest (D, t) over the targets with D not NaN, -1 when none
extern "C" void ref_feature_nn(const float* src, size_t ns, const float* tgt, size_t nt, int32_t* nn) {
#pragma omp parallel for schedule(dynamic, 16)
    for (int64_t i = 0; i < (int64_t)ns; ++i) {
        const float* s = src + i * DIM;
        float best = 0.0f;
        int32_t bt = -1;
        for (size_t t = 0; t < nt; ++t) {
            const float* q = tgt + t * DIM;
            float d = s[0] - q[0];
            float acc = d * d;
            for (int b = 1; b < DIM; ++b) {
                d = s[b] - q[b];
                acc = std::fma(d, d, acc);
            }
            if (std::isnan(acc)) continue;
            if (bt < 0 || acc < best) {
                best = acc;
                bt = (int32_t)t;
            }
        }
        nn[i] = bt;
    }
}
