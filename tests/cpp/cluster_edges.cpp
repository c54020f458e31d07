// CPU reference of the Euclidean clustering edges (DESIGN.md §3.4), for the tests only: the library's fp32 distance
// chain fma(dz, dz, fma(dy, dy, dx * dx)) against t * t.  Built by tests/cluster_reference.py with -ffp-contract=off,
// so every operation is the one written here.
#include <cmath>
#include <cstddef>
#include <cstdint>

static inline bool within(const float* pts, int64_t i, int64_t j, float t2) {
    const float* a = pts + 4 * (size_t)i;
    const float* b = pts + 4 * (size_t)j;
    const float dx = a[0] - b[0], dy = a[1] - b[1], dz = a[2] - b[2];
    return std::fma(dz, dz, std::fma(dy, dy, dx * dx)) <= t2;  // (false for NaN)
}

// keep[e] = 1 iff candidate pair (pairs[2e], pairs[2e + 1]) passes d^2 <= t * t
extern "C" void ref_pairs_within(const float* pts, const int64_t* pairs, size_t n_pairs, float t, uint8_t* keep) {
    const float t2 = t * t;
#pragma omp parallel for schedule(static)
    for (int64_t e = 0; e < (int64_t)n_pairs; ++e) keep[e] = within(pts, pairs[2 * e], pairs[2 * e + 1], t2) ? 1 : 0;
}

// Every pair i < j of finite points with d^2 <= t * t, by brute force, in (i, j) order.  Writes at most `cap` pairs to
// out and returns how many there are.
extern "C" size_t ref_brute_pairs(const float* pts, size_t n, float t, int64_t* out, size_t cap) {
    const float t2 = t * t;
    size_t m = 0;
    for (size_t i = 0; i < n; ++i) {
        const float* a = pts + 4 * i;
        if (!(std::isfinite(a[0]) && std::isfinite(a[1]) && std::isfinite(a[2]))) continue;
        for (size_t j = i + 1; j < n; ++j) {
            const float* b = pts + 4 * j;
            if (!(std::isfinite(b[0]) && std::isfinite(b[1]) && std::isfinite(b[2]))) continue;
            if (!within(pts, (int64_t)i, (int64_t)j, t2)) continue;
            if (m < cap) {
                out[2 * m] = (int64_t)i;
                out[2 * m + 1] = (int64_t)j;
            }
            ++m;
        }
    }
    return m;
}
