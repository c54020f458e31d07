// CPU reference of the radius outlier filter (DESIGN.md §3.3), for the tests only: brute force over every point with
// the library's fp32 distance chain fma(dz, dz, fma(dy, dy, dx * dx)), OpenMP over the queries.  Built by
// tests/outlier_reference.py with -ffp-contract=off, so every operation is the one written here.
#include <cmath>
#include <cstddef>
#include <cstdint>

extern "C" void ref_radius_outlier_keep(const float* pts, size_t n, const int64_t* rows, size_t n_rows, float radius,
                                        uint32_t min_neighbors, uint8_t* keep) {
    const float r2 = radius * radius;
#pragma omp parallel for schedule(dynamic, 64)
    for (int64_t t = 0; t < (int64_t)n_rows; ++t) {
        const int64_t i = rows ? rows[t] : t;
        const float* q = pts + 4 * (size_t)i;
        if (!(std::isfinite(q[0]) && std::isfinite(q[1]) && std::isfinite(q[2]))) {
            keep[t] = 0;
            continue;
        }
        uint32_t cnt = 0;
        for (size_t j = 0; j < n && cnt < min_neighbors; ++j) {
            if ((int64_t)j == i) continue;
            const float* p = pts + 4 * j;
            const float dx = q[0] - p[0], dy = q[1] - p[1], dz = q[2] - p[2];
            const float d2 = std::fma(dz, dz, std::fma(dy, dy, dx * dx));
            if (d2 <= r2) ++cnt;  // (false for NaN: non-finite points never count)
        }
        keep[t] = cnt >= min_neighbors ? 1 : 0;
    }
}
