// CPU reference of farthest point sampling (preprocess_operator/farthest_point_sampling_operator.hpp:27-94) with
// the first point given, for the tests only.  The oracle's orc_farthest_point_sampling_flags draws the first point
// from its own generator; this runs the same loop from a chosen one: the fp32 distance chain
// fma(dw, dw, fma(dz, dz, fma(dy, dy, dx * dx))), dist = fmin(dist, d), then the first of equal maxima as
// std::max_element picks it.  The update and the arg-max are split over OpenMP threads; the per-thread maxima are
// folded in thread order with the same strict `<`, so the pick is std::max_element's (dist is never NaN: it starts
// at FLT_MAX and fmin drops a NaN distance).  Built by tests/test_gpu_feature_edges.py with -ffp-contract=off, so
// every operation is the one written here.
#include <omp.h>

#include <cfloat>
#include <cmath>
#include <cstddef>
#include <cstdint>
#include <vector>

extern "C" void ref_farthest_point_sampling(const float* pts, size_t n, size_t sampling_num, size_t first,
                                            uint8_t* flags) {
    for (size_t i = 0; i < n; ++i) flags[i] = 0;
    if (n == 0 || sampling_num == 0) return;
    std::vector<float> dist(n, FLT_MAX);
    const int nt = omp_get_max_threads();
    std::vector<float> best_v(nt);
    std::vector<size_t> best_i(nt);
    size_t sel = first;
    flags[sel] = 1;
    for (size_t it = 1; it < sampling_num; ++it) {
        const float* c = pts + 4 * sel;
#pragma omp parallel num_threads(nt)
        {
            const int t = omp_get_thread_num(), used = omp_get_num_threads();
            const size_t lo = n * (size_t)t / (size_t)used, hi = n * (size_t)(t + 1) / (size_t)used;
            float bv = -1.0f;
            size_t bi = lo;
            for (size_t i = lo; i < hi; ++i) {
                const float* p = pts + 4 * i;
                const float dx = p[0] - c[0], dy = p[1] - c[1], dz = p[2] - c[2], dw = p[3] - c[3];
                const float d = std::fma(dw, dw, std::fma(dz, dz, std::fma(dy, dy, dx * dx)));
                dist[i] = std::fmin(dist[i], d);
                if (i == lo || bv < dist[i]) {
                    bv = dist[i];
                    bi = i;
                }
            }
            best_v[t] = hi > lo ? bv : -1.0f;
            best_i[t] = bi;
#pragma omp barrier
#pragma omp single
            {
                float v = best_v[0];
                size_t b = best_i[0];
                for (int u = 1; u < used; ++u)
                    if (v < best_v[u]) {
                        v = best_v[u];
                        b = best_i[u];
                    }
                sel = b;
            }
        }
        flags[sel] = 1;
    }
}
