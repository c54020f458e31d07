// segmentation::PlaneSegmentation through the C++ facade
// (include/sycl_points/algorithms/segmentation/plane_segmentation.hpp): a tilted plane of 2000 points with 500 points of
// clutter above it and a few non-finite rows, with an attribute carried along.  Run on a GPU box; prints
// "<n> checks, <f> failed".
#include <cmath>
#include <cstdio>
#include <random>
#include <stdexcept>
#include <vector>

#include "sycl_points/algorithms/segmentation/plane_segmentation.hpp"

using namespace sycl_points;
using namespace sycl_points::algorithms;

static int g_failed = 0, g_checks = 0;
#define CHECK(cond)                                                         \
    do {                                                                    \
        ++g_checks;                                                         \
        if (!(cond)) {                                                      \
            ++g_failed;                                                     \
            std::printf("  FAILED %s:%d  %s\n", __FILE__, __LINE__, #cond); \
        }                                                                   \
    } while (0)

int main() {
    sycl::device dev(sycl_utils::device_selector::default_selector_v);
    sycl_utils::DeviceQueue queue(dev);
    segmentation::PlaneSegmentation seg(queue);

    // the plane 0.1 x - 0.05 y + z + 1.5 = 0 (points within 1 cm of it), clutter 0.5 .. 3 m above it, and every 250th
    // row non-finite; row i's intensity is i
    const int n = 2500;
    std::mt19937 rng(7);
    std::uniform_real_distribution<float> xy(-10.0f, 10.0f), up(0.5f, 3.0f), jitter(-0.01f, 0.01f);
    PointCloudShared src(queue);
    src.points->resize(n);
    src.intensities->resize(n);
    std::vector<bool> on_plane(n), bad(n);
    for (int i = 0; i < n; ++i) {
        const float x = xy(rng), y = xy(rng);
        on_plane[i] = i % 5 != 4;
        const float z = -1.5f - 0.1f * x + 0.05f * y + (on_plane[i] ? jitter(rng) : up(rng));
        bad[i] = i % 250 == 3;
        (*src.points)[i] = PointType(bad[i] ? NAN : x, y, z, 1.0f);
        (*src.intensities)[i] = (float)i;
    }
    segmentation::PlaneSegmentationParams p;
    p.distance_threshold = 0.05f;
    p.max_iterations = 500;
    const auto m = seg.segment(src, p);
    CHECK(m.valid());
    const float nz = 1.0f / std::sqrt(1.0f + 0.01f + 0.0025f);
    const float sgn = m.coefficients[2] < 0 ? -1.0f : 1.0f;
    CHECK(std::fabs(sgn * m.coefficients[0] - 0.1f * nz) < 2e-3f && std::fabs(sgn * m.coefficients[1] + 0.05f * nz) < 2e-3f);
    CHECK(std::fabs(sgn * m.coefficients[3] - 1.5f * nz) < 2e-2f);
    size_t expected = 0;
    for (int i = 0; i < n; ++i) expected += on_plane[i] && !bad[i];
    CHECK(m.inliers.size() == expected && m.inliers.size() + m.remainder.size() == (size_t)n);
    for (size_t k = 0; k < m.inliers.size(); ++k) {
        CHECK(on_plane[m.inliers[k]] && !bad[m.inliers[k]] && (k == 0 || m.inliers[k] > m.inliers[k - 1]));
    }
    PointCloudShared out(queue);
    seg.extract(src, m, true, out);
    CHECK(out.size() == m.remainder.size() && out.has_intensity());
    for (size_t k = 0; k < out.size() && k < m.remainder.size(); ++k) CHECK((*out.intensities)[k] == (float)m.remainder[k]);

    // the same seed gives the same model; an axis with eps = 0 admits no plane (|n . axis| < cos 0 = 1 for every one)
    const auto again = seg.segment(src, p);
    CHECK(again.hypothesis == m.hypothesis && again.inliers.size() == m.inliers.size());
    p.use_axis = true;
    p.axis[0] = 1.0f;
    p.axis[1] = 0.0f;
    p.axis[2] = 0.1f;
    p.eps_angle = 0.0;
    const auto none = seg.segment(src, p);
    CHECK(!none.valid() && none.inliers.size() == 0 && none.remainder.size() == (size_t)n && std::isnan(none.coefficients[0]));

    // invalid arguments are refused
    bool threw = false;
    try {
        segmentation::PlaneSegmentationParams b;
        b.distance_threshold = 0.0f;
        seg.segment(src, b);
    } catch (const std::runtime_error&) {
        threw = true;
    }
    CHECK(threw);
    std::printf("%d checks, %d failed\n", g_checks, g_failed);
    return g_failed == 0 ? 0 : 1;
}
