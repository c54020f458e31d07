// filter::OutlierRemoval through the C++ facade (include/sycl_points/algorithms/filter/outlier_removal_filter.hpp):
// the four corners of a unit square plus one point 10 m away, statistical (k = 2, stddev_mul = 1) and radius filters,
// with an attribute carried along.  Run on a GPU box; prints "<n> checks, <f> failed".
#include <cmath>
#include <cstdio>
#include <stdexcept>
#include <vector>

#include "sycl_points/algorithms/filter/outlier_removal_filter.hpp"

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

static PointCloudShared square_and_far_point(const sycl_utils::DeviceQueue& q) {
    PointCloudShared c(q);
    const float xy[5][2] = {{0, 0}, {1, 0}, {0, 1}, {1, 1}, {10, 0}};
    c.points->resize(5);
    c.intensities->resize(5);
    for (int i = 0; i < 5; ++i) {
        (*c.points)[i] = PointType(xy[i][0], xy[i][1], 0.0f, 1.0f);
        (*c.intensities)[i] = 0.5f + (float)i;
    }
    return c;
}

int main() {
    sycl::device dev(sycl_utils::device_selector::default_selector_v);
    sycl_utils::DeviceQueue queue(dev);
    filter::OutlierRemoval f(queue);

    // statistical: corners have d = 1, the far point (9 + sqrt(82)) / 2; mu + sigma ~ 6.196 keeps the corners only
    {
        const PointCloudShared src = square_and_far_point(queue);
        PointCloudShared out(queue);
        f.statistical(src, out, 2, 1.0f);
        CHECK(out.size() == 4);
        CHECK(out.has_intensity() && out.intensities->size() == 4);
        for (size_t i = 0; i < out.size() && i < 4; ++i) {
            CHECK((*out.points)[i].x() == (*src.points)[i].x() && (*out.points)[i].y() == (*src.points)[i].y());
            CHECK((*out.intensities)[i] == 0.5f + (float)i);
        }
    }
    // radius 1, 2 neighbours: every corner has its two edge neighbours at exactly 1; in place
    {
        PointCloudShared c = square_and_far_point(queue);
        f.radius(c, c, 1.0f, 2);
        CHECK(c.size() == 4);
        PointCloudShared d = square_and_far_point(queue);
        f.radius(d, d, 1.0f, 3);  // the diagonal is sqrt(2): nobody has three
        CHECK(d.size() == 0);
        PointCloudShared e = square_and_far_point(queue);
        f.radius(e, e, 9.0f, 1);  // (1, 0) is exactly 9 from the far point
        CHECK(e.size() == 5);
    }
    // invalid arguments are refused
    {
        const PointCloudShared src = square_and_far_point(queue);
        PointCloudShared out(queue);
        bool threw = false;
        try {
            f.statistical(src, out, 0, 1.0f);
        } catch (const std::runtime_error&) {
            threw = true;
        }
        CHECK(threw);
        threw = false;
        try {
            f.radius(src, out, -1.0f, 1);
        } catch (const std::runtime_error&) {
            threw = true;
        }
        CHECK(threw);
    }
    std::printf("%d checks, %d failed\n", g_checks, g_failed);
    return g_failed == 0 ? 0 : 1;
}
