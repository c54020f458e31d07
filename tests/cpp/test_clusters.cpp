// segmentation::EuclideanClustering through the C++ facade
// (include/sycl_points/algorithms/segmentation/euclidean_clustering.hpp): a chain at its spacing and one fp32 step
// below, and three teeth joined through one bridge point, with an attribute carried along.  Run on a GPU box; prints
// "<n> checks, <f> failed".
#include <cmath>
#include <cstdio>
#include <stdexcept>
#include <vector>

#include "sycl_points/algorithms/segmentation/euclidean_clustering.hpp"

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

static PointCloudShared cloud(const sycl_utils::DeviceQueue& q, const std::vector<std::vector<float>>& xyz) {
    PointCloudShared c(q);
    c.points->resize(xyz.size());
    c.intensities->resize(xyz.size());
    for (size_t i = 0; i < xyz.size(); ++i) {
        (*c.points)[i] = PointType(xyz[i][0], xyz[i][1], xyz[i][2], 1.0f);
        (*c.intensities)[i] = 0.5f + (float)i;
    }
    return c;
}

int main() {
    sycl::device dev(sycl_utils::device_selector::default_selector_v);
    sycl_utils::DeviceQueue queue(dev);
    segmentation::EuclideanClustering ec(queue);

    // a chain at 0.25 m: one cluster at t = 0.25, ten singletons in index order one fp32 step below
    {
        std::vector<std::vector<float>> xyz;
        for (int i = 0; i < 10; ++i) xyz.push_back({0.25f * (float)i, 0.0f, 0.0f});
        const PointCloudShared src = cloud(queue, xyz);
        const auto one = ec.extract(src, 0.25f);
        CHECK(one.size() == 1 && one.offsets[1] == 10);
        const auto ten = ec.extract(src, std::nextafter(0.25f, 0.0f));
        CHECK(ten.size() == 10);
        for (int i = 0; i < 10 && ten.size() == 10; ++i) {
            CHECK(ten.labels[i] == i && ten.indices[i] == i && ten.offsets[i] == (uint32_t)i);
        }
    }
    // three teeth of 4 points (x = 0, 1, 2) and a bridge at (0.5, 0, 0), rows interleaved: at t = 0.5 the bridge joins
    // teeth 0 and 1 (9 points), tooth 2 stays apart (4); a size filter [5, 100] keeps the first only
    {
        std::vector<std::vector<float>> rows;
        for (float x : {0.0f, 1.0f, 2.0f})
            for (int k = 0; k < 4; ++k) rows.push_back({x, 0.0f, 0.25f * (float)k});
        rows.push_back({0.5f, 0.0f, 0.0f});
        const int order[13] = {8, 0, 4, 12, 9, 1, 5, 10, 2, 6, 11, 3, 7};
        std::vector<std::vector<float>> xyz;
        for (int r : order) xyz.push_back(rows[r]);
        const PointCloudShared src = cloud(queue, xyz);
        const auto r = ec.extract(src, 0.5f);
        const int big[9] = {1, 2, 3, 5, 6, 8, 9, 11, 12}, small[4] = {0, 4, 7, 10};
        CHECK(r.size() == 2 && r.offsets[1] == 9 && r.offsets[2] == 13);
        for (int i = 0; i < 9 && r.indices.size() == 13; ++i) CHECK(r.indices[i] == big[i] && r.labels[big[i]] == 0);
        for (int i = 0; i < 4 && r.indices.size() == 13; ++i) CHECK(r.indices[9 + i] == small[i] && r.labels[small[i]] == 1);
        PointCloudShared out(queue);
        ec.extract_cluster(src, r, 1, out);
        CHECK(out.size() == 4 && out.has_intensity());
        for (int i = 0; i < 4 && out.size() == 4; ++i) {
            CHECK((*out.points)[i].x() == 2.0f && (*out.intensities)[i] == 0.5f + (float)small[i]);
        }
        const auto f = ec.extract(src, 0.5f, 5, 100);
        CHECK(f.size() == 1 && f.offsets[1] == 9 && f.labels[0] == -1);
    }
    // invalid arguments are refused
    {
        const PointCloudShared src = cloud(queue, {{0, 0, 0}, {1, 0, 0}});
        bool threw = false;
        try {
            ec.extract(src, -1.0f);
        } catch (const std::runtime_error&) {
            threw = true;
        }
        CHECK(threw);
        threw = false;
        try {
            ec.extract(src, 1.0f, 3, 2);
        } catch (const std::runtime_error&) {
            threw = true;
        }
        CHECK(threw);
    }
    std::printf("%d checks, %d failed\n", g_checks, g_failed);
    return g_failed == 0 ? 0 : 1;
}
