// feature::FPFHEstimation, registration::match_features and registration::RANSACRegistration through the C++ facade
// (include/sycl_points/algorithms/feature/fpfh.hpp, include/sycl_points/algorithms/registration/ransac_registration.hpp):
// descriptors of a cloud of curved patches, the match of a cloud's features with themselves, RANSAC recovering a large
// rotation and translation from correspondences of which 70 % are wrong, and the argument checks.  Run on a GPU box;
// prints "<n> checks, <f> failed".
#include <cmath>
#include <cstdio>
#include <random>
#include <stdexcept>
#include <vector>

#include "sycl_points/algorithms/feature/covariance.hpp"
#include "sycl_points/algorithms/registration/ransac_registration.hpp"

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

template <class F>
static bool throws(F&& f) {
    try {
        f();
    } catch (const std::runtime_error&) {
        return true;
    }
    return false;
}

int main() {
    sycl::device dev(sycl_utils::device_selector::default_selector_v);
    sycl_utils::DeviceQueue queue(dev);

    // 3000 points on a wavy floor and two wavy walls, 20 m across; row 7 non-finite
    const int n = 3000;
    std::mt19937 rng(11);
    std::uniform_real_distribution<float> u(-10.0f, 10.0f);
    PointCloudShared src(queue);
    src.points->resize(n);
    for (int i = 0; i < n; ++i) {
        const float a = u(rng), b = u(rng), w = 0.4f * std::sin(0.7f * a) * std::cos(0.5f * b);
        const int s = i % 3;
        (*src.points)[i] = s == 0 ? PointType(a, b, w, 1.0f) : (s == 1 ? PointType(a, 10.0f + w, 0.5f * b + 5.0f, 1.0f)
                                                                        : PointType(-10.0f + w, a, 0.5f * b + 5.0f, 1.0f));
    }
    (*src.points)[7] = PointType(NAN, 0.0f, 0.0f, 1.0f);
    const auto tree = knn::KDTree::build(queue, src);
    covariance::estimate_normals_async(*tree, src, 15).wait_and_throw();
    feature::FPFHEstimation fpfh(queue);
    const auto F = fpfh.compute(src, 2.0f, 100, tree.get());
    CHECK(F.size() == (size_t)n * feature::FPFH_DIM);
    int finite_rows = 0, sums_ok = 0;
    for (int i = 0; i < n; ++i) {
        float s = 0.0f;
        bool fin = true;
        for (size_t b = 0; b < feature::FPFH_DIM; ++b) {
            fin = fin && std::isfinite(F[i * feature::FPFH_DIM + b]);
            s += F[i * feature::FPFH_DIM + b];
        }
        finite_rows += fin;
        sums_ok += fin && std::fabs(s - 600.0f) < 0.05f;  // the point's three histograms and its neighbours' three
    }
    CHECK(std::isnan(F[7 * feature::FPFH_DIM]));
    CHECK(finite_rows == n - 1 && sums_ok == n - 1);

    // the features against themselves: every finite row finds itself (or an equal row), mutual or not
    const auto self = registration::match_features(queue, F, F, true);
    CHECK(self.size() >= (size_t)(n - 1) * 99 / 100);
    int same = 0;
    for (size_t k = 0; k < self.size(); ++k) same += self.source[k] == self.target[k];
    CHECK(same >= (int)self.size() * 99 / 100);

    // RANSAC: target = T source, correspondences i -> i with 70 % of them replaced by random rows
    const float ang = 2.4f, c = std::cos(ang), s = std::sin(ang);
    const float R[3][3] = {{c, -s, 0.0f}, {s, c, 0.0f}, {0.0f, 0.0f, 1.0f}}, t[3] = {6.0f, -3.0f, 0.5f};
    PointCloudShared tgt(queue);
    tgt.points->resize(n);
    for (int i = 0; i < n; ++i) {
        const PointType& p = (*src.points)[i];
        (*tgt.points)[i] = PointType(R[0][0] * p[0] + R[0][1] * p[1] + R[0][2] * p[2] + t[0],
                                     R[1][0] * p[0] + R[1][1] * p[1] + R[1][2] * p[2] + t[1],
                                     R[2][0] * p[0] + R[2][1] * p[1] + R[2][2] * p[2] + t[2], 1.0f);
    }
    registration::FeatureCorrespondences corr;
    corr.source.resize(n);
    corr.target.resize(n);
    std::uniform_int_distribution<int> any(0, n - 1);
    std::uniform_real_distribution<float> coin(0.0f, 1.0f);
    int good = 0;
    for (int i = 0; i < n; ++i) {
        corr.source[i] = i;
        const bool ok = coin(rng) < 0.3f;
        corr.target[i] = ok ? i : any(rng);
        good += ok && i != 7;
    }
    registration::RANSACRegistration ransac(queue);
    registration::RANSACRegistrationParams p;
    p.max_correspondence_distance = 0.05f;
    p.max_iterations = 20000;
    const auto r = ransac.align(src, tgt, corr, p);
    CHECK(r.valid());
    float err = 0.0f;
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) err = std::fmax(err, std::fabs(r.T(i, j) - R[i][j]));
        err = std::fmax(err, std::fabs(r.T(i, 3) - t[i]) / 10.0f);
    }
    CHECK(err < 1e-4f);
    CHECK((int)r.inliers.size() >= good && r.fitness >= 0.29f);
    const auto again = ransac.align(src, tgt, corr, p);
    CHECK(again.hypothesis == r.hypothesis && again.inliers.size() == r.inliers.size());
    registration::FeatureCorrespondences two;
    two.source.assign(corr.source.begin(), corr.source.begin() + 2);
    two.target.assign(corr.target.begin(), corr.target.begin() + 2);
    const auto none = ransac.align(src, tgt, two, p);
    CHECK(!none.valid() && none.inliers.empty() && std::isnan(none.T(0, 0)));

    // invalid arguments are refused
    CHECK(throws([&] { fpfh.compute(src, 0.0f); }));
    CHECK(throws([&] { fpfh.compute(src, 1.0f, 101); }));
    CHECK(throws([&] { fpfh.compute(tgt, 1.0f); }));  // no normals
    CHECK(throws([&] {
        registration::RANSACRegistrationParams b;
        b.edge_length_similarity = 1.5f;
        ransac.align(src, tgt, corr, b);
    }));
    CHECK(throws([&] {
        registration::RANSACRegistrationParams b;
        b.max_iterations = 0;
        ransac.align(src, tgt, corr, b);
    }));
    std::printf("%d checks, %d failed\n", g_checks, g_failed);
    return g_failed == 0 ? 0 : 1;
}
