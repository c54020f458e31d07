// registration::RANSACRegistration and registration::match_features — global registration over FPFH correspondences
// on the device.  This interface is libspx's own, documented in INTEGRATION.md, and not a verified drop-in of any
// reference header.  Semantics are the usual feature-matching RANSAC with an edge-length check (as Open3D's
// registration_ransac_based_on_feature_matching), pinned in DESIGN.md §3.6 and include/spx.h
// (spx_feature_correspondences, spx_ransac_registration): max_iterations three-correspondence hypotheses drawn from a
// counter-based stream keyed by the seed, each posed in closed form and scored with |R p + t - q| <
// max_correspondence_distance; the most inliers win (ties: the lowest hypothesis); optimize refits the pose to the
// inliers by least squares and selects them again.  The pose is the initial guess to hand to Registration::align.
#pragma once

#include <cmath>
#include <cstdint>
#include <memory>
#include <stdexcept>

#include "sycl_points/algorithms/feature/fpfh.hpp"
#include "sycl_points/points/point_cloud.hpp"

namespace sycl_points {
namespace algorithms {
namespace registration {

struct FeatureCorrespondences {
    shared_vector<int32_t> source;  // source rows, ascending
    shared_vector<int32_t> target;  // their nearest target rows
    size_t size() const { return source.size(); }
};

/// the nearest target row of every source row by squared feature distance (ties: the lowest index; NaN rows never
/// match); mutual keeps a pair only if the reverse search picks the source row as well.  Rows are float[33].
inline FeatureCorrespondences match_features(const sycl_utils::DeviceQueue& queue, const shared_vector<float>& source,
                                             const shared_vector<float>& target, bool mutual = false) {
    if (source.size() % feature::FPFH_DIM || target.size() % feature::FPFH_DIM)
        throw std::runtime_error("[match_features] feature arrays must hold whole rows of 33");
    const size_t ns = source.size() / feature::FPFH_DIM, nt = target.size() / feature::FPFH_DIM;
    FeatureCorrespondences r;
    r.source.resize(ns);
    r.target.resize(ns);
    size_t m = 0;
    if (ns > 0) {
        queue.set_accessed_by_device(source.data(), source.size());
        queue.set_accessed_by_device(target.data(), target.size());
        queue.set_accessed_by_device(r.source.data(), ns);
        queue.set_accessed_by_device(r.target.data(), ns);
    }
    detail::spx_check(spx_feature_correspondences(queue.handle(), source.data(), ns, target.data(), nt, mutual ? 1 : 0,
                                                  r.source.data(), r.target.data(), &m));
    r.source.resize(m);
    r.target.resize(m);
    return r;
}

struct RANSACResult {
    TransformMatrix T = TransformMatrix::Identity();  // target <- source; NaN without a model
    int32_t hypothesis = -1;                          // the winning hypothesis, -1 without a model
    shared_vector<int32_t> inliers;                   // positions into the correspondence list, ascending
    float fitness = 0.0f;                             // inliers / correspondences
    bool valid() const { return hypothesis >= 0; }
};

struct RANSACRegistrationParams {
    float max_correspondence_distance = 1.0f;  // finite, > 0
    uint32_t max_iterations = 100000;          // [1, 2^20]
    float edge_length_similarity = 0.9f;       // (0, 1]
    uint64_t seed = 0;
    bool optimize = true;
};

class RANSACRegistration {
public:
    using Ptr = std::shared_ptr<RANSACRegistration>;

    RANSACRegistration(const sycl_utils::DeviceQueue& queue) : queue_(queue) {}

    /// invalid parameters throw std::runtime_error
    RANSACResult align(const PointCloudShared& source, const PointCloudShared& target,
                       const FeatureCorrespondences& correspondences, const RANSACRegistrationParams& params = {}) {
        const size_t M = correspondences.size();
        if (correspondences.target.size() != M)
            throw std::runtime_error("[RANSACRegistration] correspondence arrays differ in length");
        RANSACResult r;
        r.inliers.resize(M);
        if (M > 0) {
            this->queue_.set_accessed_by_device(source.points_ptr(), source.size());
            this->queue_.set_accessed_by_device(target.points_ptr(), target.size());
            this->queue_.set_accessed_by_device(correspondences.source.data(), M);
            this->queue_.set_accessed_by_device(correspondences.target.data(), M);
            this->queue_.set_accessed_by_device(r.inliers.data(), M);
        }
        size_t m = 0;
        detail::spx_check(spx_ransac_registration(
            this->queue_.handle(), reinterpret_cast<const float*>(source.points_ptr()), source.size(),
            reinterpret_cast<const float*>(target.points_ptr()), target.size(), correspondences.source.data(),
            correspondences.target.data(), M, params.max_correspondence_distance, params.max_iterations, params.seed,
            params.edge_length_similarity, params.optimize ? 1 : 0, r.T.data(), &r.hypothesis, r.inliers.data(), &m,
            nullptr));
        r.inliers.resize(m);
        r.fitness = M ? (float)m / (float)M : 0.0f;
        return r;
    }

private:
    sycl_utils::DeviceQueue queue_;
};

}  // namespace registration
}  // namespace algorithms
}  // namespace sycl_points
