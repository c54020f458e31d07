// segmentation::PlaneSegmentation — RANSAC plane segmentation on the device.  This interface is libspx's own,
// documented in INTEGRATION.md, and not a verified drop-in of any reference header.  Semantics are PCL's
// SACSegmentation with SACMODEL_PLANE (SACMODEL_PERPENDICULAR_PLANE when an axis is set) and SAC_RANSAC, as pinned in
// DESIGN.md §3.5 and include/spx.h (spx_plane_segment): max_iterations hypotheses drawn from a counter-based stream
// keyed by the seed, each scored over every finite point with |a x + b y + c z + d| < distance_threshold; the most
// inliers win (ties: the lowest hypothesis); optimize_coefficients refits the plane to its inliers by least squares and
// selects them again.  Inliers and remainder are listed in ascending index order; the remainder includes non-finite
// points, so it is what ground removal hands to clustering.
#pragma once

#include <cmath>
#include <cstdint>
#include <memory>
#include <stdexcept>

#include "sycl_points/algorithms/filter/gather_attributes.hpp"
#include "sycl_points/points/point_cloud.hpp"

namespace sycl_points {
namespace algorithms {
namespace segmentation {

struct PlaneModel {
    float coefficients[4] = {NAN, NAN, NAN, NAN};  // (a, b, c, d), (a, b, c) unit; NaN without a model
    int32_t hypothesis = -1;                       // the winning hypothesis, -1 without a model
    shared_vector<int32_t> inliers;                // ascending
    shared_vector<int32_t> remainder;              // every other index, ascending
    bool valid() const { return hypothesis >= 0; }
};

struct PlaneSegmentationParams {
    float distance_threshold = 0.2f;  // finite, > 0
    uint32_t max_iterations = 1000;   // [1, 2^20]
    uint64_t seed = 0;
    bool use_axis = false;            // SACMODEL_PERPENDICULAR_PLANE: the normal within eps_angle of axis
    float axis[3] = {0.0f, 0.0f, 1.0f};
    double eps_angle = 0.0;           // radians, [0, pi/2]
    bool optimize_coefficients = true;
};

class PlaneSegmentation {
public:
    using Ptr = std::shared_ptr<PlaneSegmentation>;

    PlaneSegmentation(const sycl_utils::DeviceQueue& queue) : queue_(queue) {}

    /// invalid parameters throw std::runtime_error
    PlaneModel segment(const PointCloudShared& source, const PlaneSegmentationParams& params = {}) {
        const size_t N = source.size();
        PlaneModel r;
        r.inliers.resize(N);
        r.remainder.resize(N);
        if (N > 0) {
            this->queue_.set_accessed_by_device(source.points_ptr(), N);
            this->queue_.set_accessed_by_device(r.inliers.data(), N);
            this->queue_.set_accessed_by_device(r.remainder.data(), N);
        }
        size_t m = 0;
        detail::spx_check(spx_plane_segment(this->queue_.handle(), reinterpret_cast<const float*>(source.points_ptr()), N,
                                            params.distance_threshold, params.max_iterations, params.seed,
                                            params.use_axis ? params.axis : nullptr, params.eps_angle,
                                            params.optimize_coefficients ? 1 : 0, r.coefficients, &r.hypothesis,
                                            r.inliers.data(), &m, r.remainder.data(), nullptr));
        r.inliers.resize(m);
        r.remainder.resize(N - m);
        return r;
    }

    /// output <- the inliers (negative = false) or the remainder (negative = true) of `model`, segmented from
    /// `source`: every attribute, ascending index order (PCL's ExtractIndices); output may be source
    void extract(const PointCloudShared& source, const PlaneModel& model, bool negative, PointCloudShared& output) {
        const shared_vector<int32_t>& idx = negative ? model.remainder : model.inliers;
        filter::gather_attributes(this->queue_, source, output, idx, idx.size());
    }

private:
    sycl_utils::DeviceQueue queue_;
};

}  // namespace segmentation
}  // namespace algorithms
}  // namespace sycl_points
