// filter::OutlierRemoval — statistical and radius outlier removal on the device (the reference ships a filter of this
// name at I/algorithms/filter/outlier_removal_filter.hpp).  The reference's header is not part of this repository:
// this interface is libspx's own, documented in INTEGRATION.md, and not a verified drop-in of the reference's
// signatures.  Semantics are PCL's StatisticalOutlierRemoval / RadiusOutlierRemoval as pinned in DESIGN.md §3.3 and
// include/spx.h (spx_statistical_outlier_indices, spx_radius_outlier_indices).  Both filters build the exact grid index
// over the source (KDTree::build, honouring the cloud's index hint), produce the kept indices on the device and compact
// every attribute the cloud carries, in source order (gather_attributes.hpp).  `output` may be `source`.
#pragma once

#include <cstdint>
#include <memory>

#include "sycl_points/algorithms/filter/gather_attributes.hpp"
#include "sycl_points/algorithms/knn/kdtree.hpp"
#include "sycl_points/points/point_cloud.hpp"

namespace sycl_points {
namespace algorithms {
namespace filter {

class OutlierRemoval {
public:
    using Ptr = std::shared_ptr<OutlierRemoval>;

    OutlierRemoval(const sycl_utils::DeviceQueue& queue) : queue_(queue) {}

    /// keep point i iff its mean distance to its mean_k nearest other points is at most mu + stddev_mul * sigma
    /// (mu, sigma over all valid points); 1 <= mean_k <= 127, stddev_mul finite (std::runtime_error otherwise)
    void statistical(const PointCloudShared& source, PointCloudShared& output, int mean_k, float stddev_mul) {
        const size_t N = source.size();
        if (N == 0) {
            if (&source != &output) output.clear();
            return;
        }
        const auto tree = knn::KDTree::build(this->queue_, source);
        shared_vector<int32_t> idx(N);
        this->queue_.set_accessed_by_device(source.points_ptr(), N);
        this->queue_.set_accessed_by_device(idx.data(), N);
        size_t m = 0;
        detail::spx_check(spx_statistical_outlier_indices(tree->handle(), reinterpret_cast<const float*>(source.points_ptr()),
                                                          N, mean_k, stddev_mul, nullptr, idx.data(), &m));
        gather_attributes(this->queue_, source, output, idx, m);
    }

    /// keep point i iff at least min_neighbors other points lie within `radius` (d^2 <= radius * radius in fp32);
    /// radius finite and >= 0 (std::runtime_error otherwise)
    void radius(const PointCloudShared& source, PointCloudShared& output, float radius, uint32_t min_neighbors) {
        const size_t N = source.size();
        if (N == 0) {
            if (&source != &output) output.clear();
            return;
        }
        const auto tree = knn::KDTree::build(this->queue_, source);
        shared_vector<int32_t> idx(N);
        this->queue_.set_accessed_by_device(source.points_ptr(), N);
        this->queue_.set_accessed_by_device(idx.data(), N);
        size_t m = 0;
        detail::spx_check(spx_radius_outlier_indices(tree->handle(), reinterpret_cast<const float*>(source.points_ptr()), N,
                                                     radius, min_neighbors, idx.data(), &m));
        gather_attributes(this->queue_, source, output, idx, m);
    }

private:
    sycl_utils::DeviceQueue queue_;
};

}  // namespace filter
}  // namespace algorithms
}  // namespace sycl_points
