// feature::FPFHEstimation — FPFH descriptors on the device.  This interface is libspx's own, documented in
// INTEGRATION.md, and not a verified drop-in of any reference header.  Semantics are Rusu et al. 2009 with the point's
// own SPFH term, pinned op for op in DESIGN.md §3.6 and include/spx.h (spx_fpfh): the neighbours of a point are the
// max_nn nearest within `radius` (Open3D's hybrid search), the cloud must carry normals (covariance::
// estimate_normals_async), and a point with a non-finite coordinate or normal gets a NaN row.
#pragma once

#include <cmath>
#include <cstdint>
#include <memory>
#include <stdexcept>

#include "sycl_points/algorithms/knn/kdtree.hpp"
#include "sycl_points/points/point_cloud.hpp"

namespace sycl_points {
namespace algorithms {
namespace feature {

constexpr size_t FPFH_DIM = 33;  // bins 0-10 f1 (angle), 11-21 f2, 22-32 f3

class FPFHEstimation {
public:
    using Ptr = std::shared_ptr<FPFHEstimation>;

    FPFHEstimation(const sycl_utils::DeviceQueue& queue) : queue_(queue) {}

    /// float[N][33] row-major.  radius finite and > 0, 1 <= max_nn <= 100, normals present (std::runtime_error
    /// otherwise).  tree: an index built over exactly `source`, or nullptr to build one.
    shared_vector<float> compute(const PointCloudShared& source, float radius, size_t max_nn = 100,
                                 const knn::KDTree* tree = nullptr) {
        if (!(std::isfinite(radius) && radius > 0.0f)) throw std::runtime_error("[FPFHEstimation] `radius` must be finite and > 0");
        if (max_nn < 1 || max_nn > 100) throw std::runtime_error("[FPFHEstimation] `max_nn` must be in [1, 100]");
        const size_t N = source.size();
        shared_vector<float> features;
        features.resize(N * FPFH_DIM);
        if (N == 0) return features;
        if (!source.has_normal()) throw std::runtime_error("[FPFHEstimation] the cloud has no normals");
        std::shared_ptr<knn::KDTree> owned;
        if (tree == nullptr) {
            owned = knn::KDTree::build(this->queue_, source);
            tree = owned.get();
        } else if (tree->size() != N) {
            throw std::runtime_error("[FPFHEstimation] the tree was not built over this cloud");
        }
        knn::KNNResult nn;
        tree->radius_search_async(source, max_nn, radius, nn);
        this->queue_.set_accessed_by_device(source.points_ptr(), N);
        this->queue_.set_accessed_by_device(source.normals_ptr(), N);
        this->queue_.set_accessed_by_device(features.data(), N * FPFH_DIM);
        detail::spx_check(spx_fpfh(this->queue_.handle(), reinterpret_cast<const float*>(source.points_ptr()),
                                   reinterpret_cast<const float*>(source.normals_ptr()), N, nn.indices->data(),
                                   nn.distances->data(), (int)max_nn, features.data()));
        detail::spx_check(spx_queue_sync(this->queue_.handle()));
        return features;
    }

private:
    sycl_utils::DeviceQueue queue_;
};

}  // namespace feature
}  // namespace algorithms
}  // namespace sycl_points
