// segmentation::EuclideanClustering — Euclidean cluster extraction on the device.  This interface is libspx's own,
// documented in INTEGRATION.md, and not a verified drop-in of any reference header.  Semantics are PCL's
// EuclideanClusterExtraction as pinned in DESIGN.md §3.4 and include/spx.h (spx_euclidean_clusters): clusters are the
// connected components of the graph joining two finite points at fp32 d^2 <= tolerance * tolerance; components outside
// [min_cluster_size, max_cluster_size] are dropped (not split); clusters are ordered by size descending, ties by
// smallest member, and each cluster lists its members in ascending index order.  extract builds the exact grid index
// over the source (KDTree::build, honouring the cloud's index hint).
#pragma once

#include <algorithm>
#include <cstdint>
#include <memory>
#include <stdexcept>
#include <vector>

#include "sycl_points/algorithms/filter/gather_attributes.hpp"
#include "sycl_points/algorithms/knn/kdtree.hpp"
#include "sycl_points/points/point_cloud.hpp"

namespace sycl_points {
namespace algorithms {
namespace segmentation {

struct EuclideanClusters {
    shared_vector<int32_t> labels;   // per point: its cluster, -1 for non-finite points and dropped components
    shared_vector<int32_t> indices;  // members of cluster 0, 1, ..., each ascending
    std::vector<uint32_t> offsets;   // cluster c is indices[offsets[c], offsets[c + 1]); C + 1 entries
    size_t size() const { return offsets.empty() ? 0 : offsets.size() - 1; }
};

class EuclideanClustering {
public:
    using Ptr = std::shared_ptr<EuclideanClustering>;

    EuclideanClustering(const sycl_utils::DeviceQueue& queue) : queue_(queue) {}

    /// tolerance finite and >= 0, 1 <= min_cluster_size <= max_cluster_size (std::runtime_error otherwise)
    EuclideanClusters extract(const PointCloudShared& source, float tolerance, uint32_t min_cluster_size = 1,
                              uint32_t max_cluster_size = 0x7fffffffu) {
        const size_t N = source.size();
        EuclideanClusters r;
        r.labels.resize(N);
        r.indices.resize(N);
        r.offsets.assign(1, 0u);
        if (N == 0) return r;
        const auto tree = knn::KDTree::build(this->queue_, source);
        shared_vector<uint32_t> offsets(N + 1);
        this->queue_.set_accessed_by_device(source.points_ptr(), N);
        this->queue_.set_accessed_by_device(r.labels.data(), N);
        this->queue_.set_accessed_by_device(r.indices.data(), N);
        this->queue_.set_accessed_by_device(offsets.data(), N + 1);
        size_t n_clusters = 0, n_members = 0;
        detail::spx_check(spx_euclidean_clusters(tree->handle(), reinterpret_cast<const float*>(source.points_ptr()), N,
                                                 tolerance, min_cluster_size, max_cluster_size, r.labels.data(),
                                                 r.indices.data(), offsets.data(), &n_clusters, &n_members));
        detail::spx_check(spx_queue_sync(this->queue_.handle()));
        r.indices.resize(n_members);
        r.offsets.assign(offsets.begin(), offsets.begin() + n_clusters + 1);
        return r;
    }

    /// output <- cluster c of `result` (extracted from `source`): every attribute, members in ascending index order;
    /// output may be source
    void extract_cluster(const PointCloudShared& source, const EuclideanClusters& result, size_t c,
                         PointCloudShared& output) {
        if (c >= result.size()) throw std::runtime_error("[EuclideanClustering] cluster index out of range");
        const size_t first = result.offsets[c], m = result.offsets[c + 1] - first;
        shared_vector<int32_t> idx(m);
        std::copy(result.indices.begin() + first, result.indices.begin() + first + m, idx.begin());
        filter::gather_attributes(this->queue_, source, output, idx, m);
    }

private:
    sycl_utils::DeviceQueue queue_;
};

}  // namespace segmentation
}  // namespace algorithms
}  // namespace sycl_points
