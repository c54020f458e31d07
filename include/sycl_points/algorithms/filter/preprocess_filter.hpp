// filter::PreprocessFilter — I/algorithms/filter/preprocess_filter.hpp and its operators
// (I/algorithms/filter/preprocess_operator/*.hpp): box filter, uniform / weighted / mixed random sampling, farthest
// point sampling, angle-of-incidence filter.  Every operator produces the kept indices (libspx) and compacts every
// attribute the cloud carries on the device, in source order (common/filter_by_flags.hpp:29-57).  As in the reference
// each sampling operator owns its std::mt19937 (seed 1234; set_random_seed re-seeds all of them).
#pragma once

#include <cmath>

#include <limits>
#include <memory>

#include "sycl_points/algorithms/filter/gather_attributes.hpp"
#include "sycl_points/points/point_cloud.hpp"

namespace sycl_points {
namespace algorithms {
namespace filter {

class PreprocessFilter {
public:
    using Ptr = std::shared_ptr<PreprocessFilter>;

    PreprocessFilter(const sycl_utils::DeviceQueue& queue) : queue_(queue) {
        for (spx_rng_t* r : {&rng_, &rng_weighted_, &rng_mixed_, &rng_fps_})
            detail::spx_check(spx_rng_create(1234u, r));  // random_sampling_operator.hpp:20 and siblings
    }
    ~PreprocessFilter() {
        for (spx_rng_t r : {rng_, rng_weighted_, rng_mixed_, rng_fps_})
            if (r) spx_rng_destroy(r);
    }
    PreprocessFilter(const PreprocessFilter&) = delete;
    PreprocessFilter& operator=(const PreprocessFilter&) = delete;

    /// preprocess_filter.hpp:46-51
    void set_random_seed(uint_fast32_t seed) {
        for (spx_rng_t r : {rng_, rng_weighted_, rng_mixed_, rng_fps_}) detail::spx_check(spx_rng_seed(r, (uint32_t)seed));
    }

    /// in place
    void box_filter(PointCloudShared& data, float min_distance = 1.0f,
                    float max_distance = std::numeric_limits<float>::max()) {
        this->box_filter(data, data, min_distance, max_distance);
    }
    /// keep points whose L-infinity range lies in [min_distance, max_distance]; every attribute the cloud
    /// carries is compacted with them (common/filter_by_flags.hpp:29-57), in source order
    void box_filter(const PointCloudShared& source, PointCloudShared& output, float min_distance = 1.0f,
                    float max_distance = std::numeric_limits<float>::max()) {
        const size_t N = source.size();
        if (N == 0) {
            if (&source != &output) output.clear();
            return;
        }
        shared_vector<int32_t> idx(N);
        this->queue_.set_accessed_by_device(source.points_ptr(), N);
        this->queue_.set_accessed_by_device(idx.data(), N);
        size_t m = 0;
        detail::spx_check(spx_box_filter_indices(this->queue_.handle(), reinterpret_cast<const float*>(source.points_ptr()),
                                                 N, min_distance, max_distance, idx.data(), &m));
        this->gather_all(source, output, idx, m);
    }

    /// in place
    void random_sampling(PointCloudShared& data, size_t sampling_num) {
        PointCloudShared out(this->queue_);
        this->random_sampling(data, out, sampling_num);
        data = out;
    }
    /// partial Fisher-Yates with the persistent mt19937, order-preserving compaction of every attribute
    void random_sampling(const PointCloudShared& source, PointCloudShared& output, size_t sampling_num) {
        const size_t N = source.size();
        if (N <= sampling_num) {  // keep everything (random_sampling_operator.hpp:26-30)
            output = source;
            return;
        }
        shared_vector<int32_t> idx(sampling_num);
        this->queue_.set_accessed_by_device(idx.data(), sampling_num);
        size_t m = 0;
        detail::spx_check(spx_random_sampling(this->queue_.handle(), rng_, N, sampling_num, idx.data(), &m));
        this->gather_all(source, output, idx, m);
    }

    /// weighted_sampling_operator.hpp:29-96 (in place / into `output`)
    void weighted_random_sampling(PointCloudShared& data, const shared_vector<float>& weights, size_t sampling_num) {
        PointCloudShared out(this->queue_);
        this->weighted_random_sampling(data, out, weights, sampling_num);
        data = out;
    }
    void weighted_random_sampling(const PointCloudShared& source, PointCloudShared& output,
                                  const shared_vector<float>& weights, size_t sampling_num) {
        const size_t N = source.size();
        if (N <= sampling_num) {
            output = source;
            return;
        }
        if (weights.size() != N)
            throw std::invalid_argument("[PreprocessFilter::weighted_random_sampling] weights size must match points");
        size_t positive = 0;
        for (size_t i = 0; i < N; ++i) {
            if (!std::isfinite(weights[i]) || weights[i] < 0.0f)
                throw std::invalid_argument(
                    "[PreprocessFilter::weighted_random_sampling] weights must be finite and non-negative");
            if (weights[i] > 0.0f) ++positive;
        }
        if (positive == 0)
            throw std::invalid_argument("[PreprocessFilter::weighted_random_sampling] at least one weight must be positive");
        if (sampling_num > positive)
            throw std::invalid_argument(
                "[PreprocessFilter::weighted_random_sampling] sampling_num exceeds positive-weight points");
        shared_vector<int32_t> idx(sampling_num);
        this->queue_.set_accessed_by_device(idx.data(), sampling_num);
        size_t m = 0;
        detail::spx_check(spx_weighted_random_sampling(this->queue_.handle(), rng_weighted_, weights.data(), N, sampling_num,
                                                       idx.data(), &m));
        this->gather_all(source, output, idx, m);
    }

    /// farthest_point_sampling_operator.hpp:27-94 (in place / into `output`)
    void farthest_point_sampling(PointCloudShared& data, size_t sampling_num) {
        PointCloudShared out(this->queue_);
        this->farthest_point_sampling(data, out, sampling_num);
        data = out;
    }
    void farthest_point_sampling(const PointCloudShared& source, PointCloudShared& output, size_t sampling_num) {
        const size_t N = source.size();
        if (N <= sampling_num) {
            output = source;
            return;
        }
        size_t first = 0;
        detail::spx_check(spx_rng_uniform_index(rng_fps_, N, &first));
        shared_vector<int32_t> idx(sampling_num);
        this->queue_.set_accessed_by_device(source.points_ptr(), N);
        this->queue_.set_accessed_by_device(idx.data(), sampling_num);
        size_t m = 0;
        detail::spx_check(spx_farthest_point_sampling(this->queue_.handle(),
                                                      reinterpret_cast<const float*>(source.points_ptr()), N, sampling_num,
                                                      first, idx.data(), &m));
        this->gather_all(source, output, idx, m);
    }

    /// mixed_random_sampling_operator.hpp:29-107 (in place / into `output`)
    void mixed_random_sampling(PointCloudShared& data, const shared_vector<float>& weights, size_t sampling_num,
                               float weighted_ratio) {
        PointCloudShared out(this->queue_);
        this->mixed_random_sampling(data, out, weights, sampling_num, weighted_ratio);
        data = out;
    }
    void mixed_random_sampling(const PointCloudShared& source, PointCloudShared& output,
                               const shared_vector<float>& weights, size_t sampling_num, float weighted_ratio) {
        const size_t N = source.size();
        if (N <= sampling_num) {
            output = source;
            return;
        }
        if (weights.size() != N)
            throw std::invalid_argument("[PreprocessFilter::mixed_random_sampling] weights size must match points");
        if (!std::isfinite(weighted_ratio) || weighted_ratio < 0.0f || weighted_ratio > 1.0f)
            throw std::invalid_argument("[PreprocessFilter::mixed_random_sampling] weighted_ratio must be within [0.0, 1.0]");
        for (size_t i = 0; i < N; ++i)
            if (!std::isfinite(weights[i]) || weights[i] < 0.0f)
                throw std::invalid_argument(
                    "[PreprocessFilter::mixed_random_sampling] weights must be finite and non-negative");
        shared_vector<int32_t> idx(sampling_num);
        this->queue_.set_accessed_by_device(idx.data(), sampling_num);
        size_t m = 0;
        detail::spx_check(spx_mixed_random_sampling(this->queue_.handle(), rng_mixed_, weights.data(), N, sampling_num,
                                                    weighted_ratio, idx.data(), &m));
        this->gather_all(source, output, idx, m);
    }

    /// angle_incidence_filter_operator.hpp:23-111
    void angle_incidence_filter(PointCloudShared& data, float min_angle, float max_angle) {
        this->angle_incidence_filter(data, data, min_angle, max_angle);
    }
    void angle_incidence_filter(const PointCloudShared& source, PointCloudShared& output, float min_angle,
                                float max_angle) {
        const size_t N = source.size();
        if (N == 0) return;
        if (!source.has_normal() && !source.has_cov())
            throw std::runtime_error(
                "[PreprocessFilter::angle_incidence_filter] Normal vector or covariance matrices must be "
                "pre-computed.");
        if (min_angle < 0.0f || max_angle > 3.14159265358979323846f * 0.5f || min_angle >= max_angle)
            throw std::invalid_argument("[PreprocessFilter::angle_incidence_filter] Invalid angle range");
        shared_vector<int32_t> idx(N);
        this->queue_.set_accessed_by_device(source.points_ptr(), N);
        this->queue_.set_accessed_by_device(idx.data(), N);
        size_t m = 0;
        detail::spx_check(spx_angle_incidence_indices(
            this->queue_.handle(), reinterpret_cast<const float*>(source.points_ptr()),
            source.has_normal() ? reinterpret_cast<const float*>(source.normals_ptr()) : nullptr,
            source.has_normal() ? nullptr : reinterpret_cast<const float*>(source.covs_ptr()), N, min_angle, max_angle,
            idx.data(), &m));
        this->gather_all(source, output, idx, m);
    }

private:
    void gather_all(const PointCloudShared& source, PointCloudShared& output, const shared_vector<int32_t>& idx, size_t m) {
        gather_attributes(this->queue_, source, output, idx, m);
    }

    sycl_utils::DeviceQueue queue_;
    spx_rng_t rng_ = nullptr, rng_weighted_ = nullptr, rng_mixed_ = nullptr, rng_fps_ = nullptr;
};

}  // namespace filter
}  // namespace algorithms
}  // namespace sycl_points
