// Order-preserving compaction of every per-point attribute of a cloud through a list of kept indices (the device
// counterpart of common/filter_by_flags.hpp:29-57), shared by the device filters: PreprocessFilter and OutlierRemoval.
#pragma once

#include <cstdint>

#include "sycl_points/points/point_cloud.hpp"

namespace sycl_points {
namespace algorithms {
namespace filter {

template <typename V>
inline void gather_attribute(const sycl_utils::DeviceQueue& queue, const V& src, V& dst, const shared_vector<int32_t>& idx,
                             size_t m, bool enable) {
    dst.resize(enable ? m : 0);
    if (!enable || m == 0) return;
    queue.set_accessed_by_device(src.data(), src.size());
    queue.set_accessed_by_device(dst.data(), m);
    sycl_points::detail::spx_check(
        spx_gather(queue.handle(), src.data(), sizeof(typename V::value_type), idx.data(), m, dst.data()));
}

/// output <- the m rows of source listed in idx (ascending), every attribute the source carries; output may be source
inline void gather_attributes(const sycl_utils::DeviceQueue& queue, const PointCloudShared& source, PointCloudShared& output,
                              const shared_vector<int32_t>& idx, size_t m) {
    PointCloudShared out(queue);
    gather_attribute(queue, *source.points, *out.points, idx, m, true);
    gather_attribute(queue, *source.covs, *out.covs, idx, m, source.has_cov());
    gather_attribute(queue, *source.normals, *out.normals, idx, m, source.has_normal());
    gather_attribute(queue, *source.rgb, *out.rgb, idx, m, source.has_rgb());
    gather_attribute(queue, *source.intensities, *out.intensities, idx, m, source.has_intensity());
    gather_attribute(queue, *source.timestamp_offsets, *out.timestamp_offsets, idx, m, source.has_timestamps());
    sycl_points::detail::spx_check(spx_queue_sync(queue.handle()));
    out.start_time_ms = source.start_time_ms;
    out.end_time_ms = source.end_time_ms;
    output.points.swap(out.points);
    output.covs.swap(out.covs);
    output.normals.swap(out.normals);
    output.rgb.swap(out.rgb);
    output.intensities.swap(out.intensities);
    output.timestamp_offsets.swap(out.timestamp_offsets);
    output.start_time_ms = out.start_time_ms;
    output.end_time_ms = out.end_time_ms;
}

}  // namespace filter
}  // namespace algorithms
}  // namespace sycl_points
