// Same include path as cilantro's clustering/connected_component_extraction.hpp: ConnectedComponentExtraction3f<> and
// extractConnectedComponents on top of cb_cloud_segment. The evaluator classes live in core/common_pair_evaluators.hpp.
#pragma once
#include <limits>
#include <vector>
#include "../b200_shims.hpp"
#include "../core/common_pair_evaluators.hpp"

namespace cilantro {

namespace b200 {

template <class NeighborhoodSpecT>
struct SegmentNeighborhood;  // only the three specifications of core/kd_tree.hpp map to the device path
template <typename CountT>
struct SegmentNeighborhood<KNNNeighborhoodSpecification<CountT>> {
  static void set(const KNNNeighborhoodSpecification<CountT>& nh, cb_segment_params& p) {
    p.k = (int32_t)nh.maxNumberOfNeighbors;
    p.radius2 = 0.f;
  }
};
template <typename ScalarT>
struct SegmentNeighborhood<RadiusNeighborhoodSpecification<ScalarT>> {
  static void set(const RadiusNeighborhoodSpecification<ScalarT>& nh, cb_segment_params& p) {
    p.k = 0;
    p.radius2 = (float)nh.radius;
  }
};
template <typename ScalarT, typename CountT>
struct SegmentNeighborhood<KNNInRadiusNeighborhoodSpecification<ScalarT, CountT>> {
  static void set(const KNNInRadiusNeighborhoodSpecification<ScalarT, CountT>& nh, cb_segment_params& p) {
    p.k = (int32_t)nh.maxNumberOfNeighbors;
    p.radius2 = (float)nh.radius;
  }
};

// cb_cloud_segment on a device cloud; fills the ClusteringBase maps (clustering_base.hpp:8-18)
template <typename PointIndexT, typename ClusterIndexT, class NeighborhoodSpecT, class Evaluator>
void segment_cloud(cb_cloud* cloud, size_t n, const NeighborhoodSpecT& nh, const std::vector<PointIndexT>* seeds,
                   const Evaluator& ev, size_t min_size, size_t max_size,
                   std::vector<std::vector<PointIndexT>>& clusters, std::vector<ClusterIndexT>* labels_out) {
  cb_segment_params p{};
  SegmentNeighborhood<NeighborhoodSpecT>::set(nh, p);
  SegmentEvaluator<Evaluator>::fill(ev, p);
  p.min_size = min_size;
  p.max_size = max_size;
  std::vector<uint64_t> sd;
  if (seeds) sd.assign(seeds->begin(), seeds->end());
  std::vector<uint64_t> labels(n), offsets(n + 1), points(n);
  size_t m = 0;
  check(cb_cloud_segment(Context::get(), cloud, &p, seeds ? sd.data() : nullptr, sd.size(), SegmentEvaluator<Evaluator>::normals(ev),
                         SegmentEvaluator<Evaluator>::colors(ev), labels.data(), offsets.data(), points.data(), &m, nullptr),
        "cb_cloud_segment");
  clusters.assign(m, {});
  for (size_t s = 0; s < m; s++)
    clusters[s].assign(points.begin() + (long)offsets[s], points.begin() + (long)offsets[s + 1]);
  if (labels_out) labels_out->assign(labels.begin(), labels.end());
}

}  // namespace b200

// ---- extractConnectedComponents (connected_component_extraction.hpp:162-265 and the overloads forwarding to it) ----
template <typename IndexT, class NeighborhoodSpecT, class Evaluator = AlwaysTrueEvaluator<float>>
void extractConnectedComponents(const KDTree3f<IndexT>& tree, const NeighborhoodSpecT& nh,
                                const std::vector<IndexT>& seeds_ind,
                                std::vector<std::vector<IndexT>>& segment_to_point_map,
                                const Evaluator& evaluator = Evaluator(), size_t min_segment_size = 1,
                                size_t max_segment_size = std::numeric_limits<size_t>::max()) {
  b200::segment_cloud<IndexT, size_t>(tree.b200_cloud(), tree.b200_size(), nh, &seeds_ind, evaluator, min_segment_size,
                                      max_segment_size, segment_to_point_map, nullptr);
}
template <typename IndexT, class NeighborhoodSpecT, class Evaluator = AlwaysTrueEvaluator<float>>
void extractConnectedComponents(const KDTree3f<IndexT>& tree, const NeighborhoodSpecT& nh,
                                std::vector<std::vector<IndexT>>& segment_to_point_map,
                                const Evaluator& evaluator = Evaluator(), size_t min_segment_size = 1,
                                size_t max_segment_size = std::numeric_limits<size_t>::max()) {
  b200::segment_cloud<IndexT, size_t>(tree.b200_cloud(), tree.b200_size(), nh, nullptr, evaluator, min_segment_size,
                                      max_segment_size, segment_to_point_map, nullptr);
}
template <typename IndexT = size_t, class NeighborhoodSpecT, class Evaluator = AlwaysTrueEvaluator<float>>
std::vector<std::vector<IndexT>> extractConnectedComponents(
    const ConstVectorSetMatrixMap3f& points, const NeighborhoodSpecT& nh, const std::vector<IndexT>& seeds_ind,
    const Evaluator& evaluator = Evaluator(), size_t min_segment_size = 1,
    size_t max_segment_size = std::numeric_limits<size_t>::max()) {
  std::vector<std::vector<IndexT>> out;
  extractConnectedComponents(KDTree3f<IndexT>(points), nh, seeds_ind, out, evaluator, min_segment_size,
                             max_segment_size);
  return out;
}
template <typename IndexT = size_t, class NeighborhoodSpecT, class Evaluator = AlwaysTrueEvaluator<float>>
std::vector<std::vector<IndexT>> extractConnectedComponents(
    const ConstVectorSetMatrixMap3f& points, const NeighborhoodSpecT& nh, const Evaluator& evaluator = Evaluator(),
    size_t min_segment_size = 1, size_t max_segment_size = std::numeric_limits<size_t>::max()) {
  std::vector<std::vector<IndexT>> out;
  extractConnectedComponents(KDTree3f<IndexT>(points), nh, out, evaluator, min_segment_size, max_segment_size);
  return out;
}

// ---- ConnectedComponentExtraction3f<> (connected_component_extraction.hpp:371-428) ----------------------------------
template <typename PointIndexT = size_t, typename ClusterIndexT = size_t>
class ConnectedComponentExtraction3f {
public:
  using ClusterToPointIndicesMap = std::vector<std::vector<PointIndexT>>;
  using PointToClusterIndexMap = std::vector<ClusterIndexT>;

  ConnectedComponentExtraction3f(const ConstVectorSetMatrixMap3f& points, size_t /*max_leaf_size*/ = 10)
      : n_(points.cols()), own_(points), cloud_(own_.h) {}
  ConnectedComponentExtraction3f(const KDTree3f<PointIndexT>& tree) : n_(tree.b200_size()), cloud_(tree.b200_cloud()) {}

  template <class NeighborhoodSpecT, class Evaluator = AlwaysTrueEvaluator<float>>
  ConnectedComponentExtraction3f& segment(const NeighborhoodSpecT& nh, const std::vector<PointIndexT>& seeds_ind,
                                          const Evaluator& evaluator = Evaluator(), size_t min_segment_size = 1,
                                          size_t max_segment_size = std::numeric_limits<size_t>::max()) {
    b200::segment_cloud<PointIndexT, ClusterIndexT>(cloud_, n_, nh, &seeds_ind, evaluator, min_segment_size,
                                                    max_segment_size, lists_, &labels_);
    return *this;
  }
  template <class NeighborhoodSpecT, class Evaluator = AlwaysTrueEvaluator<float>>
  ConnectedComponentExtraction3f& segment(const NeighborhoodSpecT& nh, const Evaluator& evaluator = Evaluator(),
                                          size_t min_segment_size = 1,
                                          size_t max_segment_size = std::numeric_limits<size_t>::max()) {
    b200::segment_cloud<PointIndexT, ClusterIndexT>(cloud_, n_, nh, (const std::vector<PointIndexT>*)nullptr,
                                                    evaluator, min_segment_size, max_segment_size, lists_, &labels_);
    return *this;
  }

  // ClusteringBase (clustering_base.hpp:62-99)
  const ClusterToPointIndicesMap& getClusterToPointIndicesMap() const { return lists_; }
  const PointToClusterIndexMap& getPointToClusterIndexMap() const { return labels_; }
  size_t getNumberOfClusters() const { return lists_.size(); }
  size_t getNumberOfPoints() const { return labels_.size(); }
  template <typename IndexT = PointIndexT>
  std::vector<IndexT> getLabeledPointIndices() const {
    std::vector<IndexT> r;
    for (size_t i = 0; i < labels_.size(); i++)
      if ((size_t)labels_[i] < lists_.size()) r.emplace_back((IndexT)i);
    return r;
  }
  template <typename IndexT = PointIndexT>
  std::vector<IndexT> getUnlabeledPointIndices() const {
    std::vector<IndexT> r;
    for (size_t i = 0; i < labels_.size(); i++)
      if ((size_t)labels_[i] >= lists_.size()) r.emplace_back((IndexT)i);
    return r;
  }

private:
  size_t n_;
  b200::CloudHandle own_;
  cb_cloud* cloud_;
  ClusterToPointIndicesMap lists_;
  PointToClusterIndexMap labels_;
};

}  // namespace cilantro
