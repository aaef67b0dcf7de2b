// ORACLE of connected-component segmentation — test infrastructure, not product code (tests/segment_oracle.py
// compiles it with g++ -ffp-contract=off). A serial restatement of extractConnectedComponents(tree, nh, seeds, ...)
// (clustering/connected_component_extraction.hpp:162-265) over precomputed neighbour lists: nb_idx / nb_d2 entries
// nb_off[u] .. nb_off[u+1] are what KDTree::search(points.col(u), nh) returns, ascending (d2, index). The evaluators of
// core/common_pair_evaluators.hpp:88-259 are written out literally, std::acos included; 3-term dot products and
// squared norms use Eigen's order a0 + (a1 + a2).
//
// The only liberty: segments of equal size are ordered by their smallest point index (the reference's std::sort leaves
// them unordered), so std::stable_sort on (size descending, first point ascending) replaces it.
#include <algorithm>
#include <cmath>
#include <cstddef>
#include <cstdint>
#include <limits>
#include <set>
#include <vector>

namespace {

inline float sum3(float a0, float a1, float a2) { return a0 + (a1 + a2); }

struct Evaluator {
  int kind;
  const float* normals;
  const float* colors;
  float max_distance, max_angle, max_color_diff;

  bool angle_ok(size_t i, size_t j, bool inclusive) const {
    const float* a = normals + 3 * i;
    const float* b = normals + 3 * j;
    const float angle = std::acos(sum3(a[0] * b[0], a[1] * b[1], a[2] * b[2]));
    if (max_angle >= 0.f) return inclusive ? angle <= max_angle : angle < max_angle;
    const float m = std::min(angle, (float)M_PI - angle);
    return inclusive ? m <= -max_angle : m < -max_angle;
  }
  float color_d2(size_t i, size_t j) const {
    const float* a = colors + 3 * i;
    const float* b = colors + 3 * j;
    const float d0 = a[0] - b[0], d1 = a[1] - b[1], d2 = a[2] - b[2];
    return sum3(d0 * d0, d1 * d1, d2 * d2);
  }
  bool operator()(size_t i, size_t j, float dist) const {
    switch (kind) {
      case 0:  // AlwaysTrueEvaluator
        return true;
      case 1:  // PointsProximityEvaluator
        return dist < max_distance;
      case 2:  // NormalsProximityEvaluator
        return angle_ok(i, j, true);
      case 3:  // ColorsProximityEvaluator
        return color_d2(i, j) < max_color_diff;
      case 4:  // PointsNormalsProximityEvaluator
        if (dist >= max_distance) return false;
        return angle_ok(i, j, false);
      case 5:  // PointsColorsProximityEvaluator
        return (dist < max_distance) && (color_d2(i, j) < max_color_diff);
      case 6:  // NormalsColorsProximityEvaluator
        if (color_d2(i, j) >= max_color_diff) return false;
        return angle_ok(i, j, false);
      default:  // PointsNormalsColorsProximityEvaluator
        if (dist >= max_distance || color_d2(i, j) >= max_color_diff) return false;
        return angle_ok(i, j, false);
    }
  }
};

}  // namespace

extern "C" __attribute__((visibility("default"))) size_t orc_connected_components(
    size_t n, const uint64_t* nb_off, const int64_t* nb_idx, const float* nb_d2, const uint64_t* seeds_in,
    size_t n_seeds_in, int kind, float max_distance, float max_angle, float color_thresh, const float* normals,
    const float* colors, uint64_t min_segment_size, uint64_t max_segment_size, uint64_t* labels, uint64_t* seg_offsets,
    uint64_t* seg_points) {
  const Evaluator evaluator{kind, normals, colors, max_distance, max_angle, color_thresh * color_thresh};
  std::vector<size_t> seeds_ind;
  if (seeds_in)
    seeds_ind.assign(seeds_in, seeds_in + n_seeds_in);
  else
    for (size_t i = 0; i < n; i++) seeds_ind.push_back(i);

  constexpr size_t unassigned = std::numeric_limits<size_t>::max();
  std::vector<size_t> current_label(n, unassigned);
  std::vector<size_t> frontier_set;
  frontier_set.reserve(n);
  std::vector<std::set<size_t>> seeds_to_merge_with(seeds_ind.size());
  std::vector<char> seed_active(seeds_ind.size(), 0);

  for (size_t i = 0; i < seeds_ind.size(); i++) {
    if (current_label[seeds_ind[i]] != unassigned) continue;
    seeds_to_merge_with[i].insert(i);
    frontier_set.clear();
    frontier_set.emplace_back(seeds_ind[i]);
    current_label[seeds_ind[i]] = i;
    seed_active[i] = 1;
    while (!frontier_set.empty()) {
      const size_t curr_seed = frontier_set.back();
      frontier_set.pop_back();
      for (uint64_t j = nb_off[curr_seed] + 1; j < nb_off[curr_seed + 1]; j++) {  // j >= 1 of the list
        const size_t v = (size_t)nb_idx[j];
        const size_t curr_lbl = current_label[v];
        if (curr_lbl != i && evaluator(curr_seed, v, nb_d2[j])) {
          if (curr_lbl == unassigned) {
            frontier_set.emplace_back(v);
            current_label[v] = i;
          } else {
            seeds_to_merge_with[i].insert(curr_lbl);
          }
        }
      }
    }
  }

  for (size_t i = 0; i < seeds_to_merge_with.size(); i++)
    for (auto it = seeds_to_merge_with[i].begin(); it != seeds_to_merge_with[i].end(); ++it)
      seeds_to_merge_with[*it].insert(i);

  std::vector<size_t> seed_repr(seeds_ind.size(), unassigned);
  size_t seed_cluster_num = 0;
  for (size_t i = 0; i < seeds_to_merge_with.size(); i++) {
    if (seed_active[i] == 0 || seed_repr[i] != unassigned) continue;
    frontier_set.clear();
    frontier_set.emplace_back(i);
    seed_repr[i] = seed_cluster_num;
    while (!frontier_set.empty()) {
      const size_t curr_seed = frontier_set.back();
      frontier_set.pop_back();
      for (auto it = seeds_to_merge_with[curr_seed].begin(); it != seeds_to_merge_with[curr_seed].end(); ++it) {
        if (seed_active[i] == 1 && seed_repr[*it] == unassigned) {
          frontier_set.emplace_back(*it);
          seed_repr[*it] = seed_cluster_num;
        }
      }
    }
    seed_cluster_num++;
  }

  std::vector<std::vector<size_t>> tmp(seed_cluster_num);
  for (size_t i = 0; i < current_label.size(); i++) {
    if (current_label[i] == unassigned) continue;
    const auto ind = seed_repr[current_label[i]];
    if (tmp[ind].size() <= max_segment_size) tmp[ind].emplace_back(i);
  }
  std::vector<std::vector<size_t>> segs;
  for (size_t i = 0; i < tmp.size(); i++)
    if (tmp[i].size() >= min_segment_size && tmp[i].size() <= max_segment_size) segs.emplace_back(std::move(tmp[i]));
  std::stable_sort(segs.begin(), segs.end(), [](const std::vector<size_t>& a, const std::vector<size_t>& b) {
    return a.size() > b.size() || (a.size() == b.size() && a[0] < b[0]);
  });

  // getPointToClusterIndexMap (clustering_base.hpp:8-18) and the CSR form of the cluster -> points map
  for (size_t i = 0; i < n; i++) labels[i] = segs.size();
  seg_offsets[0] = 0;
  for (size_t s = 0; s < segs.size(); s++) {
    for (size_t t = 0; t < segs[s].size(); t++) {
      labels[segs[s][t]] = s;
      seg_points[seg_offsets[s] + t] = segs[s][t];
    }
    seg_offsets[s + 1] = seg_offsets[s] + segs[s].size();
  }
  return segs.size();
}
