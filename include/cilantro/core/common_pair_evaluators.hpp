// Same include path as cilantro's core/common_pair_evaluators.hpp: the proximity evaluators (:88-259) that
// ConnectedComponentExtraction3f hands to cb_cloud_segment. Each carries its kind and thresholds (and the normals /
// colours it reads); the device applies the same predicate (cilantro_b200/csrc/segment_rule.hpp). The weight
// evaluators of the same reference file (UnityWeightEvaluator, RBFKernelWeightEvaluator) are in b200_shims.hpp.
// Any other evaluator type is rejected at compile time: arbitrary functors cannot cross the C ABI.
#pragma once
#include <type_traits>
#include "../b200_shims.hpp"

namespace cilantro {

template <typename ValueT = float>
using AlwaysTrueEvaluator = UnityWeightEvaluator<ValueT, bool>;  // :87-88

template <typename ScalarT = float>
class PointsProximityEvaluator {  // :90-103
public:
  using InputScalar = ScalarT;
  using OutputScalar = bool;
  PointsProximityEvaluator(ScalarT dist_thresh) : max_distance_(dist_thresh) {}
  bool operator()(size_t, size_t, ScalarT dist) const { return dist < max_distance_; }
  ScalarT max_distance_;
};

template <typename ScalarT = float, ptrdiff_t EigenDim = 3>
class NormalsProximityEvaluator {  // :105-127
public:
  using InputScalar = ScalarT;
  using OutputScalar = bool;
  NormalsProximityEvaluator(const ConstVectorSetMatrixMap3f& normals, ScalarT angle_thresh)
      : normals_(normals), max_angle_(angle_thresh) {}
  ConstVectorSetMatrixMap3f normals_;
  ScalarT max_angle_;
};

template <typename ScalarT = float>
class ColorsProximityEvaluator {  // :129-146
public:
  using InputScalar = ScalarT;
  using OutputScalar = bool;
  ColorsProximityEvaluator(const ConstVectorSetMatrixMap3f& colors, float dist_thresh)
      : colors_(colors), color_thresh_(dist_thresh) {}
  ConstVectorSetMatrixMap3f colors_;
  float color_thresh_;
};

template <typename ScalarT = float, ptrdiff_t EigenDim = 3>
class PointsNormalsProximityEvaluator {  // :148-172
public:
  using InputScalar = ScalarT;
  using OutputScalar = bool;
  PointsNormalsProximityEvaluator(const ConstVectorSetMatrixMap3f& normals, ScalarT dist_thresh, ScalarT angle_thresh)
      : normals_(normals), max_distance_(dist_thresh), max_angle_(angle_thresh) {}
  ConstVectorSetMatrixMap3f normals_;
  ScalarT max_distance_, max_angle_;
};

template <typename ScalarT = float, ptrdiff_t EigenDim = 3>
class PointsColorsProximityEvaluator {  // :174-194
public:
  using InputScalar = ScalarT;
  using OutputScalar = bool;
  PointsColorsProximityEvaluator(const ConstVectorSetMatrixMap3f& colors, ScalarT dist_thresh, float color_thresh)
      : colors_(colors), max_distance_(dist_thresh), color_thresh_(color_thresh) {}
  ConstVectorSetMatrixMap3f colors_;
  ScalarT max_distance_;
  float color_thresh_;
};

template <typename ScalarT = float, ptrdiff_t EigenDim = 3>
class NormalsColorsProximityEvaluator {  // :196-225
public:
  using InputScalar = ScalarT;
  using OutputScalar = bool;
  NormalsColorsProximityEvaluator(const ConstVectorSetMatrixMap3f& normals, const ConstVectorSetMatrixMap3f& colors,
                                  ScalarT angle_thresh, float color_thresh)
      : normals_(normals), colors_(colors), max_angle_(angle_thresh), color_thresh_(color_thresh) {}
  ConstVectorSetMatrixMap3f normals_, colors_;
  ScalarT max_angle_;
  float color_thresh_;
};

template <typename ScalarT = float, ptrdiff_t EigenDim = 3>
class PointsNormalsColorsProximityEvaluator {  // :227-257
public:
  using InputScalar = ScalarT;
  using OutputScalar = bool;
  PointsNormalsColorsProximityEvaluator(const ConstVectorSetMatrixMap3f& normals, const ConstVectorSetMatrixMap3f& colors,
                                        ScalarT dist_thresh, ScalarT angle_thresh, float color_thresh)
      : normals_(normals), colors_(colors), max_distance_(dist_thresh), max_angle_(angle_thresh),
        color_thresh_(color_thresh) {}
  ConstVectorSetMatrixMap3f normals_, colors_;
  ScalarT max_distance_, max_angle_;
  float color_thresh_;
};

namespace b200 {

// evaluator -> (cb_segment_evaluator, thresholds, normals, colours)
template <class Ev>
struct SegmentEvaluator {
  static_assert(!std::is_same<Ev, Ev>::value,
                "cb_cloud_segment takes AlwaysTrueEvaluator or one of the seven proximity evaluators of "
                "core/common_pair_evaluators.hpp; user-defined evaluators cannot cross the C ABI");
};
template <class E, int Kind, bool N, bool C>
struct SegmentEvaluatorBase {
  static const float* normals(const E& e) {
    if constexpr (N) return e.normals_.data();
    return nullptr;
  }
  static const float* colors(const E& e) {
    if constexpr (C) return e.colors_.data();
    return nullptr;
  }
  static void fill(const E& e, cb_segment_params& p) {
    p.evaluator = Kind;
    if constexpr (Kind == CB_SEG_POINTS || Kind == CB_SEG_POINTS_NORMALS || Kind == CB_SEG_POINTS_COLORS ||
                  Kind == CB_SEG_POINTS_NORMALS_COLORS)
      p.max_distance = (float)e.max_distance_;
    if constexpr (N) p.max_angle = (float)e.max_angle_;
    if constexpr (C) p.color_thresh = e.color_thresh_;
  }
};
template <typename V>
struct SegmentEvaluator<UnityWeightEvaluator<V, bool>>
    : SegmentEvaluatorBase<UnityWeightEvaluator<V, bool>, CB_SEG_ALWAYS_TRUE, false, false> {};
template <typename S>
struct SegmentEvaluator<PointsProximityEvaluator<S>>
    : SegmentEvaluatorBase<PointsProximityEvaluator<S>, CB_SEG_POINTS, false, false> {};
template <typename S, ptrdiff_t D>
struct SegmentEvaluator<NormalsProximityEvaluator<S, D>>
    : SegmentEvaluatorBase<NormalsProximityEvaluator<S, D>, CB_SEG_NORMALS, true, false> {};
template <typename S>
struct SegmentEvaluator<ColorsProximityEvaluator<S>>
    : SegmentEvaluatorBase<ColorsProximityEvaluator<S>, CB_SEG_COLORS, false, true> {};
template <typename S, ptrdiff_t D>
struct SegmentEvaluator<PointsNormalsProximityEvaluator<S, D>>
    : SegmentEvaluatorBase<PointsNormalsProximityEvaluator<S, D>, CB_SEG_POINTS_NORMALS, true, false> {};
template <typename S, ptrdiff_t D>
struct SegmentEvaluator<PointsColorsProximityEvaluator<S, D>>
    : SegmentEvaluatorBase<PointsColorsProximityEvaluator<S, D>, CB_SEG_POINTS_COLORS, false, true> {};
template <typename S, ptrdiff_t D>
struct SegmentEvaluator<NormalsColorsProximityEvaluator<S, D>>
    : SegmentEvaluatorBase<NormalsColorsProximityEvaluator<S, D>, CB_SEG_NORMALS_COLORS, true, true> {};
template <typename S, ptrdiff_t D>
struct SegmentEvaluator<PointsNormalsColorsProximityEvaluator<S, D>>
    : SegmentEvaluatorBase<PointsNormalsColorsProximityEvaluator<S, D>, CB_SEG_POINTS_NORMALS_COLORS, true, true> {};

}  // namespace b200
}  // namespace cilantro
