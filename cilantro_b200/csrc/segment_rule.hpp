// The pair test of connected-component segmentation (segment.cu), as ONE set of functions that compiles for the device
// (the edge and reachability kernels call pair_passes) and for the host (cb_cloud_segment builds the rule with
// make_pair_rule; tests/cpp/test_segment_rule.cpp checks angle_bounds against std::acos for every float in [-1, 1]).
//
// The proximity evaluators of core/common_pair_evaluators.hpp:88-259 compare std::acos(n_u . n_v) with an angle. acos
// cannot be reproduced on the device bit for bit, but as a function of the float dot product each angle predicate is
// true on a union of at most two intervals of floats:
//   max_angle >= 0:  acos(d) CMP max_angle                                 -> d in [up_lo, 1]
//   max_angle <  0:  min(acos(d), (float)M_PI - acos(d)) CMP -max_angle    -> d in [-1, low_hi] U [up_lo, 1]
// (CMP is <= for NormalsProximityEvaluator, < for the three combined evaluators). The interval ends are found on the
// host by bisection over float bit patterns, evaluating the predicate exactly as the evaluator writes it. A dot product
// outside [-1, 1] (two parallel unit normals can round to 1 + 2^-23) makes acos return NaN and the evaluator answer
// "not similar"; the intervals keep that: nothing is clamped.
//
// No CUDA headers: the host side needs <cmath> / <algorithm> only.
#pragma once
#if defined(__CUDACC__)
#define CB_SEG_HD __host__ __device__ __forceinline__
#else
#define CB_SEG_HD inline
#endif
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>

namespace cb {
namespace seg {

// evaluator kinds (cb_segment_evaluator in include/cilantro_b200.h)
enum Kind : int {
  kAlwaysTrue = 0,
  kPoints = 1,
  kNormals = 2,
  kColors = 3,
  kPointsNormals = 4,
  kPointsColors = 5,
  kNormalsColors = 6,
  kPointsNormalsColors = 7,
};
CB_SEG_HD bool uses_points(int k) { return k == kPoints || k == kPointsNormals || k == kPointsColors || k == kPointsNormalsColors; }
CB_SEG_HD bool uses_normals(int k) { return k == kNormals || k == kPointsNormals || k == kNormalsColors || k == kPointsNormalsColors; }
CB_SEG_HD bool uses_colors(int k) { return k == kColors || k == kPointsColors || k == kNormalsColors || k == kPointsNormalsColors; }

struct PairRule {
  int kind;
  float max_distance;  // dist < max_distance (dist = the neighbour list's squared distance)
  float max_color2;    // |c_u - c_v|^2 < color_thresh * color_thresh (the product rounded to float, as the ctor does)
  float up_lo;         // the angle test passes for dot in [up_lo, 1] ...
  float low_hi;        // ... or in [-1, low_hi]   (empty pieces: up_lo = 2, low_hi = -2)
};

#if defined(__CUDA_ARCH__)
CB_SEG_HD float s_add(float a, float b) { return __fadd_rn(a, b); }
CB_SEG_HD float s_sub(float a, float b) { return __fsub_rn(a, b); }
CB_SEG_HD float s_mul(float a, float b) { return __fmul_rn(a, b); }
#else
inline float s_add(float a, float b) { volatile float r = a + b; return r; }
inline float s_sub(float a, float b) { volatile float r = a - b; return r; }
inline float s_mul(float a, float b) { volatile float r = a * b; return r; }
#endif

// Eigen's 3-term reduction order a0 + (a1 + a2) (DESIGN §2)
CB_SEG_HD float dot3(float ax, float ay, float az, float bx, float by, float bz) {
  return s_add(s_mul(ax, bx), s_add(s_mul(ay, by), s_mul(az, bz)));
}
CB_SEG_HD float color_d2(float ax, float ay, float az, float bx, float by, float bz) {
  const float dx = s_sub(ax, bx), dy = s_sub(ay, by), dz = s_sub(az, bz);
  return s_add(s_mul(dx, dx), s_add(s_mul(dy, dy), s_mul(dz, dz)));
}

// evaluator(u, v, dist) of the selected kind; n* / c* are read only when the kind uses them
template <class V>
CB_SEG_HD bool pair_passes(const PairRule& r, float dist, const V& nu, const V& nv, const V& cu, const V& cv) {
  if (uses_points(r.kind) && !(dist < r.max_distance)) return false;
  if (uses_colors(r.kind) && !(color_d2(cu.x, cu.y, cu.z, cv.x, cv.y, cv.z) < r.max_color2)) return false;
  if (uses_normals(r.kind)) {
    const float d = dot3(nu.x, nu.y, nu.z, nv.x, nv.y, nv.z);
    return (d >= r.up_lo && d <= 1.f) || (d >= -1.f && d <= r.low_hi);
  }
  return true;
}

// ---- host only (cb_cloud_segment and the host test)
// The evaluator's angle predicate, literally (common_pair_evaluators.hpp:115-121 with inclusive = true, :153-158 with
// inclusive = false); the two pieces of the negative-angle form are its two arguments of std::min.
inline bool angle_predicate_of(float angle, float max_angle, bool inclusive) {  // angle = std::acos(dot)
  if (max_angle >= 0.f) return inclusive ? angle <= max_angle : angle < max_angle;
  const float m = std::min(angle, (float)M_PI - angle);
  return inclusive ? m <= -max_angle : m < -max_angle;
}
inline bool angle_predicate(float dot, float max_angle, bool inclusive) {
  return angle_predicate_of(std::acos(dot), max_angle, inclusive);
}

// total order of the floats as integers (-0 and +0 share a key)
inline int32_t float_key(float f) {
  int32_t b;
  std::memcpy(&b, &f, 4);
  return b >= 0 ? b : -(b & 0x7fffffff);
}
inline float key_float(int32_t k) {
  const int32_t b = k >= 0 ? k : (int32_t)(0x80000000u | (uint32_t)(-k));
  float f;
  std::memcpy(&f, &b, 4);
  return f;
}

// smallest float d in [-1, 1] with pred(d) true, for pred false-then-true over the ordered floats; 2 if pred(1) is false
template <class P>
inline float first_true(P pred) {
  int32_t lo = float_key(-1.f), hi = float_key(1.f);
  if (!pred(1.f)) return 2.f;
  if (pred(-1.f)) return -1.f;
  while (hi - lo > 1) {  // pred(lo) false, pred(hi) true
    const int32_t mid = lo + (hi - lo) / 2;
    (pred(key_float(mid)) ? hi : lo) = mid;
  }
  return key_float(hi);
}

// [up_lo, 1] U [-1, low_hi]: where the evaluator's angle test holds as a function of the float dot product
inline void angle_bounds(float max_angle, bool inclusive, float* up_lo, float* low_hi) {
  const auto cmp = [&](float a, float t) { return inclusive ? a <= t : a < t; };
  if (max_angle >= 0.f) {
    *up_lo = first_true([&](float d) { return cmp(std::acos(d), max_angle); });
    *low_hi = -2.f;
  } else if (max_angle < 0.f) {
    *up_lo = first_true([&](float d) { return cmp(std::acos(d), -max_angle); });
    // (float)M_PI - acos(d) CMP t is true-then-false over ascending d: bisect its negation
    const float f = first_true([&](float d) { return !cmp((float)M_PI - std::acos(d), -max_angle); });
    *low_hi = (f == 2.f) ? 1.f : (f == -1.f ? -2.f : key_float(float_key(f) - 1));
  } else {  // NaN angle: the evaluator's comparisons are all false
    *up_lo = 2.f;
    *low_hi = -2.f;
  }
}

inline PairRule make_pair_rule(int kind, float max_distance, float max_angle, float color_thresh) {
  PairRule r;
  r.kind = kind;
  r.max_distance = max_distance;
  r.max_color2 = color_thresh * color_thresh;
  r.up_lo = 2.f;
  r.low_hi = -2.f;
  if (uses_normals(kind)) angle_bounds(max_angle, kind == kNormals, &r.up_lo, &r.low_hi);
  return r;
}

}  // namespace seg
}  // namespace cb
