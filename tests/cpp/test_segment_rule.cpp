// Host check of the angle rule of segment_rule.hpp: for every float d in [-1, 1], for positive and negative angles and
// for both comparisons (<= of NormalsProximityEvaluator, < of the combined evaluators), the interval test the kernels
// run equals the evaluator's own predicate, std::acos and (float)M_PI included. Dot products just outside [-1, 1] and
// NaN must be rejected (acos is NaN there; nothing is clamped). Build: g++ -std=c++17 -O2 -ffp-contract=off -pthread.
#include <cstdio>
#include <thread>
#include <vector>
#include "segment_rule.hpp"

using namespace cb::seg;

int main() {
  const float kAngles[] = {0.f, (float)(2.0 * M_PI / 180.0), 0.1f, 0.7853982f, 1.5707964f, 3.0f, (float)M_PI, 4.0f,
                           -(float)(2.0 * M_PI / 180.0), -0.5f, -1.5707964f, -3.0f};
  const int na = sizeof(kAngles) / sizeof(kAngles[0]);
  std::vector<PairRule> rules;
  for (int a = 0; a < na; a++)
    for (int inclusive = 0; inclusive < 2; inclusive++) {
      PairRule r{};
      angle_bounds(kAngles[a], inclusive != 0, &r.up_lo, &r.low_hi);
      rules.push_back(r);
    }
  const auto interval = [](const PairRule& r, float d) { return (d >= r.up_lo && d <= 1.f) || (d >= -1.f && d <= r.low_hi); };
  const int32_t k0 = float_key(-1.f), k1 = float_key(1.f);
  const int nt = std::max(1u, std::thread::hardware_concurrency());
  std::vector<long long> bad(nt, 0), seen(nt, 0);
  std::vector<std::thread> th;
  for (int t = 0; t < nt; t++)
    th.emplace_back([&, t] {
      const int64_t span = (int64_t)k1 - k0 + 1;
      const int32_t b = (int32_t)(k0 + span * t / nt), e = (int32_t)(k0 + span * (t + 1) / nt);
      for (int32_t key = b; key < e; key++) {
        const float d = key_float(key);
        const float angle = std::acos(d);
        for (int a = 0; a < na; a++)
          for (int inclusive = 0; inclusive < 2; inclusive++)
            if (angle_predicate_of(angle, kAngles[a], inclusive != 0) != interval(rules[2 * a + inclusive], d)) {
              if (bad[t]++ < 5) std::printf("FAIL angle %.9g inclusive %d dot %.9g\n", kAngles[a], inclusive, d);
            }
        seen[t]++;
      }
    });
  for (auto& x : th) x.join();
  long long nbad = 0, nseen = 0;
  for (int t = 0; t < nt; t++) nbad += bad[t], nseen += seen[t];
  // outside [-1, 1] and NaN: never similar, like the evaluator
  const float outside[] = {1.00000012f, -1.00000012f, 2.f, -2.f, NAN};
  for (float d : outside)
    for (int i = 0; i < 2 * na; i++)
      if (interval(rules[i], d) || angle_predicate(d, kAngles[i / 2], i % 2)) {
        std::printf("FAIL outside dot %.9g accepted\n", d);
        nbad++;
      }
  // a NaN angle rejects everything
  float lo, hi;
  angle_bounds(NAN, true, &lo, &hi);
  if (!(lo == 2.f && hi == -2.f)) std::printf("FAIL NaN angle\n"), nbad++;
  for (int i = 0; i < 2 * na; i++)
    std::printf("angle %+.9g %s: dot in [%.9g, 1] U [-1, %.9g]\n", kAngles[i / 2], i % 2 ? "<=" : "< ", rules[i].up_lo,
                rules[i].low_hi);
  std::printf("%lld floats in [-1, 1] x %d predicates checked, %lld mismatches\n", nseen, 2 * na, nbad);
  if (nbad) return 1;
  std::printf("all segment-rule checks passed\n");
  return 0;
}
