// cilantro_b200 — header-only C++ mirror of the cilantro types on the rigid-ICP / k-means / RANSAC /
// PCA hot path, forwarding to the C ABI of libcilantro_b200.so (include/cilantro_b200.h).
//
// Same names, argument meaning and error behaviour as the reference (paths relative to
// /root/reference/include/cilantro/):
//   VectorSet3f / ConstVectorSetMatrixMap3f / Vector3f      core/data_containers.hpp:73-156
//   RigidTransform3f                                        core/space_transformations.hpp:54-57
//   Neighbor / NeighborSet                                  core/nearest_neighbors.hpp
//   Correspondence / CorrespondenceSet                      core/correspondence.hpp:9-55
//   KDTree3f<>                                              core/kd_tree.hpp:144-397
//   SimplePointToPointMetricRigidICP3f                      registration/icp_common_instances.hpp:250
//   SimpleCombinedMetricRigidICP3f                          registration/icp_common_instances.hpp:261
//   KMeans3f<>                                              clustering/kmeans.hpp:9-59,205-207
//   RigidTransformRANSACEstimator3f<>                       model_estimation/ransac_transform_estimator.hpp:9-122
//   PrincipalComponentAnalysis3f                            core/principal_component_analysis.hpp:8-89
//   NormalEstimation3f                                      core/normal_estimation.hpp:11-421
//   Points[Normals][Colors]GridDownsampler3f                core/grid_downsampler.hpp:8-340
//   PointCloud3f (points / normals / colors, size, hasNormals, transform, gridDownsample[d],
//                 estimateNormals{KNN,Radius,KNNInRadius})  utilities/point_cloud.hpp:14-22,246-420,557
//   Timer                                                   utilities/timer.hpp
// Eigen3 is an external dependency of cilantro that is absent from the build image, so the containers
// below are minimal Eigen-free stand-ins with the memory layout cilantro uses (column-major 3 x N,
// packed xyz). A cilantro maintainer keeps Eigen and only swaps the method bodies (INTEGRATION.md).
//
// Arbitrary user functors (weight / distance evaluators) cannot cross a C ABI: this path implements
// cilantro's defaults (DistanceEvaluator = identity, UnityWeightEvaluator); anything else is a
// compile-time error here, never a silent CPU fallback.
#pragma once
#include <algorithm>
#include <array>
#include <chrono>
#include <cmath>
#include <cstddef>
#include <cstdint>
#include <cstring>
#include <limits>
#include <memory>
#include <random>
#include <stdexcept>
#include <string>
#include <vector>

#include "../cilantro_b200.h"
#include "b200_ply.hpp"

// Eigen interoperability (SURVEY 7 step 2): where Eigen is installed, the stand-in containers below convert
// from / to the Eigen types real cilantro code holds (VectorSet<float,3> = Eigen::Matrix<float,3,Dynamic>,
// RigidTransform<float,3> = Eigen::Transform<float,3,Isometry>; core/data_containers.hpp:73-112,155-156,
// core/space_transformations.hpp:54-55). Eigen3 is absent from the image this repo is built and tested in, so this
// block is compiled only on a machine that has it (CILANTRO_B200_NO_EIGEN switches it off explicitly).
#if !defined(CILANTRO_B200_NO_EIGEN) && defined(__has_include)
#if __has_include(<Eigen/Dense>)
#include <Eigen/Dense>
#define CILANTRO_B200_HAS_EIGEN 1
#endif
#endif

namespace cilantro {

// ---- containers -----------------------------------------------------------------------------------
struct Vector3f {
  float v[3] = {0.f, 0.f, 0.f};
  Vector3f() = default;
  Vector3f(float x, float y, float z) : v{x, y, z} {}
  float& operator[](size_t i) { return v[i]; }
  float operator[](size_t i) const { return v[i]; }
  float* data() { return v; }
  const float* data() const { return v; }
  float norm() const { return std::sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]); }
};

// Owning 3 x N column-major float matrix (cilantro::VectorSet<float,3>).
class VectorSet3f {
public:
  VectorSet3f() = default;
  VectorSet3f(size_t rows, size_t cols) : d_(3 * cols) { (void)rows; }
  size_t rows() const { return 3; }
  size_t cols() const { return d_.size() / 3; }
  void resize(size_t /*rows*/, size_t cols) { d_.resize(3 * cols); }
  float* data() { return d_.data(); }
  const float* data() const { return d_.data(); }
  float& operator()(size_t r, size_t c) { return d_[3 * c + r]; }
  float operator()(size_t r, size_t c) const { return d_[3 * c + r]; }
  Vector3f col(size_t c) const { return Vector3f(d_[3 * c], d_[3 * c + 1], d_[3 * c + 2]); }
  void setCol(size_t c, const Vector3f& p) {
    d_[3 * c] = p[0];
    d_[3 * c + 1] = p[1];
    d_[3 * c + 2] = p[2];
  }
#ifdef CILANTRO_B200_HAS_EIGEN
  // same memory layout as Eigen::Matrix<float, 3, Dynamic> (column-major, packed xyz)
  VectorSet3f(const Eigen::Matrix<float, 3, Eigen::Dynamic>& m) : d_(m.data(), m.data() + 3 * m.cols()) {}
  Eigen::Map<Eigen::Matrix<float, 3, Eigen::Dynamic>> eigen() { return {d_.data(), 3, (Eigen::Index)cols()}; }
  Eigen::Map<const Eigen::Matrix<float, 3, Eigen::Dynamic>> eigen() const { return {d_.data(), 3, (Eigen::Index)cols()}; }
  operator Eigen::Matrix<float, 3, Eigen::Dynamic>() const { return eigen(); }
#endif

private:
  std::vector<float> d_;
};

// Non-owning view (cilantro::ConstVectorSetMatrixMap<float,3>): implicit from the same sources as
// the reference's (VectorSet, std::vector<float>, std::vector<Vector3f>, raw pointer + count).
class ConstVectorSetMatrixMap3f {
public:
  ConstVectorSetMatrixMap3f(const float* data = nullptr, size_t n = 0) : p_(data), n_(n) {}
  ConstVectorSetMatrixMap3f(const VectorSet3f& s) : p_(s.data()), n_(s.cols()) {}
  ConstVectorSetMatrixMap3f(const std::vector<float>& s) : p_(s.data()), n_(s.size() / 3) {}
  ConstVectorSetMatrixMap3f(const std::vector<Vector3f>& s)
      : p_(s.empty() ? nullptr : s[0].data()), n_(s.size()) {}
#ifdef CILANTRO_B200_HAS_EIGEN
  // the sources ConstVectorSetMatrixMap<float,3> accepts in the reference (core/data_containers.hpp:73-112)
  ConstVectorSetMatrixMap3f(const Eigen::Matrix<float, 3, Eigen::Dynamic>& m) : p_(m.data()), n_((size_t)m.cols()) {}
  ConstVectorSetMatrixMap3f(const Eigen::Map<const Eigen::Matrix<float, 3, Eigen::Dynamic>>& m)
      : p_(m.data()), n_((size_t)m.cols()) {}
  ConstVectorSetMatrixMap3f(const Eigen::Map<Eigen::Matrix<float, 3, Eigen::Dynamic>>& m)
      : p_(m.data()), n_((size_t)m.cols()) {}
  ConstVectorSetMatrixMap3f(const std::vector<Eigen::Vector3f>& s)
      : p_(s.empty() ? nullptr : s[0].data()), n_(s.size()) {}
  Eigen::Map<const Eigen::Matrix<float, 3, Eigen::Dynamic>> eigen() const { return {p_, 3, (Eigen::Index)n_}; }
#endif
  const float* data() const { return p_; }
  size_t cols() const { return n_; }
  size_t rows() const { return 3; }
  Vector3f col(size_t c) const { return Vector3f(p_[3 * c], p_[3 * c + 1], p_[3 * c + 2]); }

private:
  const float* p_;
  size_t n_;
};

// Rigid transform, row-major [R | t] storage; the accessor surface of Eigen::Transform<float,3,Isometry>
// that cilantro's examples use.
class RigidTransform3f {
public:
  RigidTransform3f() { setIdentity(); }
  explicit RigidTransform3f(const float* T12) { std::memcpy(m_, T12, sizeof(m_)); }
  static RigidTransform3f Identity() { return RigidTransform3f(); }
  void setIdentity() {
    for (float& x : m_) x = 0.f;
    m_[0] = m_[5] = m_[10] = 1.f;
  }
  float& linear(size_t r, size_t c) { return m_[4 * r + c]; }
  float linear(size_t r, size_t c) const { return m_[4 * r + c]; }
  float& translation(size_t r) { return m_[4 * r + 3]; }
  float translation(size_t r) const { return m_[4 * r + 3]; }
  const float* data() const { return m_; }
  float* data() { return m_; }
  std::array<float, 16> matrix() const {
    std::array<float, 16> M{};
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 4; c++) M[4 * r + c] = m_[4 * r + c];
    M[15] = 1.f;
    return M;
  }
  Vector3f operator*(const Vector3f& p) const {
    Vector3f q;
    for (int r = 0; r < 3; r++) q[r] = (m_[4 * r] * p[0] + (m_[4 * r + 1] * p[1] + m_[4 * r + 2] * p[2])) + m_[4 * r + 3];
    return q;
  }
  RigidTransform3f operator*(const RigidTransform3f& o) const {
    RigidTransform3f r;
    cb_compose(m_, o.m_, r.m_);
    return r;
  }
  RigidTransform3f inverse() const {
    RigidTransform3f r;
    for (int i = 0; i < 3; i++) {
      for (int j = 0; j < 3; j++) r.m_[4 * i + j] = m_[4 * j + i];
      r.m_[4 * i + 3] = -(m_[i] * m_[3] + m_[4 + i] * m_[7] + m_[8 + i] * m_[11]);
    }
    return r;
  }
#ifdef CILANTRO_B200_HAS_EIGEN
  // cilantro::RigidTransform<float,3> = Eigen::Transform<float,3,Eigen::Isometry> (core/space_transformations.hpp:54-55)
  RigidTransform3f(const Eigen::Transform<float, 3, Eigen::Isometry>& T) {
    for (int r = 0; r < 3; r++) {
      for (int c = 0; c < 3; c++) m_[4 * r + c] = T.linear()(r, c);
      m_[4 * r + 3] = T.translation()(r);
    }
  }
  operator Eigen::Transform<float, 3, Eigen::Isometry>() const {
    Eigen::Transform<float, 3, Eigen::Isometry> T = Eigen::Transform<float, 3, Eigen::Isometry>::Identity();
    for (int r = 0; r < 3; r++) {
      for (int c = 0; c < 3; c++) T.linear()(r, c) = m_[4 * r + c];
      T.translation()(r) = m_[4 * r + 3];
    }
    return T;
  }
#endif

private:
  float m_[12];
};

template <typename ScalarT = float, typename IndexT = size_t>
struct Neighbor {
  IndexT index;
  ScalarT value;
};
template <typename ScalarT = float, typename IndexT = size_t>
using NeighborSet = std::vector<Neighbor<ScalarT, IndexT>>;
template <typename ScalarT = float, typename IndexT = size_t>
using Neighborhood = NeighborSet<ScalarT, IndexT>;

// neighbourhood specifications (core/nearest_neighbors.hpp:58-87); radii are squared distances
template <typename CountT = size_t>
struct KNNNeighborhoodSpecification {
  KNNNeighborhoodSpecification(CountT k = (CountT)0) : maxNumberOfNeighbors(k) {}
  CountT maxNumberOfNeighbors;
};
template <typename ScalarT>
struct RadiusNeighborhoodSpecification {
  RadiusNeighborhoodSpecification(ScalarT r = (ScalarT)0) : radius(r) {}
  ScalarT radius;
};
template <typename ScalarT, typename CountT = size_t>
struct KNNInRadiusNeighborhoodSpecification {
  KNNInRadiusNeighborhoodSpecification(CountT k = 0, ScalarT r = (ScalarT)0) : maxNumberOfNeighbors(k), radius(r) {}
  CountT maxNumberOfNeighbors;
  ScalarT radius;
};

template <typename ScalarT = float, typename IndexT = size_t>
struct Correspondence {
  IndexT indexInFirst;
  IndexT indexInSecond;
  ScalarT value;
};
template <typename ScalarT = float, typename IndexT = size_t>
using CorrespondenceSet = std::vector<Correspondence<ScalarT, IndexT>>;

class Timer {  // utilities/timer.hpp:7-43
public:
  void start() { t0_ = std::chrono::high_resolution_clock::now(); }
  void stop() { t1_ = std::chrono::high_resolution_clock::now(); }
  double getElapsedTime() const { return std::chrono::duration<double, std::milli>(t1_ - t0_).count(); }

private:
  std::chrono::high_resolution_clock::time_point t0_, t1_;
};

// ---- library plumbing -------------------------------------------------------------------------------
namespace b200 {

inline void check(int rc, const char* what) {
  if (rc < 0) throw std::runtime_error(std::string(what) + ": " + cb_last_error());
}

// the reference seeds from std::random_device (kmeans.hpp:41, ransac_base.hpp:73); so does the
// default here, and setRandomSeed() / the seed argument make runs reproducible
inline uint32_t random_seed() { return std::random_device{}(); }

// One context per process and device (cb_context is not thread-safe: like the reference's objects,
// use one thread per set of objects).
class Context {
public:
  static cb_context* get(int device = 0) {
    static Context c(device);
    return c.ctx_;
  }

private:
  explicit Context(int device) { check(cb_context_create(device, &ctx_), "cb_context_create"); }
  ~Context() { /* process lifetime; objects holding clouds may outlive static destruction order */ }
  cb_context* ctx_ = nullptr;
};

struct CloudHandle {
  cb_cloud* h = nullptr;
  CloudHandle() = default;
  CloudHandle(const ConstVectorSetMatrixMap3f& pts, const ConstVectorSetMatrixMap3f* normals = nullptr) {
    reset(pts, normals);
  }
  void reset(const ConstVectorSetMatrixMap3f& pts, const ConstVectorSetMatrixMap3f* normals = nullptr) {
    if (h) cb_cloud_destroy(h);
    h = nullptr;
    const float* n = (normals && normals->cols() == pts.cols() && pts.cols() > 0) ? normals->data() : nullptr;
    check(cb_cloud_create(Context::get(), pts.data(), n, pts.cols(), 0, &h), "cb_cloud_create");
  }
  CloudHandle(CloudHandle&& o) noexcept : h(o.h) { o.h = nullptr; }
  CloudHandle(const CloudHandle&) = delete;
  CloudHandle& operator=(const CloudHandle&) = delete;
  ~CloudHandle() {
    if (h) cb_cloud_destroy(h);
  }
};

}  // namespace b200

// ---- KDTree3f<> ------------------------------------------------------------------------------------
// The "tree" is the device-resident uniform grid; queries are exact (same result set as the kd-tree,
// ties broken on the lower index).
template <typename IndexT = size_t>
class KDTree3f {
public:
  using NeighborResult = Neighbor<float, IndexT>;
  using NeighborhoodResult = NeighborSet<float, IndexT>;
  using NeighborhoodSetResult = std::vector<NeighborhoodResult>;

  KDTree3f(const ConstVectorSetMatrixMap3f& data, size_t /*max_leaf_size*/ = 10, size_t /*num_build_threads*/ = 1)
      : n_(data.cols()), data_map_(data), cloud_(data) {}

  bool isEmpty() const { return n_ == 0; }

  // single-point queries (core/kd_tree.hpp:181-193, 215-230, 283-299)
  NeighborResult nearestNeighborSearch(const Vector3f& q) const {
    NeighborhoodResult r = kNNInRadiusSearch(q, 1, std::numeric_limits<float>::max());
    if (r.empty()) throw std::runtime_error("nearestNeighborSearch on an empty tree");  // nanoflann.hpp:1715-1718
    return r[0];
  }
  NeighborhoodResult kNNSearch(const Vector3f& q, size_t k) const {
    return kNNInRadiusSearch(q, k, std::numeric_limits<float>::max());
  }
  NeighborhoodResult kNNInRadiusSearch(const Vector3f& q, size_t k, float radius) const {
    NeighborhoodSetResult r = kNNInRadiusSearch(ConstVectorSetMatrixMap3f(q.data(), 1), k, radius);
    return r.empty() ? NeighborhoodResult() : r[0];
  }
  // batched queries (core/kd_tree.hpp:196-213, 232-249, 301-318)
  NeighborhoodResult nearestNeighborSearch(const ConstVectorSetMatrixMap3f& queries) const {
    std::vector<int64_t> idx(queries.cols());
    std::vector<float> d2(queries.cols());
    b200::CloudHandle q(queries);
    b200::check(cb_knn1_radius(b200::Context::get(), cloud_.h, q.h, nullptr, std::numeric_limits<float>::max(),
                               idx.data(), d2.data()),
                "cb_knn1_radius");
    NeighborhoodResult out(queries.cols());
    for (size_t i = 0; i < out.size(); i++) out[i] = {static_cast<IndexT>(idx[i]), d2[i]};
    return out;
  }
  NeighborhoodSetResult kNNSearch(const ConstVectorSetMatrixMap3f& queries, size_t k) const {
    return kNNInRadiusSearch(queries, k, std::numeric_limits<float>::max());
  }
  NeighborhoodSetResult kNNInRadiusSearch(const ConstVectorSetMatrixMap3f& queries, size_t k, float radius) const {
    const size_t nq = queries.cols();
    NeighborhoodSetResult out(nq);
    if (nq == 0 || k == 0 || n_ == 0) return out;
    if (k > 256) throw std::runtime_error("cilantro_b200: kNN supports k <= 256");
    std::vector<int64_t> idx(nq * k);
    std::vector<float> d2(nq * k);
    std::vector<uint32_t> cnt(nq);
    b200::CloudHandle q(queries);
    b200::check(cb_knn_radius(b200::Context::get(), cloud_.h, q.h, nullptr, (int)k, radius, idx.data(), d2.data(),
                              cnt.data()),
                "cb_knn_radius");
    for (size_t i = 0; i < nq; i++) {
      out[i].resize(cnt[i]);
      for (uint32_t j = 0; j < cnt[i]; j++) out[i][j] = {static_cast<IndexT>(idx[i * k + j]), d2[i * k + j]};
    }
    return out;
  }
  // radiusSearch (core/kd_tree.hpp:250-278): every point with squared distance < radius, ascending distance
  NeighborhoodSetResult radiusSearch(const ConstVectorSetMatrixMap3f& queries, float radius) const {
    const size_t nq = queries.cols();
    NeighborhoodSetResult out(nq);
    if (nq == 0 || n_ == 0) return out;
    b200::CloudHandle q(queries);
    std::vector<uint64_t> off(nq + 1);
    size_t total = 0;
    b200::check(cb_radius_search(b200::Context::get(), cloud_.h, q.h, nullptr, radius, off.data(), nullptr, nullptr, 0,
                                 &total),
                "cb_radius_search");
    if (total == 0) return out;
    std::vector<int64_t> idx(total);
    std::vector<float> d2(total);
    b200::check(cb_radius_search(b200::Context::get(), cloud_.h, q.h, nullptr, radius, off.data(), idx.data(), d2.data(),
                                 total, &total),
                "cb_radius_search");
    for (size_t i = 0; i < nq; i++) {
      out[i].resize(off[i + 1] - off[i]);
      for (size_t j = off[i]; j < off[i + 1]; j++) out[i][j - off[i]] = {static_cast<IndexT>(idx[j]), d2[j]};
    }
    return out;
  }
  NeighborhoodResult radiusSearch(const Vector3f& q, float radius) const {
    NeighborhoodSetResult r = radiusSearch(ConstVectorSetMatrixMap3f(q.data(), 1), radius);
    return r.empty() ? NeighborhoodResult() : r[0];
  }
  // search(query / queries, neighbourhood specification) (core/kd_tree.hpp:320-381)
  template <typename QueryT, typename CountT>
  auto search(const QueryT& q, const KNNNeighborhoodSpecification<CountT>& nh) const {
    return kNNSearch(q, (size_t)nh.maxNumberOfNeighbors);
  }
  template <typename QueryT>
  auto search(const QueryT& q, const RadiusNeighborhoodSpecification<float>& nh) const {
    return radiusSearch(q, nh.radius);
  }
  template <typename QueryT, typename CountT>
  auto search(const QueryT& q, const KNNInRadiusNeighborhoodSpecification<float, CountT>& nh) const {
    return kNNInRadiusSearch(q, (size_t)nh.maxNumberOfNeighbors, nh.radius);
  }
  const ConstVectorSetMatrixMap3f& getPointsMatrixMap() const { return data_map_; }  // core/kd_tree.hpp:172-174
  cb_cloud* b200_cloud() const { return cloud_.h; }  // the device cloud (ConnectedComponentExtraction3f)
  size_t b200_size() const { return n_; }

private:
  size_t n_;
  ConstVectorSetMatrixMap3f data_map_;
  b200::CloudHandle cloud_;
};

// ---- ICP ---------------------------------------------------------------------------------------------
enum struct CorrespondenceSearchDirection { FIRST_TO_SECOND, SECOND_TO_FIRST, BOTH };

// CorrespondenceSearchKDTree's fluent surface (correspondence_search/correspondence_search_kd_tree.hpp:237-285).
// The defaults run the fused kernel; any other setting goes through the device-side list (icp_engine.cu).
class CorrespondenceSearchEngineB200 {
public:
  using SearchResult = CorrespondenceSet<float, size_t>;
  float getMaxDistance() const { return max_distance_; }
  CorrespondenceSearchEngineB200& setMaxDistance(float dist_thresh_squared) {
    max_distance_ = dist_thresh_squared;
    return *this;
  }
  const CorrespondenceSearchDirection& getSearchDirection() const { return dir_; }
  CorrespondenceSearchEngineB200& setSearchDirection(const CorrespondenceSearchDirection& d) {
    dir_ = d;
    return *this;
  }
  double getInlierFraction() const { return inlier_fraction_; }
  CorrespondenceSearchEngineB200& setInlierFraction(double fraction) {
    inlier_fraction_ = fraction;
    return *this;
  }
  bool getRequireReciprocality() const { return require_reciprocality_; }
  CorrespondenceSearchEngineB200& setRequireReciprocality(bool require_reciprocal) {
    require_reciprocality_ = require_reciprocal;
    return *this;
  }
  bool getOneToOne() const { return one_to_one_; }
  CorrespondenceSearchEngineB200& setOneToOne(bool one_to_one) {
    one_to_one_ = one_to_one;
    return *this;
  }
  const SearchResult& getCorrespondences() const { return corr_; }
  void fill(cb_icp_params& p) const {
    p.max_d2 = max_distance_;
    p.search_dir = dir_ == CorrespondenceSearchDirection::SECOND_TO_FIRST
                       ? CB_SECOND_TO_FIRST
                       : (dir_ == CorrespondenceSearchDirection::FIRST_TO_SECOND ? CB_FIRST_TO_SECOND : CB_BOTH);
    p.inlier_fraction = inlier_fraction_;
    p.require_reciprocal = require_reciprocality_ ? 1 : 0;
    p.one_to_one = one_to_one_ ? 1 : 0;
  }

private:
  template <int>
  friend class SimpleRigidICP3fB200;
  float max_distance_ = (float)(0.01 * 0.01);  // correspondence_search_kd_tree.hpp:49
  CorrespondenceSearchDirection dir_ = CorrespondenceSearchDirection::SECOND_TO_FIRST;
  double inlier_fraction_ = 1.0;
  bool require_reciprocality_ = false;
  bool one_to_one_ = false;
  SearchResult corr_;
};

template <int kMetric>
class SimpleRigidICP3fB200 {
public:
  using Transform = RigidTransform3f;

  // point-to-point: (dst, src); combined: (dst, dst_normals, src[, src_normals])
  SimpleRigidICP3fB200(const ConstVectorSetMatrixMap3f& dst, const ConstVectorSetMatrixMap3f& src) {
    upload(dst, nullptr, src, nullptr);
    init();
  }
  SimpleRigidICP3fB200(const ConstVectorSetMatrixMap3f& dst, const ConstVectorSetMatrixMap3f& dst_n,
                       const ConstVectorSetMatrixMap3f& src) {
    upload(dst, &dst_n, src, nullptr);
    init();
  }
  SimpleRigidICP3fB200(const ConstVectorSetMatrixMap3f& dst, const ConstVectorSetMatrixMap3f& dst_n,
                       const ConstVectorSetMatrixMap3f& src, const ConstVectorSetMatrixMap3f& src_n) {
    upload(dst, &dst_n, src, &src_n);
    init();
  }
  ~SimpleRigidICP3fB200() {
    if (icp_) cb_icp_destroy(icp_);
  }
  SimpleRigidICP3fB200(const SimpleRigidICP3fB200&) = delete;

  CorrespondenceSearchEngineB200& correspondenceSearchEngine() { return engine_; }
  const CorrespondenceSearchEngineB200& correspondenceSearchEngine() const { return engine_; }

  // IterativeClosestPointBase surface (registration/icp_base.hpp:40-106)
  size_t getMaxNumberOfIterations() const { return prm_.max_iter; }
  SimpleRigidICP3fB200& setMaxNumberOfIterations(size_t n) {
    prm_.max_iter = (int32_t)n;
    return *this;
  }
  size_t getNumberOfPerformedIterations() const { return res_.iterations; }
  float getConvergenceTolerance() const { return prm_.tol; }
  SimpleRigidICP3fB200& setConvergenceTolerance(float tol) {
    prm_.tol = tol;
    return *this;
  }
  RigidTransform3f getInitialTransform() const { return RigidTransform3f(prm_.T_init); }
  SimpleRigidICP3fB200& setInitialTransform(const RigidTransform3f& T) {
    std::memcpy(prm_.T_init, T.data(), sizeof(prm_.T_init));
    return *this;
  }
  float getLastUpdateNorm() const { return res_.last_delta; }
  bool hasConverged() const { return res_.last_delta < prm_.tol; }
  const RigidTransform3f& getTransform() const { return T_; }

  // CombinedMetricSingleTransformICP surface (icp_single_transform_combined_metric.hpp:103-141)
  float getPointToPointMetricWeight() const { return prm_.w_pt; }
  SimpleRigidICP3fB200& setPointToPointMetricWeight(float w) {
    prm_.w_pt = w;
    return *this;
  }
  float getPointToPlaneMetricWeight() const { return prm_.w_pl; }
  SimpleRigidICP3fB200& setPointToPlaneMetricWeight(float w) {
    prm_.w_pl = w;
    return *this;
  }
  size_t getMaxNumberOfOptimizationStepIterations() const { return prm_.max_opt_iter; }
  SimpleRigidICP3fB200& setMaxNumberOfOptimizationStepIterations(size_t n) {
    prm_.max_opt_iter = (int32_t)n;
    return *this;
  }
  float getOptimizationStepConvergenceTolerance() const { return prm_.opt_tol; }
  SimpleRigidICP3fB200& setOptimizationStepConvergenceTolerance(float tol) {
    prm_.opt_tol = tol;
    return *this;
  }

  SimpleRigidICP3fB200& estimate() {
    engine_.fill(prm_);
    b200::check(cb_icp_estimate(icp_, &prm_, &res_), "cb_icp_estimate");
    T_ = RigidTransform3f(res_.T);
    corr_fresh_ = false;
    return *this;
  }
  SimpleRigidICP3fB200& estimate(size_t max_iter, float conv_tol) {
    prm_.max_iter = (int32_t)max_iter;
    prm_.tol = conv_tol;
    return estimate();
  }

  // correspondenceSearchEngine().getCorrespondences() after estimate(): materialised on demand
  const CorrespondenceSet<float, size_t>& getCorrespondences() {
    if (!corr_fresh_) {
      const size_t n = cb_cloud_size(src_.h) + cb_cloud_size(dst_.h);
      std::vector<uint64_t> a(n), b(n);
      std::vector<float> v(n);
      size_t cnt = 0;
      b200::check(cb_icp_correspondences(icp_, a.data(), b.data(), v.data(), &cnt), "cb_icp_correspondences");
      engine_.corr_.resize(cnt);
      for (size_t i = 0; i < cnt; i++) engine_.corr_[i] = {(size_t)a[i], (size_t)b[i], v[i]};
      corr_fresh_ = true;
    }
    return engine_.corr_;
  }

  // getResiduals() -> computeResiduals() (icp_base.hpp:102-104): 1 x N_src
  std::vector<float> getResiduals() {
    std::vector<float> r(cb_cloud_size(src_.h));
    prm_.max_d2 = engine_.max_distance_;
    b200::check(cb_icp_residuals(icp_, &prm_, T_.data(), r.data()), "cb_icp_residuals");
    return r;
  }

  double getLastEstimateDeviceMilliseconds() const { return res_.gpu_ms_total; }

protected:
  cb_icp_params& params() { return prm_; }

private:
  // both clouds in one call: the source upload overlaps the destination's grid build (cb_cloud_create_pair)
  void upload(const ConstVectorSetMatrixMap3f& dst, const ConstVectorSetMatrixMap3f* dst_n,
              const ConstVectorSetMatrixMap3f& src, const ConstVectorSetMatrixMap3f* src_n) {
    const float* dn = (dst_n && dst_n->cols() == dst.cols() && dst.cols() > 0) ? dst_n->data() : nullptr;
    const float* sn = (src_n && src_n->cols() == src.cols() && src.cols() > 0) ? src_n->data() : nullptr;
    b200::check(cb_cloud_create_pair(b200::Context::get(), dst.data(), dn, dst.cols(), 0, src.data(), sn, src.cols(), 0,
                                     &dst_.h, &src_.h),
                "cb_cloud_create_pair");
  }
  void init() {
    cb_icp_default_params(&prm_);
    prm_.metric = kMetric;
    std::memset(&res_, 0, sizeof(res_));
    res_.last_delta = std::numeric_limits<float>::infinity();
    b200::check(cb_icp_create(b200::Context::get(), dst_.h, src_.h, &icp_), "cb_icp_create");
  }
  b200::CloudHandle dst_, src_;
  cb_icp* icp_ = nullptr;
  cb_icp_params prm_;
  cb_icp_result res_;
  RigidTransform3f T_;
  CorrespondenceSearchEngineB200 engine_;
  bool corr_fresh_ = false;
};

using SimplePointToPointMetricRigidICP3f = SimpleRigidICP3fB200<CB_ICP_POINT_TO_POINT>;
using SimpleCombinedMetricRigidICP3f = SimpleRigidICP3fB200<CB_ICP_COMBINED>;

// ---- correspondence weight evaluators (core/common_pair_evaluators.hpp) ---------------------------------------
// The two evaluators a C ABI can carry, by kind + coefficient (cb_icp_params::pt_weight_kind ...). Same class names
// and setters as the reference; operator() is kept so that host-side code calling the evaluator still compiles.
template <typename ValueT = float, typename WeightT = ValueT>
class UnityWeightEvaluator {  // :29-43
public:
  using InputScalar = ValueT;
  using OutputScalar = WeightT;
  constexpr WeightT operator()(ValueT) const { return (WeightT)1; }
  constexpr WeightT operator()(size_t, size_t, ValueT) const { return (WeightT)1; }
  static constexpr int b200_kind() { return CB_WEIGHT_UNITY; }
  float b200_coeff() const { return 0.f; }
};

template <typename ValueT = float, typename WeightT = ValueT, bool distances_are_squared = true>
class RBFKernelWeightEvaluator {  // :46-79
  static_assert(distances_are_squared, "ICP correspondences carry squared distances: only the <.., true> evaluator maps to the device path");

public:
  using InputScalar = ValueT;
  using OutputScalar = WeightT;
  RBFKernelWeightEvaluator() : coeff_(-(WeightT)(0.5)) {}
  RBFKernelWeightEvaluator(ValueT sigma) : coeff_(-(WeightT)(0.5) / (sigma * sigma)) {}
  RBFKernelWeightEvaluator& setSigma(ValueT sigma) {
    coeff_ = -(WeightT)(0.5) / (sigma * sigma);
    return *this;
  }
  WeightT operator()(ValueT dist) const { return std::exp(coeff_ * static_cast<WeightT>(dist)); }
  WeightT operator()(size_t, size_t, ValueT dist) const { return std::exp(coeff_ * static_cast<WeightT>(dist)); }
  static constexpr int b200_kind() { return CB_WEIGHT_RBF; }
  float b200_coeff() const { return (float)coeff_; }

private:
  WeightT coeff_;
};

// CombinedMetricRigidICP3f<CorrSearchT, PointToPointCorrWeightEvaluatorT, PointToPlaneCorrWeightEvaluatorT>
// (registration/icp_common_instances.hpp:29-31 over icp_single_transform_combined_metric.hpp:9-101): the general form
// with caller-owned evaluators, held by reference like the reference does (their sigma is read at every estimate()).
// The correspondence search engine argument of the reference is this object's own engine
// (correspondenceSearchEngine()); any evaluator type other than the two above is a compile-time error.
template <class PointToPointCorrWeightEvaluatorT = UnityWeightEvaluator<float, float>,
          class PointToPlaneCorrWeightEvaluatorT = UnityWeightEvaluator<float, float>>
class CombinedMetricRigidICP3f : public SimpleRigidICP3fB200<CB_ICP_COMBINED> {
  using Base = SimpleRigidICP3fB200<CB_ICP_COMBINED>;

public:
  using PointToPointCorrespondenceWeightEvaluator = PointToPointCorrWeightEvaluatorT;
  using PointToPlaneCorrespondenceWeightEvaluator = PointToPlaneCorrWeightEvaluatorT;
  CombinedMetricRigidICP3f(const ConstVectorSetMatrixMap3f& dst, const ConstVectorSetMatrixMap3f& dst_n,
                           const ConstVectorSetMatrixMap3f& src, PointToPointCorrWeightEvaluatorT& point_corr_eval,
                           PointToPlaneCorrWeightEvaluatorT& plane_corr_eval)
      : Base(dst, dst_n, src), pt_(point_corr_eval), pl_(plane_corr_eval) {}
  CombinedMetricRigidICP3f(const ConstVectorSetMatrixMap3f& dst, const ConstVectorSetMatrixMap3f& dst_n,
                           const ConstVectorSetMatrixMap3f& src, const ConstVectorSetMatrixMap3f& src_n,
                           PointToPointCorrWeightEvaluatorT& point_corr_eval, PointToPlaneCorrWeightEvaluatorT& plane_corr_eval)
      : Base(dst, dst_n, src, src_n), pt_(point_corr_eval), pl_(plane_corr_eval) {}
  PointToPointCorrWeightEvaluatorT& pointToPointCorrespondenceWeightEvaluator() { return pt_; }
  PointToPlaneCorrWeightEvaluatorT& pointToPlaneCorrespondenceWeightEvaluator() { return pl_; }
  CombinedMetricRigidICP3f& estimate() {
    this->params().pt_weight_kind = PointToPointCorrWeightEvaluatorT::b200_kind();
    this->params().pl_weight_kind = PointToPlaneCorrWeightEvaluatorT::b200_kind();
    this->params().pt_weight_coeff = pt_.b200_coeff();
    this->params().pl_weight_coeff = pl_.b200_coeff();
    Base::estimate();
    return *this;
  }
  CombinedMetricRigidICP3f& estimate(size_t max_iter, float conv_tol) {
    this->setMaxNumberOfIterations(max_iter);
    this->setConvergenceTolerance(conv_tol);
    return estimate();
  }

private:
  PointToPointCorrWeightEvaluatorT& pt_;
  PointToPlaneCorrWeightEvaluatorT& pl_;
};

// transformPoints(tform, in, out) — core/space_transformations.hpp:203-216
inline void transformPoints(const RigidTransform3f& tform, const ConstVectorSetMatrixMap3f& points, VectorSet3f& result) {
  result.resize(3, points.cols());
  b200::check(cb_transform_points(b200::Context::get(), tform.data(), points.data(), points.cols(), result.data()),
              "cb_transform_points");
}

// ---- KMeans3f<> -------------------------------------------------------------------------------------
template <typename PointIndexT = size_t, typename ClusterIndexT = size_t>
class KMeans3f {
public:
  using ClusterToPointIndicesMap = std::vector<std::vector<PointIndexT>>;
  using PointToClusterIndexMap = std::vector<ClusterIndexT>;

  KMeans3f(const ConstVectorSetMatrixMap3f& data) : n_(data.cols()), host_(data), cloud_(data) {}

  KMeans3f& cluster(const ConstVectorSetMatrixMap3f& centroids, size_t max_iter = 100,
                    float tol = std::numeric_limits<float>::epsilon(), bool use_kd_tree = false) {
    (void)use_kd_tree;  // both branches of the reference compute the same assignment; one GPU kernel here
    centroids_.resize(3, centroids.cols());
    std::memcpy(centroids_.data(), centroids.data(), 3 * centroids.cols() * sizeof(float));
    return run(max_iter, tol);
  }
  KMeans3f& cluster(size_t num_clusters, size_t max_iter = 100, float tol = std::numeric_limits<float>::epsilon(),
                    bool use_kd_tree = false, uint32_t seed = b200::random_seed()) {
    (void)use_kd_tree;
    const size_t k = std::max<size_t>(1, std::min(num_clusters, n_));  // kmeans.hpp:34-36
    std::vector<uint64_t> idx(k);
    b200::check(cb_kmeans_seed_indices(n_, k, seed, idx.data()), "cb_kmeans_seed_indices");
    centroids_.resize(3, k);
    for (size_t j = 0; j < k; j++) centroids_.setCol(j, host_.col(idx[j]));
    return run(max_iter, tol);
  }
  const VectorSet3f& getClusterCentroids() const { return centroids_; }
  size_t getNumberOfPerformedIterations() const { return iterations_; }
  const PointToClusterIndexMap& getPointToClusterIndexMap() const { return labels_; }
  const ClusterToPointIndicesMap& getClusterToPointIndicesMap() const { return lists_; }
  size_t getNumberOfClusters() const { return lists_.size(); }
  size_t getNumberOfPoints() const { return labels_.size(); }

private:
  struct std_seed_helper {};
  KMeans3f& run(size_t max_iter, float tol) {
    std::vector<uint64_t> lab(n_);
    cb_kmeans_result r;
    b200::check(cb_kmeans_cluster(b200::Context::get(), cloud_.h, centroids_.data(), centroids_.cols(), max_iter, tol,
                                  lab.data(), &r),
                "cb_kmeans_cluster");
    iterations_ = r.iterations;
    labels_.assign(lab.begin(), lab.end());
    lists_.assign(centroids_.cols(), {});  // clustering_base.hpp:22-32
    for (size_t i = 0; i < labels_.size(); i++)
      if ((size_t)labels_[i] < lists_.size()) lists_[labels_[i]].emplace_back((PointIndexT)i);
    return *this;
  }
  size_t n_;
  ConstVectorSetMatrixMap3f host_;
  b200::CloudHandle cloud_;
  VectorSet3f centroids_;
  size_t iterations_ = 0;
  PointToClusterIndexMap labels_;
  ClusterToPointIndicesMap lists_;
};

// ---- RigidTransformRANSACEstimator3f<> ----------------------------------------------------------------
template <typename IndexT = size_t>
class RigidTransformRANSACEstimator3f {
public:
  using Model = RigidTransform3f;
  using ResidualVector = std::vector<float>;
  using IndexVector = std::vector<IndexT>;

  RigidTransformRANSACEstimator3f(const ConstVectorSetMatrixMap3f& dst, const ConstVectorSetMatrixMap3f& src)
      : n_(dst.cols()), dst_(dst), src_(src) {
    defaults();
  }
  template <class CorrespondencesT>
  RigidTransformRANSACEstimator3f(const ConstVectorSetMatrixMap3f& dst, const ConstVectorSetMatrixMap3f& src,
                                  const CorrespondencesT& corr)
      : n_(corr.size()), dst_g_(gather(dst, corr, true)), src_g_(gather(src, corr, false)), dst_(dst_g_), src_(src_g_) {
    defaults();
  }

  // (dst, src, dst_ind, src_ind): pair k = (dst point dst_ind[k], src point src_ind[k])
  // (model_estimation/ransac_transform_estimator.hpp:46-59)
  template <typename IdxT>
  RigidTransformRANSACEstimator3f(const ConstVectorSetMatrixMap3f& dst, const ConstVectorSetMatrixMap3f& src,
                                  const std::vector<IdxT>& dst_ind, const std::vector<IdxT>& src_ind)
      : n_(dst_ind.size()), dst_g_(gather_ind(dst, dst_ind, dst_ind.size())), src_g_(gather_ind(src, src_ind, dst_ind.size())),
        dst_(dst_g_), src_(src_g_) {
    defaults();
  }

  // RandomSampleConsensusBase setters (model_estimation/ransac_base.hpp:29-62)
  RigidTransformRANSACEstimator3f& setMaxInlierResidual(float t) { thresh_ = t; return *this; }
  RigidTransformRANSACEstimator3f& setTargetInlierCount(size_t c) { target_ = c; return *this; }
  RigidTransformRANSACEstimator3f& setMaxNumberOfIterations(size_t n) { max_iter_ = n; return *this; }
  RigidTransformRANSACEstimator3f& setReEstimationStep(bool b) { re_estimate_ = b; return *this; }
  RigidTransformRANSACEstimator3f& setRandomSeed(uint32_t s) { seed_ = s; return *this; }  // injected (SURVEY F8)
  float getMaxInlierResidual() const { return thresh_; }
  size_t getTargetInlierCount() const { return target_; }
  size_t getMaxNumberOfIterations() const { return max_iter_; }
  bool getReEstimationStep() const { return re_estimate_; }

  RigidTransformRANSACEstimator3f& estimate() {
    cb_ransac_result r;
    std::vector<uint64_t> inl(n_);
    residuals_.resize(n_);
    b200::check(cb_ransac_rigid(b200::Context::get(), dst_.h, src_.h, seed_, target_, max_iter_, thresh_,
                                re_estimate_ ? 1 : 0, &r, inl.data(), residuals_.data()),
                "cb_ransac_rigid");
    model_ = RigidTransform3f(r.T);
    iterations_ = r.iterations;
    inliers_.assign(inl.begin(), inl.begin() + r.num_inliers);
    return *this;
  }
  RigidTransformRANSACEstimator3f& estimate(float max_residual, size_t target_inlier_count, size_t max_iter) {
    thresh_ = max_residual;
    target_ = target_inlier_count;
    max_iter_ = max_iter;
    return estimate();
  }
  const Model& getModel() const { return model_; }
  const ResidualVector& getModelResiduals() const { return residuals_; }
  const IndexVector& getModelInliers() const { return inliers_; }
  bool targetInlierCountAchieved() const { return inliers_.size() >= target_; }
  size_t getNumberOfPerformedIterations() const { return iterations_; }
  size_t getNumberOfInliers() const { return inliers_.size(); }

private:
  void defaults() {  // ransac_transform_estimator.hpp:27
    target_ = n_ / 2 + n_ % 2;
    max_iter_ = 100;
    thresh_ = 0.01f;
    re_estimate_ = true;
    seed_ = b200::random_seed();
  }
  template <class CorrespondencesT>
  static VectorSet3f gather(const ConstVectorSetMatrixMap3f& pts, const CorrespondencesT& corr, bool first) {
    VectorSet3f out(3, corr.size());  // :31-44
    for (size_t i = 0; i < corr.size(); i++) out.setCol(i, pts.col(first ? corr[i].indexInFirst : corr[i].indexInSecond));
    return out;
  }
  template <typename IdxT>
  static VectorSet3f gather_ind(const ConstVectorSetMatrixMap3f& pts, const std::vector<IdxT>& ind, size_t count) {
    VectorSet3f out(3, count);  // :53-58 (the loop runs over dst_ind.size() for both sets)
    for (size_t i = 0; i < count; i++) out.setCol(i, pts.col((size_t)ind[i]));
    return out;
  }
  size_t n_;
  VectorSet3f dst_g_, src_g_;
  b200::CloudHandle dst_, src_;
  size_t target_, max_iter_, iterations_ = 0;
  float thresh_;
  bool re_estimate_;
  uint32_t seed_;
  Model model_;
  ResidualVector residuals_;
  IndexVector inliers_;
};

// ---- PrincipalComponentAnalysis3f -----------------------------------------------------------------------
class PrincipalComponentAnalysis3f {
public:
  PrincipalComponentAnalysis3f(const ConstVectorSetMatrixMap3f& data, bool /*parallel*/ = false) {
    b200::CloudHandle c(data);
    b200::check(cb_pca(b200::Context::get(), c.h, mean_.data(), cov_.data(), evals_.data(), evecs_.data()), "cb_pca");
  }
  // subset constructor (core/principal_component_analysis.hpp:24-30): the listed points only
  template <typename ContainerT, typename = decltype(std::declval<const ContainerT&>().begin())>
  PrincipalComponentAnalysis3f(const ConstVectorSetMatrixMap3f& data, const ContainerT& subset, bool /*parallel*/ = false) {
    std::vector<float> sel;
    for (auto it = subset.begin(); it != subset.end(); ++it) {
      const Vector3f p = data.col((size_t)*it);
      sel.insert(sel.end(), {p[0], p[1], p[2]});
    }
    b200::CloudHandle c(ConstVectorSetMatrixMap3f(sel.data(), sel.size() / 3));
    b200::check(cb_pca(b200::Context::get(), c.h, mean_.data(), cov_.data(), evals_.data(), evecs_.data()), "cb_pca");
  }
  const Vector3f& getDataMean() const { return mean_; }
  const std::array<float, 9>& getDataCovariance() const { return cov_; }  // row-major 3x3
  const Vector3f& getEigenValues() const { return evals_; }               // descending
  const std::array<float, 9>& getEigenVectors() const { return evecs_; }  // row-major, columns = eigenvectors

  // project(points, target_dim) (:46-49): target_dim x N, column-major = eigenvectors.leftCols(target_dim)^T (p - mean).
  // A 3 x k map applied once after the device pass, like the reference's Eigen expression (not part of the hot path).
  std::vector<float> project(const ConstVectorSetMatrixMap3f& points, size_t target_dim) const {
    const size_t k = std::min<size_t>(target_dim, 3), n = points.cols();
    std::vector<float> out(k * n);
    for (size_t i = 0; i < n; i++) {
      const Vector3f p = points.col(i);
      const float c[3] = {p[0] - mean_[0], p[1] - mean_[1], p[2] - mean_[2]};
      for (size_t j = 0; j < k; j++) out[k * i + j] = evecs_[j] * c[0] + evecs_[3 + j] * c[1] + evecs_[6 + j] * c[2];
    }
    return out;
  }
  template <size_t DimOut>
  std::vector<float> project(const ConstVectorSetMatrixMap3f& points) const {  // :51-57
    static_assert(DimOut >= 1 && DimOut <= 3, "projection dimension of a 3-D PCA");
    return project(points, DimOut);
  }
  // reconstruct(points) (:59-70): points is dim_in x N column-major; returns 3 x N = leftCols(dim_in) * points + mean
  VectorSet3f reconstruct(const float* points, size_t dim_in, size_t n) const {
    const size_t k = std::min<size_t>(dim_in, 3);
    VectorSet3f out(3, n);
    for (size_t i = 0; i < n; i++) {
      float q[3] = {mean_[0], mean_[1], mean_[2]};
      for (size_t j = 0; j < k; j++)
        for (int r = 0; r < 3; r++) q[r] += evecs_[3 * r + j] * points[dim_in * i + j];
      out.setCol(i, Vector3f(q[0], q[1], q[2]));
    }
    return out;
  }
  VectorSet3f reconstruct(const std::vector<float>& points, size_t dim_in) const {
    return reconstruct(points.data(), dim_in, dim_in ? points.size() / dim_in : 0);
  }

private:
  Vector3f mean_, evals_;
  std::array<float, 9> cov_{}, evecs_{};
};

// ---- PointCloud3f ------------------------------------------------------------------------------------------
// ---- normal estimation (core/normal_estimation.hpp:11-421) ------------------------------------------
// Same call surface as NormalEstimation<float,3>: neighbourhoods over the cloud itself; radii are
// squared distances; fewer than 3 neighbours -> NaN; view point (default: none, :24-25) orients the
// normals; reference normals (setReferenceNormals, :63-69) take precedence over it (:281-291).
class NormalEstimation3f {
public:
  NormalEstimation3f(const ConstVectorSetMatrixMap3f& points, size_t /*max_leaf_size*/ = 10)
      : n_(points.cols()), points_(points), cloud_(points) {
    const float nan = std::numeric_limits<float>::quiet_NaN();
    view_point_ = Vector3f(nan, nan, nan);
  }
  // from an existing search tree (:30-39): the same points; the device grid is rebuilt for this object
  template <typename IndexT>
  explicit NormalEstimation3f(const KDTree3f<IndexT>& kd_tree) : NormalEstimation3f(kd_tree.getPointsMatrixMap()) {}
  // getNormals* (:71-81 and the Radius / KNNInRadius twins): return by value
  VectorSet3f getNormalsKNN(size_t k) const { return estimateNormalsKNN(k); }
  VectorSet3f getNormalsRadius(float radius) const { return estimateNormalsRadius(radius); }
  VectorSet3f getNormalsKNNInRadius(size_t k, float radius) const { return estimateNormalsKNNInRadius(k, radius); }
  const Vector3f& getViewPoint() const { return view_point_; }
  NormalEstimation3f& setViewPoint(const Vector3f& vp) {  // :52-56
    view_point_ = vp;
    return *this;
  }
  NormalEstimation3f& setReferenceNormals(const ConstVectorSetMatrixMap3f& ref_normals) {  // :63-69
    if (ref_normals.cols() == n_) {  // a copy: the caller may pass the very buffer the result goes to
      ref_normals_.assign(ref_normals.data(), ref_normals.data() + 3 * n_);
      use_ref_ = n_ > 0;
    }
    return *this;
  }
  // kNN (:83-129)
  const NormalEstimation3f& estimateNormalsAndCurvatureKNN(VectorSet3f& normals, std::vector<float>& curvature,
                                                           size_t k) const {
    return run(&normals, &curvature, k, 0.f);
  }
  const NormalEstimation3f& estimateNormalsKNN(VectorSet3f& normals, size_t k) const {
    return run(&normals, nullptr, k, 0.f);
  }
  VectorSet3f estimateNormalsKNN(size_t k) const {
    VectorSet3f n;
    run(&n, nullptr, k, 0.f);
    return n;
  }
  const NormalEstimation3f& estimateCurvatureKNN(std::vector<float>& curvature, size_t k) const {
    return run(nullptr, &curvature, k, 0.f);
  }
  // radius (:131-177)
  const NormalEstimation3f& estimateNormalsAndCurvatureRadius(VectorSet3f& normals, std::vector<float>& curvature,
                                                              float radius) const {
    return run(&normals, &curvature, 0, radius);
  }
  const NormalEstimation3f& estimateNormalsRadius(VectorSet3f& normals, float radius) const {
    return run(&normals, nullptr, 0, radius);
  }
  VectorSet3f estimateNormalsRadius(float radius) const {
    VectorSet3f n;
    run(&n, nullptr, 0, radius);
    return n;
  }
  const NormalEstimation3f& estimateCurvatureRadius(std::vector<float>& curvature, float radius) const {
    return run(nullptr, &curvature, 0, radius);
  }
  // kNN in radius (:179-232)
  const NormalEstimation3f& estimateNormalsAndCurvatureKNNInRadius(VectorSet3f& normals,
                                                                   std::vector<float>& curvature, size_t k,
                                                                   float radius) const {
    return run(&normals, &curvature, k, radius);
  }
  const NormalEstimation3f& estimateNormalsKNNInRadius(VectorSet3f& normals, size_t k, float radius) const {
    return run(&normals, nullptr, k, radius);
  }
  VectorSet3f estimateNormalsKNNInRadius(size_t k, float radius) const {
    VectorSet3f n;
    run(&n, nullptr, k, radius);
    return n;
  }
  const NormalEstimation3f& estimateCurvatureKNNInRadius(std::vector<float>& curvature, size_t k,
                                                         float radius) const {
    return run(nullptr, &curvature, k, radius);
  }

private:
  const NormalEstimation3f& run(VectorSet3f* normals, std::vector<float>* curvature, size_t k, float radius) const {
    if (k > 128) throw std::runtime_error("cilantro_b200: normal estimation supports k <= 128 neighbours");
    if (normals) normals->resize(3, n_);
    if (curvature) curvature->resize(n_);
    if (n_ == 0) return *this;
    const float nan = std::numeric_limits<float>::quiet_NaN();
    if (k == 0 && !(radius > 0.f)) {  // empty neighbourhoods: every sample is below the minimum size
      if (normals) std::fill(normals->data(), normals->data() + 3 * n_, nan);
      if (curvature) std::fill(curvature->begin(), curvature->end(), nan);
      return *this;
    }
    if (use_ref_) {  // re-upload the reference normals: the previous call overwrote the cloud's normals
      ConstVectorSetMatrixMap3f ref(ref_normals_);
      cloud_.reset(points_, &ref);
    }
    b200::check(cb_cloud_estimate_normals(b200::Context::get(), cloud_.h, (int)k, radius, view_point_.data(),
                                          use_ref_ ? 1 : 0, normals ? normals->data() : nullptr,
                                          curvature ? curvature->data() : nullptr, nullptr, nullptr),
                "cb_cloud_estimate_normals");
    return *this;
  }
  size_t n_;
  ConstVectorSetMatrixMap3f points_;
  mutable b200::CloudHandle cloud_;
  Vector3f view_point_;
  std::vector<float> ref_normals_;
  bool use_ref_ = false;
};

// ---- voxel-grid downsampling (core/grid_downsampler.hpp, core/grid_accumulator.hpp) ---------------------
// One implementation behind the four reference class names: the constructor takes the same arguments
// (points [, normals] [, colors], bin_size, parallel); parallel selects the reference's output order
// (true: bins in lexicographic (x, y, z) order, the std::map order of the parallel build; false: in order
// of first occurrence, the serial build). The per-bin sums are always the serial build's (index order).
namespace b200 {
class GridDownsampler {
public:
  GridDownsampler(const ConstVectorSetMatrixMap3f& points, const ConstVectorSetMatrixMap3f* normals,
                  const ConstVectorSetMatrixMap3f* colors, float bin_size, bool parallel)
      : points_(points), normals_(normals ? *normals : ConstVectorSetMatrixMap3f()),
        colors_(colors ? *colors : ConstVectorSetMatrixMap3f()), has_n_(normals != nullptr), has_c_(colors != nullptr),
        bin_size_(bin_size), order_(parallel ? 0 : 1) {}

protected:
  void run(VectorSet3f* ds_points, VectorSet3f* ds_normals, VectorSet3f* ds_colors, size_t min_points_in_bin) const {
    const size_t n = points_.cols();
    VectorSet3f p(3, n), nn(3, has_n_ ? n : 0), cc(3, has_c_ ? n : 0);
    size_t m = 0;
    check(cb_grid_downsample(Context::get(), points_.data(), has_n_ ? normals_.data() : nullptr,
                             has_c_ ? colors_.data() : nullptr, n, bin_size_, min_points_in_bin, order_, p.data(),
                             has_n_ ? nn.data() : nullptr, has_c_ ? cc.data() : nullptr, &m),
          "cb_grid_downsample");
    p.resize(3, m);
    if (ds_points) *ds_points = std::move(p);
    if (ds_normals && has_n_) {
      nn.resize(3, m);
      *ds_normals = std::move(nn);
    }
    if (ds_colors && has_c_) {
      cc.resize(3, m);
      *ds_colors = std::move(cc);
    }
  }
  ConstVectorSetMatrixMap3f points_, normals_, colors_;
  bool has_n_, has_c_;
  float bin_size_;
  int order_;
};
}  // namespace b200

class PointsGridDownsampler3f : public b200::GridDownsampler {  // grid_downsampler.hpp:8-44
public:
  PointsGridDownsampler3f(const ConstVectorSetMatrixMap3f& points, float bin_size, bool parallel = true)
      : GridDownsampler(points, nullptr, nullptr, bin_size, parallel) {}
  const PointsGridDownsampler3f& getDownsampledPoints(VectorSet3f& ds_points, size_t min_points_in_bin = 1) const {
    run(&ds_points, nullptr, nullptr, min_points_in_bin);
    return *this;
  }
  VectorSet3f getDownsampledPoints(size_t min_points_in_bin = 1) const {
    VectorSet3f p;
    run(&p, nullptr, nullptr, min_points_in_bin);
    return p;
  }
};

class PointsNormalsGridDownsampler3f : public b200::GridDownsampler {  // grid_downsampler.hpp:46-132
public:
  PointsNormalsGridDownsampler3f(const ConstVectorSetMatrixMap3f& points, const ConstVectorSetMatrixMap3f& normals,
                                 float bin_size, bool parallel = true)
      : GridDownsampler(points, &normals, nullptr, bin_size, parallel) {}
  const PointsNormalsGridDownsampler3f& getDownsampledPoints(VectorSet3f& p, size_t min_points_in_bin = 1) const {
    run(&p, nullptr, nullptr, min_points_in_bin);
    return *this;
  }
  const PointsNormalsGridDownsampler3f& getDownsampledNormals(VectorSet3f& nn, size_t min_points_in_bin = 1) const {
    run(nullptr, &nn, nullptr, min_points_in_bin);
    return *this;
  }
  const PointsNormalsGridDownsampler3f& getDownsampledPointsNormals(VectorSet3f& p, VectorSet3f& nn,
                                                                    size_t min_points_in_bin = 1) const {
    run(&p, &nn, nullptr, min_points_in_bin);
    return *this;
  }
};

class PointsColorsGridDownsampler3f : public b200::GridDownsampler {  // grid_downsampler.hpp:134-220
public:
  PointsColorsGridDownsampler3f(const ConstVectorSetMatrixMap3f& points, const ConstVectorSetMatrixMap3f& colors,
                                float bin_size, bool parallel = true)
      : GridDownsampler(points, nullptr, &colors, bin_size, parallel) {}
  const PointsColorsGridDownsampler3f& getDownsampledPoints(VectorSet3f& p, size_t min_points_in_bin = 1) const {
    run(&p, nullptr, nullptr, min_points_in_bin);
    return *this;
  }
  const PointsColorsGridDownsampler3f& getDownsampledColors(VectorSet3f& cc, size_t min_points_in_bin = 1) const {
    run(nullptr, nullptr, &cc, min_points_in_bin);
    return *this;
  }
  const PointsColorsGridDownsampler3f& getDownsampledPointsColors(VectorSet3f& p, VectorSet3f& cc,
                                                                  size_t min_points_in_bin = 1) const {
    run(&p, nullptr, &cc, min_points_in_bin);
    return *this;
  }
};

class PointsNormalsColorsGridDownsampler3f : public b200::GridDownsampler {  // grid_downsampler.hpp:222-340
public:
  PointsNormalsColorsGridDownsampler3f(const ConstVectorSetMatrixMap3f& points,
                                       const ConstVectorSetMatrixMap3f& normals,
                                       const ConstVectorSetMatrixMap3f& colors, float bin_size, bool parallel = true)
      : GridDownsampler(points, &normals, &colors, bin_size, parallel) {}
  const PointsNormalsColorsGridDownsampler3f& getDownsampledPoints(VectorSet3f& p, size_t min_points_in_bin = 1) const {
    run(&p, nullptr, nullptr, min_points_in_bin);
    return *this;
  }
  const PointsNormalsColorsGridDownsampler3f& getDownsampledNormals(VectorSet3f& nn,
                                                                    size_t min_points_in_bin = 1) const {
    run(nullptr, &nn, nullptr, min_points_in_bin);
    return *this;
  }
  const PointsNormalsColorsGridDownsampler3f& getDownsampledColors(VectorSet3f& cc, size_t min_points_in_bin = 1) const {
    run(nullptr, nullptr, &cc, min_points_in_bin);
    return *this;
  }
  const PointsNormalsColorsGridDownsampler3f& getDownsampledPointsNormalsColors(VectorSet3f& p, VectorSet3f& nn,
                                                                                VectorSet3f& cc,
                                                                                size_t min_points_in_bin = 1) const {
    run(&p, &nn, &cc, min_points_in_bin);
    return *this;
  }
};

struct PointCloud3f {
  VectorSet3f points, normals, colors;
  PointCloud3f() = default;
  // PLY passthrough (utilities/point_cloud.hpp:118-121, :502-543; b200_ply.hpp)
  explicit PointCloud3f(const std::string& file_name) { fromPLYFile(file_name); }
  PointCloud3f& fromPLYFile(const std::string& file_name, bool /*preload*/ = true) {
    std::vector<float> p, n, c;
    b200::ply::read(file_name, p, n, c);
    auto assign = [](VectorSet3f& dst, const std::vector<float>& src) {
      dst.resize(3, src.size() / 3);
      if (!src.empty()) std::memcpy(dst.data(), src.data(), src.size() * sizeof(float));
    };
    assign(points, p);
    assign(normals, n);
    assign(colors, c);
    return *this;
  }
  const PointCloud3f& toPLYFile(const std::string& file_name, bool binary = true) const {
    b200::ply::write(file_name, binary, size(), points.data(), hasNormals() ? normals.data() : nullptr,
                     hasColors() ? colors.data() : nullptr);
    return *this;
  }
  PointCloud3f& clear() {  // :131-136
    points.resize(3, 0);
    normals.resize(3, 0);
    colors.resize(3, 0);
    return *this;
  }
  PointCloud3f& append(const PointCloud3f& cloud) {  // :138-152
    const size_t n0 = size(), n1 = cloud.size();
    auto grow = [&](VectorSet3f& dst, const VectorSet3f& src) {
      dst.resize(3, n0 + n1);
      if (n1) std::memcpy(dst.data() + 3 * n0, src.data(), 3 * n1 * sizeof(float));
    };
    const bool keep_n = normals.cols() == n0 && cloud.hasNormals(), keep_c = colors.cols() == n0 && cloud.hasColors();
    grow(points, cloud.points);
    if (keep_n) grow(normals, cloud.normals);
    if (keep_c) grow(colors, cloud.colors);
    return *this;
  }
  // utilities/point_cloud.hpp:246-290
  PointCloud3f& gridDownsample(float bin_size, size_t min_points_in_bin = 1, bool parallel = true) {
    PointCloud3f res = gridDownsampled(bin_size, min_points_in_bin, parallel);
    *this = std::move(res);
    return *this;
  }
  PointCloud3f gridDownsampled(float bin_size, size_t min_points_in_bin = 1, bool parallel = true) const {
    PointCloud3f res;
    if (hasNormals() && hasColors()) {
      PointsNormalsColorsGridDownsampler3f(points, normals, colors, bin_size, parallel)
          .getDownsampledPointsNormalsColors(res.points, res.normals, res.colors, min_points_in_bin);
    } else if (hasNormals()) {
      PointsNormalsGridDownsampler3f(points, normals, bin_size, parallel)
          .getDownsampledPointsNormals(res.points, res.normals, min_points_in_bin);
    } else if (hasColors()) {
      PointsColorsGridDownsampler3f(points, colors, bin_size, parallel)
          .getDownsampledPointsColors(res.points, res.colors, min_points_in_bin);
    } else {
      PointsGridDownsampler3f(points, bin_size, parallel).getDownsampledPoints(res.points, min_points_in_bin);
    }
    return res;
  }
  // utilities/point_cloud.hpp:292-420: view point = origin unless the current normals serve as the
  // reference (use_current_as_ref && hasNormals())
  PointCloud3f& estimateNormalsKNN(size_t k, bool use_current_as_ref = false) {
    normal_estimator(use_current_as_ref).estimateNormalsKNN(normals, k);
    return *this;
  }
  PointCloud3f& estimateNormalsRadius(float radius, bool use_current_as_ref = false) {
    normal_estimator(use_current_as_ref).estimateNormalsRadius(normals, radius);
    return *this;
  }
  PointCloud3f& estimateNormalsKNNInRadius(size_t k, float radius, bool use_current_as_ref = false) {
    normal_estimator(use_current_as_ref).estimateNormalsKNNInRadius(normals, k, radius);
    return *this;
  }
  // overloads taking the caller's search tree (utilities/point_cloud.hpp:311-327 etc.): same result
  template <typename IndexT>
  PointCloud3f& estimateNormalsKNN(const KDTree3f<IndexT>&, size_t k, bool use_current_as_ref = false) {
    return estimateNormalsKNN(k, use_current_as_ref);
  }
  template <typename IndexT>
  PointCloud3f& estimateNormalsRadius(const KDTree3f<IndexT>&, float radius, bool use_current_as_ref = false) {
    return estimateNormalsRadius(radius, use_current_as_ref);
  }
  template <typename IndexT>
  PointCloud3f& estimateNormalsKNNInRadius(const KDTree3f<IndexT>&, size_t k, float radius,
                                           bool use_current_as_ref = false) {
    return estimateNormalsKNNInRadius(k, radius, use_current_as_ref);
  }
  NormalEstimation3f normal_estimator(bool use_current_as_ref) const {
    NormalEstimation3f ne(points);
    if (use_current_as_ref && hasNormals())
      ne.setReferenceNormals(normals);
    else
      ne.setViewPoint(Vector3f(0.f, 0.f, 0.f));
    return ne;
  }
  size_t size() const { return points.cols(); }
  bool hasNormals() const { return size() > 0 && normals.cols() == size(); }
  bool hasColors() const { return size() > 0 && colors.cols() == size(); }
  bool isEmpty() const { return size() == 0; }
  PointCloud3f& transform(const RigidTransform3f& T) {  // utilities/point_cloud.hpp (rigid overload)
    VectorSet3f out;
    transformPoints(T, points, out);
    points = out;
    if (hasNormals()) {
      RigidTransform3f R = T;
      for (int r = 0; r < 3; r++) R.translation(r) = 0.f;
      transformPoints(R, normals, out);
      normals = out;
    }
    return *this;
  }
};

}  // namespace cilantro
