/*
 * cilantro_b200 — C ABI of the B200-native (sm_100a) rigid-ICP / k-means / RANSAC / PCA hot path.
 *
 * This is the drop-in boundary (SURVEY.md §8b). cilantro itself has no FFI: its "interface" for this
 * path is a set of C++ templates over Eigen types. Each entry point below names the reference
 * function(s) it replaces (paths relative to /root/reference/include/cilantro/). The header-only C++
 * shims in include/cilantro/ re-create the reference's class names on top of these calls; see
 * INTEGRATION.md for the binding a cilantro maintainer would add.
 *
 * Conventions
 *   - Plain pointers and sizes only. Host point sets are packed xyz float32, 12 B/point — exactly the
 *     memory a ConstVectorSetMatrixMap<float,3> wraps (core/data_containers.hpp:73-112,155-156).
 *   - Rigid transforms are float32[12], row-major [R | t] (3 rows of 4).
 *   - Every function returns CB_OK (0) or a negative cb_status; cb_last_error() gives the message
 *     (thread-local). Nothing throws across this boundary.
 *   - There is NO CPU fallback: without a CUDA device cb_context_create fails with CB_ERR_NO_DEVICE.
 *     Only the cb_solve_* / cb_version helpers are host-only (they are the O(1) 3x3 / 6x6 solves the
 *     reference also runs on the host).
 *   - One cb_context per (process, device); calls on one context are serialised by the caller,
 *     like the reference's objects (not thread-safe, SURVEY.md §8b "Threading").
 */
#ifndef CILANTRO_B200_H_
#define CILANTRO_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default) /* the library is built with -fvisibility=hidden */
#endif

typedef enum cb_status {
  CB_OK = 0,
  CB_ERR_INVALID = -1,    /* bad argument */
  CB_ERR_NO_DEVICE = -2,  /* no usable CUDA device / driver */
  CB_ERR_CUDA = -3,       /* CUDA runtime error (message in cb_last_error) */
  CB_ERR_NCCL = -4,       /* NCCL missing or failed */
  CB_ERR_UNSUPPORTED = -5
} cb_status;

typedef struct cb_context cb_context;
typedef struct cb_cloud cb_cloud;
typedef struct cb_icp cb_icp;

const char* cb_last_error(void);
const char* cb_version(void);

/* ---- context -------------------------------------------------------------------------------- */
int cb_context_create(int device, cb_context** out);
void cb_context_destroy(cb_context* ctx);
int cb_context_synchronize(cb_context* ctx);
/* SM count, total HBM bytes of the context's device. */
int cb_context_device_info(cb_context* ctx, int* sm_count, size_t* hbm_bytes, char* name64);
/* Number of kernels this library has launched on the context since creation (for bench.py's
 * gpu_launches claim). */
uint64_t cb_context_kernel_launches(cb_context* ctx);
/* Evict L2 by writing a scratch buffer larger than L2 (bench hygiene; not part of any algorithm). */
int cb_context_flush_l2(cb_context* ctx);

/* Multi-GPU: one process per GPU. Rank 0 calls cb_comm_unique_id, the 128 bytes are broadcast by
 * the launcher's own channel (torch.distributed in bench.py), every rank calls cb_context_init_comm.
 * Afterwards ICP / k-means / PCA objects created from shards on this context reduce their normal
 * equations / centroid sums across ranks with ONE ncclAllReduce per iteration (SURVEY.md §8e).
 * The reference has no counterpart (single process, OpenMP reductions:
 * core/openmp_reductions.hpp:3-33, registration/transform_estimation.hpp:285-290). */
int cb_comm_unique_id(void* out_128_bytes);
int cb_context_init_comm(cb_context* ctx, const void* unique_id_128_bytes, int rank, int world);
int cb_context_comm_info(cb_context* ctx, int* rank, int* world);
/* Optional, after cb_context_init_comm: the FUSED exchange. Every rank exports a 64-byte CUDA-IPC
 * handle of its exchange table (cb_comm_ipc_handle), the launcher all-gathers them in rank order
 * (world x 64 bytes) and every rank maps its peers' tables (cb_comm_ipc_attach), then barriers.
 * From then on the ICP accumulation kernel itself all-reduces the 16/28 moments by writing them
 * straight into the peers' tables over NVLink and publishes the total to a mapped host mailbox, so an
 * iteration costs one kernel + one host poll: no ncclAllReduce, cudaMemcpy or stream synchronise.
 * If mapping fails (no peer access) the call returns an error and the NCCL path stays active. */
int cb_comm_ipc_handle(cb_context* ctx, void* out_64_bytes);
int cb_comm_ipc_attach(cb_context* ctx, const void* handles_world_x_64_bytes);
/* Back to the NCCL reduction on this rank. The launcher calls it on EVERY rank when cb_comm_ipc_attach failed
 * on any of them (the ranks must agree on the path before the first pass). */
int cb_comm_ipc_detach(cb_context* ctx);

/* ---- device-resident point sets --------------------------------------------------------------
 * Replaces: PointFeaturesAdaptor<float,3> ctor (correspondence_search/
 * common_transformable_feature_adaptors.hpp:14-17) for query sets, and the KDTree<float,3> ctor
 * (core/kd_tree.hpp:162-170 -> nanoflann buildIndex) for reference sets: the points are uploaded
 * once, binned into a uniform grid (cell-sorted float4 copy + cell-start table) and stay in HBM.
 * normals may be NULL. index_offset is added to this set's point indices in every result
 * (a rank's shard offset; 0 on a single GPU). */
int cb_cloud_create(cb_context* ctx, const float* xyz, const float* normals, size_t n, uint64_t index_offset,
                    cb_cloud** out);
/* Two clouds in one call — what the constructors of the ICP classes receive (icp_common_instances.hpp:34-44:
 * dst points [+ normals], src points [+ normals]). Same result as two cb_cloud_create calls followed by the lazy
 * index builds, but the upload of the second cloud runs on a second stream while the grid of the first is being
 * built (effective with pinned host buffers). Both clouds are indexed on return. */
int cb_cloud_create_pair(cb_context* ctx, const float* xyz_a, const float* normals_a, size_t n_a, uint64_t offset_a,
                         const float* xyz_b, const float* normals_b, size_t n_b, uint64_t offset_b, cb_cloud** out_a,
                         cb_cloud** out_b);
/* Same, from packed xyz already in device memory (used when inputs are HBM-resident). */
int cb_cloud_create_from_device(cb_context* ctx, const float* d_xyz, const float* d_normals, size_t n,
                                uint64_t index_offset, cb_cloud** out);

/* Multi-rank: a cloud EVERY rank needs in full (the replicated destination cloud of a sharded ICP —
 * SURVEY 8e) built from its contiguous blocks: each rank uploads only block [first_index, first_index + n_block) of the
 * n_total points over its own PCIe link, the blocks are exchanged over NVLink (NCCL) and every rank ends up with the
 * same cloud as cb_cloud_create(whole array) would give it, bit for bit. Collective over the context's communicator
 * (cb_context_init_comm); with world == 1 it is cb_cloud_create. Normals: present on all ranks or on none. */
int cb_cloud_create_replicated(cb_context* ctx, const float* xyz_block, const float* normals_block, size_t n_block,
                               uint64_t first_index, size_t n_total, cb_cloud** out);
void cb_cloud_destroy(cb_cloud* c);
size_t cb_cloud_size(const cb_cloud* c);
/* Grid facts for DESIGN/bench reporting: cell edge, dims[3], occupied-cell mean occupancy. */
int cb_cloud_grid_info(const cb_cloud* c, float* cell_edge, int* dims3, double* mean_occupancy);

/* ---- nearest neighbour ------------------------------------------------------------------------
 * cb_knn1_radius replaces the batched KDTree::kNNInRadiusSearch(q, k=1, r2) sweep of
 * findNNCorrespondencesUnidirectional (correspondence_search/
 * correspondence_search_kd_tree_utilities.hpp:26-33 -> core/kd_tree.hpp:284-291) with the query
 * transform of PointFeaturesAdaptor::transformFeatures fused in (T may be NULL = identity).
 * For query i (original order): idx[i] = index of the nearest ref point with d2 < max_d2 (lowest
 * index on exact ties), or -1; d2[i] = its squared distance, or max_d2.
 * max_d2 = FLT_MAX gives KDTree::nearestNeighborSearch (core/kd_tree.hpp:181-204). */
int cb_knn1_radius(cb_context* ctx, const cb_cloud* ref, const cb_cloud* qry, const float* T12, float max_d2,
                   int64_t* idx, float* d2);
/* General k (1..256; CB_ERR_UNSUPPORTED above): KDTree::kNNInRadiusSearch / kNNSearch batched (core/kd_tree.hpp:215-318).
 * idx/d2 are n_qry x k, ascending d2, unused slots idx = -1. counts (may be NULL) = found per query. */
int cb_knn_radius(cb_context* ctx, const cb_cloud* ref, const cb_cloud* qry, const float* T12, int k,
                  float max_d2, int64_t* idx, float* d2, uint32_t* counts);
/* KDTree::radiusSearch batched (core/kd_tree.hpp:250-278): for query i, every ref point with d2 < radius2,
 * ascending d2 (equal distances: ascending index; the reference leaves them to std::sort), as a CSR list:
 * entries offsets[i] .. offsets[i+1]-1 of idx / d2; offsets has n_qry + 1 entries. *total = offsets[n_qry].
 * Sizing: call with idx = d2 = NULL (or a too small capacity) -> offsets and *total are filled, nothing else
 * is written; call again with buffers of capacity >= *total. */
int cb_radius_search(cb_context* ctx, const cb_cloud* ref, const cb_cloud* qry, const float* T12, float radius2,
                     uint64_t* offsets, int64_t* idx, float* d2, size_t capacity, size_t* total);
/* ---- normal / curvature estimation -------------------------------------------------------------
 * Replaces NormalEstimation::estimateNormalsAndCurvature{KNN,Radius,KNNInRadius} (core/
 * normal_estimation.hpp:83-232 -> compute_normals_curvature_* :357-421) as called by
 * PointCloud::estimateNormals* (utilities/point_cloud.hpp:294-420). Neighbourhood of every point over
 * the cloud itself:  k > 0, radius2 <= 0 : kNN;  k > 0, radius2 > 0 : kNN within squared radius;
 * k == 0, radius2 > 0 : all points with d2 < radius2 (cilantro radii are squared distances).
 * Fewer than 3 neighbours -> NaN. view_point3 (may be NULL or non-finite = no orientation step) flips
 * each normal towards the view point (:325-329); use_current_as_ref != 0 on a cloud that has normals
 * orients by those instead (setReferenceNormals, :63-69, :351-355; takes precedence, :281-291). The normals are stored in the cloud on the device (as
 * PointCloud::normals is filled), so a combined-metric ICP can follow without a host round trip.
 * Host outputs (each may be NULL): normals 3n, curvature n, cov6 6n (xx,xy,xz,yy,yz,zz of the
 * neighbourhood covariance, diagnostic). gpu_ms (may be NULL) = device time of the kernel. k <= 128
 * (the k-best lists live in shared memory; CB_ERR_UNSUPPORTED above). */
int cb_cloud_estimate_normals(cb_context* ctx, cb_cloud* cloud, int k, float radius2, const float* view_point3,
                              int use_current_as_ref, float* normals, float* curvature, float* cov6, float* gpu_ms);
/* ---- voxel-grid downsampling -------------------------------------------------------------------
 * Replaces PointCloud::gridDownsample / gridDownsampled (utilities/point_cloud.hpp:246-290) =
 * Points[Normals][Colors]GridDownsampler (core/grid_downsampler.hpp) over GridAccumulator::build_index_
 * (core/grid_accumulator.hpp:146-199): bin = floor(p * (1 / bin_size)) per axis; per bin the point sum,
 * the sign-consistent normal sum (core/common_accumulators.hpp:122-131) and the colour sum are taken
 * in point-index order in fp32 (the serial build's arithmetic, bit for bit) and divided by the count;
 * normals are re-normalised; bins with fewer than min_points_in_bin points are dropped.
 * order = 0: bins ascending lexicographically in (x, y, z) — the std::map order the default
 *            (parallel = true) build emits (:177-181);
 * order = 1: bins in order of their first point — the serial (parallel = false) build (:194-197).
 * normals / colors (packed 3 floats per point) may be NULL; outputs are sized for n points, *out_n is
 * the number of occupied bins written. */
int cb_grid_downsample(cb_context* ctx, const float* xyz, const float* normals, const float* colors, size_t n,
                       float bin_size, size_t min_points_in_bin, int order, float* out_xyz, float* out_normals,
                       float* out_colors, size_t* out_n);
/* Same on a device-resident cloud (points + normals if it has them); the result is a new cloud that never
 * leaves HBM (downsample -> cb_cloud_estimate_normals -> cb_icp_* without host round trips). gpu_ms may be
 * NULL. */
int cb_cloud_grid_downsample(cb_context* ctx, const cb_cloud* cloud, float bin_size, size_t min_points_in_bin,
                             int order, cb_cloud** out, float* gpu_ms);
/* Copies a cloud's points (and normals, if normals != NULL and the cloud has them) back to the host in
 * original order. */
int cb_cloud_download(cb_context* ctx, const cb_cloud* cloud, float* xyz, float* normals);
/* findNNCorrespondencesUnidirectional(ref_is_first = true), compacted in query order:
 * (index_first[c], index_second[c], value[c]) = (ref idx, query idx, d2). Arrays sized n_qry. */
int cb_find_correspondences(cb_context* ctx, const cb_cloud* ref, const cb_cloud* qry, const float* T12,
                            float max_d2, uint64_t* index_first, uint64_t* index_second, float* value,
                            size_t* count);

/* ---- rigid ICP -------------------------------------------------------------------------------
 * cb_icp_* replaces SimplePointToPointMetricRigidICP3f / SimpleCombinedMetricRigidICP3f
 * (registration/icp_common_instances.hpp:34-97,250,261): IterativeClosestPointBase::estimate()
 * (registration/icp_base.hpp:68-87) with, per iteration, ONE fused kernel doing
 *   transformFeatures (common_transformable_feature_adaptors.hpp:28-34)
 * + the radius-bounded 1-NN sweep (correspondence_search_kd_tree_utilities.hpp:26-33)
 * + transformPoints (core/space_transformations.hpp:203-216)
 * + the normal-equation / Kabsch-moment accumulation
 *   (registration/transform_estimation.hpp:25-34, :298-343, :669-715),
 * then one small all-reduce when a communicator is attached, then the host-side solve
 * (transform_estimation.hpp:36-45, :346-357; core/space_transformations.hpp:43-51). */
typedef enum cb_icp_metric {
  CB_ICP_POINT_TO_POINT = 0, /* PointToPointMetricSingleTransformICP (Kabsch per iteration) */
  CB_ICP_COMBINED = 1        /* CombinedMetricSingleTransformICP; symmetric if src has normals */
} cb_icp_metric;

typedef struct cb_icp_params {
  int32_t metric;
  int32_t max_iter;     /* icp_base.hpp:24, default 15 */
  float tol;            /* icp_base.hpp:25, default 1e-5 */
  float max_d2;         /* SQUARED; correspondence_search_kd_tree.hpp:49, default 0.01*0.01 */
  float w_pt;           /* icp_single_transform_combined_metric.hpp:46, default 0 */
  float w_pl;           /* :47, default 1 */
  int32_t max_opt_iter; /* :44, default 1 */
  float opt_tol;        /* :45, default 1e-5 */
  float T_init[12];     /* icp_base.hpp:58-61 */
  int32_t flush_l2;     /* bench hygiene: evict L2 before every iteration (outside the timed events) */
  int32_t timing;       /* CUDA-event instrumentation of estimate(): 0 none (production), 1 one bracket per
                           iteration (kernel + exchange + host solve) -> gpu_ms_total / cb_icp_iteration_times,
                           2 one bracket per search kernel -> gpu_ms_search. Each cudaEventRecord costs a few us of
                           device front-end time, comparable to the ~100 us iteration, hence one mode at a time. */
  /* Correspondence-engine options (correspondence_search_kd_tree.hpp:46-50, :60-98 setters). The defaults
   * (SECOND_TO_FIRST, fraction 1, no reciprocity, not one-to-one) take the fused single-kernel path; any other
   * setting materialises the correspondence list on the device (search(es) -> union / intersection -> fraction
   * filter -> one-to-one filter, core/correspondence.hpp:57-100) and accumulates over it. With several ranks every rank runs
   * them on the whole source cloud (shards all-gathered once; create the shards with index_offset = their first global index):
   * same lists and transforms as one GPU, on every rank. */
  int32_t search_dir;          /* cb_search_dir; default CB_SECOND_TO_FIRST */
  int32_t require_reciprocal;  /* with CB_BOTH: intersection instead of union (:68-70 of ..._utilities.hpp) */
  int32_t one_to_one;          /* keep, per dst (SECOND_TO_FIRST) / src (FIRST_TO_SECOND) point, the closest pair */
  int32_t host_loop;           /* 0 (default): iterations run back to back on the device where the configuration allows it
                                  (default engine, one Gauss-Newton step per iteration); 1: host-driven loop (A/B, tests) */
  double inlier_fraction;      /* keep the llround(fraction * M) closest pairs when 0 < fraction < 1; default 1 */
  /* Correspondence weight evaluators of the combined / symmetric metric (the PointToPointCorrWeightEvaluatorT /
   * PointToPlaneCorrWeightEvaluatorT template arguments of CombinedMetricSingleTransformICP, consumed at
   * registration/transform_estimation.hpp:302-304 and :331-333): weight = metric weight * evaluator(i, j, d2).
   * Arbitrary functors cannot cross a C ABI; the two evaluators of core/common_pair_evaluators.hpp that make sense
   * here are selected by kind: CB_WEIGHT_UNITY (UnityWeightEvaluator, :29-43, the default) and CB_WEIGHT_RBF
   * (RBFKernelWeightEvaluator<float, float, true>, :46-79: exp(coeff * d2) with coeff = -0.5f / (sigma * sigma),
   * d2 = the correspondence's squared distance). */
  int32_t pt_weight_kind;
  int32_t pl_weight_kind;
  float pt_weight_coeff;
  float pl_weight_coeff;
} cb_icp_params;

typedef enum cb_weight_kind { CB_WEIGHT_UNITY = 0, CB_WEIGHT_RBF = 1 } cb_weight_kind;

typedef enum cb_search_dir {
  CB_SECOND_TO_FIRST = 0, /* queries = transformed src, tree = dst (the default) */
  CB_FIRST_TO_SECOND = 1, /* queries = dst, tree = transformed src (rebuilt every iteration) */
  CB_BOTH = 2
} cb_search_dir;

typedef struct cb_icp_result {
  float T[12];
  int32_t iterations;
  float last_delta;
  int32_t converged;
  uint64_t num_corr;    /* correspondences of the last iteration (global across ranks) */
  double gpu_ms_total;  /* sum over iterations of the CUDA-event time of the iteration's kernels */
  double gpu_ms_search; /* ... of which the fused search+accumulate kernel */
  uint64_t kernel_launches;
} cb_icp_result;

void cb_icp_default_params(cb_icp_params* p);
/* dst must carry normals for CB_ICP_COMBINED. Both clouds must outlive the icp object. */
int cb_icp_create(cb_context* ctx, const cb_cloud* dst, const cb_cloud* src, cb_icp** out);
void cb_icp_destroy(cb_icp* icp);
int cb_icp_estimate(cb_icp* icp, const cb_icp_params* prm, cb_icp_result* res);
/* Per-iteration device times of the last estimate() (ms); n = min(cap, iterations). */
int cb_icp_iteration_times(cb_icp* icp, double* ms, int cap);
/* getCorrespondences() of the engine after the last iteration (this rank's shard). Arrays hold n_src entries
 * (n_src + n_dst when search_dir == CB_BOTH). Default mode: ascending source index; other engine modes: the
 * order the reference's filters leave (ascending value after the fraction filter, ascending dst / src index
 * after the one-to-one filter, lexicographic (first, second) for CB_BOTH). */
int cb_icp_correspondences(cb_icp* icp, uint64_t* index_first, uint64_t* index_second, float* value,
                           size_t* count);
/* computeResiduals() — icp_single_transform_combined_metric.hpp:220-243 /
 * icp_single_transform_point_to_point_metric.hpp:68-85. out has n_src floats (this rank's shard). */
int cb_icp_residuals(cb_icp* icp, const cb_icp_params* prm, const float* T12, float* out);

/* One fused search+accumulate pass WITHOUT the solve: returns the reduced moments.
 * p2p: sums[16] = {n, sum d (3), sum q (3), sum d q^T (9, row-major)}
 * combined: sums[28] = {n, AtA upper triangle row-major (21), Atb (6)}. Used by the parity tests
 * and by callers that do their own reduction. */
int cb_icp_accumulate(cb_icp* icp, const cb_icp_params* prm, const float* T12, double* sums, int cap);

/* Inspection of the device-resident loop's per-query cache after cb_icp_estimate took that path (parity tests):
 * T_search12 = the transform the LAST executed iteration searched with; nearest[i] = original index of the
 * destination point the loop holds as source point i's nearest neighbour under that transform (whether or not it
 * is inside the radius), -1 = none known; searched_last = queries the last iteration had to search again.
 * Returns CB_ERR_INVALID when the last estimate() did not run on the device loop. */
int cb_icp_loop_cache(cb_icp* icp, float* T_search12, int64_t* nearest, uint64_t* searched_last);

/* Host-only O(1) solves (no device needed; exported so the N>1 logic is testable on CPU). */
/* estimateTransformPointToPointMetric from moments — transform_estimation.hpp:25-47. Returns 1 if n>=3. */
int cb_solve_kabsch_moments(const double* sums16, float* T12);
/* One Gauss-Newton update of estimateTransformCombinedMetric — :346-357: T_out = Ra ta Ra T_in. */
int cb_solve_gauss_newton(const double* sums28, const float* T_in12, float* T_out12, float* dtheta_norm);
/* LinearTransform::rotation() — core/space_transformations.hpp:43-51 (3x3 row-major in/out). */
int cb_solve_rotation(const float* L9, float* R9);
/* tform_iter * transform_ and the update norm — icp_single_transform_combined_metric.hpp:213-216. */
int cb_compose(const float* A12, const float* B12, float* out12);

/* ---- k-means ---------------------------------------------------------------------------------
 * Replaces KMeans<float,3>::cluster(centroids, max_iter, tol, use_kd_tree=false)
 * (clustering/kmeans.hpp:24-30,67-194): fused brute-force assignment (:100-119) + per-cluster
 * sums (:126-131) in one kernel, one all-reduce of K x 4 sums when a communicator is attached,
 * empty-cluster repair (:134-176) and the division (:179-181) on the host.
 * centroids: in = initial (K x 3), out = final. labels (may be NULL): n uint64, ORIGINAL order. */
typedef struct cb_kmeans_result {
  uint64_t iterations;
  double gpu_ms_total;
  uint64_t kernel_launches;
} cb_kmeans_result;
int cb_kmeans_cluster(cb_context* ctx, const cb_cloud* pts, float* centroids, size_t k, size_t max_iter,
                      float tol, uint64_t* labels, cb_kmeans_result* res);
/* One assignment sweep against given centroids (kmeans.hpp:100-119); labels n uint64. Also returns
 * the per-cluster sums (K x 3 doubles) and counts (K uint64) when non-NULL. */
int cb_kmeans_assign(cb_context* ctx, const cb_cloud* pts, const float* centroids, size_t k, uint64_t* labels,
                     double* sums, uint64_t* counts);
/* KMeans::cluster(num_clusters,...) seeding (kmeans.hpp:32-49) with an injected seed. */
int cb_kmeans_seed_indices(size_t n, size_t k, uint32_t seed, uint64_t* out_idx);

/* ---- RANSAC ----------------------------------------------------------------------------------
 * Replaces TransformRANSACEstimator<RigidTransform3f>::computeResiduals + the inlier scan of
 * RandomSampleConsensusBase::estimate (model_estimation/ransac_transform_estimator.hpp:90-98,
 * model_estimation/ransac_base.hpp:96-101): inlier COUNTS of H hypotheses over n pairs.
 * dst/src are paired clouds of equal size (pair i = point with original index i in both). */
int cb_ransac_score(cb_context* ctx, const cb_cloud* dst, const cb_cloud* src, const float* T_h, size_t H,
                    float thresh, uint32_t* counts);
/* Residuals of one model (computeResiduals) into out[n], and inlier indices (<= thresh). */
int cb_ransac_residuals(cb_context* ctx, const cb_cloud* dst, const cb_cloud* src, const float* T12,
                        float thresh, float* residuals, uint64_t* inliers, size_t* num_inliers);
typedef struct cb_ransac_result {
  float T[12];
  uint64_t iterations;
  uint64_t num_inliers;
  uint64_t best_iteration;
  double gpu_ms_total;
  uint64_t kernel_launches;
} cb_ransac_result;
/* RandomSampleConsensusBase::estimate() for rigid transforms (ransac_base.hpp:64-131) with the seed
 * injected in place of std::random_device (:73). Hypotheses are generated on the host in the
 * reference's order, scored on the device in batches, and scanned in order so that the kept model,
 * the early exit (:114) and the iteration count are those of the sequential loop. */
int cb_ransac_rigid(cb_context* ctx, const cb_cloud* dst, const cb_cloud* src, uint32_t seed,
                    size_t inlier_count_thresh, size_t max_iter, float thresh, int re_estimate,
                    cb_ransac_result* res, uint64_t* inliers, float* residuals);

/* ---- covariance / PCA ------------------------------------------------------------------------
 * Replaces Covariance<float,3>::operator() (core/covariance.hpp:31-80) and
 * PrincipalComponentAnalysis<float,3> (core/principal_component_analysis.hpp:76-84).
 * cov / evecs row-major 3x3, eigenvalues descending, evecs right-handed. Returns 1 if n >= 2,
 * else fills NaN and returns 0 (covariance.hpp:35-38). */
int cb_mean_cov(cb_context* ctx, const cb_cloud* pts, float* mean3, float* cov9);
int cb_pca(cb_context* ctx, const cb_cloud* pts, float* mean3, float* cov9, float* evals3, float* evecs9);

/* ---- connected-component segmentation -----------------------------------------------------------
 * Replaces ConnectedComponentExtraction<float,3>::segment (clustering/connected_component_extraction.hpp:371-428) =
 * extractConnectedComponents(tree, nh, seeds, ...) (:162-265; the overloads without seeds forward with every point as a
 * seed) over the proximity evaluators of core/common_pair_evaluators.hpp:88-259, and getPointToClusterIndexMap
 * (clustering/clustering_base.hpp:8-18).
 * Neighbourhood of every point over the cloud itself, encoded as for cb_cloud_estimate_normals: k > 0, radius2 <= 0:
 * kNN; k > 0, radius2 > 0: kNN within radius2; k == 0, radius2 > 0: every point with d2 < radius2; k == 0, radius2 <= 0:
 * empty (every seed is a segment of its own). u -> v is an edge when v is entry j >= 1 of u's list (ascending (d2, index),
 * the reference skips entry 0, :202) and the evaluator accepts (u, v, d2). Segments are the connected components of the
 * undirected graph over the points reachable from the seeds along edges, seeds included.
 * Output: segments of min_size <= size <= max_size, by size descending, equal sizes by smallest point index ascending;
 * labels[i] = segment of point i, or *num_segments for a point in none (n entries); the points of segment s are
 * seg_points[seg_offsets[s] .. seg_offsets[s+1]) ascending (seg_offsets has n + 1 entries, seg_points n). Point indices
 * are positions in this cloud (index_offset is not added). The result does not depend on scheduling.
 * seeds: NULL = every point (n_seeds ignored); repeated seeds are allowed, a seed >= n is CB_ERR_INVALID. normals: packed
 * 3n floats in original order, NULL = the cloud's own normals (CB_ERR_INVALID for a normals evaluator when it has none);
 * colors: packed 3n floats, required by the colour evaluators. gpu_ms (may be NULL) receives 3 floats: the device time
 * of the call, of its neighbourhood + union stage and of its finalise stage (relabelling and the segment lists). */
typedef enum cb_segment_evaluator {
  CB_SEG_ALWAYS_TRUE = 0,            /* AlwaysTrueEvaluator (the default) */
  CB_SEG_POINTS = 1,                 /* PointsProximityEvaluator: d2 < max_distance */
  CB_SEG_NORMALS = 2,                /* NormalsProximityEvaluator: angle <= max_angle */
  CB_SEG_COLORS = 3,                 /* ColorsProximityEvaluator: |dc|^2 < color_thresh^2 */
  CB_SEG_POINTS_NORMALS = 4,         /* PointsNormalsProximityEvaluator (angle < max_angle) */
  CB_SEG_POINTS_COLORS = 5,          /* PointsColorsProximityEvaluator */
  CB_SEG_NORMALS_COLORS = 6,         /* NormalsColorsProximityEvaluator (angle < max_angle) */
  CB_SEG_POINTS_NORMALS_COLORS = 7   /* PointsNormalsColorsProximityEvaluator (angle < max_angle) */
} cb_segment_evaluator;

typedef struct cb_segment_params {
  int32_t k;             /* neighbourhood (see above), k <= 256 (CB_ERR_UNSUPPORTED above) */
  float radius2;
  int32_t evaluator;     /* cb_segment_evaluator */
  float max_distance;    /* squared, compared with the list's d2 */
  float max_angle;       /* radians; negative = unoriented normals: min(angle, pi - angle) <= -max_angle */
  float color_thresh;    /* not squared (the evaluators square it) */
  uint64_t min_size;     /* :165, default 1 */
  uint64_t max_size;     /* :165, default SIZE_MAX */
} cb_segment_params;

int cb_cloud_segment(cb_context* ctx, cb_cloud* cloud, const cb_segment_params* prm, const uint64_t* seeds,
                     size_t n_seeds, const float* normals, const float* colors, uint64_t* labels,
                     uint64_t* seg_offsets, uint64_t* seg_points, size_t* num_segments, float* gpu_ms);

/* transformPoints(tform, in, out) — core/space_transformations.hpp:203-216 (host in, host out). */
int cb_transform_points(cb_context* ctx, const float* T12, const float* xyz, size_t n, float* out);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* CILANTRO_B200_H_ */
