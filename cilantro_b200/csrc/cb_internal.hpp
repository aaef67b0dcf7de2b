// Internal declarations shared by the translation units of libcilantro_b200.so.
// Product code: never includes or links anything from oracle/.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstddef>
#include <cstdio>
#include <cstdarg>
#include <vector>
#include "../../include/cilantro_b200.h"

namespace cb {

void set_error(const char* fmt, ...);

#define CB_CUDA(call)                                                                          \
  do {                                                                                         \
    cudaError_t e__ = (call);                                                                  \
    if (e__ != cudaSuccess) {                                                                  \
      cb::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__));     \
      return CB_ERR_CUDA;                                                                      \
    }                                                                                          \
  } while (0)

#define CB_CHECK(cond, status, msg)                                        \
  do {                                                                     \
    if (!(cond)) {                                                         \
      cb::set_error("%s:%d: %s", __FILE__, __LINE__, msg);                 \
      return status;                                                       \
    }                                                                      \
  } while (0)

#define CB_TRY(expr)            \
  do {                          \
    int s__ = (expr);           \
    if (s__ != CB_OK) return s__; \
  } while (0)

// Uniform grid over a cloud. Points are stored cell-sorted as float4 (x, y, z, original index bits);
// cells are x-major: id = (z * ny + y) * nx + x, so the three x-neighbours of a row are one
// contiguous range of the sorted array.
constexpr int kReduceBlock = 256;  // every kernel using grid_reduce (reduce.cuh) launches with this block size
constexpr int kReduceGroup = 64;   // blocks per first-level reduction group

constexpr int kMaxRanks = 16;      // ranks of one NVLink domain that can take part in the fused exchange
constexpr int kExchangeVals = 32;  // doubles per exchanged row (>= the largest reduced vector, 28)

// Fused epilogue of the ICP reduction (reduce.cuh, grid_reduce_async): the warp that finishes the
// grid reduction (a) all-reduces the result row with its peers by writing it straight into every
// rank's exchange table over NVLink (CUDA-IPC mapped peer memory) and summing the rows it received in
// rank order, and (b) publishes the total to mapped pinned host memory and raises a host-visible flag.
// This replaces ncclAllReduce + cudaMemcpyAsync + cudaStreamSynchronize per iteration (measured
// ~85 us at 2 GPUs) by one NVLink round trip and a host poll. enabled = 0 keeps the plain path.
struct Exchange {
  int enabled;
  int rank, world;
  unsigned long long seq;                  // pass number (> 0, +1 per pass, identical on all ranks)
  double* const* peer_vals;                // device array [world]: rank p's value table [2][world][32]
  unsigned long long* const* peer_flags;   // device array [world]: rank p's flag table  [2][world]
  double* host_vals;                       // mapped pinned [32]
  unsigned long long* host_flag;           // mapped pinned
  unsigned long long* trace;               // optional (CB_TRACE_EXCHANGE): 4 x %globaltimer stamps per pass
  unsigned long long timeout_ns;           // bound of the in-kernel wait for the peers' rows (0 = unbounded)
};

// Device scratch of the two-level grid reduction (reduce.cuh), owned by the context.
struct ReduceScratch {
  double* partials;        // [gridDim.x][NV]   one row per block
  double* gpartials;       // [ngroups][NV]     one row per group of kReduceGroup blocks
  unsigned int* counters;  // [ngroups + 1]     tickets; zero on entry, reset by their last user
  double* result;          // [NV]
  Exchange ex;             // fused exchange / host notification (grid_reduce_async only)
};

struct GridView {
  const float4* pts;           // n, cell-sorted; .w = __int_as_float(original index)
  const float4* nrm;           // n, same order (or nullptr)
  const uint32_t* cell_start;  // ncells + 1
  float ox, oy, oz;            // grid origin (bbox min)
  float inv_h;                 // 1 / cell edge
  float h_safe;                // cell edge * (1 - 2^-10): conservative edge for lower bounds
  int nx, ny, nz;
  uint32_t n;
  // Non-empty coarse blocks (kBlockCells^3 cells each): x = X, y = Y, z = Z block coordinates, w = number
  // of points. Only the far-query path (far_sweep.cuh) reads them: queries that would have to cross a lot of
  // empty space shell by shell iterate this list instead.
  const uint4* blocks;
  uint32_t nblocks;
};

constexpr int kBlockCells = 8;  // coarse block edge in cells

}  // namespace cb

struct cb_context {
  int device = 0;
  cudaStream_t stream = nullptr;
  int sm_count = 0;
  size_t l2_bytes = 0;
  size_t hbm_bytes = 0;
  char name[64] = {0};
  uint64_t launches = 0;
  // reduction scratch: per-block partials -> last block -> result
  double* d_partials = nullptr;
  size_t partials_cap = 0;  // in doubles
  unsigned int* d_counter = nullptr;  // ticket counters of the grid reduction (zero between launches)
  size_t counter_cap = 0;
  double* d_result = nullptr;  // 64 doubles
  double* h_result = nullptr;  // pinned, 64 doubles
  void* d_flush = nullptr;
  size_t flush_bytes = 0;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr;
  cudaStream_t copy_stream = nullptr;  // second stream: uploads overlapped with index builds (cb_cloud_create_pair)
  // NCCL (loaded lazily with dlopen; see nccl_dyn.cpp)
  void* nccl_comm = nullptr;
  int rank = 0, world = 1;
  // fused exchange (struct Exchange): one cudaMalloc'ed region [flags 2 x kMaxRanks u64 | values
  // 2 x kMaxRanks x 32 f64] exported to the peers with CUDA IPC, and a mapped pinned host mailbox
  void* d_xchg = nullptr;                 // this rank's region
  void* peer_xchg[cb::kMaxRanks] = {nullptr};  // every rank's region as seen from this device (self included)
  double** d_peer_vals = nullptr;         // device copies of the two pointer tables
  unsigned long long** d_peer_flags = nullptr;
  unsigned long long* h_sync = nullptr;   // mapped pinned: [0] = flag, [8..8+32) = values (as doubles)
  unsigned long long seq = 0;             // passes issued with the exchange enabled
  bool ex_ready = false;                  // tables valid for the current (rank, world)
  bool ex_attached = false;               // cb_comm_ipc_attach has mapped the peers' tables (once per context)
  bool pass_armed = false;                // the last reduction pass carried the fused exchange
};

constexpr size_t kXchgFlagBytes = 2 * cb::kMaxRanks * sizeof(unsigned long long);
constexpr size_t kXchgBytes = kXchgFlagBytes + 2 * cb::kMaxRanks * cb::kExchangeVals * sizeof(double);

struct cb_cloud {
  cb_context* ctx = nullptr;
  size_t n = 0;
  uint64_t index_offset = 0;
  float* d_raw = nullptr;      // 3n packed xyz, original order
  float* d_raw_nrm = nullptr;  // 3n packed normals or nullptr
  // grid index (built lazily by cb::ensure_index)
  bool indexed = false;
  float4* d_pts = nullptr;
  float4* d_nrm = nullptr;
  uint32_t* d_cell_start = nullptr;
  uint4* d_blocks = nullptr;  // non-empty coarse blocks (GridView::blocks)
  uint32_t nblocks = 0;
  float ox = 0, oy = 0, oz = 0, h = 1, inv_h = 1;
  int nx = 1, ny = 1, nz = 1;
  double mean_occ = 0;
};

namespace cb {

int ensure_index(cb_cloud* c);
// Finite-coordinate bounding box of n packed xyz points in device memory (synchronises the stream).
int points_bbox(cb_context* ctx, const float* d_raw, size_t n, float mn[3], float mx[3]);
// d_data has n + 1 entries; on return d_data[i] = sum_{j<i} in[j], d_data[n] = total (grid_index.cu).
int exclusive_scan_u32(cb_context* ctx, uint32_t* d_data, size_t n, uint32_t total);
// Stable LSD radix sort of (key, value) pairs on the low `bits` bits of the keys (radix_sort.cu). The
// result is left in d_keys / d_vals; d_keys_tmp / d_vals_tmp are same-sized scratch.
int radix_sort_pairs_u64(cb_context* ctx, uint64_t* d_keys, uint32_t* d_vals, uint64_t* d_keys_tmp,
                         uint32_t* d_vals_tmp, size_t n, int bits);
GridView grid_view(const cb_cloud* c);
// k-best lists of a cloud against itself, n x k in original order (knn_k.cu; used by segment.cu).
int knn_lists_self(cb_context* ctx, const cb_cloud* c, int k, float max_d2, int* d_idx, float* d_d2, uint32_t* d_cnt);
// Scratch for a grid_reduce over `blocks` blocks of `nv` values each (grown on demand).
int get_reduce_scratch(cb_context* ctx, int blocks, int nv, ReduceScratch* out);
// Arms the fused exchange for the next pass (bumps ctx->seq) when the tables are ready; returns
// whether it did. wait_exchange() then blocks the host until that pass published its totals.
bool arm_exchange(cb_context* ctx, Exchange* ex);
bool exchange_available(const cb_context* ctx);  // fused exchange usable (tables mapped, not switched off)
int wait_exchange(cb_context* ctx, int count, double* out);

// Scoped stream-ordered scratch: everything alloc()ed is cudaFreeAsync()ed on the context's stream when the
// object goes out of scope, unless release()d to the caller.
struct DeviceScope {
  cb_context* ctx;
  std::vector<void*> ptrs;
  explicit DeviceScope(cb_context* c) : ctx(c) {}
  DeviceScope(const DeviceScope&) = delete;
  DeviceScope& operator=(const DeviceScope&) = delete;
  template <class T>
  int alloc(T** p, size_t count) {
    *p = nullptr;
    CB_CUDA(cudaMallocAsync((void**)p, (count ? count : 1) * sizeof(T), ctx->stream));
    ptrs.push_back(*p);
    return CB_OK;
  }
  void release(void* p) {
    for (size_t i = 0; i < ptrs.size(); i++)
      if (ptrs[i] == p) {
        ptrs.erase(ptrs.begin() + (long)i);
        return;
      }
  }
  ~DeviceScope() {
    for (void* p : ptrs) cudaFreeAsync(p, ctx->stream);
  }
};

// A pair of CUDA events that is destroyed on every exit path.
struct ScopedEvents {
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  ScopedEvents() = default;
  ScopedEvents(const ScopedEvents&) = delete;
  ScopedEvents& operator=(const ScopedEvents&) = delete;
  int create() {
    CB_CUDA(cudaEventCreate(&e0));
    CB_CUDA(cudaEventCreate(&e1));
    return CB_OK;
  }
  ~ScopedEvents() {
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
  }
};

// Correspondence list of the non-default engine modes (icp_engine.cu): device arrays of `count` pairs in
// the reference's list order, ORIGINAL indices (first = dst point, second = src point).
struct EnginePairs {
  uint32_t* first = nullptr;
  uint32_t* second = nullptr;
  float* d2 = nullptr;
  uint32_t count = 0;
};
inline bool engine_mode(const cb_icp_params* p) {
  return p->search_dir != CB_SECOND_TO_FIRST || p->one_to_one != 0 ||
         (p->inlier_fraction > 0.0 && p->inlier_fraction < 1.0);
}
// findCorrespondences(tform) of CorrespondenceSearchKDTree (correspondence_search_kd_tree.hpp:107-229) for
// the current estimate T: searches, union / intersection, fraction and one-to-one filters. Replaces *pairs.
int engine_find_pairs(cb_context* ctx, const cb_cloud* dst, const cb_cloud* src, const cb_icp_params* prm,
                      const float* T12, EnginePairs* pairs);
void engine_release_pairs(cb_context* ctx, EnginePairs* pairs);

// nccl_dyn.cpp
int nccl_unique_id(void* out128);
int nccl_init(cb_context* ctx, const void* id128, int rank, int world);
int nccl_allreduce_sum_f64(cb_context* ctx, double* d_buf, size_t count);
int nccl_allreduce_sum_u32(cb_context* ctx, uint32_t* d_buf, size_t count);
void nccl_destroy(cb_context* ctx);

}  // namespace cb
