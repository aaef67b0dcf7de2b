// General-k nearest neighbours over the grid (product code, sm_100a).
// Replaces the batched KDTree::kNNInRadiusSearch / kNNSearch (core/kd_tree.hpp:215-318) for k <= 256 (the k-best list is a
// per-thread array: registers for small k, L1-resident local memory for large k; the reference is unbounded in k):
// same shell sweep as nn_search.cuh, with a per-thread sorted list of the k best (d2, index) pairs
// whose worst entry plays the role of nanoflann's worstDist() (kd_tree.hpp:101).
#include "cb_internal.hpp"
#include "grid_sweep.cuh"
#include <algorithm>
#include <vector>

using namespace cb;

namespace {

constexpr int kMaxK = 256;
constexpr int kBlock = 128;

struct KBest {
  float d2[kMaxK];
  int idx[kMaxK];
};

// insertion keeping ascending (d2, idx); entries with d2 >= bound never enter. Ties on d2 are ordered
// by original index so that the result is independent of the visiting order.
template <int K>
__device__ __forceinline__ void kbest_insert(float (&bd)[K], int (&bi)[K], int k, int& count, float r, int pi) {
  // reject if not better than the current k-th
  if (count == k) {
    if (!(r < bd[k - 1] || (r == bd[k - 1] && pi < bi[k - 1]))) return;
  }
  int pos = (count < k) ? count : k - 1;
  while (pos > 0 && (bd[pos - 1] > r || (bd[pos - 1] == r && bi[pos - 1] > pi))) {
    bd[pos] = bd[pos - 1];
    bi[pos] = bi[pos - 1];
    --pos;
  }
  bd[pos] = r;
  bi[pos] = pi;
  if (count < k) ++count;
}

template <int K>
__global__ void __launch_bounds__(kBlock) knn_k_kernel(const GridView g, const float4* __restrict__ qry, uint32_t nq,
                                                       const Rigid T, int k, float max_d2, int* __restrict__ out_idx,
                                                       float* __restrict__ out_d2, uint32_t* __restrict__ out_cnt) {
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t qi = blockIdx.x * blockDim.x + threadIdx.x; qi < nq; qi += stride) {
    const float4 s = __ldg(qry + qi);
    const int oi = __float_as_int(s.w);
    float qx, qy, qz;
    apply_rigid(T, s.x, s.y, s.z, qx, qy, qz);
    float bd[K];
    int bi[K];
    int count = 0;
    // bound = current worst admissible squared distance (strict): max_d2 until k found
    auto bound = [&]() { return (count == k) ? bd[k - 1] : max_d2; };
    auto scan = [&](uint32_t b, uint32_t e) {
      for (uint32_t j = b; j < e; ++j) {
        const float4 p = __ldg(g.pts + j);
        const float dx = __fsub_rn(qx, p.x), dy = __fsub_rn(qy, p.y), dz = __fsub_rn(qz, p.z);
        float r = __fmul_rn(dx, dx);
        r = __fadd_rn(r, __fmul_rn(dy, dy));
        r = __fadd_rn(r, __fmul_rn(dz, dz));
        if (r < max_d2) kbest_insert<K>(bd, bi, k, count, r, __float_as_int(p.w));
      }
    };
    grid_sweep(g, qx, qy, qz, bound, scan, [&]() { count = 0; }, (uint32_t)k);
    for (int j = 0; j < k; j++) {
      out_idx[(size_t)oi * k + j] = (j < count) ? bi[j] : -1;
      out_d2[(size_t)oi * k + j] = (j < count) ? bd[j] : max_d2;
    }
    if (out_cnt) out_cnt[oi] = (uint32_t)count;
  }
}

}  // namespace

namespace cb {

// k-best lists of every point of `c` against `c` itself (the neighbourhoods of segment.cu): d_idx / d_d2 are n x k in
// original order, d_cnt[i] = entries of list i. Stream-ordered; no synchronise.
int knn_lists_self(cb_context* ctx, const cb_cloud* c, int k, float max_d2, int* d_idx, float* d_d2, uint32_t* d_cnt) {
  CB_CHECK(k >= 1 && k <= kMaxK, CB_ERR_UNSUPPORTED, "k must be in [1, 256]");
  const size_t n = c->n;
  if (n == 0) return CB_OK;
  const Rigid T = rigid_from_t12(nullptr);
  const int blocks = (int)std::max<size_t>(1, std::min<size_t>((size_t)ctx->sm_count * 8, (n + kBlock - 1) / kBlock));
  const GridView g = grid_view(c);
  if (k <= 4)
    knn_k_kernel<4><<<blocks, kBlock, 0, ctx->stream>>>(g, c->d_pts, (uint32_t)n, T, k, max_d2, d_idx, d_d2, d_cnt);
  else if (k <= 16)
    knn_k_kernel<16><<<blocks, kBlock, 0, ctx->stream>>>(g, c->d_pts, (uint32_t)n, T, k, max_d2, d_idx, d_d2, d_cnt);
  else if (k <= 32)
    knn_k_kernel<32><<<blocks, kBlock, 0, ctx->stream>>>(g, c->d_pts, (uint32_t)n, T, k, max_d2, d_idx, d_d2, d_cnt);
  else if (k <= 64)
    knn_k_kernel<64><<<blocks, kBlock, 0, ctx->stream>>>(g, c->d_pts, (uint32_t)n, T, k, max_d2, d_idx, d_d2, d_cnt);
  else if (k <= 128)
    knn_k_kernel<128><<<blocks, kBlock, 0, ctx->stream>>>(g, c->d_pts, (uint32_t)n, T, k, max_d2, d_idx, d_d2, d_cnt);
  else
    knn_k_kernel<256><<<blocks, kBlock, 0, ctx->stream>>>(g, c->d_pts, (uint32_t)n, T, k, max_d2, d_idx, d_d2, d_cnt);
  ctx->launches += 1;
  CB_CUDA(cudaGetLastError());
  return CB_OK;
}

}  // namespace cb

extern "C" int cb_knn_radius(cb_context* ctx, const cb_cloud* ref, const cb_cloud* qry, const float* T12, int k,
                             float max_d2, int64_t* idx, float* d2, uint32_t* counts) {
  CB_CHECK(ctx && ref && qry && idx && d2, CB_ERR_INVALID, "null argument");
  CB_CHECK(k >= 1 && k <= kMaxK, CB_ERR_UNSUPPORTED, "k must be in [1, 256]");
  CB_CHECK(ref->ctx == ctx && qry->ctx == ctx, CB_ERR_INVALID, "cloud belongs to another context");
  CB_CUDA(cudaSetDevice(ctx->device));
  CB_TRY(ensure_index(const_cast<cb_cloud*>(ref)));
  CB_TRY(ensure_index(const_cast<cb_cloud*>(qry)));
  const size_t nq = qry->n;
  if (nq == 0) return CB_OK;
  const Rigid T = rigid_from_t12(T12);
  int* d_idx = nullptr;
  float* d_d2 = nullptr;
  uint32_t* d_cnt = nullptr;
  CB_CUDA(cudaMallocAsync(&d_idx, nq * k * sizeof(int), ctx->stream));
  CB_CUDA(cudaMallocAsync(&d_d2, nq * k * sizeof(float), ctx->stream));
  CB_CUDA(cudaMallocAsync(&d_cnt, nq * sizeof(uint32_t), ctx->stream));
  const int blocks = (int)std::max<size_t>(1, std::min<size_t>((size_t)ctx->sm_count * 8, (nq + kBlock - 1) / kBlock));
  const GridView g = grid_view(ref);
  if (k <= 4)
    knn_k_kernel<4><<<blocks, kBlock, 0, ctx->stream>>>(g, qry->d_pts, (uint32_t)nq, T, k, max_d2, d_idx, d_d2, d_cnt);
  else if (k <= 16)
    knn_k_kernel<16><<<blocks, kBlock, 0, ctx->stream>>>(g, qry->d_pts, (uint32_t)nq, T, k, max_d2, d_idx, d_d2, d_cnt);
  else if (k <= 32)
    knn_k_kernel<32><<<blocks, kBlock, 0, ctx->stream>>>(g, qry->d_pts, (uint32_t)nq, T, k, max_d2, d_idx, d_d2, d_cnt);
  else if (k <= 64)
    knn_k_kernel<64><<<blocks, kBlock, 0, ctx->stream>>>(g, qry->d_pts, (uint32_t)nq, T, k, max_d2, d_idx, d_d2, d_cnt);
  else if (k <= 128)
    knn_k_kernel<128><<<blocks, kBlock, 0, ctx->stream>>>(g, qry->d_pts, (uint32_t)nq, T, k, max_d2, d_idx, d_d2, d_cnt);
  else
    knn_k_kernel<256><<<blocks, kBlock, 0, ctx->stream>>>(g, qry->d_pts, (uint32_t)nq, T, k, max_d2, d_idx, d_d2, d_cnt);
  ctx->launches += 1;
  CB_CUDA(cudaGetLastError());
  std::vector<int> h_idx(nq * k);
  CB_CUDA(cudaMemcpyAsync(h_idx.data(), d_idx, nq * k * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CB_CUDA(cudaMemcpyAsync(d2, d_d2, nq * k * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  if (counts) CB_CUDA(cudaMemcpyAsync(counts, d_cnt, nq * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  CB_CUDA(cudaFreeAsync(d_idx, ctx->stream));
  CB_CUDA(cudaFreeAsync(d_d2, ctx->stream));
  CB_CUDA(cudaFreeAsync(d_cnt, ctx->stream));
  CB_CUDA(cudaStreamSynchronize(ctx->stream));
  for (size_t i = 0; i < nq * k; i++) idx[i] = h_idx[i] < 0 ? -1 : (int64_t)h_idx[i] + (int64_t)ref->index_offset;
  return CB_OK;
}

// ---- radius neighbourhoods (variable length) ---------------------------------------------------------
// KDTree::radiusSearch batched (core/kd_tree.hpp:250-278): every ref point with d2 < radius2, ascending
// distance (RadiusSearchResultAdaptor + std::sort by value, :111-141, :254). Three kernels over the same
// sweep: count per query -> exclusive scan -> fill, then one thread per query heap-sorts its segment on
// (d2, original index) — a total order, so the result does not depend on the visiting order (the reference
// leaves the order of equal distances to std::sort).
namespace {

template <bool kFill>
__global__ void __launch_bounds__(kBlock) radius_kernel(const GridView g, const float4* __restrict__ qry, uint32_t nq,
                                                        const Rigid T, float r2, uint32_t* __restrict__ counts,
                                                        const uint32_t* __restrict__ offsets, int* __restrict__ out_idx,
                                                        float* __restrict__ out_d2) {
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t qi = blockIdx.x * blockDim.x + threadIdx.x; qi < nq; qi += stride) {
    const float4 s = __ldg(qry + qi);
    const int oi = __float_as_int(s.w);
    float qx, qy, qz;
    apply_rigid(T, s.x, s.y, s.z, qx, qy, qz);
    uint32_t n = 0;
    const uint32_t base = kFill ? offsets[oi] : 0u;
    grid_sweep(
        g, qx, qy, qz, [&]() { return r2; },
        [&](uint32_t b, uint32_t e) {
          for (uint32_t j = b; j < e; ++j) {
            const float4 p = __ldg(g.pts + j);
            const float dx = __fsub_rn(qx, p.x), dy = __fsub_rn(qy, p.y), dz = __fsub_rn(qz, p.z);
            float r = __fmul_rn(dx, dx);
            r = __fadd_rn(r, __fmul_rn(dy, dy));
            r = __fadd_rn(r, __fmul_rn(dz, dz));
            if (r < r2) {
              if (kFill) {
                out_idx[base + n] = __float_as_int(p.w);
                out_d2[base + n] = r;
              }
              ++n;
            }
          }
        },
        [&]() { n = 0; }, 0u);
    if (!kFill) counts[oi] = n;
  }
}

__device__ __forceinline__ bool nb_less(float da, int ia, float db, int ib) { return da < db || (da == db && ia < ib); }

__global__ void segment_heapsort_kernel(const uint32_t* __restrict__ offsets, uint32_t nq, int* __restrict__ idx,
                                        float* __restrict__ d2) {
  for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += gridDim.x * blockDim.x) {
    const uint32_t b = offsets[q], m = offsets[q + 1] - b;
    if (m < 2) continue;
    int* I = idx + b;
    float* D = d2 + b;
    auto sift = [&](uint32_t root, uint32_t end) {  // max-heap on (d2, idx)
      const float dv = D[root];
      const int iv = I[root];
      for (;;) {
        uint32_t c = 2 * root + 1;
        if (c >= end) break;
        if (c + 1 < end && nb_less(D[c], I[c], D[c + 1], I[c + 1])) ++c;
        if (!nb_less(dv, iv, D[c], I[c])) break;
        D[root] = D[c];
        I[root] = I[c];
        root = c;
      }
      D[root] = dv;
      I[root] = iv;
    };
    for (uint32_t s = m / 2; s-- > 0;) sift(s, m);
    for (uint32_t e = m - 1; e > 0; --e) {
      const float dt = D[0];
      const int it = I[0];
      D[0] = D[e];
      I[0] = I[e];
      D[e] = dt;
      I[e] = it;
      sift(0, e);
    }
  }
}

}  // namespace

extern "C" int cb_radius_search(cb_context* ctx, const cb_cloud* ref, const cb_cloud* qry, const float* T12,
                                float radius2, uint64_t* offsets, int64_t* idx, float* d2, size_t capacity,
                                size_t* total) {
  CB_CHECK(ctx && ref && qry && offsets && total, CB_ERR_INVALID, "null argument");
  CB_CHECK(ref->ctx == ctx && qry->ctx == ctx, CB_ERR_INVALID, "cloud belongs to another context");
  CB_CUDA(cudaSetDevice(ctx->device));
  CB_TRY(ensure_index(const_cast<cb_cloud*>(ref)));
  CB_TRY(ensure_index(const_cast<cb_cloud*>(qry)));
  const size_t nq = qry->n;
  *total = 0;
  offsets[0] = 0;
  if (nq == 0) return CB_OK;
  const Rigid T = rigid_from_t12(T12);
  uint32_t* d_off = nullptr;
  CB_CUDA(cudaMallocAsync(&d_off, (nq + 2) * sizeof(uint32_t), ctx->stream));
  CB_CUDA(cudaMemsetAsync(d_off, 0, (nq + 2) * sizeof(uint32_t), ctx->stream));
  const int blocks = (int)std::max<size_t>(1, std::min<size_t>((size_t)ctx->sm_count * 8, (nq + kBlock - 1) / kBlock));
  const GridView g = grid_view(ref);
  radius_kernel<false><<<blocks, kBlock, 0, ctx->stream>>>(g, qry->d_pts, (uint32_t)nq, T, radius2, d_off, nullptr,
                                                          nullptr, nullptr);
  ctx->launches += 1;
  // counts are 32-bit: sum them on the host in 64 bits before trusting the 32-bit scan
  std::vector<uint32_t> h_cnt(nq);
  CB_CUDA(cudaMemcpyAsync(h_cnt.data(), d_off, nq * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  CB_CUDA(cudaStreamSynchronize(ctx->stream));
  uint64_t sum = 0;
  for (size_t i = 0; i < nq; i++) {
    offsets[i] = sum;
    sum += h_cnt[i];
  }
  offsets[nq] = sum;
  *total = (size_t)sum;
  if (sum == 0 || !idx || !d2 || capacity < sum) {
    CB_CUDA(cudaFreeAsync(d_off, ctx->stream));
    return CB_OK;  // sizing call, or the caller's buffers are too small: *total says what is needed
  }
  if (sum >= (1ull << 32)) {
    cudaFreeAsync(d_off, ctx->stream);
    CB_CHECK(false, CB_ERR_UNSUPPORTED, "radius search: more than 2^32 - 1 neighbour pairs in one call");
  }
  CB_TRY(exclusive_scan_u32(ctx, d_off, nq + 1, 0u));
  int* d_idx = nullptr;
  float* d_d2 = nullptr;
  CB_CUDA(cudaMallocAsync(&d_idx, sum * sizeof(int), ctx->stream));
  CB_CUDA(cudaMallocAsync(&d_d2, sum * sizeof(float), ctx->stream));
  radius_kernel<true><<<blocks, kBlock, 0, ctx->stream>>>(g, qry->d_pts, (uint32_t)nq, T, radius2, nullptr, d_off, d_idx,
                                                         d_d2);
  segment_heapsort_kernel<<<blocks, kBlock, 0, ctx->stream>>>(d_off, (uint32_t)nq, d_idx, d_d2);
  ctx->launches += 2;
  CB_CUDA(cudaGetLastError());
  std::vector<int> h_idx(sum);
  CB_CUDA(cudaMemcpyAsync(h_idx.data(), d_idx, sum * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CB_CUDA(cudaMemcpyAsync(d2, d_d2, sum * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  CB_CUDA(cudaFreeAsync(d_idx, ctx->stream));
  CB_CUDA(cudaFreeAsync(d_d2, ctx->stream));
  CB_CUDA(cudaFreeAsync(d_off, ctx->stream));
  CB_CUDA(cudaStreamSynchronize(ctx->stream));
  for (size_t i = 0; i < sum; i++) idx[i] = (int64_t)h_idx[i] + (int64_t)ref->index_offset;
  return CB_OK;
}
