// Connected-component segmentation on the device (product code, sm_100a).
// Replaces extractConnectedComponents(tree, nh, seeds, ...) (clustering/connected_component_extraction.hpp:162-265).
//
// The reference grows one region per seed with a frontier stack and one kd-tree search per popped point, recording
// label merges in std::sets. Every point of R (the points reachable from the seeds along the directed edges u -> L(u)[j],
// j >= 1, that the evaluator accepts) is popped exactly once, and each of its passing edges either adopts v or records a
// merge with v's label; so its segments are the connected components of the undirected graph on R with those edges.
// That is what is computed here, in an order-free way:
//   * edges: one thread per point of the cell-sorted copy runs the grid sweep (grid_sweep.cuh) with the fixed bound
//     radius2, or walks its kNN list (knn_k.cu), and calls union for every passing pair;
//   * union-find over original indices: lock-free hooking of the higher root under the lower (atomicCAS), path halving,
//     a final compression pass (ECL-CC). Work is O(edges) and does not grow with the depth of the graph. A root is
//     always the smallest index of its component;
//   * seed lists: a frontier traversal over the directed edges. A thread keeps expanding what it claims from a small
//     private stack (the oldest entry spills to the next frontier when it is full), so a chain is walked by one thread
//     in one launch. Unions are made on the way: every u in R is expanded once, which is the union pass restricted to R.
//     No kernel waits on another block; the host launches until the frontier is empty;
//   * finalise: component sizes (atomicAdd), the min / max filter, the surviving roots compacted in ascending order and
//     sorted stably by (n - size), so equal sizes keep ascending smallest index; labels from the sort rank; the
//     segment -> points lists from a stable sort of the labels over ascending point indices.
// The partition, the filter and both sorts are determined by the graph alone: two runs are bit-identical.
//
// All seeds and a radius neighbourhood: L(u)[0] is the lowest index w with d2(u, w) == 0, so w <= u, and every
// evaluator is symmetric bit for bit; the dropped direction u -> w is present as w -> u. The undirected edge set is
// then {u != v : d2 < radius2, evaluator}, and each pair is visited once (v > u). With a seed list the dropped direction
// matters (seed u of duplicates w < u reaches no w), so the traversal skips w = first[u] explicitly.
#include "cb_internal.hpp"
#include "grid_sweep.cuh"
#include "segment_rule.hpp"
#include <algorithm>
#include <vector>

using namespace cb;

namespace {

constexpr int kBlock = 128;
constexpr int kMinBlocks = 8;  // without a minimum, ptxas caps the sweep kernels at 32 registers and spills
constexpr uint32_t kStack = 16;  // private stack of the reachability kernel (a power of two: it is a ring)
constexpr uint32_t kNone = 0xffffffffu;

struct Attr {  // per-point evaluator inputs in cell-sorted order; nullptr when the evaluator does not read them
  const float4* nrm;
  const float4* col;
};

__device__ __forceinline__ float4 ld_attr(const float4* a, uint32_t pos) {
  return a ? __ldg(a + pos) : make_float4(0.f, 0.f, 0.f, 0.f);
}

__device__ __forceinline__ float self_d2(float qx, float qy, float qz, const float4& p) {
  const float dx = __fsub_rn(qx, p.x), dy = __fsub_rn(qy, p.y), dz = __fsub_rn(qz, p.z);
  float r = __fmul_rn(dx, dx);
  r = __fadd_rn(r, __fmul_rn(dy, dy));
  return __fadd_rn(r, __fmul_rn(dz, dz));
}

__device__ __forceinline__ uint32_t ld_parent(const uint32_t* p) { return *(const volatile uint32_t*)p; }

// root of x; parent[x] <= x always, so a root is the smallest index of its tree
__device__ __forceinline__ uint32_t uf_find(uint32_t* parent, uint32_t x) {
  for (;;) {
    const uint32_t p = ld_parent(parent + x);
    if (p == x) return x;
    const uint32_t g = ld_parent(parent + p);
    if (g == p) return p;
    *(volatile uint32_t*)(parent + x) = g;  // path halving: x is not a root, so no hook can race with this store
    x = g;
  }
}

__device__ __forceinline__ void uf_union(uint32_t* parent, uint32_t a, uint32_t b) {
  for (;;) {
    a = uf_find(parent, a);
    b = uf_find(parent, b);
    if (a == b) return;
    if (a > b) {
      const uint32_t t = a;
      a = b;
      b = t;
    }
    const uint32_t old = atomicCAS(parent + b, b, a);  // hook the higher root under the lower
    if (old == b) return;
    b = old;
  }
}

__global__ void seg_init_kernel(const float4* __restrict__ pts, uint32_t n, uint32_t* __restrict__ parent,
                                uint32_t* __restrict__ pos_of) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    parent[i] = i;
    pos_of[__float_as_uint(__ldg(pts + i).w)] = i;
  }
}

// packed 3n floats in original order -> float4 in cell-sorted order
__global__ void seg_permute_kernel(const float4* __restrict__ pts, uint32_t n, const float* __restrict__ raw,
                                   float4* __restrict__ out) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const size_t o = __float_as_uint(__ldg(pts + i).w);
    out[i] = make_float4(raw[3 * o], raw[3 * o + 1], raw[3 * o + 2], 0.f);
  }
}

// all seeds, radius lists: union every accepted pair {u, v}, u < v, d2 < r2
__global__ void __launch_bounds__(kBlock, kMinBlocks) seg_radius_union_kernel(const GridView g, float r2, const seg::PairRule rule,
                                                                  const Attr at, uint32_t* __restrict__ parent) {
  for (uint32_t pos = blockIdx.x * blockDim.x + threadIdx.x; pos < g.n; pos += gridDim.x * blockDim.x) {
    const float4 s = __ldg(g.pts + pos);
    const uint32_t u = __float_as_uint(s.w);
    const float4 nu = ld_attr(at.nrm, pos), cu = ld_attr(at.col, pos);
    grid_sweep(
        g, s.x, s.y, s.z, [&]() { return r2; },
        [&](uint32_t b, uint32_t e) {
          for (uint32_t j = b; j < e; ++j) {
            const float4 p = __ldg(g.pts + j);
            const uint32_t v = __float_as_uint(p.w);
            if (v <= u) continue;
            const float d2 = self_d2(s.x, s.y, s.z, p);
            if (d2 < r2 && seg::pair_passes(rule, d2, nu, ld_attr(at.nrm, j), cu, ld_attr(at.col, j)))
              uf_union(parent, u, v);
          }
        },
        [&]() {}, 0u);  // a restarted sweep only repeats unions
  }
}

// all seeds, kNN lists: union u with every accepted L(u)[j], j >= 1
__global__ void __launch_bounds__(kBlock, kMinBlocks) seg_knn_union_kernel(uint32_t n, int k, const int* __restrict__ lists,
                                                               const float* __restrict__ ld2,
                                                               const uint32_t* __restrict__ lcnt,
                                                               const uint32_t* __restrict__ pos_of,
                                                               const seg::PairRule rule, const Attr at,
                                                               uint32_t* __restrict__ parent) {
  for (uint32_t u = blockIdx.x * blockDim.x + threadIdx.x; u < n; u += gridDim.x * blockDim.x) {
    const uint32_t c = lcnt[u];
    if (c < 2) continue;
    const uint32_t pu = pos_of[u];
    const float4 nu = ld_attr(at.nrm, pu), cu = ld_attr(at.col, pu);
    for (uint32_t j = 1; j < c; ++j) {
      const size_t e = (size_t)u * k + j;
      const uint32_t v = (uint32_t)lists[e];
      const uint32_t pv = pos_of[v];
      if (seg::pair_passes(rule, ld2[e], nu, ld_attr(at.nrm, pv), cu, ld_attr(at.col, pv))) uf_union(parent, u, v);
    }
  }
}

// radius lists with a seed list: first[u] = L(u)[0], the lowest index at computed distance 0 from u
__global__ void __launch_bounds__(kBlock, kMinBlocks) seg_first_kernel(const GridView g, uint32_t* __restrict__ first) {
  for (uint32_t pos = blockIdx.x * blockDim.x + threadIdx.x; pos < g.n; pos += gridDim.x * blockDim.x) {
    const float4 s = __ldg(g.pts + pos);
    uint32_t w = __float_as_uint(s.w);
    grid_sweep(
        g, s.x, s.y, s.z, [&]() { return 1.17549435e-38f; },  // only d2 == 0 is wanted: the smallest normal float
        [&](uint32_t b, uint32_t e) {
          for (uint32_t j = b; j < e; ++j) {
            const float4 p = __ldg(g.pts + j);
            if (self_d2(s.x, s.y, s.z, p) == 0.f) w = min(w, __float_as_uint(p.w));
          }
        },
        [&]() {}, 0u);
    first[__float_as_uint(s.w)] = w;
  }
}

__global__ void seg_seed_kernel(const uint64_t* __restrict__ seeds, size_t ns, uint32_t* __restrict__ visited,
                                uint32_t* __restrict__ frontier, uint32_t* __restrict__ count) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < ns; i += (size_t)gridDim.x * blockDim.x) {
    const uint32_t s = (uint32_t)seeds[i];
    if (atomicExch(visited + s, 1u) == 0u) frontier[atomicAdd(count, 1u)] = s;
  }
}

// Expands the frontier (original indices) along the directed edges: unions every accepted edge u -> v and claims
// unvisited v. kKnn: the lists of knn_k.cu; otherwise the radius sweep, skipping first[u].
template <bool kKnn>
__global__ void __launch_bounds__(kBlock, kMinBlocks) seg_reach_kernel(const GridView g, float r2, const seg::PairRule rule,
                                                           const Attr at, const uint32_t* __restrict__ pos_of,
                                                           const uint32_t* __restrict__ first, int k,
                                                           const int* __restrict__ lists, const float* __restrict__ ld2,
                                                           const uint32_t* __restrict__ lcnt, uint32_t* visited,
                                                           uint32_t* parent, const uint32_t* __restrict__ frontier,
                                                           uint32_t nf, uint32_t* __restrict__ next,
                                                           uint32_t* __restrict__ next_count) {
  for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < nf; t += gridDim.x * blockDim.x) {
    uint32_t st[kStack];
    uint32_t lo = 0, cnt = 1;
    st[0] = frontier[t];
    while (cnt > 0) {
      --cnt;
      const uint32_t u = st[(lo + cnt) & (kStack - 1)];
      const uint32_t pu = pos_of[u];
      const float4 nu = ld_attr(at.nrm, pu), cu = ld_attr(at.col, pu);
      auto visit = [&](uint32_t v, uint32_t pv, float d2) {
        if (!seg::pair_passes(rule, d2, nu, ld_attr(at.nrm, pv), cu, ld_attr(at.col, pv))) return;
        uf_union(parent, u, v);
        if (atomicExch(visited + v, 1u) != 0u) return;
        if (cnt == kStack) {  // full: the oldest entry goes to the next frontier, the walk goes on with the newest
          next[atomicAdd(next_count, 1u)] = st[lo];
          lo = (lo + 1) & (kStack - 1);
          --cnt;
        }
        st[(lo + cnt) & (kStack - 1)] = v;
        ++cnt;
      };
      if (kKnn) {
        const uint32_t c = lcnt[u];
        for (uint32_t j = 1; j < c; ++j) {
          const size_t e = (size_t)u * k + j;
          const uint32_t v = (uint32_t)lists[e];
          visit(v, pos_of[v], ld2[e]);
        }
      } else {
        const float4 s = __ldg(g.pts + pu);
        const uint32_t w = first[u];
        grid_sweep(
            g, s.x, s.y, s.z, [&]() { return r2; },
            [&](uint32_t b, uint32_t e) {
              for (uint32_t j = b; j < e; ++j) {
                const float4 p = __ldg(g.pts + j);
                const uint32_t v = __float_as_uint(p.w);
                if (v == w) continue;
                const float d2 = self_d2(s.x, s.y, s.z, p);
                if (d2 < r2) visit(v, j, d2);
              }
            },
            [&]() {}, 0u);
      }
    }
  }
}

// Final compression: parent[i] = root. No path halving here: a halving store of another thread could overwrite an
// entry already compressed with an older (non-root) ancestor. Only thread i writes parent[i]; readers see the old
// or the new value of an entry, both ancestors, and reach the same root.
__global__ void seg_compress_kernel(uint32_t n, uint32_t* parent) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    uint32_t r = i, p;
    while ((p = ld_parent(parent + r)) != r) r = p;
    *(volatile uint32_t*)(parent + i) = r;
  }
}

// visited == nullptr: every point is in R
__global__ void seg_size_kernel(uint32_t n, const uint32_t* __restrict__ parent, const uint32_t* __restrict__ visited,
                                uint32_t* __restrict__ size) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    if (!visited || visited[i]) atomicAdd(size + parent[i], 1u);
}

__global__ void seg_keep_kernel(uint32_t n, const uint32_t* __restrict__ parent, const uint32_t* __restrict__ size,
                                unsigned long long min_size, unsigned long long max_size, uint32_t* __restrict__ flag) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t s = size[i];  // 0 for non-roots and for points outside R
    flag[i] = (parent[i] == i && s > 0 && s >= min_size && s <= max_size) ? 1u : 0u;
  }
}

// kept roots in ascending order: key n - size (sorted stably next), value the root
__global__ void seg_emit_kernel(uint32_t n, const uint32_t* __restrict__ scan, const uint32_t* __restrict__ size,
                                uint64_t* __restrict__ keys, uint32_t* __restrict__ vals) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t j = scan[i];
    if (scan[i + 1] != j) {
      keys[j] = (uint64_t)(n - size[i]);
      vals[j] = i;
    }
  }
}

__global__ void seg_rank_kernel(uint32_t m, const uint32_t* __restrict__ roots, uint32_t* __restrict__ rank_of) {
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < m; j += gridDim.x * blockDim.x) rank_of[roots[j]] = j;
}

__global__ void seg_label_kernel(uint32_t n, uint32_t m, const uint32_t* __restrict__ parent,
                                 const uint32_t* __restrict__ visited, const uint32_t* __restrict__ rank_of,
                                 uint64_t* __restrict__ labels, uint64_t* __restrict__ lkeys,
                                 uint32_t* __restrict__ lvals) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    uint32_t r = (!visited || visited[i]) ? rank_of[parent[i]] : kNone;
    if (r == kNone) r = m;
    labels[i] = r;
    lkeys[i] = r;
    lvals[i] = i;
  }
}

int bit_length(uint64_t x) {
  int b = 0;
  while (x) {
    ++b;
    x >>= 1;
  }
  return b;
}

}  // namespace

extern "C" int cb_cloud_segment(cb_context* ctx, cb_cloud* cloud, const cb_segment_params* prm, const uint64_t* seeds,
                                size_t n_seeds, const float* normals, const float* colors, uint64_t* labels,
                                uint64_t* seg_offsets, uint64_t* seg_points, size_t* num_segments, float* gpu_ms) {
  CB_CHECK(ctx && cloud && prm && num_segments && seg_offsets, CB_ERR_INVALID, "null argument");
  CB_CHECK(cloud->ctx == ctx, CB_ERR_INVALID, "cloud belongs to another context");
  CB_CHECK(prm->k >= 0, CB_ERR_INVALID, "k must be >= 0");
  CB_CHECK(prm->k <= 256, CB_ERR_UNSUPPORTED, "k must be in [0, 256]");
  CB_CHECK(prm->evaluator >= seg::kAlwaysTrue && prm->evaluator <= seg::kPointsNormalsColors, CB_ERR_INVALID,
           "unknown evaluator kind");
  const size_t n = cloud->n;
  CB_CHECK(n == 0 || (labels && seg_points), CB_ERR_INVALID, "null argument");
  *num_segments = 0;
  seg_offsets[0] = 0;
  if (gpu_ms) gpu_ms[0] = gpu_ms[1] = gpu_ms[2] = 0.f;
  if (seeds)
    for (size_t i = 0; i < n_seeds; i++) CB_CHECK(seeds[i] < n, CB_ERR_INVALID, "seed index out of range");
  const int kind = prm->evaluator;
  CB_CHECK(!seg::uses_colors(kind) || colors || n == 0, CB_ERR_INVALID, "the evaluator needs colours");
  if (n == 0) return CB_OK;
  CB_CUDA(cudaSetDevice(ctx->device));
  CB_TRY(ensure_index(cloud));
  CB_CHECK(!seg::uses_normals(kind) || normals || cloud->d_nrm, CB_ERR_INVALID,
           "the evaluator needs normals and the cloud has none");
  const seg::PairRule rule = seg::make_pair_rule(kind, prm->max_distance, prm->max_angle, prm->color_thresh);
  const bool seeded = seeds != nullptr;
  const int k = prm->k;
  const bool radius = k == 0 && prm->radius2 > 0.f;
  const bool knn = k > 0;
  const uint32_t n32 = (uint32_t)n;
  const int blocks = (int)std::max<size_t>(1, std::min<size_t>((size_t)ctx->sm_count * 8, (n + kBlock - 1) / kBlock));
  cudaStream_t s = ctx->stream;
  DeviceScope sc(ctx);

  ScopedEvents ev;
  cudaEvent_t e_mid = nullptr;
  if (gpu_ms) {
    CB_TRY(ev.create());
    CB_CUDA(cudaEventCreate(&e_mid));
    CB_CUDA(cudaEventRecord(ev.e0, s));
  }
  struct EventGuard {
    cudaEvent_t e;
    ~EventGuard() {
      if (e) cudaEventDestroy(e);
    }
  } mid_guard{e_mid};

  uint32_t *parent, *pos_of;
  CB_TRY(sc.alloc(&parent, n));
  CB_TRY(sc.alloc(&pos_of, n));
  seg_init_kernel<<<blocks, kBlock, 0, s>>>(cloud->d_pts, n32, parent, pos_of);
  ctx->launches += 1;
  Attr at{nullptr, nullptr};
  if (seg::uses_normals(kind)) {
    if (normals) {
      float* d_raw;
      float4* d_n;
      CB_TRY(sc.alloc(&d_raw, 3 * n));
      CB_TRY(sc.alloc(&d_n, n));
      CB_CUDA(cudaMemcpyAsync(d_raw, normals, 3 * n * sizeof(float), cudaMemcpyHostToDevice, s));
      seg_permute_kernel<<<blocks, kBlock, 0, s>>>(cloud->d_pts, n32, d_raw, d_n);
      ctx->launches += 1;
      at.nrm = d_n;
    } else {
      at.nrm = cloud->d_nrm;
    }
  }
  if (seg::uses_colors(kind)) {
    float* d_raw;
    float4* d_c;
    CB_TRY(sc.alloc(&d_raw, 3 * n));
    CB_TRY(sc.alloc(&d_c, n));
    CB_CUDA(cudaMemcpyAsync(d_raw, colors, 3 * n * sizeof(float), cudaMemcpyHostToDevice, s));
    seg_permute_kernel<<<blocks, kBlock, 0, s>>>(cloud->d_pts, n32, d_raw, d_c);
    ctx->launches += 1;
    at.col = d_c;
  }
  int* lists = nullptr;
  float* ld2 = nullptr;
  uint32_t* lcnt = nullptr;
  if (knn) {
    CB_TRY(sc.alloc(&lists, n * (size_t)k));
    CB_TRY(sc.alloc(&ld2, n * (size_t)k));
    CB_TRY(sc.alloc(&lcnt, n));
    CB_TRY(knn_lists_self(ctx, cloud, k, prm->radius2 > 0.f ? prm->radius2 : 3.402823466e38f, lists, ld2, lcnt));
  }
  const GridView g = grid_view(cloud);
  uint32_t* visited = nullptr;
  if (!seeded) {
    if (radius) {
      seg_radius_union_kernel<<<blocks, kBlock, 0, s>>>(g, prm->radius2, rule, at, parent);
      ctx->launches += 1;
    } else if (knn) {
      seg_knn_union_kernel<<<blocks, kBlock, 0, s>>>(n32, k, lists, ld2, lcnt, pos_of, rule, at, parent);
      ctx->launches += 1;
    }
  } else {
    uint32_t *front, *next, *counter, *first = nullptr;
    uint64_t* d_seeds;
    CB_TRY(sc.alloc(&visited, n));
    CB_TRY(sc.alloc(&front, n));
    CB_TRY(sc.alloc(&next, n));
    CB_TRY(sc.alloc(&counter, 1));
    CB_TRY(sc.alloc(&d_seeds, n_seeds));
    CB_CUDA(cudaMemsetAsync(visited, 0, n * sizeof(uint32_t), s));
    CB_CUDA(cudaMemsetAsync(counter, 0, sizeof(uint32_t), s));
    uint32_t nf = 0;
    if (n_seeds) {
      CB_CUDA(cudaMemcpyAsync(d_seeds, seeds, n_seeds * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
      const int sb = (int)std::max<size_t>(1, std::min<size_t>((size_t)ctx->sm_count * 8, (n_seeds + 255) / 256));
      seg_seed_kernel<<<sb, 256, 0, s>>>(d_seeds, n_seeds, visited, front, counter);
      ctx->launches += 1;
      CB_CUDA(cudaMemcpyAsync(&nf, counter, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
      CB_CUDA(cudaStreamSynchronize(s));
    }
    if (radius) {
      CB_TRY(sc.alloc(&first, n));
      seg_first_kernel<<<blocks, kBlock, 0, s>>>(g, first);
      ctx->launches += 1;
    }
    // level-synchronous launches; the host stops when no thread spilled anything to the next frontier
    while (nf > 0 && (radius || knn)) {
      CB_CUDA(cudaMemsetAsync(counter, 0, sizeof(uint32_t), s));
      const int fb = (int)std::max<uint32_t>(1, std::min<uint32_t>((uint32_t)ctx->sm_count * 8, (nf + kBlock - 1) / kBlock));
      if (knn)
        seg_reach_kernel<true><<<fb, kBlock, 0, s>>>(g, 0.f, rule, at, pos_of, nullptr, k, lists, ld2, lcnt, visited,
                                                     parent, front, nf, next, counter);
      else
        seg_reach_kernel<false><<<fb, kBlock, 0, s>>>(g, prm->radius2, rule, at, pos_of, first, 0, nullptr, nullptr,
                                                      nullptr, visited, parent, front, nf, next, counter);
      ctx->launches += 1;
      CB_CUDA(cudaGetLastError());
      CB_CUDA(cudaMemcpyAsync(&nf, counter, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
      CB_CUDA(cudaStreamSynchronize(s));
      std::swap(front, next);
    }
  }
  if (gpu_ms) CB_CUDA(cudaEventRecord(e_mid, s));

  // ---- finalise
  uint32_t *size, *scan;
  CB_TRY(sc.alloc(&size, n));
  CB_TRY(sc.alloc(&scan, n + 2));
  CB_CUDA(cudaMemsetAsync(size, 0, n * sizeof(uint32_t), s));
  CB_CUDA(cudaMemsetAsync(scan, 0, (n + 2) * sizeof(uint32_t), s));
  seg_compress_kernel<<<blocks, kBlock, 0, s>>>(n32, parent);
  seg_size_kernel<<<blocks, kBlock, 0, s>>>(n32, parent, visited, size);
  seg_keep_kernel<<<blocks, kBlock, 0, s>>>(n32, parent, size, (unsigned long long)prm->min_size,
                                            (unsigned long long)prm->max_size, scan);
  ctx->launches += 3;
  CB_CUDA(cudaGetLastError());
  CB_TRY(exclusive_scan_u32(ctx, scan, n + 1, 0u));
  uint32_t m = 0;
  CB_CUDA(cudaMemcpyAsync(&m, scan + n, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  CB_CUDA(cudaStreamSynchronize(s));

  std::vector<uint64_t> h_keys(m);
  std::vector<uint32_t> h_pts;
  if (m > 0) {
    uint64_t *keys, *keys_tmp, *lkeys, *lkeys_tmp;
    uint32_t *roots, *roots_tmp, *rank_of, *lvals, *lvals_tmp;
    uint64_t* d_labels;
    CB_TRY(sc.alloc(&keys, m));
    CB_TRY(sc.alloc(&keys_tmp, m));
    CB_TRY(sc.alloc(&roots, m));
    CB_TRY(sc.alloc(&roots_tmp, m));
    seg_emit_kernel<<<blocks, kBlock, 0, s>>>(n32, scan, size, keys, roots);
    ctx->launches += 1;
    CB_TRY(radix_sort_pairs_u64(ctx, keys, roots, keys_tmp, roots_tmp, m, bit_length(n)));
    CB_TRY(sc.alloc(&rank_of, n));
    CB_CUDA(cudaMemsetAsync(rank_of, 0xff, n * sizeof(uint32_t), s));
    seg_rank_kernel<<<blocks, kBlock, 0, s>>>(m, roots, rank_of);
    CB_TRY(sc.alloc(&d_labels, n));
    CB_TRY(sc.alloc(&lkeys, n));
    CB_TRY(sc.alloc(&lkeys_tmp, n));
    CB_TRY(sc.alloc(&lvals, n));
    CB_TRY(sc.alloc(&lvals_tmp, n));
    seg_label_kernel<<<blocks, kBlock, 0, s>>>(n32, m, parent, visited, rank_of, d_labels, lkeys, lvals);
    ctx->launches += 2;
    CB_CUDA(cudaGetLastError());
    CB_TRY(radix_sort_pairs_u64(ctx, lkeys, lvals, lkeys_tmp, lvals_tmp, n, bit_length(m)));
    if (gpu_ms) CB_CUDA(cudaEventRecord(ev.e1, s));
    h_pts.resize(n);
    CB_CUDA(cudaMemcpyAsync(h_keys.data(), keys, m * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
    CB_CUDA(cudaMemcpyAsync(labels, d_labels, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
    CB_CUDA(cudaMemcpyAsync(h_pts.data(), lvals, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    CB_CUDA(cudaStreamSynchronize(s));
  } else {
    if (gpu_ms) CB_CUDA(cudaEventRecord(ev.e1, s));
    CB_CUDA(cudaStreamSynchronize(s));
    std::fill(labels, labels + n, (uint64_t)0);
  }
  uint64_t total = 0;
  for (uint32_t j = 0; j < m; j++) {
    total += n - h_keys[j];
    seg_offsets[j + 1] = total;
  }
  for (uint64_t t = 0; t < total; t++) seg_points[t] = h_pts[t];
  *num_segments = m;
  if (gpu_ms) {
    CB_CUDA(cudaEventElapsedTime(&gpu_ms[0], ev.e0, ev.e1));
    CB_CUDA(cudaEventElapsedTime(&gpu_ms[1], ev.e0, e_mid));
    CB_CUDA(cudaEventElapsedTime(&gpu_ms[2], e_mid, ev.e1));
  }
  return CB_OK;
}
