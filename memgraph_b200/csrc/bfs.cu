// memgraph_b200/csrc/bfs.cu -- direction-optimising breadth-first expansion for sm_100a (include/mgb200_bfs.h).
//
// Semantics: SingleSourceShortestPathCursor, src/query/plan/operator.cpp:2692-2912 (restated and pinned in
// oracle/bfs_oracle.c).  Distances are integers and order-independent, so parity is bit-exact whatever the
// traversal strategy; the strategy is chosen per level for speed (Beamer et al.):
//   top-down   small frontiers: one warp per (frontier vertex, <=1024-edge segment), lanes stride the adjacency,
//              discovery by atomicCAS on the depth array, warp-aggregated pushes into the next queue;
//   bottom-up  large frontiers: every unvisited vertex scans its REVERSE adjacency for a parent in the
//              frontier bitmap (2 MiB at scale-24: L1/L2 resident) and stops at the first hit.
// HBM-bound integer work: coalesced adjacency reads, random 4-byte depth / 1-bit frontier probes.
//
// MGB200_BFS_STRATEGY, read at every mgb200_bfs_run call, pins the strategy so that tests can reach every path on
// small graphs: unset or "auto" = the switch above; "top_down" / "bottom_up" = that strategy at every level (bottom-up
// from level 0, a one-vertex frontier); "alternate" = top-down on even levels, bottom-up on odd ones, so both hand-offs
// between queue and bitmap run.  Any other value is refused, so that a typo cannot quietly run the default.
#include <algorithm>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cub/cub.cuh>
#include <new>
#include <vector>

#include "core.hpp"
#include "mgb200_bfs.h"

struct mgb200_bfs_graph {
  int device = 0;
  int sm_count = 0;
  cudaStream_t stream = nullptr;
  uint64_t n = 0, m = 0;
  uint64_t *out_ptr = nullptr, *in_ptr = nullptr;   // [n + 1]
  uint32_t *out_adj = nullptr, *in_adj = nullptr;   // [m], sorted inside a row
  int32_t *depth = nullptr;                         // [n]
  uint32_t *queue[2] = {nullptr, nullptr};          // [n] frontier vertex lists
  uint32_t *bitmap[2] = {nullptr, nullptr};         // [ceil(n/32)]
  uint64_t *seg_count = nullptr, *seg_scan = nullptr;  // [n + 1]
  unsigned long long *counters = nullptr;           // device: [0] next size [1] frontier degree sum [2] inspected [3] items
  unsigned long long *host_counters = nullptr;      // pinned
  void *cub_tmp = nullptr;
  size_t cub_tmp_bytes = 0;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
};

namespace mgb200 {
namespace {

constexpr int kThreads = 256;
constexpr uint32_t kSegEdges = 1024;
constexpr unsigned kFull = 0xffffffffu;

inline int blocks_for(uint64_t items, int sm_count, int per_sm = 16) {
  const uint64_t want = (items + kThreads - 1) / kThreads;
  return static_cast<int>(std::max<uint64_t>(1, std::min<uint64_t>(want, static_cast<uint64_t>(sm_count) * per_sm)));
}

struct Adj {  // the adjacency a direction walks: `a` first, then `b` (BOTH)
  const uint64_t *a_ptr;
  const uint32_t *a_adj;
  const uint64_t *b_ptr;  // nullptr unless BOTH
  const uint32_t *b_adj;
  __device__ __forceinline__ uint64_t degree(uint32_t u) const {
    uint64_t d = a_ptr[u + 1] - a_ptr[u];
    if (b_ptr) d += b_ptr[u + 1] - b_ptr[u];
    return d;
  }
  // k-th neighbour of u in the concatenation
  __device__ __forceinline__ uint32_t neighbour(uint32_t u, uint64_t k) const {
    const uint64_t a0 = a_ptr[u], da = a_ptr[u + 1] - a0;
    if (k < da) return a_adj[a0 + k];
    return b_adj[b_ptr[u] + (k - da)];
  }
};

__global__ void degree_count_kernel(uint64_t m, uint64_t n, const uint32_t *from, const uint32_t *to,
                                    unsigned long long *out_deg, unsigned long long *in_deg, int *bad) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (uint64_t e = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; e < m; e += stride) {
    const uint32_t s = from[e], d = to[e];
    if (s >= n || d >= n) {
      *bad = 1;
      continue;
    }
    atomicAdd(out_deg + s, 1ull);
    atomicAdd(in_deg + d, 1ull);
  }
}
__global__ void pair_key_kernel(uint64_t m, const uint32_t *hi, const uint32_t *lo, uint64_t *key) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (uint64_t e = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; e < m; e += stride)
    key[e] = (static_cast<uint64_t>(hi[e]) << 32) | lo[e];
}
__global__ void low_half_kernel(uint64_t m, const uint64_t *key, uint32_t *out) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (uint64_t e = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; e < m; e += stride)
    out[e] = static_cast<uint32_t>(key[e]);
}

__global__ void init_depth_kernel(uint64_t n, uint32_t source, int32_t *depth, uint32_t *queue0,
                                  unsigned long long *counters) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (uint64_t v = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; v < n; v += stride)
    depth[v] = v == source ? 0 : -1;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    queue0[0] = source;
    counters[0] = counters[1] = counters[2] = counters[3] = 0ull;
  }
}

// segments per frontier vertex + the frontier's degree sum (Beamer's m_f)
__global__ void frontier_segments_kernel(uint64_t nf, const uint32_t *queue, Adj adj, uint64_t *seg_count,
                                         unsigned long long *counters) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  unsigned long long deg_sum = 0;
  for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < nf; i += stride) {
    const uint64_t d = adj.degree(queue[i]);
    seg_count[i] = (d + kSegEdges - 1) / kSegEdges;
    deg_sum += d;
  }
  for (int o = 16; o > 0; o >>= 1) deg_sum += __shfl_xor_sync(kFull, deg_sum, o);
  if ((threadIdx.x & 31) == 0 && deg_sum) atomicAdd(counters + 1, deg_sum);
}

// top-down: one warp per (frontier vertex, segment)
__global__ void __launch_bounds__(kThreads) top_down_kernel(uint64_t nf, const uint32_t *queue, const uint64_t *seg_scan,
                                                            Adj adj, int32_t next_depth, int32_t *depth,
                                                            uint32_t *next_queue, unsigned long long *counters) {
  const int lane = threadIdx.x & 31;
  const uint64_t warps_total = static_cast<uint64_t>(gridDim.x) * (kThreads / 32);
  const uint64_t total_items = seg_scan[nf];
  unsigned long long inspected = 0;
  for (uint64_t item = static_cast<uint64_t>(blockIdx.x) * (kThreads / 32) + (threadIdx.x >> 5); item < total_items;
       item += warps_total) {
    // largest i with seg_scan[i] <= item
    uint64_t lo = 0, hi = nf;
    while (lo + 1 < hi) {
      const uint64_t mid = (lo + hi) >> 1;
      if (seg_scan[mid] <= item) lo = mid; else hi = mid;
    }
    const uint32_t u = queue[lo];
    const uint64_t deg = adj.degree(u);
    const uint64_t k0 = (item - seg_scan[lo]) * kSegEdges;
    const uint64_t k1 = (k0 + kSegEdges < deg) ? k0 + kSegEdges : deg;
    for (uint64_t kb = k0; kb < k1; kb += 32) {
      const uint64_t k = kb + lane;
      bool found = false;
      uint32_t v = 0;
      if (k < k1) {
        v = adj.neighbour(u, k);
        ++inspected;
        if (depth[v] == -1) found = atomicCAS(depth + v, -1, next_depth) == -1;
      }
      const unsigned ballot = __ballot_sync(kFull, found);
      if (ballot) {
        unsigned long long base = 0;
        const int leader = __ffs(ballot) - 1;
        if (lane == leader) base = atomicAdd(counters + 0, static_cast<unsigned long long>(__popc(ballot)));
        base = __shfl_sync(kFull, base, leader);
        if (found) next_queue[base + __popc(ballot & ((1u << lane) - 1u))] = v;
      }
    }
  }
  for (int o = 16; o > 0; o >>= 1) inspected += __shfl_xor_sync(kFull, inspected, o);
  if (lane == 0 && inspected) atomicAdd(counters + 2, inspected);
}

__global__ void clear_words_kernel(uint64_t words, uint32_t *bitmap) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (uint64_t w = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; w < words; w += stride) bitmap[w] = 0u;
}
__global__ void queue_to_bitmap_kernel(uint64_t nf, const uint32_t *queue, uint32_t *bitmap) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < nf; i += stride) {
    const uint32_t v = queue[i];
    atomicOr(bitmap + (v >> 5), 1u << (v & 31));
  }
}

// bottom-up: every unvisited vertex looks for a parent in the frontier along its reverse adjacency
__global__ void __launch_bounds__(kThreads) bottom_up_kernel(uint64_t n, Adj reverse, const uint32_t *frontier_bits,
                                                             int32_t next_depth, int32_t *depth,
                                                             uint32_t *next_queue, unsigned long long *counters) {
  const int lane = threadIdx.x & 31;
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  const uint64_t n_round = (n + 31) / 32 * 32;
  unsigned long long inspected = 0;
  for (uint64_t v = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; v < n_round; v += stride) {
    bool found = false;
    if (v < n && depth[v] == -1) {
      const uint64_t deg = reverse.degree(static_cast<uint32_t>(v));
      for (uint64_t k = 0; k < deg; ++k) {
        const uint32_t u = reverse.neighbour(static_cast<uint32_t>(v), k);
        ++inspected;
        if ((frontier_bits[u >> 5] >> (u & 31)) & 1u) {
          found = true;
          break;
        }
      }
      if (found) depth[v] = next_depth;
    }
    const unsigned ballot = __ballot_sync(kFull, found);
    if (ballot) {
      unsigned long long base = 0;
      const int leader = __ffs(ballot) - 1;
      if (lane == leader) base = atomicAdd(counters + 0, static_cast<unsigned long long>(__popc(ballot)));
      base = __shfl_sync(kFull, base, leader);
      if (found) next_queue[base + __popc(ballot & ((1u << lane) - 1u))] = static_cast<uint32_t>(v);
    }
  }
  for (int o = 16; o > 0; o >>= 1) inspected += __shfl_xor_sync(kFull, inspected, o);
  if (lane == 0 && inspected) atomicAdd(counters + 2, inspected);
}

__global__ void finalize_kernel(uint64_t n, uint32_t source, const int32_t *depth, long long lower, long long upper,
                                int32_t *dist) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (uint64_t v = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; v < n; v += stride) {
    const int32_t d = depth[v];
    dist[v] = (v != source && d > 0 && d >= lower && d <= upper) ? d : -1;  // operator.cpp:2833,2874
  }
}

struct Scratch {
  std::vector<void *> ptrs;
  ~Scratch() {
    for (void *p : ptrs) cudaFree(p);
  }
  template <typename T>
  cudaError_t alloc(T **out, uint64_t count) {
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, std::max<uint64_t>(count, 1) * sizeof(T));
    if (e == cudaSuccess) ptrs.push_back(p);
    *out = static_cast<T *>(p);
    return e;
  }
};

// rows sorted by (row, neighbour): ptr from the degree counts, adj from the sorted keys
int build_side(mgb200_bfs_graph &g, Scratch &tmp, const uint32_t *row, const uint32_t *col,
               const unsigned long long *deg, uint64_t **ptr_out, uint32_t **adj_out) {
  const uint64_t n = g.n, m = g.m;
  cudaStream_t st = g.stream;
  MGB_CUDA(cudaMalloc(ptr_out, (n + 1) * sizeof(uint64_t)));
  MGB_CUDA(cudaMalloc(adj_out, std::max<uint64_t>(m, 1) * sizeof(uint32_t)));
  {
    size_t bytes = 0;
    MGB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, bytes, deg, *ptr_out, n, st));
    void *t = nullptr;
    MGB_CUDA(tmp.alloc(reinterpret_cast<char **>(&t), bytes));
    MGB_CUDA(cub::DeviceScan::ExclusiveSum(t, bytes, deg, *ptr_out, n, st));
    MGB_CUDA(cudaMemcpyAsync(*ptr_out + n, &g.m, sizeof(uint64_t), cudaMemcpyHostToDevice, st));
  }
  if (m == 0) return MGB200_OK;
  uint64_t *key = nullptr, *alt = nullptr;
  MGB_CUDA(tmp.alloc(&key, m));
  MGB_CUDA(tmp.alloc(&alt, m));
  pair_key_kernel<<<blocks_for(m, g.sm_count), kThreads, 0, st>>>(m, row, col, key);
  cub::DoubleBuffer<uint64_t> kb(key, alt);
  size_t bytes = 0;
  int bits = 1;
  while (bits < 32 && (n >> bits) != 0) ++bits;
  MGB_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, bytes, kb, m, 0, 32 + bits, st));
  void *t = nullptr;
  MGB_CUDA(tmp.alloc(reinterpret_cast<char **>(&t), bytes));
  MGB_CUDA(cub::DeviceRadixSort::SortKeys(t, bytes, kb, m, 0, 32 + bits, st));
  low_half_kernel<<<blocks_for(m, g.sm_count), kThreads, 0, st>>>(m, kb.Current(), *adj_out);
  MGB_CUDA(cudaGetLastError());
  MGB_CUDA(cudaStreamSynchronize(st));
  return MGB200_OK;
}

enum class Strategy { kAuto, kTopDown, kBottomUp, kAlternate };

int read_strategy(Strategy *out) {
  const char *s = getenv("MGB200_BFS_STRATEGY");
  if (!s || !strcmp(s, "auto")) *out = Strategy::kAuto;
  else if (!strcmp(s, "top_down")) *out = Strategy::kTopDown;
  else if (!strcmp(s, "bottom_up")) *out = Strategy::kBottomUp;
  else if (!strcmp(s, "alternate")) *out = Strategy::kAlternate;
  else {
    set_error(std::string("bfs: unknown MGB200_BFS_STRATEGY '") + s + "' (auto, top_down, bottom_up or alternate)");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  return MGB200_OK;
}

int read_counters(mgb200_bfs_graph &g) {
  MGB_CUDA(cudaMemcpyAsync(g.host_counters, g.counters, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, g.stream));
  MGB_CUDA(cudaStreamSynchronize(g.stream));
  return MGB200_OK;
}

}  // namespace
}  // namespace mgb200

using namespace mgb200;

extern "C" {

void mgb200_bfs_graph_destroy(mgb200_bfs_graph *g) {
  if (!g) return;
  cudaSetDevice(g->device);
  void *ptrs[] = {g->out_ptr, g->in_ptr, g->out_adj, g->in_adj, g->depth, g->queue[0], g->queue[1], g->bitmap[0],
                  g->bitmap[1], g->seg_count, g->seg_scan, g->counters, g->cub_tmp};
  for (void *p : ptrs)
    if (p) cudaFree(p);
  if (g->host_counters) cudaFreeHost(g->host_counters);
  if (g->ev0) cudaEventDestroy(g->ev0);
  if (g->ev1) cudaEventDestroy(g->ev1);
  if (g->stream) cudaStreamDestroy(g->stream);
  delete g;
}

int mgb200_bfs_graph_create_device(int device, uint64_t n, uint64_t m, const uint32_t *d_from, const uint32_t *d_to,
                                   mgb200_bfs_graph **out) {
  if (!out) return MGB200_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  if (n >= 0xFFFFFFFFull || (m > 0 && (!d_from || !d_to))) {
    set_error("bfs: n must be < 2^32 - 1 and the edge arrays non-null");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  int count = 0;
  cudaError_t ce = cudaGetDeviceCount(&count);
  if (ce != cudaSuccess) return cuda_fail(ce, "cudaGetDeviceCount", __FILE__, __LINE__);
  if (count <= 0 || device < 0 || device >= count) {
    set_error("CUDA error: no usable CUDA device (this library has no CPU fallback)");
    return MGB200_ERR_CUDA;
  }
  auto *g = new (std::nothrow) mgb200_bfs_graph();
  if (!g) return MGB200_ERR_INVALID_ARGUMENT;
  g->device = device;
  g->n = n;
  g->m = m;
  auto fail = [&](int rc) {
    mgb200_bfs_graph_destroy(g);
    return rc;
  };
  auto body = [&]() -> int {
    MGB_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop{};
    MGB_CUDA(cudaGetDeviceProperties(&prop, device));
    g->sm_count = prop.multiProcessorCount;
    MGB_CUDA(cudaStreamCreateWithFlags(&g->stream, cudaStreamNonBlocking));
    MGB_CUDA(cudaEventCreate(&g->ev0));
    MGB_CUDA(cudaEventCreate(&g->ev1));
    cudaStream_t st = g->stream;
    Scratch tmp;
    unsigned long long *out_deg = nullptr, *in_deg = nullptr;
    int *bad = nullptr;
    MGB_CUDA(tmp.alloc(&out_deg, n + 1));
    MGB_CUDA(tmp.alloc(&in_deg, n + 1));
    MGB_CUDA(tmp.alloc(&bad, 1));
    MGB_CUDA(cudaMemsetAsync(out_deg, 0, (n + 1) * sizeof(unsigned long long), st));
    MGB_CUDA(cudaMemsetAsync(in_deg, 0, (n + 1) * sizeof(unsigned long long), st));
    MGB_CUDA(cudaMemsetAsync(bad, 0, sizeof(int), st));
    if (m) degree_count_kernel<<<blocks_for(m, g->sm_count), kThreads, 0, st>>>(m, n, d_from, d_to, out_deg, in_deg, bad);
    int bad_host = 0;
    MGB_CUDA(cudaMemcpyAsync(&bad_host, bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    MGB_CUDA(cudaStreamSynchronize(st));
    if (bad_host) {
      set_error("edge endpoint out of range (>= number_of_nodes)");
      return MGB200_ERR_INVALID_ARGUMENT;
    }
    int rc = build_side(*g, tmp, d_from, d_to, out_deg, &g->out_ptr, &g->out_adj);
    if (rc) return rc;
    rc = build_side(*g, tmp, d_to, d_from, in_deg, &g->in_ptr, &g->in_adj);
    if (rc) return rc;
    const uint64_t words = (n + 31) / 32 + 1;
    MGB_CUDA(cudaMalloc(&g->depth, std::max<uint64_t>(n, 1) * sizeof(int32_t)));
    for (int i = 0; i < 2; ++i) {
      MGB_CUDA(cudaMalloc(&g->queue[i], std::max<uint64_t>(n, 1) * sizeof(uint32_t)));
      MGB_CUDA(cudaMalloc(&g->bitmap[i], words * sizeof(uint32_t)));
    }
    MGB_CUDA(cudaMalloc(&g->seg_count, (n + 1) * sizeof(uint64_t)));
    MGB_CUDA(cudaMalloc(&g->seg_scan, (n + 2) * sizeof(uint64_t)));
    MGB_CUDA(cudaMalloc(&g->counters, 4 * sizeof(unsigned long long)));
    MGB_CUDA(cudaMallocHost(reinterpret_cast<void **>(&g->host_counters), 4 * sizeof(unsigned long long)));
    MGB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, g->cub_tmp_bytes, g->seg_count, g->seg_scan, n + 1, st));
    MGB_CUDA(cudaMalloc(&g->cub_tmp, std::max<size_t>(g->cub_tmp_bytes, 16)));
    return MGB200_OK;
  };
  const int rc = body();
  if (rc) return fail(rc);
  *out = g;
  return MGB200_OK;
}

int mgb200_bfs_graph_create_host(int device, uint64_t n, uint64_t m, const uint64_t *from, const uint64_t *to,
                                 mgb200_bfs_graph **out) {
  if (!out) return MGB200_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  if (n >= 0xFFFFFFFFull || (m > 0 && (!from || !to))) {
    set_error("bfs: n must be < 2^32 - 1 and the edge arrays non-null");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  std::vector<uint32_t> f(m), t(m);
  for (uint64_t e = 0; e < m; ++e) {
    if (from[e] >= n || to[e] >= n) {
      set_error("edge endpoint out of range (>= number_of_nodes)");
      return MGB200_ERR_INVALID_ARGUMENT;
    }
    f[e] = static_cast<uint32_t>(from[e]);
    t[e] = static_cast<uint32_t>(to[e]);
  }
  int count = 0;
  cudaError_t ce = cudaGetDeviceCount(&count);
  if (ce != cudaSuccess) return cuda_fail(ce, "cudaGetDeviceCount", __FILE__, __LINE__);
  if (count <= 0 || device < 0 || device >= count) {
    set_error("CUDA error: no usable CUDA device (this library has no CPU fallback)");
    return MGB200_ERR_CUDA;
  }
  MGB_CUDA(cudaSetDevice(device));
  uint32_t *d_f = nullptr, *d_t = nullptr;
  MGB_CUDA(cudaMalloc(&d_f, std::max<uint64_t>(m, 1) * 4));
  cudaError_t e2 = cudaMalloc(&d_t, std::max<uint64_t>(m, 1) * 4);
  if (e2 != cudaSuccess) {
    cudaFree(d_f);
    return cuda_fail(e2, "cudaMalloc", __FILE__, __LINE__);
  }
  int rc = MGB200_OK;
  if (m) {
    cudaError_t a = cudaMemcpy(d_f, f.data(), m * 4, cudaMemcpyHostToDevice);
    cudaError_t b = cudaMemcpy(d_t, t.data(), m * 4, cudaMemcpyHostToDevice);
    if (a != cudaSuccess || b != cudaSuccess) rc = cuda_fail(a != cudaSuccess ? a : b, "cudaMemcpy(COO)", __FILE__, __LINE__);
  }
  if (!rc) rc = mgb200_bfs_graph_create_device(device, n, m, d_f, d_t, out);
  cudaFree(d_f);
  cudaFree(d_t);
  return rc;
}

int mgb200_bfs_run(mgb200_bfs_graph *g, uint64_t source, int direction, int64_t lower_bound, int64_t upper_bound,
                   int32_t *dist_out, int dist_on_device, mgb200_bfs_stats *stats_out) {
  if (!g || (g->n > 0 && !dist_out) || direction < MGB200_BFS_OUT || direction > MGB200_BFS_BOTH) {
    set_error("bfs: invalid argument");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  if (source >= g->n) {
    set_error("bfs: source vertex out of range");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  Strategy strategy = Strategy::kAuto;
  if (int rc = read_strategy(&strategy)) return rc;
  MGB_CUDA(cudaSetDevice(g->device));
  cudaStream_t st = g->stream;
  const uint64_t n = g->n;
  mgb200_bfs_stats stats{};
  Adj forward{}, reverse{};
  if (direction == MGB200_BFS_OUT) {
    forward = Adj{g->out_ptr, g->out_adj, nullptr, nullptr};
    reverse = Adj{g->in_ptr, g->in_adj, nullptr, nullptr};
  } else if (direction == MGB200_BFS_IN) {
    forward = Adj{g->in_ptr, g->in_adj, nullptr, nullptr};
    reverse = Adj{g->out_ptr, g->out_adj, nullptr, nullptr};
  } else {
    forward = Adj{g->out_ptr, g->out_adj, g->in_ptr, g->in_adj};
    reverse = Adj{g->in_ptr, g->in_adj, g->out_ptr, g->out_adj};
  }
  const uint64_t m_dir = direction == MGB200_BFS_BOTH ? 2 * g->m : g->m;
  const uint64_t words = (n + 31) / 32;

  MGB_CUDA(cudaEventRecord(g->ev0, st));
  init_depth_kernel<<<blocks_for(n, g->sm_count), kThreads, 0, st>>>(n, static_cast<uint32_t>(source), g->depth,
                                                                     g->queue[0], g->counters);
  stats.kernel_launches++;
  uint64_t nf = 1;
  uint64_t explored_degree = 0;  // sum of degrees of every vertex expanded so far
  int cur = 0;
  int32_t level = 0;
  const bool bounds_empty = upper_bound < 1 || lower_bound > upper_bound;  // operator.cpp:2830
  while (!bounds_empty && nf > 0 && static_cast<int64_t>(level) < upper_bound && level < INT_MAX - 1) {
    // frontier statistics: segments per vertex and degree sum (m_f)
    frontier_segments_kernel<<<blocks_for(nf, g->sm_count), kThreads, 0, st>>>(nf, g->queue[cur], forward, g->seg_count,
                                                                                g->counters);
    int rc = read_counters(*g);
    if (rc) return rc;
    const uint64_t m_f = g->host_counters[1];
    const uint64_t m_u = m_dir > explored_degree ? m_dir - explored_degree : 0;
    explored_degree += m_f;
    stats.kernel_launches++;
    // Beamer's switch: go bottom-up when the frontier's edges outnumber 1/14 of the unexplored ones
    bool bottom_up = m_f > m_u / 14 && nf > 1024;
    if (strategy == Strategy::kTopDown) bottom_up = false;
    else if (strategy == Strategy::kBottomUp) bottom_up = true;
    else if (strategy == Strategy::kAlternate) bottom_up = (level & 1) != 0;
    MGB_CUDA(cudaMemsetAsync(g->counters, 0, 2 * sizeof(unsigned long long), st));
    if (bottom_up) {
      clear_words_kernel<<<blocks_for(words, g->sm_count), kThreads, 0, st>>>(words, g->bitmap[0]);
      queue_to_bitmap_kernel<<<blocks_for(nf, g->sm_count), kThreads, 0, st>>>(nf, g->queue[cur], g->bitmap[0]);
      bottom_up_kernel<<<blocks_for(n, g->sm_count, 32), kThreads, 0, st>>>(n, reverse, g->bitmap[0], level + 1, g->depth,
                                                                            g->queue[cur ^ 1], g->counters);
      stats.kernel_launches += 3;
      stats.bottom_up_levels++;
    } else {
      MGB_CUDA(cub::DeviceScan::ExclusiveSum(g->cub_tmp, g->cub_tmp_bytes, g->seg_count, g->seg_scan, nf + 1, st));
      top_down_kernel<<<g->sm_count * 8, kThreads, 0, st>>>(nf, g->queue[cur], g->seg_scan, forward, level + 1, g->depth,
                                                            g->queue[cur ^ 1], g->counters);
      stats.kernel_launches += 2;
      stats.top_down_levels++;
    }
    MGB_CUDA(cudaGetLastError());
    rc = read_counters(*g);
    if (rc) return rc;
    nf = g->host_counters[0];
    stats.edges_inspected = g->host_counters[2];
    stats.reached += nf;
    cur ^= 1;
    if (nf > 0) ++level;
  }
  MGB_CUDA(cudaEventRecord(g->ev1, st));
  stats.levels = static_cast<uint32_t>(level);
  if (n > 0) {
    int32_t *d_out = dist_out;
    if (!dist_on_device) MGB_CUDA(cudaMalloc(&d_out, n * sizeof(int32_t)));
    finalize_kernel<<<blocks_for(n, g->sm_count), kThreads, 0, st>>>(n, static_cast<uint32_t>(source), g->depth,
                                                                    static_cast<long long>(lower_bound),
                                                                    static_cast<long long>(upper_bound), d_out);
    stats.kernel_launches++;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess && !dist_on_device)
      e = cudaMemcpyAsync(dist_out, d_out, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st);
    cudaError_t e2 = cudaStreamSynchronize(st);
    if (!dist_on_device) cudaFree(d_out);
    if (e != cudaSuccess) return cuda_fail(e, "bfs finalize", __FILE__, __LINE__);
    if (e2 != cudaSuccess) return cuda_fail(e2, "cudaStreamSynchronize", __FILE__, __LINE__);
  }
  float ms = 0.f;
  MGB_CUDA(cudaEventElapsedTime(&ms, g->ev0, g->ev1));
  stats.traverse_ms = ms;
  if (stats_out) *stats_out = stats;
  return MGB200_OK;
}

}  // extern "C"
