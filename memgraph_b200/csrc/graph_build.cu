// memgraph_b200/csrc/graph_build.cu -- COO on the device -> degree-sorted SELL-32 + segmented CSC.
//
// This is the device-side counterpart of the reference's graph constructors
// (PageRankGraph(n, m, edges), pagerank.cpp:165-181; CreatePageRankGraph, pagerank_module.cpp:18-54):
// they produce a source-ordered edge list plus out-degrees for a CPU push loop; this produces the
// pull layout the sm_100a kernels stream.  It runs once per graph and is outside the timed
// iteration (SURVEY 8d); sorting and scanning use CUB (library code, like cuBLAS for a plain GEMM),
// the layout kernels are ours.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cub/cub.cuh>
#include <vector>

#include "core.hpp"

namespace mgb200 {
namespace {

constexpr int kThreads = 256;

inline int blocks_for(uint64_t items, int sm_count) {
  const uint64_t want = (items + kThreads - 1) / kThreads;
  const uint64_t cap = static_cast<uint64_t>(sm_count) * 16;
  return static_cast<int>(std::max<uint64_t>(1, std::min(want, cap)));
}

// ---- degrees ----------------------------------------------------------------------------------------

__global__ void degree_kernel(uint64_t m, uint64_t n, const uint32_t *from, const uint32_t *to, uint32_t *outdeg,
                              uint32_t *indeg, int *bad) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (uint64_t e = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; e < m; e += stride) {
    const uint32_t s = from[e], d = to[e];
    if (s >= n || d >= n) {
      *bad = 1;
      continue;
    }
    atomicAdd(outdeg + s, 1u);
    atomicAdd(indeg + d, 1u);
  }
}

// sort key: in-degree descending, then out-degree descending (stable sort keeps original id order)
__global__ void sort_key_kernel(uint64_t n, const uint32_t *indeg, const uint32_t *outdeg, uint64_t *key,
                                uint32_t *id) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (uint64_t v = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; v < n; v += stride) {
    key[v] = (static_cast<uint64_t>(~indeg[v]) << 32) | static_cast<uint64_t>(~outdeg[v]);
    id[v] = static_cast<uint32_t>(v);
  }
}

struct Dealer {  // sorted position -> global label when positions are dealt round-robin to P owners
  uint64_t n;
  uint32_t world;
  __host__ __device__ uint64_t count(uint32_t q) const { return (n + world - 1 - q) / world; }
  __host__ __device__ uint64_t start(uint32_t q) const {
    // sum_{r<q} count(r): the first (n % world) owners hold one extra row
    const uint64_t base = n / world, extra = n % world;
    return static_cast<uint64_t>(q) * base + (q < extra ? q : extra);
  }
  __host__ __device__ uint64_t label(uint64_t pos) const {
    const uint32_t owner = static_cast<uint32_t>(pos % world);
    return start(owner) + pos / world;
  }
};

__global__ void label_kernel(RowMap map, const uint32_t *sorted_id, const uint32_t *indeg, const uint32_t *outdeg,
                             uint32_t *label_of, uint32_t *indeg_l, uint32_t *outdeg_l, uint32_t *vertex_of_label) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (uint64_t pos = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; pos < map.n; pos += stride) {
    const uint32_t v = sorted_id[pos];
    const uint64_t l = map.label_of_pos(pos);
    label_of[v] = static_cast<uint32_t>(l);
    indeg_l[l] = indeg[v];
    outdeg_l[l] = outdeg[v];
    vertex_of_label[l] = v;
  }
}

// ---- edges owned by this partition -> (local row, source label) keys ---------------------------------

__global__ void edge_key_all_kernel(uint64_t m, const uint32_t *from, const uint32_t *to, const uint32_t *label_of,
                                    uint64_t *key) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (uint64_t e = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; e < m; e += stride)
    key[e] = (static_cast<uint64_t>(label_of[to[e]]) << 32) | label_of[from[e]];
}

__global__ void out_weight_kernel(uint64_t n, const double *outw, const uint32_t *label_of, double *outw_l) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (uint64_t v = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; v < n; v += stride)
    outw_l[label_of[v]] = outw[v];
}

__global__ void edge_key_owned_kernel(uint64_t m, const uint32_t *from, const uint32_t *to, const uint32_t *label_of,
                                      RowMap map, uint64_t row_hi, uint64_t *key,
                                      unsigned long long *cursor) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  const int lane = threadIdx.x & 31;
  const uint64_t m_round = (m + 31) / 32 * 32;  // keep whole warps in the loop for the ballot
  for (uint64_t e = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; e < m_round; e += stride) {
    uint64_t dl = 0;
    bool mine = false;
    if (e < m) {
      dl = label_of[to[e]];
      mine = map.global_order ? map.owner(dl) == map.rank : (dl >= map.row_lo && dl < row_hi);
    }
    const unsigned ballot = __ballot_sync(0xffffffffu, mine);
    if (ballot == 0) continue;
    unsigned long long base = 0;
    if (lane == __ffs(ballot) - 1) base = atomicAdd(cursor, static_cast<unsigned long long>(__popc(ballot)));
    base = __shfl_sync(0xffffffffu, base, __ffs(ballot) - 1);
    if (mine) {
      const unsigned before = __popc(ballot & ((1u << lane) - 1u));
      const uint64_t local = map.global_order ? map.local_of(dl) : dl - map.row_lo;
      key[base + before] = (local << 32) | label_of[from[e]];
    }
  }
}

// ---- class boundaries: rows are sorted by in-degree descending ----------------------------------------

__global__ void class_count_kernel(uint64_t rows, const uint32_t *indeg_local, uint32_t heavy_min,
                                   unsigned long long *counts /* [0]=heavy, [1]=nonzero, [2]=edges */) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  unsigned long long h = 0, nz = 0, ed = 0;
  for (uint64_t r = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < rows; r += stride) {
    const uint32_t d = indeg_local[r];
    h += d >= heavy_min;
    nz += d > 0;
    ed += d;
  }
  for (int o = 16; o > 0; o >>= 1) {
    h += __shfl_xor_sync(0xffffffffu, h, o);
    nz += __shfl_xor_sync(0xffffffffu, nz, o);
    ed += __shfl_xor_sync(0xffffffffu, ed, o);
  }
  if ((threadIdx.x & 31) == 0) {
    if (h) atomicAdd(counts + 0, h);
    if (nz) atomicAdd(counts + 1, nz);
    if (ed) atomicAdd(counts + 2, ed);
  }
}

// non-zero in-degree rows per partition: label l belongs to the partition whose [start, start+count) holds it
__global__ void nonzero_per_partition_kernel(Dealer deal, const uint32_t *indeg_l, unsigned long long *nz) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (uint32_t q = 0; q < deal.world; ++q) {
    const uint64_t lo = deal.start(q), hi = lo + deal.count(q);
    unsigned long long c = 0;
    for (uint64_t l = lo + static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; l < hi; l += stride)
      c += indeg_l[l] > 0;
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(nz + q, c);
  }
}

// Which partitions gather the contribution of an owned row?  Every partition sees the whole edge list, so this is local
// work: edge u -> v makes owner(v) a reader of u.  At P = 8 on RMAT only 48 % of the (vertex, peer) pairs are readers
// (scripts/push_need.py): the other half of the NVLink pushes is never looked at.
__global__ void need_mask_kernel(uint64_t m, const uint32_t *from, const uint32_t *to, const uint32_t *label_of,
                                 RowMap map, uint32_t *words) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (uint64_t e = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; e < m; e += stride) {
    const uint64_t ul = label_of[from[e]];
    if (map.owner(ul) != map.rank) continue;
    const uint32_t q = map.owner(label_of[to[e]]);
    if (q == map.rank) continue;
    const uint64_t row = map.local_of(ul);
    const uint32_t bit = (1u << q) << ((row & 3u) * 8u);
    uint32_t *w = words + (row >> 2);
    if ((*reinterpret_cast<volatile uint32_t *>(w) & bit) == 0) atomicOr(w, bit);  // hubs: one atomic, then reads
  }
}

struct U32ToU64 {
  __host__ __device__ uint64_t operator()(uint32_t v) const { return v; }
};

// ---- heavy class ---------------------------------------------------------------------------------------

// Hotness of a source label (core.hpp kIdxL2Hot / kIdxL1Hot), decided once per stored index instead of once per
// gather per iteration: local = label - first label of the owning partition (the dealt labelling gives every
// partition's range its own hottest-first order), compared with the thresholds the gather window uses.
struct IndexFlags {
  Dealer deal;
  uint32_t l1_hot, l2_hot;  // Graph::l1_hot_labels() (kNoL1Hints -> no L1 flag is ever read), l2_hot_labels()
  uint32_t enabled;
  uint32_t table_per_owner;  // > 0: the hottest labels of every owner live in the SELL kernel's shared-memory table;
                             // their stored index is code 01 in bits 31/30 + the table slot (owner * per_owner + local)
  __device__ uint32_t operator()(uint32_t label) const {
    if (!enabled) return label;
    if (label >= deal.n) return label | kIdxL2Hot | kIdxL1Hot;  // the pad slot: one address, read by every slice
    uint32_t s0 = 0, owner = 0;
    for (uint32_t q = 1; q < deal.world; ++q) {
      const uint32_t s = static_cast<uint32_t>(deal.start(q));
      if (label >= s) {
        s0 = s;
        owner = q;
      }
    }
    const uint32_t local = label - s0;
    if (local < table_per_owner) return kIdxL1Hot | (owner * table_per_owner + local);
    return label | (local < l2_hot ? kIdxL2Hot : 0u) | (l1_hot != kNoL1Hints && local < l1_hot ? kIdxL1Hot : 0u);
  }
};

__global__ void low32_kernel(uint64_t count, const uint64_t *key, IndexFlags flags, uint32_t *out) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (uint64_t e = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; e < count; e += stride)
    out[e] = flags(static_cast<uint32_t>(key[e]));
}

struct SegCount {
  uint32_t seg;
  __host__ __device__ uint64_t operator()(uint32_t deg) const { return (static_cast<uint64_t>(deg) + seg - 1) / seg; }
};

__global__ void segment_fill_kernel(uint64_t n_heavy, const uint64_t *heavy_ptr, const uint64_t *seg_first,
                                    uint32_t seg_edges, uint32_t *seg_row, uint64_t *seg_begin) {
  // one warp per heavy row; lanes stride over that row's segments
  const int lane = threadIdx.x & 31;
  const uint64_t warps_total = static_cast<uint64_t>(gridDim.x) * (blockDim.x >> 5);
  for (uint64_t r = static_cast<uint64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5); r < n_heavy;
       r += warps_total) {
    const uint64_t s0 = seg_first[r], s1 = seg_first[r + 1], e0 = heavy_ptr[r];
    for (uint64_t s = s0 + lane; s < s1; s += 32) {
      seg_row[s] = static_cast<uint32_t>(r);
      seg_begin[s] = e0 + (s - s0) * seg_edges;
    }
  }
}

// ---- SELL class ------------------------------------------------------------------------------------------

__global__ void slice_width_kernel(uint64_t n_slices, const uint32_t *indeg_local, uint64_t first_row,
                                   uint64_t *width) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (uint64_t s = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; s < n_slices; s += stride)
    width[s] = indeg_local[first_row + s * kSliceRows];  // rows sorted descending: lane 0 is the widest
}

__global__ void sell_fill_kernel(uint64_t n_slices, uint64_t first_row, uint64_t end_row, const uint64_t *row_ptr,
                                 const uint64_t *key, const uint64_t *colbase, uint32_t pad, IndexFlags flags,
                                 uint32_t *sell_idx, const double *w_sorted, double *sell_w) {
  const int lane = threadIdx.x & 31;
  const uint64_t warps_total = static_cast<uint64_t>(gridDim.x) * (blockDim.x >> 5);
  for (uint64_t s = static_cast<uint64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5); s < n_slices;
       s += warps_total) {
    const uint64_t c0 = colbase[s];
    const uint32_t width = static_cast<uint32_t>(colbase[s + 1] - c0);
    const uint64_t row = first_row + s * kSliceRows + lane;
    uint64_t e0 = 0;
    uint32_t deg = 0;
    if (row < end_row) {
      e0 = row_ptr[row];
      deg = static_cast<uint32_t>(row_ptr[row + 1] - e0);
    }
    uint32_t *dst = sell_idx + c0 * kSliceRows + lane;
    for (uint32_t k = 0; k < width; ++k)
      dst[static_cast<size_t>(k) * kSliceRows] = flags(k < deg ? static_cast<uint32_t>(key[e0 + k]) : pad);
    if (sell_w) {
      double *wd = sell_w + c0 * kSliceRows + lane;
      for (uint32_t k = 0; k < width; ++k) wd[static_cast<size_t>(k) * kSliceRows] = k < deg ? w_sorted[e0 + k] : 0.0;
    }
  }
}

// work items for the streaming SELL kernel: item i starts at the first slice whose column base is
// >= i * total_cols / n_items (binary search over the slice column bases)
__global__ void sell_items_kernel(uint32_t n_items, uint64_t n_slices, const uint64_t *colbase, uint64_t total_cols,
                                  uint64_t slice_cost, uint64_t *item_begin) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n_items) return;
  if (i == n_items) {
    item_begin[i] = n_slices;
    return;
  }
  // cost of slices [0, s) = their columns + slice_cost per slice; item i starts where that reaches i/n_items of the total
  const unsigned __int128 t = static_cast<unsigned __int128>(total_cols + slice_cost * n_slices) * i;
  const uint64_t target = static_cast<uint64_t>(t / n_items);
  uint64_t lo = 0, hi = n_slices;  // first s in [0, n_slices] with cost(s) >= target
  while (lo < hi) {
    const uint64_t mid = (lo + hi) >> 1;
    if (colbase[mid] + slice_cost * mid < target) lo = mid + 1; else hi = mid;
  }
  item_begin[i] = lo;
}

__global__ void work_item_kernel(uint32_t n_items, const uint64_t *item_begin, const uint64_t *colbase, WorkItem *out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_items) return;
  const uint64_t b = item_begin[i], e = item_begin[i + 1];
  WorkItem w{b, e, 0, 0};
  if (b < e) {
    w.col_begin = colbase[b];
    w.col_end = colbase[e];
  }
  out[i] = w;
}

// by_local[r] = by_label[label of this partition's local row r]  (original vertex ids, in-degrees)
__global__ void gather_local_u32_kernel(uint64_t rows, RowMap map, const uint32_t *by_label, uint32_t *by_local) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (uint64_t r = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < rows; r += stride)
    by_local[r] = by_label[map.label_of_local(r)];
}

__global__ void narrow_kernel(uint64_t count, uint64_t n, const uint64_t *in, uint32_t *out, int *bad) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (uint64_t e = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; e < count; e += stride) {
    const uint64_t v = in[e];
    if (v >= n) *bad = 1;
    out[e] = static_cast<uint32_t>(v);
  }
}

// RAII-free scratch tracker: everything pushed here is freed when the build returns.
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
  void release(void *p) {
    for (auto &q : ptrs)
      if (q == p) {
        cudaFree(p);
        q = nullptr;
      }
  }
};

template <typename T>
cudaError_t keep_alloc(Graph &g, T **out, uint64_t count) {
  void *p = nullptr;
  const uint64_t bytes = std::max<uint64_t>(count, 1) * sizeof(T);
  cudaError_t e = cudaMalloc(&p, bytes);
  if (e == cudaSuccess) g.resident_bytes += bytes;
  *out = static_cast<T *>(p);
  return e;
}

// peak device memory in use during the build (whole device, so other handles of the process count too)
void note_mem(Graph &g) {
  size_t free_b = 0, total_b = 0;
  if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) g.build_peak_bytes = std::max<uint64_t>(g.build_peak_bytes, total_b - free_b);
}

uint32_t env_u32(const char *name, uint32_t fallback) {
  const char *s = getenv(name);
  if (!s || !*s) return fallback;
  const unsigned long v = strtoul(s, nullptr, 10);
  return v ? static_cast<uint32_t>(v) : fallback;
}

uint32_t env_u32_zero(const char *name, uint32_t fallback) {  // like env_u32, but "0" is a value
  const char *s = getenv(name);
  return (s && *s) ? static_cast<uint32_t>(strtoul(s, nullptr, 10)) : fallback;
}

int bits_for(uint64_t v) {  // number of bits needed to represent values < v
  int b = 0;
  while (b < 64 && (v >> b) != 0) ++b;
  return std::max(b, 1);
}

}  // namespace

int narrow_edges_u64_to_u32(int device, cudaStream_t stream, uint64_t n, uint64_t count, const uint64_t *d_in,
                            uint32_t *d_out, int *d_bad_flag) {
  MGB_CUDA(cudaSetDevice(device));
  if (count == 0) return MGB200_OK;
  narrow_kernel<<<static_cast<int>(std::min<uint64_t>((count + kThreads - 1) / kThreads, 148 * 16)), kThreads, 0,
                  stream>>>(count, n, d_in, d_out, d_bad_flag);
  MGB_CUDA(cudaGetLastError());
  return MGB200_OK;
}

void free_graph(Graph &g) {
  cudaSetDevice(g.device);
  for (int q = 0; q < kMaxPeers; ++q)
    if (g.peer_mapped[q]) cudaIpcCloseMemHandle(g.peer_mapped[q]);
  if (g.sell_item_begin) cudaFree(g.sell_item_begin);
  if (g.sell_work_begin) cudaFree(g.sell_work_begin);
  if (g.sell_work_items) cudaFree(g.sell_work_items);
  if (g.queue) cudaFree(g.queue);
  if (g.sell_sums) cudaFree(g.sell_sums);
  if (g.out_stage) cudaFree(g.out_stage);
  if (g.need_mask) cudaFree(g.need_mask);
  if (g.heavy_w) cudaFree(g.heavy_w);
  if (g.sell_w) cudaFree(g.sell_w);
  if (g.outw_l) cudaFree(g.outw_l);
  void *ptrs[] = {g.label_of,  g.outdeg_l,  g.local_vertex, g.heavy_ptr,    g.heavy_idx, g.seg_row,     g.seg_begin,
                  g.seg_first, g.seg_partial, g.heavy_sums, g.sell_colbase, g.sell_idx,     g.rank,      g.window,      g.state,
                  g.sum_partials};
  for (void *p : ptrs)
    if (p) cudaFree(p);
  if (g.host_state) cudaFreeHost(g.host_state);
  for (auto &e : g.ev)
    if (e) cudaEventDestroy(e);
  for (auto &e : g.kev)
    if (e) cudaEventDestroy(e);
  if (g.fork_ev) cudaEventDestroy(g.fork_ev);
  if (g.join_ev) cudaEventDestroy(g.join_ev);
  if (g.stream2) cudaStreamDestroy(g.stream2);
  if (g.stream) cudaStreamDestroy(g.stream);
}

int build_graph(Graph &g, EdgeSource &edges) {
  MGB_CUDA(cudaSetDevice(g.device));
  cudaDeviceProp prop{};
  MGB_CUDA(cudaGetDeviceProperties(&prop, g.device));
  g.sm_count = prop.multiProcessorCount;
  MGB_CUDA(cudaStreamCreateWithFlags(&g.stream, cudaStreamNonBlocking));
  {  // the side stream carries the SELL epilogue + peer push: highest priority, so that its few CTAs are placed before
     // the heavy-row kernel's when both become ready at the end of the SELL kernel
    int prio_low = 0, prio_high = 0;
    MGB_CUDA(cudaDeviceGetStreamPriorityRange(&prio_low, &prio_high));
    MGB_CUDA(cudaStreamCreateWithPriority(&g.stream2, cudaStreamNonBlocking, prio_high));
  }
  MGB_CUDA(cudaEventCreateWithFlags(&g.fork_ev, cudaEventDisableTiming));
  MGB_CUDA(cudaEventCreateWithFlags(&g.join_ev, cudaEventDisableTiming));
  {
    const char *s = getenv("MGB200_OVERLAP_EPILOGUE");
    g.overlap_epilogue = !(s && s[0] == '0');
    if ((s = getenv("MGB200_L2_HOT_MB")) != nullptr) g.tun.l2_hot_mb = static_cast<uint64_t>(std::max(0l, strtol(s, nullptr, 10)));
    if ((s = getenv("MGB200_L1_HOT_K")) != nullptr) g.tun.l1_hot_k = strtol(s, nullptr, 10);
    if ((s = getenv("MGB200_MULTI_AWARE")) != nullptr) g.tun.multi_aware = s[0] != '0';
    if ((s = getenv("MGB200_FORCE_MULTI_PATH")) != nullptr) g.tun.force_multi_path = s[0] == '1';
    if ((s = getenv("MGB200_SELL_KERNEL")) != nullptr) g.tun.stream_kernel = strcmp(s, "stream") == 0;
    if ((s = getenv("MGB200_IDX_FLAGS")) != nullptr) g.tun.idx_flags = atoi(s);
    if ((s = getenv("MGB200_SELL_MODE")) != nullptr) g.tun.sell_mode = atoi(s);
    if ((s = getenv("MGB200_PUSH_CTAS")) != nullptr) g.tun.push_ctas = std::max(0, atoi(s));
    if ((s = getenv("MGB200_SMEM_TABLE_KB")) != nullptr) g.tun.smem_table_kb = static_cast<uint32_t>(std::min(224, std::max(0, atoi(s))));
    if ((s = getenv("MGB200_LABELLING")) != nullptr) g.tun.global_order = strcmp(s, "global") == 0;
    if ((s = getenv("MGB200_PUSH_MASK")) != nullptr) g.tun.push_mask = s[0] == '1';
    if ((s = getenv("MGB200_LONE_PARTITION")) != nullptr) g.tun.lone_partition = s[0] == '1';
    if ((s = getenv("MGB200_BARRIER_TIMEOUT_MS")) != nullptr) {
      const unsigned long long ms = strtoull(s, nullptr, 10);
      if (ms) g.tun.barrier_timeout_ms = ms;
    }
  }
  for (auto &e : g.ev) MGB_CUDA(cudaEventCreate(&e));
  cudaStream_t st = g.stream;
  const uint64_t n = g.n, m = g.m;
  g.heavy_min_degree = env_u32("MGB200_HEAVY_MIN_DEGREE", 1024);
  g.segment_edges = env_u32("MGB200_SEGMENT_EDGES", 4096);

  MGB_CUDA(cudaEventRecord(g.ev[0], st));
  Scratch tmp;
  const Dealer deal{n, g.part_world};
  RowMap &map = g.map;
  map = RowMap{};
  map.n = n;
  map.world = g.part_world;
  map.rank = g.part_rank;
  map.global_order = (g.tun.global_order && g.part_world > 1) ? 1u : 0u;  // one partition: both labellings coincide
  // Hot flags in the stored indices replace the per-gather owner lookup on several partitions (default there);
  // on one partition the range policy already costs nothing per gather, so flags are opt-in (MGB200_IDX_FLAGS=1).
  // They need two index bits (n < 2^30) and partition-aware thresholds; the TMA stream kernel reads raw indices.
  g.idx_flagged = (g.tun.idx_flags > 0 || (g.tun.idx_flags < 0 && g.part_world > 1)) && g.tun.multi_aware &&
                  !g.tun.global_order && !g.tun.stream_kernel && n < (1ull << 30);
  // (table_labels() needs idx_flagged, set just above; the heavy-row kernel has no table, so its indices keep labels)
  const IndexFlags idx_flags_heavy{deal, g.l1_hot_labels(), g.l2_hot_labels(), g.idx_flagged ? 1u : 0u, 0u};
  const IndexFlags idx_flags{deal, g.l1_hot_labels(), g.l2_hot_labels(), g.idx_flagged ? 1u : 0u,
                             g.idx_flagged ? g.table_labels() / g.part_world : 0u};
  g.row_lo = 0;
  g.local_rows = 0;  // known once the degrees are (global order: depends on the heavy-row count of the whole graph)

  // iteration state and exchange window exist even for an empty graph
  MGB_CUDA(keep_alloc(g, &g.state, 1));
  MGB_CUDA(cudaMemsetAsync(g.state, 0, sizeof(IterState), st));
  MGB_CUDA(cudaMallocHost(reinterpret_cast<void **>(&g.host_state), sizeof(IterState)));
  MGB_CUDA(keep_alloc(g, &g.sum_partials, kSumBlocks));
  MGB_CUDA(keep_alloc(g, &g.queue, 1));
  MGB_CUDA(cudaMemsetAsync(g.queue, 0, sizeof(WorkQueue), st));
  g.contrib_stride = ((n + 1) * sizeof(double) + 255) / 256 * 256;
  g.window_bytes = kFlagPageBytes + 2 * g.contrib_stride;
  MGB_CUDA(cudaMalloc(&g.window, g.window_bytes));
  g.resident_bytes += g.window_bytes;
  MGB_CUDA(cudaMemsetAsync(g.window, 0, g.window_bytes, st));
  for (int q = 0; q < kMaxPeers; ++q) {
    g.peers.contrib[0][q] = g.peers.contrib[1][q] = nullptr;
    g.peers.flags[q] = nullptr;
  }
  g.peers.contrib[0][g.part_rank] = g.contrib(0);
  g.peers.contrib[1][g.part_rank] = g.contrib(1);
  g.peers.flags[g.part_rank] = g.flags();
  MGB_CUDA(keep_alloc(g, &g.label_of, n));
  MGB_CUDA(keep_alloc(g, &g.outdeg_l, n));

  if (n == 0) {
    MGB_CUDA(keep_alloc(g, &g.rank, 0));
    MGB_CUDA(keep_alloc(g, &g.local_vertex, 0));
    MGB_CUDA(cudaEventRecord(g.ev[1], st));
    MGB_CUDA(cudaStreamSynchronize(st));
    return MGB200_OK;
  }

  // 1. degrees in original id space
  uint32_t *outdeg = nullptr, *indeg = nullptr;
  int *bad = nullptr;
  MGB_CUDA(tmp.alloc(&outdeg, n));
  MGB_CUDA(tmp.alloc(&indeg, n));
  MGB_CUDA(tmp.alloc(&bad, 1));
  MGB_CUDA(cudaMemsetAsync(outdeg, 0, n * sizeof(uint32_t), st));
  MGB_CUDA(cudaMemsetAsync(indeg, 0, n * sizeof(uint32_t), st));
  MGB_CUDA(cudaMemsetAsync(bad, 0, sizeof(int), st));
  const uint64_t chunk_cap = std::max<uint64_t>(1, std::min<uint64_t>(edges.chunk_edges ? edges.chunk_edges : m, std::max<uint64_t>(m, 1)));
  for (uint64_t first = 0; first < m; first += chunk_cap) {  // pass 1 over the edge list: degrees
    const uint64_t cnt = std::min(chunk_cap, m - first);
    const uint32_t *d_from = nullptr, *d_to = nullptr;
    const int grc = edges.get(first, cnt, &d_from, &d_to, st);
    if (grc) return grc;
    degree_kernel<<<blocks_for(cnt, g.sm_count), kThreads, 0, st>>>(cnt, n, d_from, d_to, outdeg, indeg, bad);
  }
  int bad_host = 0;
  MGB_CUDA(cudaMemcpyAsync(&bad_host, bad, sizeof(int), cudaMemcpyDeviceToHost, st));
  MGB_CUDA(cudaStreamSynchronize(st));
  if (bad_host) {
    set_error("edge endpoint out of range (>= number_of_nodes)");
    return MGB200_ERR_INVALID_ARGUMENT;
  }

  // 1b. who owns what.  Global-order labelling deals the heavy rows singly and the rest in blocks of 32 labels, so it
  // needs the heavy-row count (and, for the zero-row tail, the non-zero count) of the WHOLE graph first.
  uint64_t nonzero_global = 0;
  if (map.global_order) {
    unsigned long long *gc = nullptr;
    MGB_CUDA(tmp.alloc(&gc, 3));
    MGB_CUDA(cudaMemsetAsync(gc, 0, 3 * sizeof(unsigned long long), st));
    class_count_kernel<<<blocks_for(n, g.sm_count), kThreads, 0, st>>>(n, indeg, g.heavy_min_degree, gc);
    unsigned long long gc_host[3] = {0, 0, 0};
    MGB_CUDA(cudaMemcpyAsync(gc_host, gc, sizeof(gc_host), cudaMemcpyDeviceToHost, st));
    MGB_CUDA(cudaStreamSynchronize(st));
    map.heavy = gc_host[0];
    nonzero_global = std::max<uint64_t>(gc_host[1], gc_host[0]);
  }
  map.finalize();
  g.row_lo = map.row_lo;
  g.local_rows = map.local_rows(g.part_rank);
  const uint64_t row_hi = g.row_lo + g.local_rows;
  MGB_CUDA(keep_alloc(g, &g.rank, g.local_rows));
  MGB_CUDA(keep_alloc(g, &g.local_vertex, g.local_rows));

  // 2. global order: in-degree desc, out-degree desc, id asc (stable radix sort)
  uint64_t *vkey = nullptr, *vkey_alt = nullptr;
  uint32_t *vid = nullptr, *vid_alt = nullptr;
  MGB_CUDA(tmp.alloc(&vkey, n));
  MGB_CUDA(tmp.alloc(&vkey_alt, n));
  MGB_CUDA(tmp.alloc(&vid, n));
  MGB_CUDA(tmp.alloc(&vid_alt, n));
  sort_key_kernel<<<blocks_for(n, g.sm_count), kThreads, 0, st>>>(n, indeg, outdeg, vkey, vid);
  {
    cub::DoubleBuffer<uint64_t> kb(vkey, vkey_alt);
    cub::DoubleBuffer<uint32_t> vb(vid, vid_alt);
    size_t bytes = 0;
    MGB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, bytes, kb, vb, n, 0, 64, st));
    void *cub_tmp = nullptr;
    MGB_CUDA(tmp.alloc(reinterpret_cast<char **>(&cub_tmp), bytes));
    MGB_CUDA(cub::DeviceRadixSort::SortPairs(cub_tmp, bytes, kb, vb, n, 0, 64, st));
    vid = vb.Current();
  }

  // 3. labels, degrees by label
  uint32_t *indeg_l = nullptr, *vertex_of_label = nullptr;
  MGB_CUDA(tmp.alloc(&indeg_l, n));
  MGB_CUDA(tmp.alloc(&vertex_of_label, n));
  label_kernel<<<blocks_for(n, g.sm_count), kThreads, 0, st>>>(map, vid, indeg, outdeg, g.label_of, indeg_l,
                                                              g.outdeg_l, vertex_of_label);
  gather_local_u32_kernel<<<blocks_for(g.local_rows, g.sm_count), kThreads, 0, st>>>(g.local_rows, map, vertex_of_label,
                                                                                    g.local_vertex);
  const uint32_t *indeg_local = indeg_l + g.row_lo;  // dealt ranges: the owned labels are contiguous
  if (map.global_order) {
    uint32_t *gathered = nullptr;
    MGB_CUDA(tmp.alloc(&gathered, g.local_rows));
    gather_local_u32_kernel<<<blocks_for(g.local_rows, g.sm_count), kThreads, 0, st>>>(g.local_rows, map, indeg_l,
                                                                                      gathered);
    indeg_local = gathered;
  }
  if (g.tun.push_mask && g.part_world > 1 && m > 0 && g.local_rows > 0) {
    const uint64_t words = (g.local_rows + 3) / 4;
    MGB_CUDA(keep_alloc(g, &g.need_mask, words));
    MGB_CUDA(cudaMemsetAsync(g.need_mask, 0, words * sizeof(uint32_t), st));
    // filled in pass 2 over the edge list, next to the owned-edge extraction
  }

  // 4. class boundaries and local edge count
  unsigned long long *counts = nullptr;
  MGB_CUDA(tmp.alloc(&counts, 4));
  MGB_CUDA(cudaMemsetAsync(counts, 0, 4 * sizeof(unsigned long long), st));
  class_count_kernel<<<blocks_for(g.local_rows, g.sm_count), kThreads, 0, st>>>(g.local_rows, indeg_local,
                                                                               g.heavy_min_degree, counts);
  unsigned long long counts_host[4] = {0, 0, 0, 0};
  MGB_CUDA(cudaMemcpyAsync(counts_host, counts, sizeof(counts_host), cudaMemcpyDeviceToHost, st));
  MGB_CUDA(cudaStreamSynchronize(st));
  g.any_zero_rows = false;
  uint64_t sell_rows_global_order = 0;
  if (map.global_order) {
    // Blocks [0, nz_blocks) hold at least one row with in-edges: they are SELL slices (the zero rows of the one mixed
    // block are ordinary SELL rows of width 0).  Every label from zero_first on is a zero row on whichever partition
    // owns it: ONE global tail range, the same on every partition.
    const uint64_t nz_blocks = nonzero_global > map.heavy ? (nonzero_global - map.heavy + kSliceRows - 1) / kSliceRows : 0;
    const uint64_t zero_first = std::min<uint64_t>(n, map.heavy + nz_blocks * kSliceRows);
    sell_rows_global_order = map.rows_in_blocks(g.part_rank, nz_blocks);
    for (uint32_t q = 0; q < g.part_world; ++q) g.part_start[q] = g.zero_lo[q] = g.zero_hi[q] = 0;
    g.zero_lo[0] = zero_first;
    g.zero_hi[0] = n;
    g.any_zero_rows = zero_first < n;
  } else {
    unsigned long long *nz = nullptr;
    MGB_CUDA(tmp.alloc(&nz, kMaxPeers));
    MGB_CUDA(cudaMemsetAsync(nz, 0, kMaxPeers * sizeof(unsigned long long), st));
    nonzero_per_partition_kernel<<<blocks_for(n / g.part_world + 1, g.sm_count), kThreads, 0, st>>>(deal, indeg_l, nz);
    unsigned long long nz_host[kMaxPeers] = {};
    MGB_CUDA(cudaMemcpyAsync(nz_host, nz, sizeof(nz_host), cudaMemcpyDeviceToHost, st));
    MGB_CUDA(cudaStreamSynchronize(st));
    for (uint32_t q = 0; q < g.part_world; ++q) {
      g.part_start[q] = deal.start(q);
      g.zero_lo[q] = deal.start(q) + nz_host[q];
      g.zero_hi[q] = deal.start(q) + deal.count(q);
      if (g.zero_hi[q] > g.zero_lo[q]) g.any_zero_rows = true;
    }
  }
  g.n_heavy = counts_host[0];
  if (map.global_order && g.n_heavy != map.heavy_q) {
    set_error("internal: heavy rows owned (" + std::to_string(g.n_heavy) + ") != dealt (" + std::to_string(map.heavy_q) + ")");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  g.n_sell = map.global_order ? sell_rows_global_order : counts_host[1] - counts_host[0];
  g.n_zero = g.local_rows - g.n_heavy - g.n_sell;
  g.local_edges = counts_host[2];

  // 5. keys of the owned edges, sorted by (local row, source label)
  uint64_t *ekey = nullptr, *ekey_alt = nullptr;
  MGB_CUDA(tmp.alloc(&ekey, g.local_edges));
  MGB_CUDA(tmp.alloc(&ekey_alt, g.local_edges));
  const bool weighted = edges.weighted();
  if (weighted && g.part_world > 1) {
    set_error("edge weights are supported on a single partition only");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  double *eval = nullptr, *eval_alt = nullptr;  // weights travelling with the edge keys through the sort
  if (weighted) {
    if (!edges.out_weights()) {
      set_error("internal: a weighted edge source must supply its out-weight sums");
      return MGB200_ERR_INVALID_ARGUMENT;
    }
    MGB_CUDA(tmp.alloc(&eval, g.local_edges));
    MGB_CUDA(tmp.alloc(&eval_alt, g.local_edges));
    MGB_CUDA(keep_alloc(g, &g.outw_l, n));
    out_weight_kernel<<<blocks_for(n, g.sm_count), kThreads, 0, st>>>(n, edges.out_weights(), g.label_of, g.outw_l);
  }
  if (m && g.part_world > 1) MGB_CUDA(cudaMemsetAsync(counts + 3, 0, sizeof(unsigned long long), st));
  for (uint64_t first = 0; first < m; first += chunk_cap) {  // pass 2 over the edge list: who reads what, owned edges
    const uint64_t cnt = std::min(chunk_cap, m - first);
    const uint32_t *d_from = nullptr, *d_to = nullptr;
    const int grc = edges.get(first, cnt, &d_from, &d_to, st);
    if (grc) return grc;
    if (g.need_mask)
      need_mask_kernel<<<blocks_for(cnt, g.sm_count), kThreads, 0, st>>>(cnt, d_from, d_to, g.label_of, map, g.need_mask);
    if (g.part_world == 1) {
      edge_key_all_kernel<<<blocks_for(cnt, g.sm_count), kThreads, 0, st>>>(cnt, d_from, d_to, g.label_of, ekey + first);
      if (weighted)
        MGB_CUDA(cudaMemcpyAsync(eval + first, edges.weights(), cnt * sizeof(double), cudaMemcpyDeviceToDevice, st));
    } else {
      edge_key_owned_kernel<<<blocks_for(cnt, g.sm_count), kThreads, 0, st>>>(cnt, d_from, d_to, g.label_of, map, row_hi,
                                                                             ekey, counts + 3);
    }
  }
  note_mem(g);
  if (g.local_edges) {
    cub::DoubleBuffer<uint64_t> kb(ekey, ekey_alt);
    size_t bytes = 0;
    const int end_bit = std::min(64, 32 + bits_for(g.local_rows));
    void *cub_tmp = nullptr;
    if (weighted) {
      cub::DoubleBuffer<double> vb(eval, eval_alt);
      MGB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, bytes, kb, vb, g.local_edges, 0, end_bit, st));
      MGB_CUDA(tmp.alloc(reinterpret_cast<char **>(&cub_tmp), bytes));
      MGB_CUDA(cub::DeviceRadixSort::SortPairs(cub_tmp, bytes, kb, vb, g.local_edges, 0, end_bit, st));
      eval = vb.Current();
    } else {
      MGB_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, bytes, kb, g.local_edges, 0, end_bit, st));
      MGB_CUDA(tmp.alloc(reinterpret_cast<char **>(&cub_tmp), bytes));
      MGB_CUDA(cub::DeviceRadixSort::SortKeys(cub_tmp, bytes, kb, g.local_edges, 0, end_bit, st));
    }
    note_mem(g);
    ekey = kb.Current();
  }

  // 6. row pointers over the local rows (uint64)
  uint64_t *row_ptr = nullptr;
  MGB_CUDA(tmp.alloc(&row_ptr, g.local_rows + 1));
  {
    cub::TransformInputIterator<uint64_t, U32ToU64, const uint32_t *> it(indeg_local, U32ToU64());
    size_t bytes = 0;
    MGB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, bytes, it, row_ptr, g.local_rows, st));
    void *cub_tmp = nullptr;
    MGB_CUDA(tmp.alloc(reinterpret_cast<char **>(&cub_tmp), bytes));
    MGB_CUDA(cub::DeviceScan::ExclusiveSum(cub_tmp, bytes, it, row_ptr, g.local_rows, st));
    MGB_CUDA(cudaMemcpyAsync(row_ptr + g.local_rows, &g.local_edges, sizeof(uint64_t), cudaMemcpyHostToDevice, st));
  }

  // 7. heavy class: CSC prefix + segments
  if (g.n_heavy) {
    MGB_CUDA(cudaMemcpyAsync(&g.heavy_edges, row_ptr + g.n_heavy, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    MGB_CUDA(cudaStreamSynchronize(st));
    if (!getenv("MGB200_SEGMENT_EDGES")) {
      // one warp per segment: aim for >= 8 segments per resident warp (64 warps/SM) so the tail is short
      // when a partition holds few heavy edges (multi-GPU), capped at 4096 edges
      const uint64_t resident_warps = static_cast<uint64_t>(g.sm_count) * 64;
      uint64_t seg = g.heavy_edges / (resident_warps * 8);
      seg = (seg / 256) * 256;
      g.segment_edges = static_cast<uint32_t>(std::min<uint64_t>(4096, std::max<uint64_t>(256, seg)));
    }
    MGB_CUDA(keep_alloc(g, &g.heavy_ptr, g.n_heavy + 1));
    MGB_CUDA(cudaMemcpyAsync(g.heavy_ptr, row_ptr, (g.n_heavy + 1) * sizeof(uint64_t), cudaMemcpyDeviceToDevice, st));
    MGB_CUDA(keep_alloc(g, &g.heavy_idx, g.heavy_edges));
    low32_kernel<<<blocks_for(g.heavy_edges, g.sm_count), kThreads, 0, st>>>(g.heavy_edges, ekey, idx_flags_heavy,
                                                                                   g.heavy_idx);
    if (weighted) {  // rows are sorted, heavy rows first: their weights are the prefix of the sorted weights
      MGB_CUDA(keep_alloc(g, &g.heavy_w, g.heavy_edges));
      MGB_CUDA(cudaMemcpyAsync(g.heavy_w, eval, g.heavy_edges * sizeof(double), cudaMemcpyDeviceToDevice, st));
    }
    MGB_CUDA(keep_alloc(g, &g.seg_first, g.n_heavy + 1));
    {
      cub::TransformInputIterator<uint64_t, SegCount, const uint32_t *> it(indeg_local, SegCount{g.segment_edges});
      size_t bytes = 0;
      MGB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, bytes, it, g.seg_first, g.n_heavy, st));
      void *cub_tmp = nullptr;
      MGB_CUDA(tmp.alloc(reinterpret_cast<char **>(&cub_tmp), bytes));
      MGB_CUDA(cub::DeviceScan::ExclusiveSum(cub_tmp, bytes, it, g.seg_first, g.n_heavy, st));
    }
    // total = seg_first[n_heavy-1] + segs(last row)
    uint64_t last_first = 0;
    uint32_t last_deg = 0;
    MGB_CUDA(cudaMemcpyAsync(&last_first, g.seg_first + g.n_heavy - 1, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    MGB_CUDA(cudaMemcpyAsync(&last_deg, indeg_local + g.n_heavy - 1, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    MGB_CUDA(cudaStreamSynchronize(st));
    g.n_seg = last_first + (static_cast<uint64_t>(last_deg) + g.segment_edges - 1) / g.segment_edges;
    MGB_CUDA(cudaMemcpyAsync(g.seg_first + g.n_heavy, &g.n_seg, sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    MGB_CUDA(keep_alloc(g, &g.seg_row, g.n_seg));
    MGB_CUDA(keep_alloc(g, &g.seg_begin, g.n_seg));
    MGB_CUDA(keep_alloc(g, &g.seg_partial, g.n_seg));
    MGB_CUDA(keep_alloc(g, &g.heavy_sums, g.n_heavy));
    segment_fill_kernel<<<blocks_for(g.n_heavy * 32, g.sm_count), kThreads, 0, st>>>(
        g.n_heavy, g.heavy_ptr, g.seg_first, g.segment_edges, g.seg_row, g.seg_begin);
  }

  // 8. SELL class
  if (g.n_sell) {
    g.n_slices = (g.n_sell + kSliceRows - 1) / kSliceRows;
    uint64_t *width = nullptr;
    MGB_CUDA(tmp.alloc(&width, g.n_slices));
    slice_width_kernel<<<blocks_for(g.n_slices, g.sm_count), kThreads, 0, st>>>(g.n_slices, indeg_local, g.n_heavy,
                                                                               width);
    MGB_CUDA(keep_alloc(g, &g.sell_colbase, g.n_slices + 1));
    {
      size_t bytes = 0;
      MGB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, bytes, width, g.sell_colbase, g.n_slices, st));
      void *cub_tmp = nullptr;
      MGB_CUDA(tmp.alloc(reinterpret_cast<char **>(&cub_tmp), bytes));
      MGB_CUDA(cub::DeviceScan::ExclusiveSum(cub_tmp, bytes, width, g.sell_colbase, g.n_slices, st));
    }
    uint64_t last_base = 0, last_width = 0;
    MGB_CUDA(cudaMemcpyAsync(&last_base, g.sell_colbase + g.n_slices - 1, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    MGB_CUDA(cudaMemcpyAsync(&last_width, width + g.n_slices - 1, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    MGB_CUDA(cudaStreamSynchronize(st));
    const uint64_t total_cols = last_base + last_width;
    MGB_CUDA(cudaMemcpyAsync(g.sell_colbase + g.n_slices, &total_cols, sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    g.sell_entries = total_cols * kSliceRows;
    MGB_CUDA(keep_alloc(g, &g.sell_idx, g.sell_entries));
    if (weighted) MGB_CUDA(keep_alloc(g, &g.sell_w, g.sell_entries));
    sell_fill_kernel<<<blocks_for(g.n_slices * 32, g.sm_count), kThreads, 0, st>>>(
        g.n_slices, g.n_heavy, g.n_heavy + g.n_sell, row_ptr, ekey, g.sell_colbase, static_cast<uint32_t>(n),
        idx_flags, g.sell_idx, eval, g.sell_w);
    MGB_CUDA(keep_alloc(g, &g.sell_sums, g.n_sell));
    g.sell_items = env_u32("MGB200_SELL_ITEMS", static_cast<uint32_t>(g.sm_count) * 32u);
    MGB_CUDA(keep_alloc(g, &g.sell_item_begin, static_cast<uint64_t>(g.sell_items) + 1));
    sell_items_kernel<<<(g.sell_items + 1 + kThreads - 1) / kThreads, kThreads, 0, st>>>(
        g.sell_items, g.n_slices, g.sell_colbase, total_cols, 0, g.sell_item_begin);
    // Work items of sell_rows_kernel (contiguous slice runs of ~equal cost = columns + kSliceCost per slice).
    // Measured on scale-26 partitions (profiles/r02_sell_schedule.md): with >= 64 slices per resident warp the ticket
    // queue over ~16 items per warp wins (whole graph 2.12 vs 2.51 ms), below that every extra run start costs more
    // than the balance gains and ONE (or two) contiguous runs per warp, dealt statically, are fastest
    // (1/8 partition: 0.37 vs 0.56 ms; 1/4: 0.68 vs 0.77 ms).
    const uint64_t kSliceCost = env_u32_zero("MGB200_SLICE_COST", 8);
    const uint64_t resident_warps = static_cast<uint64_t>(g.sm_count) * 32u;  // 4 CTAs x 8 warps per SM
    const uint64_t per_warp = g.n_slices / resident_warps;
    g.sell_static = g.tun.sell_mode >= 0 ? g.tun.sell_mode == 1 : per_warp < 64;
    const uint64_t items_default = !g.sell_static ? resident_warps * 16 : (per_warp < 32 ? resident_warps : resident_warps * 2);
    g.sell_work = static_cast<uint32_t>(std::min<uint64_t>(
        g.n_slices, env_u32("MGB200_SELL_WORK_ITEMS", static_cast<uint32_t>(items_default))));
    MGB_CUDA(keep_alloc(g, &g.sell_work_begin, static_cast<uint64_t>(g.sell_work) + 1));
    sell_items_kernel<<<(g.sell_work + 1 + kThreads - 1) / kThreads, kThreads, 0, st>>>(
        g.sell_work, g.n_slices, g.sell_colbase, total_cols, kSliceCost, g.sell_work_begin);
    MGB_CUDA(keep_alloc(g, &g.sell_work_items, g.sell_work));
    work_item_kernel<<<(g.sell_work + kThreads - 1) / kThreads, kThreads, 0, st>>>(g.sell_work, g.sell_work_begin,
                                                                                  g.sell_colbase, g.sell_work_items);
  }
  note_mem(g);
  MGB_CUDA(cudaGetLastError());
  MGB_CUDA(cudaEventRecord(g.ev[1], st));
  MGB_CUDA(cudaStreamSynchronize(st));
  float ms = 0.f;
  MGB_CUDA(cudaEventElapsedTime(&ms, g.ev[0], g.ev[1]));
  g.build_ms = ms;
  return MGB200_OK;
}

}  // namespace mgb200
