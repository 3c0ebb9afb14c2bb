// memgraph_b200/csrc/pagerank_kernels.cu -- the power iteration as hand-written sm_100a kernels.
//
// What is computed (reference: mage/cpp/pagerank_module/algorithm/pagerank.cpp):
//   r_{k+1}[v] = (1-d)/N + d * sum_{(u->v) in E} r_k[u] / outdeg(u)          :86-96, :104-112, :221-226
//   continue iff k+1 != max_iterations and max_v |r_{k+1}[v] - r_k[v]| > eps  :138-150
//   result = r_K / sum(r_K)                                                   :156-161
// The reference pushes along source-ordered edges into per-thread N-vectors; here the same sum is
// PULLED per destination row from contrib[u] = r_k[u]/outdeg(u), which is computed once per vertex
// with an IEEE division (bit-identical to the reference's per-edge quotient).  Only the order of
// the additions inside a row differs from the reference (ascending source label here).
//
// Roofline: HBM-bound sparse gather, no tensor cores.  Algorithmic bytes per iteration
// 12*E + 24*N (SURVEY 8d).  Per edge: one coalesced 4-byte index read (streamed, evict-first) and
// one 8-byte gather of contrib[]; per row: rank RMW in place, out-degree read, contrib write.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "core.hpp"

namespace mgb200 {
namespace {

constexpr int kBlockThreads = 256;
constexpr int kWarpsPerBlock = kBlockThreads / 32;
constexpr unsigned kFull = 0xffffffffu;
#ifndef MGB_UNROLL
#define MGB_UNROLL 8   // heavy-row segments: gathers in flight per lane
#endif
constexpr int kUnroll = MGB_UNROLL;

// ---- small PTX helpers ---------------------------------------------------------------------------

// Streaming read of an index word: read once per iteration, keep it out of the way of the
// gathered vector in L1/L2 (ld.global.nc, no L1 allocation, L2 evict-first policy).
__device__ __forceinline__ uint64_t make_evict_first_policy() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
#ifndef MGB_IDX_HINT
#define MGB_IDX_HINT 1     // 1: index stream no L1 allocation + L2 evict_first, 0: plain read-only loads
#endif
#ifndef MGB_EPI_HINT
#define MGB_EPI_HINT 1     // 1: rank / out-degree / contrib_out traffic evict_first, 0: default policy
#endif
#ifndef MGB_GATHER_POLICY
#define MGB_GATHER_POLICY 1  // 0: plain ld.global.nc, 1: range(evict_last hot prefix, evict_first tail), 2: all evict_last
#endif
__device__ __forceinline__ uint32_t ld_index(const uint32_t *p, uint64_t pol) {
#if MGB_IDX_HINT
  uint32_t v;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
  return v;
#else
  (void)pol;
  return __ldg(p);
#endif
}
// Gather of one contribution: read-only path; reuse across CTAs lives in L2.
__device__ __forceinline__ double ld_contrib(const double *p, uint64_t pol) {
#if MGB_GATHER_POLICY
  double v;
  asm volatile("ld.global.nc.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(pol));
  return v;
#else
  (void)pol;
  return __ldg(p);
#endif
}
// L2 / L1 residency plan (measured, scripts/l2_bench.cu, scripts/gather_bench.cu): random gathers run at
// ~275 G/s while the gathered set fits ~64 MiB of L2 and at ~49 G/s from HBM; an SM issues one L2 request per
// cycle, so every L1 hit is a request saved, and with plain LRU the 86 % of gathers that miss evict the hottest
// lines (14 % L1 hit rate).  Labels are sorted by degree, so "hot" is a property of the label alone:
//   one partition : the hot vertices are the PREFIX of contrib[]            -> local index = label
//   P partitions  : sorted positions are dealt round-robin, every partition's label range starts with ITS
//                   hottest vertices                                          -> local index = label - start[owner]
// local < l2_hot: L2 evict_last, else evict_first (like every other stream: indices, rank, out-degree, contrib_out);
// local < l1_hot: may allocate in L1 (evict_last), else bypasses it.
struct GatherWindow {
  uint32_t hot_bytes;    // single partition: primary (evict_last) span of the range policy, from contrib_in
  uint32_t total_bytes;  // whole vector (secondary span: evict_first)
  uint32_t l1_hot;       // local indices below this may allocate in L1
  uint32_t l2_hot;       // local indices below this are L2 evict_last (multi-partition form)
  uint32_t world;        // number of partitions
  uint32_t table_n;      // labels held in the shared-memory hot table (0 = none); P partitions: table_n / P per owner
  uint32_t path;         // kernel instantiation: kPathRange / kPathLookup / kPathFlags (below)
  uint32_t start[kMaxPeers];  // first global label of every partition
};
constexpr uint32_t kL1Plain = kNoL1Hints;  // GatherWindow::l1_hot value meaning "no L1 hints"
// How a gather learns whether its source is hot:
//   kPathRange  one partition: a createpolicy.range over the prefix decides L2, `label < l1_hot` decides L1;
//   kPathLookup P partitions, plain indices: owner found by <= 7 compare/selects per gather (costs 4.7 %,
//               profiles/r01_multi_gpu.md), kept for graphs with >= 2^30 vertices and as the A/B baseline;
//   kPathFlags  the hotness was computed ONCE at build time and rides in bits 31/30 of the stored index
//               (graph_build.cu IndexFlags): two bit tests per gather, no per-partition table in the kernel.
constexpr int kPathRange = 0, kPathLookup = 1, kPathFlags = 2;
struct GatherPolicy {
  uint64_t hot;   // single partition: the range policy; else fractional evict_last
  uint64_t cold;  // fractional evict_first
};
__device__ __forceinline__ GatherPolicy make_gather_policy(const double *contrib_in, const GatherWindow &w) {
  GatherPolicy p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p.cold));
  if (w.path == kPathRange) {  // single partition, or partition-unaware legacy mode: one range policy over the prefix
    asm volatile("createpolicy.range.global.L2::evict_last.L2::evict_first.b64 %0, [%1], %2, %3;"
                 : "=l"(p.hot)
                 : "l"(contrib_in), "r"(w.hot_bytes), "r"(w.total_bytes));
  } else {
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p.hot));
  }
  return p;
}
// The hottest labels live in shared memory (kTable): an L2 request is what the SMs run out of (one per SM per clock,
// r01), and the degree-sorted labelling makes "hottest" a prefix -- 21 % of all gathers of RMAT-26 go to the first 16 K
// labels, 27 % to the first 28 K (profiles/r01_topk_share.txt).  One partition: slot = label (label < table_n).  Several
// partitions: the build stored the slot in the index itself, code 01 in bits 31/30 (graph_build.cu IndexFlags).
template <int kPath, bool kSelectL2 = true, bool kTable = false>
__device__ __forceinline__ double ld_contrib_at(const double *base, uint32_t src, const GatherPolicy &gp,
                                                const GatherWindow &w, const double *table = nullptr) {
  if (kTable) {
    if (kPath == kPathFlags) {
      if ((src >> 30) == 1u) return table[src & kIdxLabelMask];
    } else if (src < w.table_n) {
      return table[src];
    }
  }
  uint32_t label = src;
  uint64_t pol = gp.hot;
  bool l1_hot;
  if (kPath == kPathFlags) {
    label = src & kIdxLabelMask;
    if (kSelectL2) pol = (src & kIdxL2Hot) ? gp.hot : gp.cold;  // else: every gather of this kernel evict_last
    l1_hot = (src & kIdxL1Hot) != 0;
  } else if (kPath == kPathLookup) {
    uint32_t s0 = 0;
#pragma unroll
    for (int q = 1; q < kMaxPeers; ++q)
      if (q < static_cast<int>(w.world) && src >= w.start[q]) s0 = w.start[q];
    const uint32_t local = src - s0;
    pol = local < w.l2_hot ? gp.hot : gp.cold;
    l1_hot = local < w.l1_hot;
  } else {
    l1_hot = src < w.l1_hot;
  }
  const double *p = base + label;
  double v;
  if (w.l1_hot == kL1Plain) {  // default L1 policy for every gather
    asm volatile("ld.global.nc.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(pol));
  } else if (l1_hot) {
    asm volatile("ld.global.nc.L1::evict_last.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(pol));
  } else {
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(pol));
  }
  return v;
}
__device__ __forceinline__ double ld_stream_f64(const double *p, uint64_t pol) {
#if MGB_EPI_HINT
  double v;
  asm volatile("ld.global.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(pol));
  return v;
#else
  (void)pol;
  return *p;
#endif
}
__device__ __forceinline__ void st_stream_f64(double *p, double v, uint64_t pol) {
#if MGB_EPI_HINT
  asm volatile("st.global.L2::cache_hint.f64 [%0], %1, %2;" ::"l"(p), "d"(v), "l"(pol) : "memory");
#else
  (void)pol;
  *p = v;
#endif
}

__device__ __forceinline__ int ld_volatile_int(const int *p) { return *reinterpret_cast<const volatile int *>(p); }

__device__ __forceinline__ void st_release_sys_u64(unsigned long long *p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed_sys_u64(unsigned long long *p, unsigned long long v) {
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long *p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long global_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// ---- mbarrier / TMA bulk-copy helpers (hot table fill here, index ring in sell_stream.cuh) ---------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
  }
}
// TMA bulk copy global -> shared (1-D, bytes multiple of 16), completion counted on the mbarrier.
__device__ __forceinline__ void tma_load_1d(uint32_t dst_smem, const void *src, uint32_t bytes, uint32_t bar,
                                            uint64_t pol) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
      ::"r"(dst_smem), "l"(src), "r"(bytes), "r"(bar), "l"(pol)
      : "memory");
}

// ---- per-row epilogue ------------------------------------------------------------------------------

struct RowEpilogue {
  double base;     // (1 - d) / N
  double damping;  // d
  double *rank;            // [local_rows]
  const uint32_t *outdeg;  // [n] by global label
  RowMap map;              // local row -> global label
  double *contrib_out[kMaxPeers];  // this iteration's output buffer on every partition (self included)
  int world;
  int self;                // this partition
  const uint8_t *need;     // [local_rows] bit q: partition q gathers this row's contribution; nullptr = everyone
  uint32_t store_mask;     // bit q: the epilogue stores into partition q's buffer (all ones; self only in the lone-partition profiling mode)
};

// max over the block of the rows' |delta| (callers start from -1.0 = "none seen"; NaN deltas never replace it, like
// the reference's `abs(...) > eps` is false for NaN) -> one atomicMax on bits + 1, so that 0 keeps meaning "none".
__device__ __forceinline__ void block_max_to_state(double local_max, IterState *state) {
  __shared__ double warp_max[kWarpsPerBlock];
  for (int o = 16; o > 0; o >>= 1) {
    const double other = __shfl_xor_sync(kFull, local_max, o);
    if (other > local_max) local_max = other;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) warp_max[warp] = local_max;
  __syncthreads();
  if (threadIdx.x == 0) {
    double m = warp_max[0];
    for (int w = 1; w < kWarpsPerBlock; ++w)
      if (warp_max[w] > m) m = warp_max[w];
    if (m >= 0.0) atomicMax(&state->diff_bits, static_cast<unsigned long long>(__double_as_longlong(m)) + 1ull);
  }
}

// ---- init -------------------------------------------------------------------------------------------

// Zero in-degree rows never receive anything: their rank is (1-d)/N after the first iteration and stays
// there, and their contribution is (that rank)/outdeg.  Every partition knows every partition's zero-row
// label ranges (graph_build.cu), so all of it is set up locally -- no kernel in the iteration loop, no
// NVLink traffic: init writes rank = (1-d)/N for the own zero rows, contrib[0] = (1/N)/outdeg for every
// label and contrib[1] = ((1-d)/N)/outdeg for all zero-row labels; zero_refresh_kernel rewrites contrib[0]
// for the zero-row labels during iteration 1.  Their one-time delta |(1-d)/N - 1/N| enters iteration 0's
// L-infinity test through iter_end_kernel (extra_diff_bits).
struct ZeroRanges {
  uint64_t lo[kMaxPeers];
  uint64_t hi[kMaxPeers];
  int world;
};

// rank = 1/N (:199); contrib[0] = (1/N)/outdeg for EVERY label (each partition fills its own full
// copy, so iteration 0 needs no exchange); pad slots = 0.
__global__ void __launch_bounds__(kBlockThreads) init_kernel(uint64_t n, uint64_t local_rows, uint64_t local_nonzero,
                                                             double zero_rank, double *rank, const uint32_t *outdeg,
                                                             double *contrib0, double *contrib1, ZeroRanges zr,
                                                             IterState *state) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  const uint64_t tid = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const double r0 = 1.0 / static_cast<double>(n);
  for (uint64_t i = tid; i < n; i += stride) {
    const uint32_t od = outdeg[i];
    if (od) contrib0[i] = __ddiv_rn(r0, static_cast<double>(od));
  }
  for (int q = 0; q < kMaxPeers; ++q) {
    if (q >= zr.world) break;
    for (uint64_t i = zr.lo[q] + tid; i < zr.hi[q]; i += stride) {
      const uint32_t od = outdeg[i];
      if (od) contrib1[i] = __ddiv_rn(zero_rank, static_cast<double>(od));
    }
  }
  for (uint64_t i = tid; i < local_rows; i += stride) rank[i] = i < local_nonzero ? r0 : zero_rank;
  if (tid == 0) {
    contrib0[n] = 0.0;
    contrib1[n] = 0.0;
    state->diff_bits = 0ull;
    state->iterations = 0ull;
    state->last_diff = 0.0;
    state->local_sum = 0.0;
    state->rank_sum = 0.0;
    state->done = 0;
    state->error = 0;
    state->abort_req = 0;
    state->aborted = 0;
  }
}

// iteration 1 only: contrib[0] of the zero-row labels moves from (1/N)/outdeg to ((1-d)/N)/outdeg
__global__ void __launch_bounds__(kBlockThreads) zero_refresh_kernel(double zero_rank, const uint32_t *outdeg,
                                                                     double *contrib0, ZeroRanges zr,
                                                                     IterState *state) {
  if (ld_volatile_int(&state->done)) return;
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  const uint64_t tid = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const uint64_t pol = make_evict_first_policy();
  for (int q = 0; q < kMaxPeers; ++q) {
    if (q >= zr.world) break;
    for (uint64_t i = zr.lo[q] + tid; i < zr.hi[q]; i += stride) {
      const uint32_t od = ld_index(outdeg + i, pol);
      if (od) st_stream_f64(contrib0 + i, __ddiv_rn(zero_rank, static_cast<double>(od)), pol);
    }
  }
}

// ---- SELL-32 rows: one lane per row, coalesced column-major index reads -----------------------------

// Row epilogue as a separate, perfectly coalesced elementwise pass over rows [first_row, end_row) whose gathered sums
// lie in sums[r - first_row]; used for the SELL class (its own kernel on the side stream) and for the heavy rows
// (after heavy_rowsum_kernel).  History: fused into the gather kernels it cost 2.9 ms of 5.2 ms at scale-26
// (profiles/r01_attribution.md): the rank and out-degree loads, the FP64 division and the stores sit at the end of
// every slice's dependency chain and drain the warp's memory pipeline once per ~24 columns.  The first split version
// walked one row per thread per trip through two dependent DRAM round trips (sums -> rank / out-degree) with
// asm-volatile loads, which pin the issue order; this one takes kEpiRows rows per trip and issues every load of the
// trip before the first use, as plain streaming loads (ld/st.global.cs) the compiler may hoist
// (profiles/r02_epilogue.md: 0.28 -> 0.19 ms at scale-26, 0.26 -> 0.025 ms on a 1/8 partition).
//
//   rank_next = base + d * acc as two separately rounded operations, like the reference's
//   `rank_next[i] += damping_factor * block[i]` compiled without FMA contraction (:109-111);
//   contribution = rank_next / outdeg with an IEEE division (:93), once per vertex instead of once per edge.
constexpr int kEpiRows = 4;
__global__ void __launch_bounds__(kBlockThreads) row_epilogue_kernel(uint64_t first_row, uint64_t end_row,
                                                                     const double *sums, IterState *state,
                                                                     const RowEpilogue ep) {
  if (ld_volatile_int(&state->done)) return;
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  double local_max = -1.0;
  for (uint64_t r0 = first_row + static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r0 < end_row;
       r0 += stride * kEpiRows) {
    double acc[kEpiRows], prev[kEpiRows];
    uint32_t od[kEpiRows], need[kEpiRows];
    uint64_t label[kEpiRows];
#pragma unroll
    for (int j = 0; j < kEpiRows; ++j) {
      const uint64_t r = r0 + j * stride;
      const bool ok = r < end_row;
      label[j] = ep.map.label_of_local(ok ? r : first_row);
      acc[j] = ok ? __ldcs(sums + (r - first_row)) : 0.0;
      prev[j] = ok ? __ldcs(ep.rank + r) : 0.0;
      od[j] = ok ? __ldcs(ep.outdeg + label[j]) : 0u;
      // push only to the partitions that have an in-edge from this vertex (graph_build.cu need_mask_kernel)
      need[j] = (ok && ep.need) ? (static_cast<uint32_t>(__ldcs(ep.need + r)) | (1u << ep.self)) : 0xFFu;
    }
#pragma unroll
    for (int j = 0; j < kEpiRows; ++j) {
      const uint64_t r = r0 + j * stride;
      if (r < end_row) {
        const double next = __dadd_rn(ep.base, __dmul_rn(ep.damping, acc[j]));
        __stcs(ep.rank + r, next);
        // A vertex without out-edges is never a gather source, so its contribution is never read: no division, no
        // store, and -- what matters across GPUs -- no NVLink push.  Labels are sorted by (in-degree, out-degree)
        // descending, so these vertices are the contiguous tail of every in-degree class: whole warps skip.
        if (od[j] != 0) {
          const double c = __ddiv_rn(next, static_cast<double>(od[j]));
          const uint32_t to = need[j] & ep.store_mask;
#pragma unroll
          for (int q = 0; q < kMaxPeers; ++q)
            if (q < ep.world && ((to >> q) & 1u)) __stcs(ep.contrib_out[q] + label[j], c);  // q != self: NVLink store
        }
        const double d = fabs(next - prev[j]);
        if (d > local_max) local_max = d;  // NaN never replaces it, like the reference's `abs(...) > eps`
      }
    }
  }
  block_max_to_state(local_max, state);
}

struct SellArgs {
  const uint64_t *colbase;
  const uint32_t *idx;
  const double *w;       // edge weights parallel to idx (weighted variants only, else nullptr)
  const WorkItem *work;  // [n_work] contiguous slice runs of ~equal cost, descending width (graph_build.cu)
  uint32_t n_work;
  WorkQueue *queue;      // ticket counter of this launch (rewound by the last CTA to leave)
  uint32_t mode;         // 0 tickets in list order (default), 1 static round-robin (A/B baseline)
  uint64_t first_row;    // local row of slice 0, lane 0
  uint64_t end_row;      // first local row past the SELL class
  const double *contrib_in;
  GatherWindow window;
  IterState *state;
  double *sums;  // [n_sell] per-row sums of gathered contributions (consumed by row_epilogue_kernel)
};

// Tunables (compile-time; sweeps: profiles/r02_sell_variants.md)
#ifndef MGB_SELL_UNROLL
#define MGB_SELL_UNROLL 8      // columns per batch (gathers in flight per lane)
#endif
#ifndef MGB_SELL_MIN_BLOCKS
#define MGB_SELL_MIN_BLOCKS 4  // resident CTAs/SM requested from ptxas (register cap = 65536 / (256 * this))
#endif
constexpr int kSellUnroll = MGB_SELL_UNROLL;

// SELL-32 rows: one lane per row, a warp walks a WORK ITEM = a contiguous run of slices, i.e. one contiguous span of
// sell_idx, as ONE stream of columns: index batch k+1 is requested before the gathers of batch k are consumed, across
// slice boundaries -- a boundary only decides where the running sum is stored.  (The first version restarted its
// pipeline at every slice: an exposed round trip per slice, 22 per warp on a 1/8 partition, and every run of narrow
// slices degenerated to `width` gathers in flight.)  Items have about equal cost and are handed out in descending-width
// order through a ticket counter, so a warp that drew cheap work (or sits on an SM with the longer way to L2) simply takes
// more; the queue is software-pipelined (record of item i+1 and ticket of item i+2 in flight while item i is gathered).
// mode 1 deals the items round-robin instead (no atomics) -- the A/B baseline of profiles/r02_sell_tickets.md.
template <int kPath, bool kTable, bool kWeighted = false>
__device__ __forceinline__ void sell_walk(const SellArgs &a, const double *table) {
  const int lane = threadIdx.x & 31;
  const int warps_per_block = static_cast<int>(blockDim.x >> 5);
  const uint64_t pol = make_evict_first_policy();
  const GatherPolicy gpol = make_gather_policy(a.contrib_in, a.window);
  unsigned long long static_next = static_cast<unsigned long long>(blockIdx.x) * warps_per_block + (threadIdx.x >> 5);
  const unsigned long long warps_total = static_cast<unsigned long long>(gridDim.x) * warps_per_block;
  auto draw = [&]() -> unsigned long long {
    if (a.mode == 1) {
      const unsigned long long t = static_next;
      static_next += warps_total;
      return t;
    }
    return lane == 0 ? atomicAdd(&a.queue->ticket, 1ull) : 0ull;
  };
  // lanes 0..3 fetch the four words of an item record (one 32-byte sector)
  auto fetch = [&](uint32_t t) -> uint64_t {
    return (lane < 4 && t < a.n_work) ? reinterpret_cast<const uint64_t *>(a.work + t)[lane] : 0ull;
  };
  uint32_t t_cur = static_cast<uint32_t>(min(__shfl_sync(kFull, draw(), 0), static_cast<unsigned long long>(a.n_work)));
  unsigned long long pending = draw();  // ticket of the item after the first
  uint64_t rec = fetch(t_cur);
  while (t_cur < a.n_work) {
    const uint64_t s_begin = __shfl_sync(kFull, rec, 0), s_end = __shfl_sync(kFull, rec, 1);
    const uint64_t col_begin = __shfl_sync(kFull, rec, 2), col_end = __shfl_sync(kFull, rec, 3);
    // next item: its ticket was drawn one item ago; request its record now, and draw the ticket after it
    t_cur = static_cast<uint32_t>(min(__shfl_sync(kFull, pending, 0), static_cast<unsigned long long>(a.n_work)));
    rec = fetch(t_cur);
    pending = draw();
    if (s_begin >= s_end) continue;
    // slice ends: lane l holds colbase[block + l + 1] for a block of 32 slices (one coalesced load per 32 slices)
    uint64_t s = s_begin, s_block = s_begin;
    uint64_t ends = (s_block + lane + 1 <= s_end) ? a.colbase[s_block + lane + 1] : col_end;
    uint64_t slice_end = __shfl_sync(kFull, ends, 0);
    const uint32_t *p = a.idx + col_begin * kSliceRows + lane;  // column c of the span: p[(c - col_begin) * 32]
    const uint64_t ncols = col_end - col_begin;
    double acc = 0.0;
    uint32_t nxt[kSellUnroll];
#pragma unroll
    for (int j = 0; j < kSellUnroll; ++j)
      if (static_cast<uint64_t>(j) < ncols) nxt[j] = ld_index(p + static_cast<size_t>(j) * kSliceRows, pol);
    for (uint64_t k = 0; k < ncols; k += kSellUnroll) {
      uint32_t src[kSellUnroll];
      double v[kSellUnroll];
#pragma unroll
      for (int j = 0; j < kSellUnroll; ++j) src[j] = nxt[j];
#pragma unroll
      for (int j = 0; j < kSellUnroll; ++j)  // the next batch of indices travels while this batch is gathered
        if (k + kSellUnroll + j < ncols) nxt[j] = ld_index(p + static_cast<size_t>(k + kSellUnroll + j) * kSliceRows, pol);
      double wv[kSellUnroll];
      if (kWeighted) {
        const double *pw = a.w + col_begin * kSliceRows + lane;
#pragma unroll
        for (int j = 0; j < kSellUnroll; ++j)
          if (k + j < ncols) wv[j] = ld_stream_f64(pw + static_cast<size_t>(k + j) * kSliceRows, pol);
      }
#pragma unroll
      for (int j = 0; j < kSellUnroll; ++j)
        if (k + j < ncols) v[j] = ld_contrib_at<kPath, true, kTable>(a.contrib_in, src[j], gpol, a.window, table);
      if (kWeighted) {
#pragma unroll
        for (int j = 0; j < kSellUnroll; ++j)
          if (k + j < ncols) v[j] = __dmul_rn(wv[j], v[j]);
      }
#pragma unroll
      for (int j = 0; j < kSellUnroll; ++j) {
        if (k + j < ncols) {
          acc += v[j];  // fixed order inside a row: ascending source label
          const uint64_t col_next = col_begin + k + j + 1;
          while (col_next == slice_end && s < s_end) {  // (a zero-width slice would store 0 for its rows right here)
            const uint64_t row = a.first_row + s * kSliceRows + lane;
            if (row < a.end_row) a.sums[row - a.first_row] = acc;  // epilogue runs as its own elementwise kernel
            acc = 0.0;
            ++s;
            if (s < s_end) {
              if (s - s_block == 32) {
                s_block = s;
                ends = (s_block + lane + 1 <= s_end) ? a.colbase[s_block + lane + 1] : col_end;
              }
              slice_end = __shfl_sync(kFull, ends, static_cast<int>(s - s_block));
            }
          }
        }
      }
    }
  }
  if (a.mode == 1) return;
  // the last CTA to leave rewinds the queue for the next launch (every ticket of this launch has been drawn by then)
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int left = atomicAdd(&a.queue->ctas_done, 1u);
    if (left == gridDim.x - 1) {
      a.queue->ticket = 0ull;
      a.queue->ctas_done = 0u;
      __threadfence();
    }
  }
}


template <int kPath>
__global__ void __launch_bounds__(kBlockThreads, MGB_SELL_MIN_BLOCKS) sell_rows_kernel(const SellArgs a) {
  if (ld_volatile_int(&a.state->done)) return;
  sell_walk<kPath, false>(a, nullptr);
}

// every gathered value multiplied by its edge weight (cuGraph-semantics variants, one partition); no hot table
template <int kPath>
__global__ void __launch_bounds__(kBlockThreads, MGB_SELL_MIN_BLOCKS) sell_rows_weighted_kernel(const SellArgs a) {
  if (ld_volatile_int(&a.state->done)) return;
  sell_walk<kPath, false, true>(a, nullptr);
}

// The same walk with the hot table: ONE 1024-thread CTA per SM (the same 32 warps as 4 x 256 threads) so that the SM
// holds one copy of the table; filled once per launch -- one partition: TMA bulk copies (cp.async.bulk, 32 KiB each,
// completion on an mbarrier, L2 evict-last) of the contiguous label prefix; several partitions: one window per owner,
// whose first label is only 8-byte aligned, so the threads load it cooperatively.
constexpr int kTableThreads = 1024;
template <int kPath>
__global__ void __launch_bounds__(kTableThreads, 1) sell_rows_table_kernel(const SellArgs a) {
  extern __shared__ __align__(128) unsigned char table_smem[];
  __shared__ __align__(8) unsigned long long fill_bar;
  if (ld_volatile_int(&a.state->done)) return;
  double *table = reinterpret_cast<double *>(table_smem);
  const uint32_t table_n = a.window.table_n;
  if (kPath == kPathFlags) {
    const uint32_t per = table_n / a.window.world;
    for (uint32_t q = 0; q < a.window.world; ++q)
      for (uint32_t i = threadIdx.x; i < per; i += blockDim.x)
        table[q * per + i] = __ldg(a.contrib_in + a.window.start[q] + i);
    __syncthreads();
  } else {
    const uint32_t bar = smem_u32(&fill_bar);
    if (threadIdx.x == 0) {
      mbar_init(bar, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
      uint64_t keep;
      asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(keep));
      const uint32_t bytes = table_n * static_cast<uint32_t>(sizeof(double));
      mbar_expect_tx(bar, bytes);
      for (uint32_t off = 0; off < bytes; off += 32768u)
        tma_load_1d(smem_u32(table_smem + off), reinterpret_cast<const unsigned char *>(a.contrib_in) + off,
                    min(32768u, bytes - off), bar, keep);
    }
    __syncthreads();  // the barrier is initialised before anyone waits on it
    mbar_wait(bar, 0);
  }
  sell_walk<kPath, true>(a, table);
}

#include "sell_stream.cuh"

// ---- heavy rows: one warp per fixed-size edge segment, then one warp per row ------------------------

struct HeavyArgs {
  const uint64_t *heavy_ptr;
  const uint32_t *heavy_idx;
  const double *heavy_w;  // edge weights parallel to heavy_idx (weighted variants only)
  const uint32_t *seg_row;
  const uint64_t *seg_begin;
  const uint64_t *seg_first;
  double *seg_partial;
  double *row_sums;  // [n_heavy]
  uint64_t n_seg;
  uint64_t n_heavy;
  uint32_t segment_edges;
  const double *contrib_in;
  GatherWindow window;
  IterState *state;
};

#ifndef MGB_HEAVY_MIN_BLOCKS
#define MGB_HEAVY_MIN_BLOCKS 8  // 32 registers: occupancy beats the 8-16 B of spill (measured, r01_multi_gpu.md)
#endif
#ifndef MGB_HEAVY_PREFETCH
#define MGB_HEAVY_PREFETCH 0    // 1: request the next batch of segment indices before consuming the current gathers
#endif
#ifndef MGB_HEAVY_FLAGS_L2
#define MGB_HEAVY_FLAGS_L2 1    // flagged indices: 1 = per-load L2 hot/cold selection, 0 = L1 flag only
#endif
template <int kPath, bool kWeighted = false>
__global__ void __launch_bounds__(kBlockThreads, MGB_HEAVY_MIN_BLOCKS) heavy_segments_kernel(const HeavyArgs a) {
  constexpr bool kSelL2 = MGB_HEAVY_FLAGS_L2 != 0;
  if (ld_volatile_int(&a.state->done)) return;
  const int lane = threadIdx.x & 31;
  const uint64_t warps_total = static_cast<uint64_t>(gridDim.x) * kWarpsPerBlock;
  const uint64_t warp0 = static_cast<uint64_t>(blockIdx.x) * kWarpsPerBlock + (threadIdx.x >> 5);
  const uint64_t pol = make_evict_first_policy();
  const GatherPolicy gpol = make_gather_policy(a.contrib_in, a.window);
  for (uint64_t g = warp0; g < a.n_seg; g += warps_total) {
    const uint32_t r = a.seg_row[g];
    const uint64_t e0 = a.seg_begin[g];
    const uint64_t row_end = a.heavy_ptr[r + 1];
    const uint64_t e1 = (e0 + a.segment_edges < row_end) ? e0 + a.segment_edges : row_end;
    double acc = 0.0;
    uint64_t e = e0 + lane;
#if MGB_HEAVY_PREFETCH
    // software pipeline like the SELL walk: the indices of batch k+1 are requested before the gathers of batch k are consumed
    uint32_t nxt[kUnroll];
    if (e + 32ull * (kUnroll - 1) < e1) {
#pragma unroll
      for (int j = 0; j < kUnroll; ++j) nxt[j] = ld_index(a.heavy_idx + e + 32ull * j, pol);
    }
#endif
    for (; e + 32ull * (kUnroll - 1) < e1; e += 32ull * kUnroll) {
      uint32_t src[kUnroll];
      double v[kUnroll];
#if MGB_HEAVY_PREFETCH
#pragma unroll
      for (int j = 0; j < kUnroll; ++j) src[j] = nxt[j];
      if (e + 32ull * kUnroll + 32ull * (kUnroll - 1) < e1) {
#pragma unroll
        for (int j = 0; j < kUnroll; ++j) nxt[j] = ld_index(a.heavy_idx + e + 32ull * kUnroll + 32ull * j, pol);
      }
#else
#pragma unroll
      for (int j = 0; j < kUnroll; ++j) src[j] = ld_index(a.heavy_idx + e + 32ull * j, pol);
#endif
#pragma unroll
      for (int j = 0; j < kUnroll; ++j) v[j] = ld_contrib_at<kPath, kSelL2>(a.contrib_in, src[j], gpol, a.window);
      if (kWeighted) {
#pragma unroll
        for (int j = 0; j < kUnroll; ++j) v[j] = __dmul_rn(ld_stream_f64(a.heavy_w + e + 32ull * j, pol), v[j]);
      }
#pragma unroll
      for (int j = 0; j < kUnroll; ++j) acc += v[j];
    }
    for (; e < e1; e += 32) {
      double v1 = ld_contrib_at<kPath, kSelL2>(a.contrib_in, ld_index(a.heavy_idx + e, pol), gpol, a.window);
      if (kWeighted) v1 = __dmul_rn(ld_stream_f64(a.heavy_w + e, pol), v1);
      acc += v1;
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(kFull, acc, o);  // fixed tree
    if (lane == 0) a.seg_partial[g] = acc;
  }
}

// per heavy row: segment partials summed in segment order (lane-strided, fixed shuffle tree) -> row_sums[r];
// the row epilogue then runs as row_epilogue_kernel over [0, n_heavy)
__global__ void __launch_bounds__(kBlockThreads) heavy_rowsum_kernel(const HeavyArgs a) {
  if (ld_volatile_int(&a.state->done)) return;
  const int lane = threadIdx.x & 31;
  const uint64_t warps_total = static_cast<uint64_t>(gridDim.x) * kWarpsPerBlock;
  const uint64_t warp0 = static_cast<uint64_t>(blockIdx.x) * kWarpsPerBlock + (threadIdx.x >> 5);
  for (uint64_t r = warp0; r < a.n_heavy; r += warps_total) {
    const uint64_t s0 = a.seg_first[r], s1 = a.seg_first[r + 1];
    double acc = 0.0;
    for (uint64_t s = s0 + lane; s < s1; s += 32) acc += a.seg_partial[s];
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(kFull, acc, o);
    if (lane == 0) a.row_sums[r] = acc;
  }
}

// ---- cross-partition barrier over the flag pages (P == 1: degenerates to nothing) ---------------------

struct BarrierArgs {
  IterState *state;
  FlagPage *mine;
  FlagPage *peer[kMaxPeers];  // peer[q] = partition q's flag page as mapped on THIS device (self included)
  int rank, world;
  unsigned long long timeout_ns;
};

// One warp.  Publishes `payload_bits`/`payload_sum` into slot [rank] of every partition's flag page,
// then waits until every partition has arrived at the same sequence number.  All stores issued by
// earlier kernels of this stream (including remote contribution stores) are ordered before the
// release store by the kernel boundary plus the system-scope fence.
__device__ __forceinline__ bool warp_barrier_exchange(const BarrierArgs &b, unsigned long long seq,
                                                      unsigned long long payload_bits, double payload_sum) {
  const int lane = threadIdx.x & 31;
  const int par = static_cast<int>(seq & 1ull);
  bool ok = true;
  if (lane < b.world) {
    FlagPage *dst = b.peer[lane];
    st_relaxed_sys_u64(&dst->diff_bits[par][b.rank], payload_bits);
    st_relaxed_sys_u64(reinterpret_cast<unsigned long long *>(&dst->rank_sum[par][b.rank]),
                       static_cast<unsigned long long>(__double_as_longlong(payload_sum)));
    __threadfence_system();
    st_release_sys_u64(&dst->arrive[b.rank], seq);
    const unsigned long long t0 = global_timer_ns();
    while (ld_acquire_sys_u64(&b.mine->arrive[lane]) < seq) {
      if (global_timer_ns() - t0 > b.timeout_ns) {
        ok = false;
        break;
      }
      __nanosleep(64);
    }
  }
  return __all_sync(kFull, ok);
}

struct IterEndArgs {
  BarrierArgs bar;
  unsigned long long max_iterations;
  double eps;
  unsigned long long extra_diff_bits;  // iteration 0: the zero rows' |(1-d)/N - 1/N| (same on every partition)
};

// End of one iteration: all-reduce(max) of the L-infinity delta across partitions, then the
// reference's CheckContinueIterate (:138-150) evaluated identically on every partition.
__global__ void iter_end_kernel(const IterEndArgs a) {
  IterState *st = a.bar.state;
  if (ld_volatile_int(&st->done)) return;
  const int lane = threadIdx.x & 31;
  unsigned long long bits = st->diff_bits;  // bits(max delta) + 1, 0 = none
  if (a.extra_diff_bits > bits) bits = a.extra_diff_bits;
  // Abort is a COLLECTIVE decision: a partition whose host asked to stop publishes kAbortBits instead of its delta;
  // the max-reduce hands it to everyone, so all partitions leave the loop in the same iteration and their barrier
  // counters stay in step (a partition that returned on its own would leave the others waiting, then run ahead).
  if (ld_volatile_int(&st->abort_req)) bits = kAbortBits;
  bool ok = true;
  unsigned long long seq = st->barrier_seq;
  if (a.bar.world > 1) {
    seq += 1;
    ok = warp_barrier_exchange(a.bar, seq, bits, 0.0);
    unsigned long long other = 0ull;
    if (lane < a.bar.world) other = a.bar.mine->diff_bits[seq & 1ull][lane];
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long t = __shfl_xor_sync(kFull, other, o);
      if (t > other) other = t;
    }
    bits = other;
  }
  if (lane == 0) {
    st->barrier_seq = seq;
    const bool abort_all = bits == kAbortBits;
    const bool any_delta = bits != 0ull && !abort_all;
    const double diff = any_delta ? __longlong_as_double(static_cast<long long>(bits - 1ull)) : 0.0;
    st->iterations += 1ull;
    st->last_diff = diff;
    // :138-150 -- continue iff the cap is not reached and SOME element has |delta| > eps (all-NaN: none has)
    const bool cont = (st->iterations != a.max_iterations) && any_delta && (diff > a.eps);
    st->diff_bits = 0ull;
    if (!ok) st->error = 1;
    if (abort_all) st->aborted = 1;
    if (!cont || !ok || abort_all) st->done = 1;
  }
}

__global__ void barrier_kernel(const BarrierArgs b) {
  if (b.world <= 1) return;
  IterState *st = b.state;
  const unsigned long long seq = st->barrier_seq + 1;
  const bool ok = warp_barrier_exchange(b, seq, 0ull, 0.0);
  if ((threadIdx.x & 31) == 0) {
    st->barrier_seq = seq;
    if (!ok) {
      st->error = 1;
      st->done = 1;
    }
  }
}

// ---- normalise (:156-161): deterministic two-stage sum, then divide ----------------------------------

__global__ void __launch_bounds__(kBlockThreads) partial_sum_kernel(const double *rank, uint64_t count,
                                                                    double *partials) {
  // block b sums the contiguous chunk [b*chunk, (b+1)*chunk): thread-strided partials, fixed tree.
  const uint64_t chunk = (count + gridDim.x - 1) / gridDim.x;
  const uint64_t lo = chunk * blockIdx.x;
  const uint64_t hi = (lo + chunk < count) ? lo + chunk : count;
  double acc = 0.0;
  for (uint64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) acc += rank[i];
  __shared__ double sm[kBlockThreads];
  sm[threadIdx.x] = acc;
  __syncthreads();
  for (int o = kBlockThreads / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) sm[threadIdx.x] += sm[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) partials[blockIdx.x] = sm[0];
}

__global__ void final_sum_kernel(const double *partials, int count, const BarrierArgs b) {
  __shared__ double sm[kSumBlocks];
  for (int i = threadIdx.x; i < kSumBlocks; i += blockDim.x) sm[i] = i < count ? partials[i] : 0.0;
  __syncthreads();
  for (int o = kSumBlocks / 2; o > 0; o >>= 1) {
    for (int i = threadIdx.x; i < o; i += blockDim.x) sm[i] += sm[i + o];
    __syncthreads();
  }
  IterState *st = b.state;
  if (threadIdx.x < 32) {
    const double local = sm[0];
    double total = local;
    bool ok = true;
    unsigned long long seq = st->barrier_seq;
    if (b.world > 1) {
      seq += 1;
      ok = warp_barrier_exchange(b, seq, 0ull, local);
      total = 0.0;
      for (int q = 0; q < b.world; ++q) total += b.mine->rank_sum[seq & 1ull][q];  // same order everywhere
    }
    if (threadIdx.x == 0) {
      st->barrier_seq = seq;
      st->local_sum = local;
      st->rank_sum = total;
      if (!ok) st->error = 1;
    }
  }
}

__global__ void __launch_bounds__(kBlockThreads) write_original_order_kernel(uint64_t n, const uint32_t *label_of,
                                                                             const double *rank,
                                                                             const IterState *state, double *out) {
  const double sum = state->rank_sum;
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (uint64_t v = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; v < n; v += stride)
    out[v] = __ddiv_rn(rank[label_of[v]], sum);  // :158-160
}

__global__ void __launch_bounds__(kBlockThreads) write_local_kernel(uint64_t local_rows, const double *rank,
                                                                    const uint32_t *local_vertex,
                                                                    const IterState *state, double *out,
                                                                    uint32_t *vertex_out) {
  const double sum = state->rank_sum;
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (uint64_t r = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < local_rows; r += stride) {
    out[r] = __ddiv_rn(rank[r], sum);
    if (vertex_out) vertex_out[r] = local_vertex[r];
  }
}

// ---- host-side launch helpers -------------------------------------------------------------------------

// a whole number of resident waves on the SMs; the occupancy query is made once per kernel per graph handle (it used
// to be ~6 driver calls per iteration, ADVICE r1)
int grid_for(const Graph &g, const void *kernel, int threads = kBlockThreads) {
  for (int i = 0; i < g.occ_cached; ++i)
    if (g.occ_kernel[i] == kernel) return g.sm_count * g.occ_blocks[i];
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, 0) != cudaSuccess || per_sm < 1) per_sm = 4;
  if (g.occ_cached < Graph::kOccSlots) {
    g.occ_kernel[g.occ_cached] = kernel;
    g.occ_blocks[g.occ_cached] = per_sm;
    ++g.occ_cached;
  }
  return g.sm_count * per_sm;
}

uint64_t ceil_div(uint64_t a, uint64_t b) { return (a + b - 1) / b; }

RowEpilogue make_epilogue(const Graph &g, uint64_t it, const IterateConfig &cfg) {
  RowEpilogue ep{};
  ep.base = (1.0 - cfg.damping) / static_cast<double>(g.n);
  ep.damping = cfg.damping;
  ep.rank = g.rank;
  ep.outdeg = g.outdeg_l;
  ep.map = g.map;
  ep.world = static_cast<int>(g.part_world);
  ep.self = static_cast<int>(g.part_rank);
  ep.need = reinterpret_cast<const uint8_t *>(g.need_mask);
  ep.store_mask = g.tun.lone_partition ? (1u << g.part_rank) : 0xFFFFFFFFu;
  const int out_parity = static_cast<int>((it + 1) & 1ull);
  for (int q = 0; q < kMaxPeers; ++q) ep.contrib_out[q] = q < ep.world ? g.peers.contrib[out_parity][q] : nullptr;
  return ep;
}

// Tunables are read from the environment once per graph (graph_build.cu, Graph::tun) -- no process-wide statics,
// so concurrent calls from several sessions never race on them.
GatherWindow make_window(const Graph &g) {
  const uint64_t hot_mb = g.tun.l2_hot_mb;
  const uint64_t total = std::min<uint64_t>((g.n + 1) * sizeof(double), 0xFFFFFF00ull);
  GatherWindow w{};
  w.total_bytes = static_cast<uint32_t>(total);
  w.hot_bytes = static_cast<uint32_t>(std::min<uint64_t>(total, hot_mb << 20));
  w.world = g.part_world;
  w.l1_hot = g.l1_hot_labels();
  w.l2_hot = g.l2_hot_labels();
  w.table_n = g.table_labels();
  // global-order labelling: "hot" is one label prefix on every partition -> the exact single-partition code
  w.path = g.idx_flagged ? kPathFlags
           : (g.tun.multi_aware && !g.map.global_order && (g.part_world > 1 || g.tun.force_multi_path)) ? kPathLookup
                                                                                                        : kPathRange;
  for (uint32_t q = 0; q < static_cast<uint32_t>(kMaxPeers); ++q)
    w.start[q] = q < g.part_world ? static_cast<uint32_t>(g.part_start[q]) : 0xFFFFFFFFu;
  return w;
}

BarrierArgs make_barrier(const Graph &g) {
  BarrierArgs b{};
  b.state = g.state;
  b.mine = g.flags();
  b.rank = static_cast<int>(g.part_rank);
  b.world = static_cast<int>(g.part_world);
  for (int q = 0; q < kMaxPeers; ++q) b.peer[q] = q < b.world ? g.peers.flags[q] : nullptr;
  if (g.tun.lone_partition) {  // profiling: a barrier of one over the own flag page
    b.rank = 0;
    b.world = 1;
    for (int q = 0; q < kMaxPeers; ++q) b.peer[q] = q == 0 ? g.flags() : nullptr;
  }
  b.timeout_ns = g.tun.barrier_timeout_ms * 1000000ull;
  return b;
}

}  // namespace

ZeroRanges make_zero_ranges(const Graph &g) {
  ZeroRanges zr{};
  zr.world = static_cast<int>(g.part_world);
  for (int q = 0; q < kMaxPeers; ++q) {
    zr.lo[q] = q < zr.world ? g.zero_lo[q] : 0;
    zr.hi[q] = q < zr.world ? g.zero_hi[q] : 0;
  }
  return zr;
}

// the rank of a zero in-degree row once the loop has run at least once ((1-d)/N); 1/N if it never runs
double zero_row_rank(const Graph &g, const IterateConfig &cfg) {
  return cfg.max_iterations == 0 ? 1.0 / static_cast<double>(g.n) : (1.0 - cfg.damping) / static_cast<double>(g.n);
}

// SELL rows: the plain kernel (4 x 256 threads per SM) or, with a hot table, one 1024-thread CTA per SM
int launch_sell_rows(Graph &g, const SellArgs &s) {
  const uint32_t table_n = s.window.table_n;
  if (s.w != nullptr) {
    void (*const fn)(SellArgs) = s.window.path == kPathFlags    ? sell_rows_weighted_kernel<kPathFlags>
                                 : s.window.path == kPathLookup ? sell_rows_weighted_kernel<kPathLookup>
                                                                : sell_rows_weighted_kernel<kPathRange>;
    const int grid = static_cast<int>(std::min(static_cast<uint64_t>(grid_for(g, reinterpret_cast<const void *>(fn))),
                                               ceil_div(g.sell_work, kWarpsPerBlock)));
    fn<<<grid, kBlockThreads, 0, g.stream>>>(s);
  } else if (table_n > 0 && s.window.path != kPathLookup) {
    void (*const fn)(SellArgs) = s.window.path == kPathFlags ? sell_rows_table_kernel<kPathFlags> : sell_rows_table_kernel<kPathRange>;
    const int bytes = static_cast<int>(table_n * sizeof(double));
    if (g.table_attr_bytes[s.window.path == kPathFlags] < bytes) {
      MGB_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
      g.table_attr_bytes[s.window.path == kPathFlags] = bytes;
    }
    const int grid = static_cast<int>(std::min<uint64_t>(g.sm_count, ceil_div(g.sell_work, kTableThreads / 32)));
    fn<<<grid, kTableThreads, bytes, g.stream>>>(s);
  } else {
    void (*const sell_fn)(SellArgs) = s.window.path == kPathFlags    ? sell_rows_kernel<kPathFlags>
                                      : s.window.path == kPathLookup ? sell_rows_kernel<kPathLookup>
                                                                     : sell_rows_kernel<kPathRange>;
    const int grid = static_cast<int>(std::min(
        static_cast<uint64_t>(grid_for(g, reinterpret_cast<const void *>(sell_fn))), ceil_div(g.sell_work, kWarpsPerBlock)));
    sell_fn<<<grid, kBlockThreads, 0, g.stream>>>(s);
  }
  MGB_CUDA(cudaGetLastError());
  return MGB200_OK;
}

int launch_init(Graph &g, const IterateConfig &cfg) {
  MGB_CUDA(cudaSetDevice(g.device));
  const int grid = grid_for(g, reinterpret_cast<const void *>(init_kernel));
  init_kernel<<<grid, kBlockThreads, 0, g.stream>>>(g.n, g.local_rows, g.n_heavy + g.n_sell, zero_row_rank(g, cfg),
                                                     g.rank, g.outdeg_l, g.contrib(0), g.contrib(1),
                                                     make_zero_ranges(g), g.state);
  MGB_CUDA(cudaGetLastError());
  return MGB200_OK;
}

int launch_barrier(Graph &g) {
  if (g.part_world <= 1) return MGB200_OK;
  barrier_kernel<<<1, 32, 0, g.stream>>>(make_barrier(g));
  MGB_CUDA(cudaGetLastError());
  return MGB200_OK;
}

// One iteration.  Main stream: (iteration 1: zero-row contribution refresh) -> SELL rows -> heavy segments ->
// heavy finish -> [join] -> iteration end.  Side stream: the SELL epilogue, forked after the SELL rows:
// it is the kernel that pushes contributions to the peer GPUs (NVLink-bound), so it overlaps with the
// heavy-row kernels (L2-gather-bound) instead of queueing behind them.  Every kernel returns immediately
// once state->done is set, so the host may enqueue iterations ahead of the convergence decision.
int launch_iteration(Graph &g, uint64_t it, const IterateConfig &cfg, uint64_t *launch_count,
                     uint64_t *spmv_count) {
  const RowEpilogue ep = make_epilogue(g, it, cfg);
  const double *contrib_in = g.contrib(static_cast<int>(it & 1ull));
  uint64_t launches = 0;
  const bool timed = g.time_spmv && g.timed_launches < Graph::kMaxTimedLaunches;
  auto tick = [&](int cls, int edge, cudaStream_t st) -> cudaError_t {
    if (!timed) return cudaSuccess;
    return cudaEventRecord(g.kev[(g.timed_launches * Graph::kClasses + cls) * 2 + edge], st);
  };
  if (it == 1 && g.any_zero_rows) {
    MGB_CUDA(tick(Graph::kClsZero, 0, g.stream));
    zero_refresh_kernel<<<grid_for(g, reinterpret_cast<const void *>(zero_refresh_kernel)), kBlockThreads, 0,
                          g.stream>>>(zero_row_rank(g, cfg), g.outdeg_l, g.contrib(0), make_zero_ranges(g), g.state);
    MGB_CUDA(tick(Graph::kClsZero, 1, g.stream));
    ++launches;
  }
  bool forked = false;
  if (g.n_slices > 0) {
    SellArgs s{};
    s.colbase = g.sell_colbase;
    s.idx = g.sell_idx;
    s.work = g.sell_work_items;
    s.n_work = g.sell_work;
    s.queue = g.queue;
    s.mode = g.sell_static ? 1u : 0u;
    s.first_row = g.n_heavy;
    s.end_row = g.n_heavy + g.n_sell;
    s.contrib_in = contrib_in;
    s.window = make_window(g);
    s.state = g.state;
    s.sums = g.sell_sums;
    // "rows" (default): ticketed warp-per-slice kernel, gathers through LDG; "stream": TMA index ring + LDGSTS gathers
    // (sell_stream.cuh) -- correct, but measured slower (3.4 vs 2.4 ms at scale-26, profiles/r01_stream_vs_rows.md)
    const bool stream_kernel = g.tun.stream_kernel && g.sell_items > 0;
    cudaStream_t es = g.overlap_epilogue ? g.stream2 : g.stream;
    MGB_CUDA(tick(Graph::kClsSell, 0, g.stream));
    if (stream_kernel) {
      if (!g.stream_attr_set) {  // per device, so per graph handle
        MGB_CUDA(cudaFuncSetAttribute(sell_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      kStreamSmemBytes));
        g.stream_attr_set = true;
      }
      SellStreamArgs t{};
      t.colbase = g.sell_colbase;
      t.idx = g.sell_idx;
      t.item_begin = g.sell_item_begin;
      t.n_items = g.sell_items;
      t.first_row = s.first_row;
      t.end_row = s.end_row;
      t.contrib_in = contrib_in;
      t.window = s.window;
      t.state = g.state;
      t.sums = g.sell_sums;
      const int sgrid = static_cast<int>(std::min<uint64_t>(g.sm_count, ceil_div(g.sell_items, kStreamWarps)));
      sell_stream_kernel<<<sgrid, kStreamThreads, kStreamSmemBytes, g.stream>>>(t);
    } else {
      const int rc = launch_sell_rows(g, s);
      if (rc) return rc;
    }
    ++launches;
    MGB_CUDA(tick(Graph::kClsSell, 1, g.stream));
    // the epilogue (+ NVLink push to the peers) of the SELL rows runs on the side stream, next to the heavy-row kernels
    if (g.overlap_epilogue) {
      MGB_CUDA(cudaEventRecord(g.fork_ev, g.stream));
      MGB_CUDA(cudaStreamWaitEvent(g.stream2, g.fork_ev, 0));
      forked = true;
    }
    // Across GPUs this kernel IS the exchange (one NVLink store per peer per row): it is bound by the links, not by the
    // SMs, and it must run NEXT TO the heavy-row kernels, not before or after them.  A full grid (4 CTAs/SM x 63
    // registers) takes the whole register file, so the heavy kernel (8 CTAs/SM x 32 registers, also the whole file)
    // only starts when it drains -- measured at 8 GPUs: 0.47 ms for the pair = 0.25 push + 0.22 heavy in sequence
    // (profiles/r02_multi_gpu.md).  A small grid (MGB200_PUSH_CTAS per SM, default 1) leaves 6 of the heavy kernel's 8
    // CTA slots free and keeps enough stores in flight to fill the links.
    uint64_t egrid_cap = static_cast<uint64_t>(grid_for(g, reinterpret_cast<const void *>(row_epilogue_kernel)));
    if (g.part_world > 1 && g.overlap_epilogue && g.tun.push_ctas > 0)
      egrid_cap = std::min<uint64_t>(egrid_cap, static_cast<uint64_t>(g.sm_count) * g.tun.push_ctas);
    const int egrid = static_cast<int>(std::min(egrid_cap, ceil_div(g.n_sell, kBlockThreads * kEpiRows)));
    MGB_CUDA(tick(Graph::kClsSellEpi, 0, es));
    row_epilogue_kernel<<<egrid, kBlockThreads, 0, es>>>(s.first_row, s.end_row, g.sell_sums, g.state, ep);
    MGB_CUDA(tick(Graph::kClsSellEpi, 1, es));
    ++launches;
    if (forked) MGB_CUDA(cudaEventRecord(g.join_ev, g.stream2));
    if (spmv_count) *spmv_count += 1;
  }
  if (g.n_seg > 0) {
    HeavyArgs h{};
    h.heavy_ptr = g.heavy_ptr;
    h.heavy_idx = g.heavy_idx;
    h.seg_row = g.seg_row;
    h.seg_begin = g.seg_begin;
    h.seg_first = g.seg_first;
    h.seg_partial = g.seg_partial;
    h.n_seg = g.n_seg;
    h.n_heavy = g.n_heavy;
    h.segment_edges = g.segment_edges;
    h.contrib_in = contrib_in;
    h.window = make_window(g);
    h.row_sums = g.heavy_sums;
    h.state = g.state;
    void (*const heavy_fn)(HeavyArgs) = h.window.path == kPathFlags    ? heavy_segments_kernel<kPathFlags>
                                        : h.window.path == kPathLookup ? heavy_segments_kernel<kPathLookup>
                                                                       : heavy_segments_kernel<kPathRange>;
    const void *hfn = reinterpret_cast<const void *>(heavy_fn);
    uint64_t hgrid_cap = static_cast<uint64_t>(grid_for(g, hfn));
    // leave register-file room for the push kernel's CTAs (63 registers x 256 threads each) next to this one
    if (forked && g.part_world > 1 && g.tun.push_ctas > 0 && hgrid_cap > static_cast<uint64_t>(g.sm_count) * 2)
      hgrid_cap -= static_cast<uint64_t>(g.sm_count) * 2;
    int grid = static_cast<int>(std::min(hgrid_cap, ceil_div(g.n_seg, kWarpsPerBlock)));
    MGB_CUDA(tick(Graph::kClsHeavySeg, 0, g.stream));
    heavy_fn<<<grid, kBlockThreads, 0, g.stream>>>(h);
    MGB_CUDA(tick(Graph::kClsHeavySeg, 1, g.stream));
    grid = static_cast<int>(
        std::min(static_cast<uint64_t>(grid_for(g, reinterpret_cast<const void *>(heavy_rowsum_kernel))),
                 ceil_div(g.n_heavy, kWarpsPerBlock)));
    MGB_CUDA(tick(Graph::kClsHeavyFin, 0, g.stream));
    heavy_rowsum_kernel<<<grid, kBlockThreads, 0, g.stream>>>(h);
    grid = static_cast<int>(
        std::min(static_cast<uint64_t>(grid_for(g, reinterpret_cast<const void *>(row_epilogue_kernel))),
                 ceil_div(g.n_heavy, kBlockThreads * kEpiRows)));
    row_epilogue_kernel<<<grid, kBlockThreads, 0, g.stream>>>(0, g.n_heavy, g.heavy_sums, g.state, ep);
    MGB_CUDA(tick(Graph::kClsHeavyFin, 1, g.stream));
    ++launches;
    launches += 2;
  }
  if (forked) MGB_CUDA(cudaStreamWaitEvent(g.stream, g.join_ev, 0));
  IterEndArgs e{};
  e.bar = make_barrier(g);
  e.max_iterations = cfg.max_iterations;
  e.eps = cfg.eps;
  e.extra_diff_bits = 0ull;
  if (g.any_zero_rows) {
    // the zero rows are elements of the reference's stop test too: |(1-d)/N - 1/N| in iteration 0, exactly 0 afterwards
    const double zr = zero_row_rank(g, cfg);
    const double zd = it == 0 ? fabs(zr - 1.0 / static_cast<double>(g.n)) : fabs(zr - zr);
    if (zd >= 0.0) {  // NaN contributes nothing, like the per-row test; same bits + 1 encoding as the rows' deltas
      memcpy(&e.extra_diff_bits, &zd, sizeof(zd));
      e.extra_diff_bits += 1ull;
    }
  }
  MGB_CUDA(tick(Graph::kClsIterEnd, 0, g.stream));
  iter_end_kernel<<<1, 32, 0, g.stream>>>(e);
  MGB_CUDA(tick(Graph::kClsIterEnd, 1, g.stream));
  ++launches;
  MGB_CUDA(cudaGetLastError());
  if (timed) ++g.timed_launches;
  if (launch_count) *launch_count += launches;
  return MGB200_OK;
}

// The gather phase alone, over an arbitrary per-label vector vec_in[n + 1] (slot n must hold 0): SELL row sums into
// g.sell_sums, heavy segment partials into g.seg_partial (summed per row by the caller in segment order).  This is
// y = A^T x for the rows of this partition with PageRank's kernels and cache policies; other SpMV-shaped paths hang
// their own epilogue on it (Katz: omega_i = A^T omega_{i-1}, katz.cu).  Kernels return at once while state->done is set.
int launch_gather_phase(Graph &g, const double *vec_in, uint64_t *launch_count, bool heavy_row_sums, bool weighted) {
  uint64_t launches = 0;
  const GatherWindow window = make_window(g);
  // (partitioned handles never carry weights: build_graph refuses them)
  if (weighted && ((g.n_slices > 0 && !g.sell_w) || (g.n_seg > 0 && !g.heavy_w))) {
    set_error("this graph handle carries no edge weights");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  if (g.n_slices > 0) {
    SellArgs s{};
    s.colbase = g.sell_colbase;
    s.idx = g.sell_idx;
    s.w = weighted ? g.sell_w : nullptr;
    s.work = g.sell_work_items;
    s.n_work = g.sell_work;
    s.queue = g.queue;
    s.mode = g.sell_static ? 1u : 0u;
    s.first_row = g.n_heavy;
    s.end_row = g.n_heavy + g.n_sell;
    s.contrib_in = vec_in;
    s.window = window;
    s.state = g.state;
    s.sums = g.sell_sums;
    const int rc = launch_sell_rows(g, s);
    if (rc) return rc;
    ++launches;
  }
  if (g.n_seg > 0) {
    HeavyArgs h{};
    h.heavy_ptr = g.heavy_ptr;
    h.heavy_idx = g.heavy_idx;
    h.heavy_w = weighted ? g.heavy_w : nullptr;
    h.seg_row = g.seg_row;
    h.seg_begin = g.seg_begin;
    h.seg_first = g.seg_first;
    h.seg_partial = g.seg_partial;
    h.n_seg = g.n_seg;
    h.n_heavy = g.n_heavy;
    h.segment_edges = g.segment_edges;
    h.contrib_in = vec_in;
    h.window = window;
    h.state = g.state;
    void (*const heavy_fn)(HeavyArgs) =
        weighted ? (window.path == kPathFlags    ? heavy_segments_kernel<kPathFlags, true>
                    : window.path == kPathLookup ? heavy_segments_kernel<kPathLookup, true>
                                                 : heavy_segments_kernel<kPathRange, true>)
                 : (window.path == kPathFlags    ? heavy_segments_kernel<kPathFlags>
                    : window.path == kPathLookup ? heavy_segments_kernel<kPathLookup>
                                                 : heavy_segments_kernel<kPathRange>);
    const int grid = static_cast<int>(std::min(static_cast<uint64_t>(grid_for(g, reinterpret_cast<const void *>(heavy_fn))),
                                               ceil_div(g.n_seg, kWarpsPerBlock)));
    heavy_fn<<<grid, kBlockThreads, 0, g.stream>>>(h);
    ++launches;
    if (heavy_row_sums) {
      h.row_sums = g.heavy_sums;
      const int rgrid = static_cast<int>(
          std::min(static_cast<uint64_t>(grid_for(g, reinterpret_cast<const void *>(heavy_rowsum_kernel))),
                   ceil_div(g.n_heavy, kWarpsPerBlock)));
      heavy_rowsum_kernel<<<rgrid, kBlockThreads, 0, g.stream>>>(h);
      ++launches;
    }
  }
  MGB_CUDA(cudaGetLastError());
  if (launch_count) *launch_count += launches;
  return MGB200_OK;
}

int launch_sum_and_exchange(Graph &g) {
  const int blocks = static_cast<int>(std::min<uint64_t>(kSumBlocks, g.local_rows ? ceil_div(g.local_rows, 4096) : 1));
  partial_sum_kernel<<<blocks, kBlockThreads, 0, g.stream>>>(g.rank, g.local_rows, g.sum_partials);
  final_sum_kernel<<<1, 256, 0, g.stream>>>(g.sum_partials, blocks, make_barrier(g));
  MGB_CUDA(cudaGetLastError());
  return MGB200_OK;
}

int launch_write_ranks_original_order(Graph &g, double *d_out) {
  if (g.n == 0) return MGB200_OK;
  const int grid = static_cast<int>(
      std::min(static_cast<uint64_t>(grid_for(g, reinterpret_cast<const void *>(write_original_order_kernel))),
          ceil_div(g.n, kBlockThreads)));
  write_original_order_kernel<<<grid, kBlockThreads, 0, g.stream>>>(g.n, g.label_of, g.rank, g.state, d_out);
  MGB_CUDA(cudaGetLastError());
  return MGB200_OK;
}

int launch_write_ranks_local(Graph &g, double *d_rank_out, uint32_t *d_vertex_out) {
  if (g.local_rows == 0) return MGB200_OK;
  const int grid = static_cast<int>(
      std::min(static_cast<uint64_t>(grid_for(g, reinterpret_cast<const void *>(write_local_kernel))),
          ceil_div(g.local_rows, kBlockThreads)));
  write_local_kernel<<<grid, kBlockThreads, 0, g.stream>>>(g.local_rows, g.rank, g.local_vertex, g.state,
                                                           d_rank_out, d_vertex_out);
  MGB_CUDA(cudaGetLastError());
  return MGB200_OK;
}

int kernel_occupancy_report(Graph &g, char *buf, size_t cap) {
  int a = 0, b = 0, c = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&a, sell_rows_kernel<kPathRange>, kBlockThreads, 0);
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, heavy_segments_kernel<kPathRange>, kBlockThreads, 0);
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&c, heavy_rowsum_kernel, kBlockThreads, 0);
  snprintf(buf, cap, "sm=%d blocks/SM: sell=%d heavy_seg=%d heavy_fin=%d (block=%d threads)", g.sm_count, a, b, c,
           kBlockThreads);
  return MGB200_OK;
}

}  // namespace mgb200
