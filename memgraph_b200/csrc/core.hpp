// memgraph_b200/csrc/core.hpp -- internal types shared by the build, the kernels and the C ABI.
//
// HBM layout of one partition (see DESIGN.md "Data layout"):
//   vertices are relabelled once at ingest: global order = in-degree descending, ties by
//   out-degree descending, then original id; with P partitions the sorted positions are dealt
//   round-robin to the P owners and each owner's vertices become one contiguous label range, so
//   every owner holds an in-degree-sorted slice with ~E/P in-edges and ~N/P rows.
//   Local rows fall into three classes by in-degree:
//     heavy  [0, n_heavy)                 deg >= heavy_min_degree : CSC + fixed-size edge segments
//     sell   [n_heavy, n_heavy + n_sell)  0 < deg < heavy_min    : SELL-32 slices (column-major per 32 rows)
//     zero   the rest                     deg == 0                : rank is the constant (1-d)/N
//   contrib[b][label] = rank/out_degree of the vertex with that label for iteration parity b
//   (full length N + 1, slot N is the zero read by SELL padding entries).
#pragma once

#include <cuda_runtime.h>

#include <cstdint>
#include <string>
#include <vector>

#include "mgb200_pagerank.h"

namespace mgb200 {

constexpr int kMaxPeers = 8;
constexpr int kSliceRows = 32;
// When Graph::idx_flagged, a stored source index (heavy_idx / sell_idx) carries the hotness of its label:
constexpr uint32_t kIdxL2Hot = 0x80000000u;     // keep in L2 (evict_last), else evict_first
constexpr uint32_t kIdxL1Hot = 0x40000000u;     // may allocate in L1, else bypass
constexpr uint32_t kIdxLabelMask = 0x3FFFFFFFu; // the label itself: flagged graphs have n < 2^30
constexpr uint32_t kNoL1Hints = 0xFFFFFFFFu;    // l1_hot_labels() when MGB200_L1_HOT_K < 0

// Which labels a partition owns and how its local rows (ascending label) map onto them.
//   dealt ranges (default): sorted position p -> owner p % P, label = start(owner) + p / P.  Every partition owns ONE
//     contiguous label range whose prefix is its hot part ("hot" = P windows in label space).
//   global order (MGB200_LABELLING=global): label = sorted position.  The `heavy` first labels (the heavy rows of the
//     whole graph) are owned round-robin, label % P; after them, BLOCKS of 32 consecutive labels -- one SELL slice, one
//     256-byte coalesced push per warp -- are owned round-robin.  "Hot" is one global label prefix on every partition,
//     so the single-partition gather code (range policy, label < l1_hot) is exact everywhere, with no owner lookup.
//     In-edge balance at P = 8: 1.0135 vs 1.0127 max/mean for the dealt ranges (profiles/r01_partition_balance.txt).
#define MGB_HD __host__ __device__ __forceinline__
struct RowMap {
  uint64_t n = 0;
  uint64_t heavy = 0;  // global order: number of heavy rows of the WHOLE graph (labels [0, heavy))
  uint32_t world = 1, rank = 0;
  uint32_t global_order = 0;
  uint64_t row_lo = 0;   // dealt ranges: first label owned by `rank`             (set by finalize())
  uint64_t heavy_q = 0;  // global order: heavy rows owned by `rank`               (set by finalize())

  // ---- dealt ranges ----
  MGB_HD uint64_t dealt_count(uint32_t q) const { return (n + world - 1 - q) / world; }
  MGB_HD uint64_t dealt_start(uint32_t q) const {  // sum_{r<q} count(r): the first (n % world) owners hold one extra row
    const uint64_t base = n / world, extra = n % world;
    return static_cast<uint64_t>(q) * base + (q < extra ? q : extra);
  }
  // ---- global order ----
  MGB_HD uint64_t heavy_rows(uint32_t q) const { return (heavy + world - 1 - q) / world; }  // labels q, q+P, .. < heavy
  MGB_HD uint64_t blocks() const { return (n - heavy + kSliceRows - 1) / kSliceRows; }
  // rows `q` owns in blocks [0, first_blocks) of the block sequence
  MGB_HD uint64_t rows_in_blocks(uint32_t q, uint64_t first_blocks) const {
    if (first_blocks == 0) return 0;
    uint64_t rows = ((first_blocks + world - 1 - q) / world) * kSliceRows;
    const uint64_t nb = blocks();
    if (first_blocks == nb && (nb - 1) % world == q) rows -= nb * kSliceRows - (n - heavy);  // last block may be partial
    return rows;
  }
  // ---- both ----
  MGB_HD uint64_t local_rows(uint32_t q) const {
    return global_order ? heavy_rows(q) + rows_in_blocks(q, blocks()) : dealt_count(q);
  }
  MGB_HD uint64_t label_of_pos(uint64_t pos) const {
    return global_order ? pos : dealt_start(static_cast<uint32_t>(pos % world)) + pos / world;
  }
  MGB_HD uint32_t owner(uint64_t label) const {
    if (global_order)
      return static_cast<uint32_t>(label < heavy ? label % world : ((label - heavy) / kSliceRows) % world);
    uint32_t q = 0;
    for (uint32_t r = 1; r < world; ++r)
      if (label >= dealt_start(r)) q = r;
    return q;
  }
  MGB_HD uint64_t local_of(uint64_t label) const {  // local row of `label` on its owner
    if (!global_order) return label - dealt_start(owner(label));
    if (label < heavy) return label / world;
    const uint64_t b = (label - heavy) / kSliceRows;
    return heavy_rows(static_cast<uint32_t>(b % world)) + (b / world) * kSliceRows + (label - heavy) % kSliceRows;
  }
  MGB_HD uint64_t label_of_local(uint64_t r) const {  // local row of THIS partition -> label
    if (!global_order) return row_lo + r;
    if (r < heavy_q) return r * world + rank;
    const uint64_t k = r - heavy_q;
    return heavy + ((k / kSliceRows) * world + rank) * kSliceRows + k % kSliceRows;
  }
  void finalize() {
    row_lo = (!global_order && n) ? dealt_start(rank) : 0;
    heavy_q = global_order ? heavy_rows(rank) : 0;
  }
};

// Written by iteration kernels, read by the host between batches (plain device memory).
struct IterState {
  unsigned long long diff_bits;   // running max |delta| of the current iteration as bits(double >= 0) + 1; 0 = no
                                  // non-NaN delta seen yet (CheckContinueIterate finds no element > eps then)
  unsigned long long iterations;  // completed iterations (the reference's number_of_iterations)
  unsigned long long barrier_seq; // cross-GPU barrier sequence number (monotonic over the handle's life)
  double last_diff;
  double local_sum;               // sum of this partition's un-normalised ranks
  double rank_sum;                // global sum (NormalizeRank divisor)
  int done;                       // set when CheckContinueIterate would return false
  int error;                      // 1: peer barrier timed out
  int abort_req;                  // written by THIS partition's host between batches: should_abort said stop
  int aborted;                    // set on EVERY partition in the same iteration once any partition asked to abort
};
constexpr unsigned long long kAbortBits = ~0ull;  // published instead of the delta by a partition that wants to abort

// Ticket counter of the SELL kernel's work items (pagerank_kernels.cu sell_rows_kernel).
struct WorkQueue {
  unsigned long long ticket;
  unsigned int ctas_done;
  unsigned int pad;
};

// One work item of the SELL kernel: slices [slice_begin, slice_end) and the column base of its first two slices, so a
// warp that draws the item needs ONE 32-byte record before its first index load.
struct WorkItem {
  uint64_t slice_begin, slice_end, col_begin, col_end;  // columns = 32-entry columns of sell_idx (colbase units)
};

// First page of the exchange window; every slot [q] is written by peer q (remote store over NVLink).
struct FlagPage {
  unsigned long long arrive[kMaxPeers];
  unsigned long long diff_bits[2][kMaxPeers];
  double rank_sum[2][kMaxPeers];
};
constexpr size_t kFlagPageBytes = 4096;
static_assert(sizeof(FlagPage) <= kFlagPageBytes, "flag page overflow");

struct PeerTable {
  double *contrib[2][kMaxPeers];  // [parity][peer] -> that peer's contrib buffer (index = global label)
  FlagPage *flags[kMaxPeers];
};

struct Graph {
  int device = 0;
  cudaStream_t stream = nullptr;
  int sm_count = 0;
  uint64_t n = 0, m = 0;
  uint32_t part_rank = 0, part_world = 1;
  uint64_t row_lo = 0;       // first global label owned (dealt ranges; 0 under global-order labelling)
  RowMap map;                // label <-> (owner, local row)
  uint64_t local_rows = 0;
  uint64_t local_edges = 0;
  uint64_t n_heavy = 0, n_sell = 0, n_zero = 0;
  uint32_t heavy_min_degree = 0, segment_edges = 0;
  uint64_t part_start[kMaxPeers] = {};  // first global label of every partition
  uint64_t zero_lo[kMaxPeers] = {}, zero_hi[kMaxPeers] = {};  // global label range of every partition's zero rows
  bool any_zero_rows = false;

  // label-space metadata
  uint32_t *label_of = nullptr;     // [n]  original id -> global label
  uint32_t *outdeg_l = nullptr;     // [n]  out-degree by global label
  uint32_t *local_vertex = nullptr; // [local_rows] original id of each owned row
  uint32_t *need_mask = nullptr;    // [ceil(local_rows / 4)] one BYTE per owned row: bit q = partition q gathers this
                                    // row's contribution (has an in-edge from it); nullptr = push to every peer

  // heavy class
  uint64_t heavy_edges = 0;
  uint64_t *heavy_ptr = nullptr;  // [n_heavy + 1]
  uint32_t *heavy_idx = nullptr;  // [heavy_edges] source labels (+ hot flags if idx_flagged), ascending inside a row
  uint64_t n_seg = 0;
  uint32_t *seg_row = nullptr;    // [n_seg] local heavy row
  uint64_t *seg_begin = nullptr;  // [n_seg] first edge
  uint64_t *seg_first = nullptr;  // [n_heavy + 1] first segment of each heavy row
  double *seg_partial = nullptr;  // [n_seg]
  double *heavy_sums = nullptr;   // [n_heavy] per-row gathered sums of the current iteration
  // optional edge weights (cuGraph-semantics variants only; one partition): parallel to heavy_idx / sell_idx, pad = 0
  double *heavy_w = nullptr, *sell_w = nullptr;
  double *outw_l = nullptr;       // [n] sum of the out-edge weights by label (EdgeSource::out_weights, input order)

  // SELL class
  uint64_t n_slices = 0;
  uint64_t sell_entries = 0;
  uint64_t *sell_colbase = nullptr;  // [n_slices + 1] in units of 32-entry columns
  uint32_t *sell_idx = nullptr;      // [sell_entries] source labels (+ hot flags if idx_flagged), pad = n
  bool idx_flagged = false;          // bits 31/30 of every stored index = L2-hot / L1-hot (graph_build.cu IndexFlags)
  double *sell_sums = nullptr;       // [n_sell] per-row gathered sums of the current iteration
  uint32_t sell_items = 0;           // work items of the streaming kernel: contiguous slice runs, ~equal columns
  uint64_t *sell_item_begin = nullptr;  // [sell_items + 1] first slice of each item
  uint32_t sell_work = 0;            // work items of sell_rows_kernel: contiguous slice runs of ~equal cost
  uint64_t *sell_work_begin = nullptr;  // [sell_work + 1]
  WorkItem *sell_work_items = nullptr;  // [sell_work]
  WorkQueue *queue = nullptr;        // ticket counter (zero between launches)
  bool sell_static = false;          // items dealt round-robin instead of drawn by ticket (small partitions)

  // iteration state
  double *rank = nullptr;      // [local_rows] un-normalised ranks, updated in place
  void *window = nullptr;      // exchange window: FlagPage | contrib[0] | contrib[1]
  size_t window_bytes = 0;
  size_t contrib_stride = 0;   // bytes between contrib[0] and contrib[1]
  IterState *state = nullptr;
  IterState *host_state = nullptr;  // pinned
  double *sum_partials = nullptr;   // [kSumBlocks]
  double *out_stage = nullptr;      // [n] device staging of the normalised ranks for host-output runs (lazy)
  PeerTable peers{};                // device pointers valid on THIS device
  void *peer_mapped[kMaxPeers] = {};  // IPC mappings to close
  bool peers_connected = false;
  bool poisoned = false;  // a peer barrier timed out: the partitions' barrier counters may disagree; runs are refused

  uint64_t resident_bytes = 0;
  uint64_t build_peak_bytes = 0;  // highest device memory in use seen during the build (transients included)
  double build_ms = 0.0;
  double upload_ms = 0.0;  // host COO -> device (mgb200_graph_create_host*), wall clock
  cudaEvent_t ev[4] = {};
  // side stream for the SELL epilogue (overlaps the peer push with the heavy-row kernels)
  cudaStream_t stream2 = nullptr;
  cudaEvent_t fork_ev = nullptr;
  cudaEvent_t join_ev = nullptr;
  bool overlap_epilogue = true;
  bool stream_attr_set = false;
  static constexpr int kOccSlots = 24;  // occupancy of every kernel launched on this handle, asked once (grid_for)
  mutable const void *occ_kernel[kOccSlots] = {};
  mutable int occ_blocks[kOccSlots] = {};
  mutable int occ_cached = 0;
  int table_attr_bytes[2] = {0, 0};  // dynamic shared memory already granted to sell_rows_table_kernel<range / flags>
  struct Tunables {  // environment, read once per graph in build_graph()
    uint64_t l2_hot_mb = 64;     // MGB200_L2_HOT_MB: evict-last window of the gathered vector (64 = effective L2, l2_bench)
    long l1_hot_k = 16;          // MGB200_L1_HOT_K: hottest labels (x1024) allowed to allocate in L1; <0 = no L1 hints
    bool multi_aware = true;     // MGB200_MULTI_AWARE=0: legacy "global label prefix is hot" on every partition
    bool force_multi_path = false;  // MGB200_FORCE_MULTI_PATH=1: run the multi-partition gather code on one GPU (measurement)
    bool stream_kernel = false;  // MGB200_SELL_KERNEL=stream
    uint32_t smem_table_kb = 0;  // MGB200_SMEM_TABLE_KB: shared-memory hot table of the SELL kernel (0 = off)
    int push_ctas = 2;           // MGB200_PUSH_CTAS: CTAs per SM of the SELL epilogue + peer push on several partitions (0 = full grid)
    int sell_mode = -1;          // MGB200_SELL_MODE: 0 ticket queue, 1 static deal, -1 (default) by partition size
    bool global_order = false;   // MGB200_LABELLING=global: label = global degree order, blocks of 32 dealt (RowMap)
    bool push_mask = true;       // MGB200_PUSH_MASK=0: push every contribution to every peer (default: only to the partitions that gather it)
    bool lone_partition = false; // MGB200_LONE_PARTITION=1 (profiling only): run ONE partition of part_world without its
                                 // peers -- no stores to them, barrier of one; timings/ncu are real, ranks are NOT
    int idx_flags = -1;          // MGB200_IDX_FLAGS: 1 bake hotness into the indices, 0 never, -1 (default) see build_graph
    unsigned long long barrier_timeout_ms = 20000;  // MGB200_BARRIER_TIMEOUT_MS
  } tun;
  // hot thresholds in LOCAL label units (label - first label of the owning partition); one definition for the
  // build-time index flags and the run-time gather window
  uint32_t hot_divisor() const { return (tun.multi_aware && !map.global_order) ? part_world : 1u; }
  uint32_t l1_hot_labels() const {
    if (tun.l1_hot_k < 0) return kNoL1Hints;
    const uint64_t v = static_cast<uint64_t>(tun.l1_hot_k) * 1024 / hot_divisor();
    return static_cast<uint32_t>(v < 0xFFFFFFF0ull ? v : 0xFFFFFFF0ull);
  }
  // labels in the shared-memory hot table: a multiple of 2 * partitions (every owner's window has an even size, a whole
  // number of 16-byte TMA units on one partition); only with 30-bit labels on several partitions (the slot rides in
  // the stored index), never with the per-gather owner lookup
  uint32_t table_labels() const {
    if (tun.smem_table_kb == 0 || tun.stream_kernel) return 0;
    if (part_world > 1 && (!idx_flagged || map.global_order)) return 0;
    if (part_world == 1 && (idx_flagged || tun.force_multi_path)) return 0;
    const uint64_t unit = 2ull * part_world;
    uint64_t labels = std::min<uint64_t>(static_cast<uint64_t>(tun.smem_table_kb) * 1024 / sizeof(double), n);
    labels = labels / unit * unit;
    return static_cast<uint32_t>(labels);
  }
  uint32_t l2_hot_labels() const {
    if (!tun.multi_aware) return 0xFFFFFFFFu;
    const uint64_t v = (tun.l2_hot_mb << 20) / sizeof(double) / hot_divisor();
    return static_cast<uint32_t>(v < 0xFFFFFFFFull ? v : 0xFFFFFFFFull);
  }
  // optional per-launch timing: an event pair around every kernel of the first kMaxTimedLaunches iterations
  static constexpr int kMaxTimedLaunches = 64;
  static constexpr int kClasses = 6;
  enum { kClsZero = 0, kClsSell, kClsSellEpi, kClsHeavySeg, kClsHeavyFin, kClsIterEnd };
  bool time_spmv = false;
  int timed_launches = 0;  // iterations whose kernels carry event pairs
  cudaEvent_t kev[2 * kClasses * kMaxTimedLaunches] = {};

  double *contrib(int parity) const {
    return reinterpret_cast<double *>(static_cast<char *>(window) + kFlagPageBytes + parity * contrib_stride);
  }
  FlagPage *flags() const { return static_cast<FlagPage *>(window); }
};

// error plumbing (capi.cu)
void set_error(const std::string &msg);
int cuda_fail(cudaError_t e, const char *what, const char *file, int line);
#define MGB_CUDA(expr)                                                        \
  do {                                                                        \
    cudaError_t _e = (expr);                                                  \
    if (_e != cudaSuccess) return ::mgb200::cuda_fail(_e, #expr, __FILE__, __LINE__); \
  } while (0)

// Where the build reads the COO from, a chunk at a time (graph_build.cu walks it twice: degrees, then the edges this
// partition owns).  With several partitions nobody has to hold the whole edge list on a device: the transient is one
// chunk plus the owned edges, so the graph size scales with the number of GPUs.
struct EdgeSource {
  uint64_t m = 0;            // edges in total
  uint64_t chunk_edges = 0;  // largest count the build may ask for
  virtual ~EdgeSource() = default;
  // device pointers to edges [first, first + count), valid until the next call (work is enqueued on `st`)
  virtual int get(uint64_t first, uint64_t count, const uint32_t **from, const uint32_t **to, cudaStream_t st) = 0;
  // optional edge weights of the chunk last returned by get() (nullptr: unweighted graph)
  virtual const double *weights() const { return nullptr; }
  virtual bool weighted() const { return false; }
  // weighted graphs: device array [n] by original vertex id, each vertex's out-edge weights summed left to right in
  // input edge order -- the producer has seen every edge already, and one fixed order makes the sums reproducible
  virtual const double *out_weights() const { return nullptr; }
};

// graph_build.cu
int build_graph(Graph &g, EdgeSource &edges);
void free_graph(Graph &g);
int narrow_edges_u64_to_u32(int device, cudaStream_t stream, uint64_t n, uint64_t count, const uint64_t *d_in,
                            uint32_t *d_out, int *d_bad_flag);

// pagerank_kernels.cu
struct IterateConfig {
  uint64_t max_iterations;
  double damping;
  double eps;
};
constexpr int kSumBlocks = 1024;
int launch_init(Graph &g, const IterateConfig &cfg);
int launch_iteration(Graph &g, uint64_t it, const IterateConfig &cfg, uint64_t *launch_count, uint64_t *spmv_count);
// SELL sums + heavy segment partials (heavy_row_sums: also the heavy rows' sums, into g.heavy_sums)
int launch_gather_phase(Graph &g, const double *vec_in, uint64_t *launch_count, bool heavy_row_sums = false,
                        bool weighted = false);  // weighted: multiply every gathered value by its edge weight
int launch_barrier(Graph &g);
int launch_sum_and_exchange(Graph &g);
int launch_write_ranks_original_order(Graph &g, double *d_out);                   // single partition
int launch_write_ranks_local(Graph &g, double *d_rank_out, uint32_t *d_vertex_out);  // partitioned
int kernel_occupancy_report(Graph &g, char *buf, size_t cap);

// katz.cu
struct KatzResult {
  uint64_t iterations = 0, max_out_degree = 0, launches = 0, tie_order_runs = 0;
  double gamma = 0.0, iterate_ms = 0.0;
  bool converged = false;
};
int katz_iterate(Graph &g, double alpha, double epsilon, uint64_t max_iterations, double *d_out_original_order,
                 KatzResult *res);

// rmat.cu
int rmat_device(int device, uint32_t scale, uint64_t first_edge, uint64_t count, uint64_t seed, double a, double b,
                double c, uint32_t *d_from, uint32_t *d_to);

}  // namespace mgb200
