// memgraph_b200/csrc/capi.cu -- implementation of include/mgb200_pagerank.h (host orchestration).
//
// The host side only sequences work: ingest -> device build (graph_build.cu) -> batches of
// iteration launches (pagerank_kernels.cu) with a device-side convergence flag, so the host
// synchronises once per batch instead of once per iteration -> normalise -> copy out.
// There is no CPU compute path: every entry point that needs a device fails with
// MGB200_ERR_CUDA when none is usable.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "core.hpp"
#include "mgb200_katz.h"
#include "mgb200_personalized.h"
#include "rmat.hpp"

struct mgb200_graph {
  mgb200::Graph g;
};

namespace mgb200 {

namespace {
thread_local std::string tls_error;
}

void set_error(const std::string &msg) { tls_error = msg; }

int cuda_fail(cudaError_t e, const char *what, const char *file, int line) {
  char buf[512];
  const char *base = strrchr(file, '/');
  snprintf(buf, sizeof(buf), "CUDA error: %s (%s) at %s:%d [%s]", cudaGetErrorString(e), cudaGetErrorName(e),
           base ? base + 1 : file, line, what);
  set_error(buf);
  cudaGetLastError();  // clear the sticky-less error so the next call reports its own
  return MGB200_ERR_CUDA;
}

namespace {

__global__ void rmat_kernel(uint32_t scale, uint64_t first_edge, uint64_t count, uint64_t seed, RmatThresholds t,
                            uint32_t *from, uint32_t *to) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < count; i += stride) {
    uint32_t s, d;
    rmat_edge(scale, first_edge + i, seed, t, s, d);
    from[i] = s;
    to[i] = d;
  }
}

// ---- edge sources of the build (core.hpp EdgeSource) ------------------------------------------------------------
uint64_t build_chunk_edges(uint64_t fallback) {
  const char *s = getenv("MGB200_BUILD_CHUNK_EDGES");  // tests shrink it to force many chunks
  const unsigned long long v = s ? strtoull(s, nullptr, 10) : 0ull;
  return v ? v : fallback;
}

struct DeviceArrays final : EdgeSource {  // the whole COO is resident: chunks are views
  const uint32_t *from, *to;
  const double *weight;  // nullable
  const double *outw;    // [n] out-weight sums by vertex (with weight)
  uint64_t last_first = 0;
  DeviceArrays(uint64_t count, const uint32_t *f, const uint32_t *t, const double *w = nullptr, const double *ow = nullptr)
      : from(f), to(t), weight(w), outw(ow) {
    m = count;
    chunk_edges = build_chunk_edges(count);
  }
  int get(uint64_t first, uint64_t, const uint32_t **f, const uint32_t **t, cudaStream_t) override {
    *f = from + first;
    *t = to + first;
    last_first = first;
    return MGB200_OK;
  }
  const double *weights() const override { return weight ? weight + last_first : nullptr; }
  bool weighted() const override { return weight != nullptr; }
  const double *out_weights() const override { return outw; }
};

struct RmatStream final : EdgeSource {  // the synthetic workload, generated chunk by chunk: no COO is ever materialised
  uint32_t scale;
  uint64_t seed;
  RmatThresholds thr;
  uint32_t *buf_from = nullptr, *buf_to = nullptr;
  RmatStream(uint32_t scale_, uint64_t count, uint64_t seed_, double a, double b, double c)
      : scale(scale_), seed(seed_), thr(rmat_thresholds(a, b, c)) {
    m = count;
    chunk_edges = std::min<uint64_t>(std::max<uint64_t>(count, 1), build_chunk_edges(1ull << 27));
  }
  ~RmatStream() override {
    cudaFree(buf_from);
    cudaFree(buf_to);
  }
  int get(uint64_t first, uint64_t count, const uint32_t **f, const uint32_t **t, cudaStream_t st) override {
    if (!buf_from) {
      MGB_CUDA(cudaMalloc(&buf_from, chunk_edges * sizeof(uint32_t)));
      MGB_CUDA(cudaMalloc(&buf_to, chunk_edges * sizeof(uint32_t)));
    }
    const int blocks = static_cast<int>(std::min<uint64_t>((count + 255) / 256, 148ull * 32));
    rmat_kernel<<<blocks, 256, 0, st>>>(scale, first, count, seed, thr, buf_from, buf_to);
    MGB_CUDA(cudaGetLastError());
    *f = buf_from;
    *t = buf_to;
    return MGB200_OK;
  }
};

int check_device(int device) {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess) return cuda_fail(e, "cudaGetDeviceCount", __FILE__, __LINE__);
  if (count <= 0) {
    set_error("CUDA error: no CUDA device available (this library has no CPU fallback)");
    return MGB200_ERR_CUDA;
  }
  if (device < 0 || device >= count) {
    set_error("invalid device ordinal " + std::to_string(device) + " (device count " + std::to_string(count) + ")");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  return MGB200_OK;
}

int validate_sizes(uint64_t n, uint32_t part_rank, uint32_t part_world) {
  if (n >= 0xFFFFFFFFull) {
    set_error("number_of_nodes must be < 2^32 - 1 (32-bit vertex labels)");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  if (part_world == 0 || part_world > static_cast<uint32_t>(kMaxPeers) || part_rank >= part_world) {
    set_error("invalid partition: rank " + std::to_string(part_rank) + " of " + std::to_string(part_world));
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  return MGB200_OK;
}

// Iteration loop shared by the single- and multi-partition entry points.
int iterate(Graph &g, const mgb200_run_params &p, mgb200_run_stats &stats) {
  MGB_CUDA(cudaSetDevice(g.device));
  if (g.poisoned) {
    set_error("this partition handle saw a peer time-out earlier; its barrier state is undefined -- destroy and rebuild it");
    return MGB200_ERR_COMM;
  }
  IterateConfig cfg{p.max_iterations, p.damping_factor, p.stop_epsilon};
  stats = mgb200_run_stats{};
  if (g.n == 0) {
    // The reference runs one pass over empty vectors when max_iterations != 0 (pagerank.cpp:201-231).
    stats.iterations = p.max_iterations != 0 ? 1 : 0;
    return MGB200_OK;
  }
  g.time_spmv = p.time_spmv_kernel != 0;
  g.timed_launches = 0;
  if (g.time_spmv) {
    // fresh events every run: a never-recorded event marks "kernel class not launched in that iteration"
    for (auto &e : g.kev) {
      if (e) cudaEventDestroy(e);
      MGB_CUDA(cudaEventCreate(&e));
    }
  }
  MGB_CUDA(cudaEventRecord(g.ev[2], g.stream));  // timed region starts with the rank = 1/N initialisation (:199)
  int rc = launch_init(g, cfg);
  if (rc) return rc;
  rc = launch_barrier(g);  // peers have initialised before anyone pushes into their buffers
  if (rc) return rc;
  uint64_t launches = 0, spmv = 0;
  uint64_t it = 0;
  bool done = p.max_iterations == 0;
  bool abort_sent = false;
  const uint64_t batch_cap = 32;
  while (!done) {
    uint64_t batch = batch_cap;
    if (p.max_iterations - it < batch) batch = p.max_iterations - it;
    for (uint64_t b = 0; b < batch; ++b, ++it) {
      rc = launch_iteration(g, it, cfg, &launches, &spmv);
      if (rc) return rc;
    }
    MGB_CUDA(cudaMemcpyAsync(g.host_state, g.state, sizeof(IterState), cudaMemcpyDeviceToHost, g.stream));
    MGB_CUDA(cudaStreamSynchronize(g.stream));
    if (g.host_state->error) {
      g.poisoned = true;
      set_error("multi-GPU barrier timed out waiting for a peer partition");
      return MGB200_ERR_COMM;
    }
    if (g.host_state->aborted) {  // some partition's host asked to stop: every partition left the loop in the same iteration
      set_error("aborted by the host (mgp_must_abort)");
      return MGB200_ERR_ABORTED;
    }
    done = g.host_state->done != 0 || it >= p.max_iterations;
    if (!done && !abort_sent && p.should_abort && p.should_abort(p.abort_user)) {
      // publish the request; the next iteration end turns it into a collective stop (pagerank_kernels.cu iter_end_kernel)
      static const int one = 1;
      MGB_CUDA(cudaMemcpyAsync(&g.state->abort_req, &one, sizeof(int), cudaMemcpyHostToDevice, g.stream));
      abort_sent = true;
    }
  }
  rc = launch_sum_and_exchange(g);
  launches += 2;
  if (rc) return rc;
  MGB_CUDA(cudaEventRecord(g.ev[3], g.stream));
  MGB_CUDA(cudaMemcpyAsync(g.host_state, g.state, sizeof(IterState), cudaMemcpyDeviceToHost, g.stream));
  MGB_CUDA(cudaStreamSynchronize(g.stream));
  if (g.host_state->error) {
    g.poisoned = true;
    set_error("multi-GPU barrier timed out waiting for a peer partition");
    return MGB200_ERR_COMM;
  }
  float ms = 0.f;
  MGB_CUDA(cudaEventElapsedTime(&ms, g.ev[2], g.ev[3]));
  stats.iterations = g.host_state->iterations;
  stats.last_diff = g.host_state->last_diff;
  stats.rank_sum = g.host_state->rank_sum;
  stats.iterate_ms = ms;
  stats.kernel_launches = launches;
  // launches past the convergence point return immediately; report the ones that did work
  stats.spmv_launches = std::min<uint64_t>(spmv, stats.iterations);
  const int timed = static_cast<int>(std::min<uint64_t>(g.timed_launches, stats.iterations));
  for (int i = 0; i < timed; ++i) {
    for (int c = 0; c < Graph::kClasses; ++c) {
      cudaEvent_t e0 = g.kev[(i * Graph::kClasses + c) * 2], e1 = g.kev[(i * Graph::kClasses + c) * 2 + 1];
      if (cudaEventQuery(e0) != cudaSuccess || cudaEventQuery(e1) != cudaSuccess) {
        cudaGetLastError();
        continue;  // this kernel class was not launched in that iteration
      }
      float kms = 0.f;
      if (cudaEventElapsedTime(&kms, e0, e1) != cudaSuccess) {
        cudaGetLastError();
        continue;
      }
      stats.class_ms[c] += kms;
    }
  }
  stats.kernel_ms = stats.class_ms[Graph::kClsSell];
  stats.kernel_timed_launches = g.n_slices > 0 ? timed : 0;
  return MGB200_OK;
}

}  // namespace
}  // namespace mgb200

namespace mgb200 {
int cugraph_pagerank_iterate(Graph &g, const mgb200_cugraph_params &prm, double *d_out_original_order,
                             mgb200_cugraph_stats *stats);
}

using namespace mgb200;

extern "C" {

const char *mgb200_last_error(void) { return tls_error.c_str(); }

int mgb200_device_count(int *count_out) {
  if (!count_out) return MGB200_ERR_INVALID_ARGUMENT;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess) {
    *count_out = 0;
    return cuda_fail(e, "cudaGetDeviceCount", __FILE__, __LINE__);
  }
  *count_out = count;
  return MGB200_OK;
}

int mgb200_graph_create_device(int device, uint64_t n, uint64_t m, const uint32_t *d_from, const uint32_t *d_to,
                               uint32_t part_rank, uint32_t part_world, mgb200_graph **out) {
  if (!out) return MGB200_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  if (m > 0 && (!d_from || !d_to)) {
    set_error("null edge arrays");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  int rc = validate_sizes(n, part_rank, part_world);
  if (rc) return rc;
  rc = check_device(device);
  if (rc) return rc;
  auto *h = new (std::nothrow) mgb200_graph();
  if (!h) {
    set_error("out of host memory");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  h->g.device = device;
  h->g.n = n;
  h->g.m = m;
  h->g.part_rank = part_rank;
  h->g.part_world = part_world;
  DeviceArrays source(m, d_from, d_to);
  rc = build_graph(h->g, source);
  if (rc) {
    free_graph(h->g);
    delete h;
    return rc;
  }
  *out = h;
  return MGB200_OK;
}

int mgb200_graph_create_host_weighted_u32(int device, uint64_t n, uint64_t m, const uint32_t *from, const uint32_t *to,
                                         const double *weight, mgb200_graph **out) {
  if (!out) return MGB200_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  if (m > 0 && (!from || !to || !weight)) {
    set_error("null edge arrays");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  int rc = validate_sizes(n, 0, 1);
  if (rc) return rc;
  rc = check_device(device);
  if (rc) return rc;
  MGB_CUDA(cudaSetDevice(device));
  // out-weight sums, left to right in input edge order (cuGraph's out_w of every vertex): one fixed order, so the
  // sums -- and every rank divided by them -- do not depend on the build's chunking or on thread timing
  std::vector<double> outw;
  try {
    outw.assign(n, 0.0);
  } catch (const std::bad_alloc &) {
    set_error("out of host memory");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  for (uint64_t e = 0; e < m; ++e) {
    if (from[e] >= n || to[e] >= n) {
      set_error("edge endpoint out of range (>= number_of_nodes)");
      return MGB200_ERR_INVALID_ARGUMENT;
    }
    if (!(weight[e] >= 0.0)) {  // cuGraph expects non-negative weights; NaN fails this test too
      set_error("edge weights must be non-negative numbers");
      return MGB200_ERR_INVALID_ARGUMENT;
    }
    outw[from[e]] += weight[e];
  }
  uint32_t *d_from = nullptr, *d_to = nullptr;
  double *d_w = nullptr, *d_outw = nullptr;
  auto cleanup = [&]() {
    cudaFree(d_from);
    cudaFree(d_to);
    cudaFree(d_w);
    cudaFree(d_outw);
  };
  cudaError_t e;
  const uint64_t cnt = std::max<uint64_t>(m, 1);
  if ((e = cudaMalloc(&d_from, cnt * 4)) != cudaSuccess || (e = cudaMalloc(&d_to, cnt * 4)) != cudaSuccess ||
      (e = cudaMalloc(&d_w, cnt * 8)) != cudaSuccess ||
      (e = cudaMalloc(&d_outw, std::max<uint64_t>(n, 1) * 8)) != cudaSuccess ||
      (e = cudaMemcpy(d_from, from, m * 4, cudaMemcpyHostToDevice)) != cudaSuccess ||
      (e = cudaMemcpy(d_to, to, m * 4, cudaMemcpyHostToDevice)) != cudaSuccess ||
      (e = cudaMemcpy(d_w, weight, m * 8, cudaMemcpyHostToDevice)) != cudaSuccess ||
      (e = cudaMemcpy(d_outw, outw.data(), n * 8, cudaMemcpyHostToDevice)) != cudaSuccess) {
    cleanup();
    return cuda_fail(e, "weighted COO upload", __FILE__, __LINE__);
  }
  auto *h = new (std::nothrow) mgb200_graph();
  if (!h) {
    cleanup();
    set_error("out of host memory");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  h->g.device = device;
  h->g.n = n;
  h->g.m = m;
  h->g.part_rank = 0;
  h->g.part_world = 1;
  {
    DeviceArrays source(m, d_from, d_to, d_w, d_outw);
    rc = build_graph(h->g, source);
  }
  cleanup();
  if (rc) {
    free_graph(h->g);
    delete h;
    return rc;
  }
  *out = h;
  return MGB200_OK;
}

int mgb200_graph_create_rmat(int device, uint32_t scale, uint64_t edge_count, uint64_t seed, double a, double b, double c,
                             uint32_t part_rank, uint32_t part_world, mgb200_graph **out) {
  if (!out) return MGB200_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  if (scale == 0 || scale > 31) {
    set_error("rmat: scale must be in [1, 31]");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  const uint64_t n = 1ull << scale;
  int rc = validate_sizes(n, part_rank, part_world);
  if (rc) return rc;
  rc = check_device(device);
  if (rc) return rc;
  auto *h = new (std::nothrow) mgb200_graph();
  if (!h) {
    set_error("out of host memory");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  h->g.device = device;
  h->g.n = n;
  h->g.m = edge_count;
  h->g.part_rank = part_rank;
  h->g.part_world = part_world;
  cudaSetDevice(device);
  {
    RmatStream source(scale, edge_count, seed, a, b, c);
    rc = build_graph(h->g, source);
  }
  if (rc) {
    free_graph(h->g);
    delete h;
    return rc;
  }
  *out = h;
  return MGB200_OK;
}

}  // extern "C"

namespace {

// ---- host COO -> device uint32 COO: pinned, double-buffered, single pass ------------------------------------------
// The reference's ingest ends in host vectors (pagerank_module.cpp:18-54); this is the hop from there to the device.
// r01 staged pageable uint64 chunks synchronously, twice (16 B per edge over PCIe at the driver's single-threaded
// pageable rate).  Now a few host threads narrow (or copy) chunk c into pinned buffer c & 1 -- validating the
// endpoints on the way -- while the copy engine ships buffer (c - 1) & 1: 8 B per edge on the link, both endpoints
// of an edge in the same pass.  The pinned staging (4 x 64 MiB) is kept for the life of the process: allocating it
// costs more than the upload of a small graph.
constexpr uint64_t kIngestChunk = 1ull << 24;  // edges per staging buffer

struct IngestStaging {
  std::mutex busy;
  uint32_t *pinned[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};  // [buffer][from / to]
  cudaEvent_t shipped[2] = {nullptr, nullptr};
  cudaStream_t stream = nullptr;
  int device = -1;
  int ensure(int dev) {
    if (device == dev && pinned[0][0]) return MGB200_OK;
    release();
    MGB_CUDA(cudaSetDevice(dev));
    for (auto &buf : pinned)
      for (auto &p : buf) MGB_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&p), kIngestChunk * sizeof(uint32_t), cudaHostAllocDefault));
    for (auto &e : shipped) MGB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    MGB_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    device = dev;
    return MGB200_OK;
  }
  void release() {
    for (auto &buf : pinned)
      for (auto &p : buf) {
        if (p) cudaFreeHost(p);
        p = nullptr;
      }
    for (auto &e : shipped) {
      if (e) cudaEventDestroy(e);
      e = nullptr;
    }
    if (stream) cudaStreamDestroy(stream);
    stream = nullptr;
    device = -1;
  }
};
IngestStaging g_staging;  // one upload at a time per process; a second concurrent caller allocates its own

unsigned ingest_threads() {
  const char *s = getenv("MGB200_INGEST_THREADS");
  if (s && atoi(s) > 0) return static_cast<unsigned>(std::min(atoi(s), 64));
  const unsigned hw = std::thread::hardware_concurrency();
  return std::max(1u, std::min(32u, hw / 2));
}

template <typename T>
int upload_coo(int device, uint64_t n, uint64_t m, const T *from, const T *to, uint32_t *d_from, uint32_t *d_to) {
  std::unique_lock<std::mutex> lock(g_staging.busy, std::try_to_lock);
  IngestStaging local;
  IngestStaging &st = lock.owns_lock() ? g_staging : local;
  int rc = st.ensure(device);
  if (rc) return rc;
  const unsigned threads = ingest_threads();
  std::atomic<int> bad{0};
  for (uint64_t off = 0, c = 0; off < m; off += kIngestChunk, ++c) {
    const uint64_t cnt = std::min(kIngestChunk, m - off);
    const int b = static_cast<int>(c & 1);
    if (c >= 2) MGB_CUDA(cudaEventSynchronize(st.shipped[b]));  // the copy that last read this buffer is done
    auto work = [&, b, off, cnt](unsigned t, unsigned nt) {
      const uint64_t lo = cnt * t / nt, hi = cnt * (t + 1) / nt;
      uint32_t *pf = st.pinned[b][0], *pt = st.pinned[b][1];
      T worst = 0;
      for (uint64_t i = lo; i < hi; ++i) {
        const T f = from[off + i], d = to[off + i];
        worst = std::max(worst, std::max(f, d));
        pf[i] = static_cast<uint32_t>(f);
        pt[i] = static_cast<uint32_t>(d);
      }
      if (static_cast<uint64_t>(worst) >= n) bad.store(1, std::memory_order_relaxed);
    };
    const unsigned nt = cnt < (1u << 16) ? 1u : threads;
    if (nt == 1) {
      work(0, 1);
    } else {
      std::vector<std::thread> pool;
      for (unsigned t = 1; t < nt; ++t) pool.emplace_back(work, t, nt);
      work(0, nt);
      for (auto &th : pool) th.join();
    }
    if (bad.load(std::memory_order_relaxed)) break;
    MGB_CUDA(cudaMemcpyAsync(d_from + off, st.pinned[b][0], cnt * sizeof(uint32_t), cudaMemcpyHostToDevice, st.stream));
    MGB_CUDA(cudaMemcpyAsync(d_to + off, st.pinned[b][1], cnt * sizeof(uint32_t), cudaMemcpyHostToDevice, st.stream));
    MGB_CUDA(cudaEventRecord(st.shipped[b], st.stream));
  }
  MGB_CUDA(cudaStreamSynchronize(st.stream));
  if (!lock.owns_lock()) local.release();
  if (bad.load()) {
    set_error("edge endpoint out of range (>= number_of_nodes)");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  return MGB200_OK;
}

template <typename T>
int create_from_host(int device, uint64_t n, uint64_t m, const T *from, const T *to, uint32_t part_rank,
                     uint32_t part_world, mgb200_graph **out) {
  if (!out) return MGB200_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  if (m > 0 && (!from || !to)) {
    set_error("null edge arrays");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  int rc = validate_sizes(n, part_rank, part_world);
  if (rc) return rc;
  rc = check_device(device);
  if (rc) return rc;
  MGB_CUDA(cudaSetDevice(device));
  uint32_t *d_from = nullptr, *d_to = nullptr;
  cudaError_t e;
  if ((e = cudaMalloc(&d_from, std::max<uint64_t>(m, 1) * sizeof(uint32_t))) != cudaSuccess ||
      (e = cudaMalloc(&d_to, std::max<uint64_t>(m, 1) * sizeof(uint32_t))) != cudaSuccess) {
    cudaFree(d_from);
    return cuda_fail(e, "cudaMalloc(COO)", __FILE__, __LINE__);
  }
  const auto t0 = std::chrono::steady_clock::now();
  rc = upload_coo(device, n, m, from, to, d_from, d_to);
  const double upload_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  if (!rc) rc = mgb200_graph_create_device(device, n, m, d_from, d_to, part_rank, part_world, out);
  cudaFree(d_from);
  cudaFree(d_to);
  if (!rc) (*out)->g.upload_ms = upload_ms;
  return rc;
}

}  // namespace

extern "C" {

int mgb200_graph_create_host(int device, uint64_t n, uint64_t m, const uint64_t *from, const uint64_t *to,
                             uint32_t part_rank, uint32_t part_world, mgb200_graph **out) {
  return create_from_host(device, n, m, from, to, part_rank, part_world, out);
}

int mgb200_graph_create_host_u32(int device, uint64_t n, uint64_t m, const uint32_t *from, const uint32_t *to,
                                 uint32_t part_rank, uint32_t part_world, mgb200_graph **out) {
  return create_from_host(device, n, m, from, to, part_rank, part_world, out);
}

// 128-bit fingerprint of a dense COO (order-sensitive), for callers that keep a device graph across calls and need to
// know whether the graph they just pulled is the one already resident (the mgp ABI carries no graph version).
int mgb200_coo_fingerprint_u32(uint64_t n, uint64_t m, const uint32_t *from, const uint32_t *to, uint64_t out[2]) {
  if (!out || (m > 0 && (!from || !to))) return MGB200_ERR_INVALID_ARGUMENT;
  const unsigned threads = m < (1u << 18) ? 1u : ingest_threads();
  std::vector<uint64_t> part(static_cast<size_t>(threads) * 2, 0);
  auto work = [&](unsigned t) {
    const uint64_t lo = m * t / threads, hi = m * (t + 1) / threads;
    uint64_t a = 0x9E3779B97F4A7C15ull ^ lo, b = 0xC2B2AE3D27D4EB4Full ^ hi;
    for (uint64_t i = lo; i < hi; ++i) {
      const uint64_t v = (static_cast<uint64_t>(from[i]) << 32) | to[i];
      a = (a ^ v) * 0xBF58476D1CE4E5B9ull;
      a ^= a >> 29;
      b = (b + v) * 0x94D049BB133111EBull;
      b ^= b >> 31;
    }
    part[2 * t] = a;
    part[2 * t + 1] = b;
  };
  std::vector<std::thread> pool;
  for (unsigned t = 1; t < threads; ++t) pool.emplace_back(work, t);
  work(0);
  for (auto &th : pool) th.join();
  uint64_t a = n * 0xD6E8FEB86659FD93ull + m, b = m ^ 0xA24BAED4963EE407ull;
  for (unsigned t = 0; t < threads; ++t) {  // fixed combination order; the thread count is part of the definition
    a = (a ^ part[2 * t]) * 0xBF58476D1CE4E5B9ull + t;
    b = (b + part[2 * t + 1]) * 0x94D049BB133111EBull + threads;
  }
  out[0] = a;
  out[1] = b;
  return MGB200_OK;
}

void mgb200_graph_destroy(mgb200_graph *g) {
  if (!g) return;
  free_graph(g->g);
  delete g;
}

int mgb200_graph_get_info(const mgb200_graph *h, mgb200_graph_info *info) {
  if (!h || !info) return MGB200_ERR_INVALID_ARGUMENT;
  const Graph &g = h->g;
  info->node_count = g.n;
  info->edge_count = g.m;
  info->part_rank = g.part_rank;
  info->part_world = g.part_world;
  info->local_rows = g.local_rows;
  info->local_edges = g.local_edges;
  info->heavy_rows = g.n_heavy;
  info->heavy_edges = g.heavy_edges;
  info->heavy_segments = g.n_seg;
  info->sell_rows = g.n_sell;
  info->sell_slices = g.n_slices;
  info->sell_entries = g.sell_entries;
  info->zero_rows = g.n_zero;
  info->resident_bytes = g.resident_bytes;
  info->build_ms = g.build_ms;
  info->upload_ms = g.upload_ms;
  info->build_peak_bytes = g.build_peak_bytes;
  return MGB200_OK;
}

int mgb200_pagerank_run(mgb200_graph *h, const mgb200_run_params *params, double *rank_out,
                        mgb200_run_stats *stats_out) {
  if (!h || !params) return MGB200_ERR_INVALID_ARGUMENT;
  Graph &g = h->g;
  if (g.part_world != 1) {
    set_error("mgb200_pagerank_run needs a single-partition graph; use mgb200_pagerank_run_partition");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  if (g.n > 0 && !rank_out) {
    set_error("rank_out is null");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  mgb200_run_stats stats{};
  int rc = iterate(g, *params, stats);
  if (rc) return rc;
  if (g.n > 0) {
    double *d_out = rank_out;
    if (!params->rank_out_on_device) {
      if (!g.out_stage) MGB_CUDA(cudaMalloc(&g.out_stage, g.n * sizeof(double)));  // kept for the handle's life
      d_out = g.out_stage;
    }
    rc = launch_write_ranks_original_order(g, d_out);
    if (!rc && !params->rank_out_on_device) {
      cudaError_t e = cudaMemcpyAsync(rank_out, d_out, g.n * sizeof(double), cudaMemcpyDeviceToHost, g.stream);
      if (e != cudaSuccess) rc = cuda_fail(e, "cudaMemcpyAsync(ranks D2H)", __FILE__, __LINE__);
    }
    cudaError_t e = cudaStreamSynchronize(g.stream);
    if (!rc && e != cudaSuccess) rc = cuda_fail(e, "cudaStreamSynchronize", __FILE__, __LINE__);
    if (rc) return rc;
  }
  if (stats_out) *stats_out = stats;
  return MGB200_OK;
}

int mgb200_pagerank_run_partition(mgb200_graph *h, const mgb200_run_params *params, double *rank_out,
                                  uint32_t *vertex_out, mgb200_run_stats *stats_out) {
  if (!h || !params) return MGB200_ERR_INVALID_ARGUMENT;
  Graph &g = h->g;
  if (g.part_world > 1 && !g.peers_connected && !g.tun.lone_partition) {
    set_error("partition is not connected to its peers (mgb200_graph_connect_peers)");
    return MGB200_ERR_COMM;
  }
  mgb200_run_stats stats{};
  int rc = iterate(g, *params, stats);
  if (rc) return rc;
  if (g.local_rows > 0 && rank_out) {
    double *d_out = rank_out;
    uint32_t *d_vtx = vertex_out;
    if (!params->rank_out_on_device) {
      // staging buffer kept for the handle's life (sized n in the single-partition path, local_rows here)
      if (!g.out_stage) MGB_CUDA(cudaMalloc(&g.out_stage, std::max<uint64_t>(g.local_rows, g.part_world == 1 ? g.n : 0) * sizeof(double)));
      d_out = g.out_stage;
      d_vtx = nullptr;
    }
    rc = launch_write_ranks_local(g, d_out, d_vtx);
    cudaError_t e = cudaSuccess;
    if (!rc && !params->rank_out_on_device) {
      e = cudaMemcpyAsync(rank_out, d_out, g.local_rows * sizeof(double), cudaMemcpyDeviceToHost, g.stream);
      if (e == cudaSuccess && vertex_out)
        e = cudaMemcpyAsync(vertex_out, g.local_vertex, g.local_rows * sizeof(uint32_t), cudaMemcpyDeviceToHost,
                            g.stream);
      if (e != cudaSuccess) rc = cuda_fail(e, "cudaMemcpyAsync(ranks D2H)", __FILE__, __LINE__);
    }
    e = cudaStreamSynchronize(g.stream);
    if (!rc && e != cudaSuccess) rc = cuda_fail(e, "cudaStreamSynchronize", __FILE__, __LINE__);
    if (rc) return rc;
  }
  if (stats_out) *stats_out = stats;
  return MGB200_OK;
}

int mgb200_parallel_iterative_pagerank(uint64_t n, uint64_t m, const uint64_t *from, const uint64_t *to,
                                       uint64_t max_iterations, double damping_factor, double stop_epsilon,
                                       uint32_t number_of_threads, double *rank_out, uint64_t *iterations_out) {
  // pagerank.cpp:195-197: the thread count is clamped, then zero is rejected before any work.
  if (number_of_threads == 0) {
    set_error(MGB200_MSG_ZERO_THREADS);
    return MGB200_ERR_ZERO_THREADS;
  }
  if (n == 0) {
    if (iterations_out) *iterations_out = max_iterations != 0 ? 1 : 0;
    // still require a device: the product has no CPU path, even a trivial one
    int count = 0;
    int rc = mgb200_device_count(&count);
    if (rc) return rc;
    if (count <= 0) {
      set_error("CUDA error: no CUDA device available (this library has no CPU fallback)");
      return MGB200_ERR_CUDA;
    }
    return MGB200_OK;
  }
  const char *dev_env = getenv("MGB200_DEVICE");
  const int device = dev_env ? atoi(dev_env) : 0;
  mgb200_graph *g = nullptr;
  int rc = mgb200_graph_create_host(device, n, m, from, to, 0, 1, &g);
  if (rc) return rc;
  mgb200_run_params p{};
  p.max_iterations = max_iterations;
  p.damping_factor = damping_factor;
  p.stop_epsilon = stop_epsilon;
  mgb200_run_stats stats{};
  rc = mgb200_pagerank_run(g, &p, rank_out, &stats);
  mgb200_graph_destroy(g);
  if (rc) return rc;
  if (iterations_out) *iterations_out = stats.iterations;
  return MGB200_OK;
}

}  // extern "C"

namespace {
int poll_flag(void *user) { return static_cast<std::atomic<int> *>(user)->load(std::memory_order_relaxed); }

template <typename T>
int pagerank_multi_impl(uint64_t n, uint64_t m, const T *from, const T *to, const mgb200_run_params *params,
                        uint32_t number_of_threads, uint32_t gpu_count, const int *devices, double *rank_out,
                        uint64_t *iterations_out) {
  if (!params) return MGB200_ERR_INVALID_ARGUMENT;
  if (params->rank_out_on_device) {
    set_error("mgb200_pagerank_multi gathers into host memory (rank_out_on_device must be 0)");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  if (number_of_threads == 0) {
    set_error(MGB200_MSG_ZERO_THREADS);
    return MGB200_ERR_ZERO_THREADS;
  }
  if (gpu_count > static_cast<uint32_t>(kMaxPeers)) {
    set_error("at most " + std::to_string(kMaxPeers) + " GPUs per graph");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  if (gpu_count <= 1 || n == 0) {
    if (n == 0)
      return mgb200_parallel_iterative_pagerank(n, 0, nullptr, nullptr, params->max_iterations, params->damping_factor,
                                                params->stop_epsilon, number_of_threads, rank_out, iterations_out);
    const char *dev_env = getenv("MGB200_DEVICE");
    const int device = devices ? devices[0] : (dev_env ? atoi(dev_env) : 0);
    mgb200_graph *g = nullptr;
    int rc = create_from_host(device, n, m, from, to, 0, 1, &g);
    if (rc) return rc;
    mgb200_run_stats stats{};
    rc = mgb200_pagerank_run(g, params, rank_out, &stats);
    mgb200_graph_destroy(g);
    if (!rc && iterations_out) *iterations_out = stats.iterations;
    return rc;
  }
  std::vector<mgb200_graph *> parts(gpu_count, nullptr);
  auto destroy_all = [&]() {
    for (auto *p : parts) mgb200_graph_destroy(p);
  };
  for (uint32_t q = 0; q < gpu_count; ++q) {
    const int dev = devices ? devices[q] : static_cast<int>(q);
    const int rc = create_from_host(dev, n, m, from, to, q, gpu_count, &parts[q]);
    if (rc) {
      destroy_all();
      return rc;
    }
  }
  for (uint32_t q = 0; q < gpu_count; ++q) {
    const int rc = mgb200_graph_connect_peers(parts[q], nullptr, parts.data());
    if (rc) {
      destroy_all();
      return rc;
    }
  }
  // One host thread per GPU: the partitions meet in device-side barriers, so they must all be launched.  The caller's
  // should_abort hook may only be used from the CALLING thread (mgp_* functions are not thread-safe, mg_procedure.h:75-81),
  // so this thread polls it while the workers run and hands the answer to them through an atomic flag; the device side
  // turns the first partition's request into a collective stop.
  std::atomic<int> abort_flag{0};
  std::atomic<uint32_t> finished{0};
  std::vector<int> rcs(gpu_count, MGB200_OK);
  std::vector<std::string> messages(gpu_count);
  std::vector<std::vector<double>> ranks(gpu_count);
  std::vector<std::vector<uint32_t>> vertices(gpu_count);
  std::vector<mgb200_run_stats> stats(gpu_count);
  std::vector<std::thread> workers;
  for (uint32_t q = 0; q < gpu_count; ++q) {
    workers.emplace_back([&, q]() {
      mgb200_run_params p = *params;
      p.should_abort = params->should_abort ? poll_flag : nullptr;
      p.abort_user = &abort_flag;
      p.rank_out_on_device = 0;
      const uint64_t rows = parts[q]->g.local_rows;
      ranks[q].resize(rows);
      vertices[q].resize(rows);
      rcs[q] = mgb200_pagerank_run_partition(parts[q], &p, ranks[q].data(), vertices[q].data(), &stats[q]);
      if (rcs[q]) messages[q] = mgb200_last_error();
      finished.fetch_add(1, std::memory_order_release);
    });
  }
  while (finished.load(std::memory_order_acquire) < gpu_count) {
    if (params->should_abort && !abort_flag.load(std::memory_order_relaxed) && params->should_abort(params->abort_user))
      abort_flag.store(1, std::memory_order_relaxed);
    std::this_thread::sleep_for(std::chrono::milliseconds(2));
  }
  for (auto &w : workers) w.join();
  destroy_all();
  for (uint32_t q = 0; q < gpu_count; ++q) {
    if (rcs[q]) {
      set_error(messages[q]);
      return rcs[q];
    }
  }
  for (uint32_t q = 0; q < gpu_count; ++q)
    for (size_t r = 0; r < ranks[q].size(); ++r) rank_out[vertices[q][r]] = ranks[q][r];
  if (iterations_out) *iterations_out = stats[0].iterations;
  return MGB200_OK;
}

}  // namespace

extern "C" {

int mgb200_pagerank_multi(uint64_t n, uint64_t m, const uint64_t *from, const uint64_t *to,
                          const mgb200_run_params *params, uint32_t number_of_threads, uint32_t gpu_count,
                          const int *devices, double *rank_out, uint64_t *iterations_out) {
  return pagerank_multi_impl(n, m, from, to, params, number_of_threads, gpu_count, devices, rank_out, iterations_out);
}

int mgb200_pagerank_multi_u32(uint64_t n, uint64_t m, const uint32_t *from, const uint32_t *to,
                              const mgb200_run_params *params, uint32_t number_of_threads, uint32_t gpu_count,
                              const int *devices, double *rank_out, uint64_t *iterations_out) {
  return pagerank_multi_impl(n, m, from, to, params, number_of_threads, gpu_count, devices, rank_out, iterations_out);
}

int mgb200_parallel_iterative_pagerank_multi(uint64_t n, uint64_t m, const uint64_t *from, const uint64_t *to,
                                             uint64_t max_iterations, double damping_factor, double stop_epsilon,
                                             uint32_t number_of_threads, uint32_t gpu_count, const int *devices,
                                             double *rank_out, uint64_t *iterations_out) {
  if (gpu_count <= 1) {
    return mgb200_parallel_iterative_pagerank(n, m, from, to, max_iterations, damping_factor, stop_epsilon,
                                              number_of_threads, rank_out, iterations_out);
  }
  mgb200_run_params p{};
  p.max_iterations = max_iterations;
  p.damping_factor = damping_factor;
  p.stop_epsilon = stop_epsilon;
  return mgb200_pagerank_multi(n, m, from, to, &p, number_of_threads, gpu_count, devices, rank_out, iterations_out);
}

// ---- Katz centrality (include/mgb200_katz.h; kernels in katz.cu) -----------------------------------------

int mgb200_katz_run(mgb200_graph *h, double alpha, double epsilon, uint64_t max_iterations, double *centrality_out,
                    mgb200_katz_stats *stats_out) {
  if (!h) return MGB200_ERR_INVALID_ARGUMENT;
  Graph &g = h->g;
  if (g.n > 0 && !centrality_out) {
    set_error("centrality_out is null");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  MGB_CUDA(cudaSetDevice(g.device));
  if (g.n > 0 && !g.out_stage) MGB_CUDA(cudaMalloc(&g.out_stage, g.n * sizeof(double)));  // kept for the handle's life
  KatzResult res;
  int rc = katz_iterate(g, alpha, epsilon, max_iterations, g.out_stage, &res);
  if (rc) return rc;
  if (g.n > 0) {
    cudaError_t e = cudaMemcpyAsync(centrality_out, g.out_stage, g.n * sizeof(double), cudaMemcpyDeviceToHost, g.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(g.stream);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpyAsync(centralities D2H)", __FILE__, __LINE__);
  }
  if (stats_out) {
    stats_out->iterations = res.iterations;
    stats_out->max_out_degree = res.max_out_degree;
    stats_out->gamma = res.gamma;
    stats_out->iterate_ms = res.iterate_ms;
    stats_out->kernel_launches = res.launches;
    stats_out->tie_order_runs = res.tie_order_runs;
  }
  if (!res.converged) {
    set_error("Katz centrality: max_iterations reached before the ranking separated");
    return MGB200_KATZ_NOT_CONVERGED;
  }
  return MGB200_OK;
}

int mgb200_katz_centrality(uint64_t n, uint64_t m, const uint64_t *from, const uint64_t *to, double alpha,
                           double epsilon, uint64_t max_iterations, double *centrality_out, uint64_t *iterations_out) {
  const char *dev_env = getenv("MGB200_DEVICE");
  const int device = dev_env ? atoi(dev_env) : 0;
  mgb200_graph *g = nullptr;
  int rc = mgb200_graph_create_host(device, n, m, from, to, 0, 1, &g);  // fails without a device, also for n == 0
  if (rc) return rc;
  mgb200_katz_stats stats{};
  rc = mgb200_katz_run(g, alpha, epsilon, max_iterations, centrality_out, &stats);
  mgb200_graph_destroy(g);
  if (iterations_out) *iterations_out = stats.iterations;
  return rc;
}

// ---- cuGraph-semantics PageRank (include/mgb200_personalized.h; kernels in personalized.cu) ---------------------

int mgb200_cugraph_pagerank_run(mgb200_graph *h, const mgb200_cugraph_params *params, double *rank_out,
                                mgb200_cugraph_stats *stats_out) {
  if (!h || !params) return MGB200_ERR_INVALID_ARGUMENT;
  Graph &g = h->g;
  if (g.part_world != 1) {
    set_error("mgb200_cugraph_pagerank_run needs a single-partition graph");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  if (g.n > 0 && !rank_out) {
    set_error("rank_out is null");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  if (params->n_personalization && (!params->personalization_vertices || !params->personalization_values)) {
    set_error("null personalization arrays");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  MGB_CUDA(cudaSetDevice(g.device));
  if (g.n > 0 && !g.out_stage) MGB_CUDA(cudaMalloc(&g.out_stage, g.n * sizeof(double)));  // kept for the handle's life
  mgb200_cugraph_stats stats{};
  int rc = cugraph_pagerank_iterate(g, *params, g.out_stage, &stats);
  if (rc) return rc;
  if (g.n > 0) {
    cudaError_t e = cudaMemcpyAsync(rank_out, g.out_stage, g.n * sizeof(double), cudaMemcpyDeviceToHost, g.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(g.stream);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpyAsync(ranks D2H)", __FILE__, __LINE__);
  }
  if (stats_out) *stats_out = stats;
  return MGB200_OK;
}

int mgb200_partition_range(uint64_t n, uint32_t part_world, uint32_t part_rank, uint64_t *first_label_out,
                           uint64_t *rows_out) {
  if (part_world == 0 || part_world > static_cast<uint32_t>(kMaxPeers) || part_rank >= part_world) {
    set_error("invalid partition: rank " + std::to_string(part_rank) + " of " + std::to_string(part_world));
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  // same arithmetic as Dealer in graph_build.cu: sorted position p belongs to owner p % world
  const uint64_t base = n / part_world, extra = n % part_world;
  if (first_label_out) *first_label_out = static_cast<uint64_t>(part_rank) * base + std::min<uint64_t>(part_rank, extra);
  if (rows_out) *rows_out = base + (part_rank < extra ? 1 : 0);
  return MGB200_OK;
}

namespace {
int make_row_map(uint64_t n, uint64_t heavy_rows, uint32_t part_world, int global_order, uint32_t part_rank,
                 RowMap *map) {
  if (part_world == 0 || part_world > static_cast<uint32_t>(kMaxPeers) || part_rank >= part_world ||
      (global_order && heavy_rows > n)) {
    set_error("invalid partition: rank " + std::to_string(part_rank) + " of " + std::to_string(part_world));
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  *map = RowMap{};
  map->n = n;
  map->heavy = global_order ? heavy_rows : 0;
  map->world = part_world;
  map->rank = part_rank;
  map->global_order = global_order ? 1u : 0u;
  map->finalize();
  return MGB200_OK;
}
}  // namespace

int mgb200_partition_locate(uint64_t n, uint64_t heavy_rows, uint32_t part_world, int global_order, uint64_t label,
                            uint32_t *owner_out, uint64_t *local_row_out) {
  RowMap map;
  const int rc = make_row_map(n, heavy_rows, part_world, global_order, 0, &map);
  if (rc != MGB200_OK) return rc;
  if (label >= n) {
    set_error("label out of range");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  if (owner_out) *owner_out = map.owner(label);
  if (local_row_out) *local_row_out = map.local_of(label);
  return MGB200_OK;
}

int mgb200_partition_label(uint64_t n, uint64_t heavy_rows, uint32_t part_world, int global_order, uint32_t part_rank,
                           uint64_t local_row, uint64_t *label_out, uint64_t *rows_out) {
  RowMap map;
  const int rc = make_row_map(n, heavy_rows, part_world, global_order, part_rank, &map);
  if (rc != MGB200_OK) return rc;
  const uint64_t rows = map.local_rows(part_rank);
  if (rows_out) *rows_out = rows;
  if (label_out) {
    if (local_row >= rows) {
      set_error("local row out of range");
      return MGB200_ERR_INVALID_ARGUMENT;
    }
    *label_out = map.label_of_local(local_row);
  }
  return MGB200_OK;
}

// ---- multi-GPU wiring ---------------------------------------------------------------------------------

int mgb200_graph_export_window(mgb200_graph *h, void *ipc_handle_out) {
  if (!h || !ipc_handle_out) return MGB200_ERR_INVALID_ARGUMENT;
  static_assert(sizeof(cudaIpcMemHandle_t) == MGB200_IPC_HANDLE_BYTES, "IPC handle size");
  MGB_CUDA(cudaSetDevice(h->g.device));
  cudaIpcMemHandle_t handle;
  MGB_CUDA(cudaIpcGetMemHandle(&handle, h->g.window));
  memcpy(ipc_handle_out, &handle, sizeof(handle));
  return MGB200_OK;
}

int mgb200_graph_connect_peers(mgb200_graph *h, const void *const *ipc_handles, mgb200_graph *const *peer_graphs) {
  if (!h) return MGB200_ERR_INVALID_ARGUMENT;
  Graph &g = h->g;
  MGB_CUDA(cudaSetDevice(g.device));
  for (uint32_t q = 0; q < g.part_world; ++q) {
    if (q == g.part_rank) continue;
    void *base = nullptr;
    if (peer_graphs && peer_graphs[q]) {
      const Graph &pg = peer_graphs[q]->g;
      if (pg.n != g.n || pg.part_world != g.part_world || pg.part_rank != q) {
        set_error("peer graph does not belong to the same partitioned graph");
        return MGB200_ERR_COMM;
      }
      if (pg.device != g.device) {
        int can = 0;
        MGB_CUDA(cudaDeviceCanAccessPeer(&can, g.device, pg.device));
        if (!can) {
          set_error("devices " + std::to_string(g.device) + " and " + std::to_string(pg.device) +
                    " are not NVLink/P2P peers");
          return MGB200_ERR_COMM;
        }
        cudaError_t e = cudaDeviceEnablePeerAccess(pg.device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
          return cuda_fail(e, "cudaDeviceEnablePeerAccess", __FILE__, __LINE__);
        cudaGetLastError();
      }
      base = pg.window;
    } else if (ipc_handles && ipc_handles[q]) {
      cudaIpcMemHandle_t handle;
      memcpy(&handle, ipc_handles[q], sizeof(handle));
      MGB_CUDA(cudaIpcOpenMemHandle(&base, handle, cudaIpcMemLazyEnablePeerAccess));
      g.peer_mapped[q] = base;
    } else {
      set_error("no handle for peer partition " + std::to_string(q));
      return MGB200_ERR_COMM;
    }
    char *bytes = static_cast<char *>(base);
    g.peers.flags[q] = reinterpret_cast<FlagPage *>(bytes);
    g.peers.contrib[0][q] = reinterpret_cast<double *>(bytes + kFlagPageBytes);
    g.peers.contrib[1][q] = reinterpret_cast<double *>(bytes + kFlagPageBytes + g.contrib_stride);
  }
  // a fresh connection starts every partition's barrier counter from zero (all partitions reconnect together, before
  // any run): this is also how a set of handles recovers after a peer time-out poisoned them
  MGB_CUDA(cudaMemset(g.window, 0, kFlagPageBytes));
  MGB_CUDA(cudaMemset(&g.state->barrier_seq, 0, sizeof(unsigned long long)));
  g.poisoned = false;
  g.peers_connected = true;
  return MGB200_OK;
}

// ---- synthetic workload ------------------------------------------------------------------------------

int mgb200_rmat_generate_device(int device, uint32_t scale, uint64_t first_edge, uint64_t count, uint64_t seed,
                                double a, double b, double c, uint32_t *d_from, uint32_t *d_to) {
  if (scale == 0 || scale > 31 || (count > 0 && (!d_from || !d_to))) {
    set_error("rmat: scale must be in [1, 31] and outputs non-null");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  int rc = check_device(device);
  if (rc) return rc;
  MGB_CUDA(cudaSetDevice(device));
  if (count == 0) return MGB200_OK;
  const RmatThresholds t = rmat_thresholds(a, b, c);
  const int blocks = static_cast<int>(std::min<uint64_t>((count + 255) / 256, 148ull * 32));
  rmat_kernel<<<blocks, 256>>>(scale, first_edge, count, seed, t, d_from, d_to);
  MGB_CUDA(cudaGetLastError());
  MGB_CUDA(cudaDeviceSynchronize());
  return MGB200_OK;
}

int mgb200_rmat_generate_host(uint32_t scale, uint64_t first_edge, uint64_t count, uint64_t seed, double a, double b,
                              double c, uint64_t *from, uint64_t *to) {
  if (scale == 0 || scale > 31 || (count > 0 && (!from || !to))) {
    set_error("rmat: scale must be in [1, 31] and outputs non-null");
    return MGB200_ERR_INVALID_ARGUMENT;
  }
  const RmatThresholds t = rmat_thresholds(a, b, c);
  for (uint64_t i = 0; i < count; ++i) {
    uint32_t s, d;
    rmat_edge(scale, first_edge + i, seed, t, s, d);
    from[i] = s;
    to[i] = d;
  }
  return MGB200_OK;
}

// ---- device-memory helpers -----------------------------------------------------------------------------

int mgb200_device_malloc(int device, size_t bytes, void **ptr_out) {
  if (!ptr_out) return MGB200_ERR_INVALID_ARGUMENT;
  *ptr_out = nullptr;
  int rc = check_device(device);
  if (rc) return rc;
  MGB_CUDA(cudaSetDevice(device));
  MGB_CUDA(cudaMalloc(ptr_out, bytes ? bytes : 1));
  return MGB200_OK;
}

int mgb200_device_free(int device, void *ptr) {
  int rc = check_device(device);
  if (rc) return rc;
  MGB_CUDA(cudaSetDevice(device));
  MGB_CUDA(cudaFree(ptr));
  return MGB200_OK;
}

int mgb200_copy_to_device(int device, void *dst_device, const void *src_host, size_t bytes) {
  int rc = check_device(device);
  if (rc) return rc;
  MGB_CUDA(cudaSetDevice(device));
  MGB_CUDA(cudaMemcpy(dst_device, src_host, bytes, cudaMemcpyHostToDevice));
  return MGB200_OK;
}

int mgb200_copy_to_host(int device, void *dst_host, const void *src_device, size_t bytes) {
  int rc = check_device(device);
  if (rc) return rc;
  MGB_CUDA(cudaSetDevice(device));
  MGB_CUDA(cudaMemcpy(dst_host, src_device, bytes, cudaMemcpyDeviceToHost));
  return MGB200_OK;
}

int mgb200_device_info(int device, char *name_out, size_t name_cap, int *sm_count, size_t *total_bytes) {
  int rc = check_device(device);
  if (rc) return rc;
  cudaDeviceProp prop{};
  MGB_CUDA(cudaGetDeviceProperties(&prop, device));
  if (name_out && name_cap) {
    strncpy(name_out, prop.name, name_cap - 1);
    name_out[name_cap - 1] = '\0';
  }
  if (sm_count) *sm_count = prop.multiProcessorCount;
  if (total_bytes) *total_bytes = prop.totalGlobalMem;
  return MGB200_OK;
}

}  // extern "C"
