// memgraph_b200/csrc/personalized.cu -- cuGraph-semantics PageRank (uniform or personalised teleport, dangling mass
// redistributed, L1 stop test) on the PageRank graph layout; include/mgb200_personalized.h has the recurrence and the
// reference call sites.  The gather phase is PageRank's (launch_gather_phase: SELL row sums, heavy row sums, same cache
// policies); only the vector preparation (contribution + dangling mass) and the row epilogue differ:
//   prepare : contrib[l] = pr[l] / outdeg[l] (0 for sinks), dangling = sum of pr over sinks      one pass over N labels
//   epilogue: new[r] = alpha * gathered[r] + (alpha * dangling + 1 - alpha) * p[r], L1 diff       one pass over N rows
// Both reductions are two-stage with a fixed tree (per-block partials, then one block), every row is gathered in a
// fixed order, and the out-weight sums of a weighted handle are summed on the host in input edge order
// (mgb200_graph_create_host_weighted_u32): results are bit-reproducible run to run and handle to handle, whatever the
// gather configuration or build chunking, which cuGraph itself is not.  One partition: label == local row, so pr, p and
// the gathered sums share one index space.
#include <algorithm>
#include <vector>

#include "core.hpp"
#include "mgb200_personalized.h"

namespace mgb200 {
namespace {

constexpr int kThreads = 256;
constexpr int kPartials = 1024;

inline int blocks_for(uint64_t items) {
  return static_cast<int>(std::max<uint64_t>(1, std::min<uint64_t>((items + kThreads * 4 - 1) / (kThreads * 4), kPartials)));
}

__device__ __forceinline__ double block_sum(double v) {
  __shared__ double sm[kThreads];
  sm[threadIdx.x] = v;
  __syncthreads();
  for (int o = kThreads / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) sm[threadIdx.x] += sm[threadIdx.x + o];
    __syncthreads();
  }
  return sm[0];
}

__global__ void __launch_bounds__(kThreads) ppr_init_kernel(uint64_t n, double *pr, double *contrib_pad, IterState *state) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  const double r0 = 1.0 / static_cast<double>(n);
  for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) pr[i] = r0;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    contrib_pad[n] = 0.0;  // the slot SELL padding entries read
    state->done = 0;       // the gather kernels return at once while this is set
    state->error = 0;
  }
}

// chunked like partial_sum_kernel: block b owns one contiguous chunk, so the partials do not depend on the grid's timing
__global__ void __launch_bounds__(kThreads) ppr_prepare_kernel(uint64_t n, const double *pr, const uint32_t *outdeg,
                                                               const double *out_weight, double *contrib, double *partials) {
  const uint64_t chunk = (n + gridDim.x - 1) / gridDim.x;
  const uint64_t lo = chunk * blockIdx.x, hi = min(lo + chunk, n);
  double dangling = 0.0;
  for (uint64_t l = lo + threadIdx.x; l < hi; l += blockDim.x) {
    // out-weight sum: the weights' sum on a weighted handle, the out-degree otherwise (every edge counts 1)
    const double ow = out_weight ? out_weight[l] : static_cast<double>(outdeg[l]);
    const double r = pr[l];
    contrib[l] = ow != 0.0 ? __ddiv_rn(r, ow) : 0.0;
    if (ow == 0.0) dangling += r;
  }
  const double s = block_sum(dangling);
  if (threadIdx.x == 0) partials[blockIdx.x] = s;
}

__global__ void __launch_bounds__(kThreads) ppr_reduce_kernel(const double *partials, int count, double *out) {
  double acc = 0.0;
  for (int i = threadIdx.x; i < count; i += blockDim.x) acc += partials[i];
  const double s = block_sum(acc);
  if (threadIdx.x == 0) *out = s;
}

struct PprRows {
  uint64_t n, n_heavy, n_sell;
  const double *heavy_sums, *sell_sums;
  const double *pr;
  const double *p;  // nullptr: uniform 1/N
  double *pr_new;
  double alpha;
  const double *dangling;
};

__global__ void __launch_bounds__(kThreads) ppr_epilogue_kernel(PprRows a, double *partials) {
  const uint64_t chunk = (a.n + gridDim.x - 1) / gridDim.x;
  const uint64_t lo = chunk * blockIdx.x, hi = min(lo + chunk, a.n);
  const double spread = a.alpha * (*a.dangling) + (1.0 - a.alpha);
  const double uniform = 1.0 / static_cast<double>(a.n);
  double diff = 0.0;
  for (uint64_t r = lo + threadIdx.x; r < hi; r += blockDim.x) {
    const double gathered = r < a.n_heavy ? a.heavy_sums[r] : (r < a.n_heavy + a.n_sell ? a.sell_sums[r - a.n_heavy] : 0.0);
    const double nw = a.alpha * gathered + spread * (a.p ? a.p[r] : uniform);
    diff += fabs(nw - a.pr[r]);
    a.pr_new[r] = nw;
  }
  const double s = block_sum(diff);
  if (threadIdx.x == 0) partials[blockIdx.x] = s;
}

__global__ void __launch_bounds__(kThreads) ppr_write_kernel(uint64_t n, const uint32_t *label_of, const double *pr,
                                                             double *out) {
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (uint64_t v = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; v < n; v += stride) out[v] = pr[label_of[v]];
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

}  // namespace

int cugraph_pagerank_iterate(Graph &g, const mgb200_cugraph_params &prm, double *d_out_original_order,
                             mgb200_cugraph_stats *stats) {
  MGB_CUDA(cudaSetDevice(g.device));
  const uint64_t n = g.n;
  *stats = mgb200_cugraph_stats{};
  stats->converged = 1;
  if (n == 0) return MGB200_OK;
  cudaStream_t st = g.stream;
  Scratch tmp;
  double *pr_new = nullptr, *p = nullptr, *partials = nullptr, *scalars = nullptr;  // scalars: [0] dangling, [1] diff
  MGB_CUDA(tmp.alloc(&pr_new, n));
  MGB_CUDA(tmp.alloc(&partials, kPartials));
  MGB_CUDA(tmp.alloc(&scalars, 2));
  if (prm.n_personalization) {
    // p by label, built on the host from the (few) seeds: normalised values, duplicates add up
    double sum = 0.0;
    for (uint64_t i = 0; i < prm.n_personalization; ++i) {
      if (prm.personalization_vertices[i] >= n) {
        set_error("personalization vertex out of range");
        return MGB200_ERR_INVALID_ARGUMENT;
      }
      sum += prm.personalization_values[i];
    }
    if (!(sum > 0.0)) {
      set_error("personalization values must sum to a positive number");
      return MGB200_ERR_INVALID_ARGUMENT;
    }
    MGB_CUDA(tmp.alloc(&p, n));
    MGB_CUDA(cudaMemsetAsync(p, 0, n * sizeof(double), st));
    std::vector<uint32_t> labels(prm.n_personalization);
    std::vector<uint32_t> ids(prm.n_personalization);
    for (uint64_t i = 0; i < prm.n_personalization; ++i) ids[i] = static_cast<uint32_t>(prm.personalization_vertices[i]);
    // label_of lives on the device: fetch the seeds' labels one by one (seed lists are short)
    for (uint64_t i = 0; i < prm.n_personalization; ++i)
      MGB_CUDA(cudaMemcpyAsync(&labels[i], g.label_of + ids[i], sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    MGB_CUDA(cudaStreamSynchronize(st));
    std::vector<std::pair<uint32_t, double>> seeds;
    for (uint64_t i = 0; i < prm.n_personalization; ++i) seeds.emplace_back(labels[i], prm.personalization_values[i] / sum);
    std::sort(seeds.begin(), seeds.end(), [](const auto &a, const auto &b) { return a.first < b.first; });
    for (size_t i = 0; i < seeds.size();) {  // duplicates add up, in a fixed order
      double v = 0.0;
      size_t j = i;
      for (; j < seeds.size() && seeds[j].first == seeds[i].first; ++j) v += seeds[j].second;
      MGB_CUDA(cudaMemcpyAsync(p + seeds[i].first, &v, sizeof(double), cudaMemcpyHostToDevice, st));
      MGB_CUDA(cudaStreamSynchronize(st));  // `v` is a stack temporary
      i = j;
    }
  }
  double *pr = g.rank;  // [n] at one partition
  double *contrib = g.contrib(0);
  uint64_t launches = 0;
  MGB_CUDA(cudaEventRecord(g.ev[2], st));
  ppr_init_kernel<<<blocks_for(n), kThreads, 0, st>>>(n, pr, contrib, g.state);
  ++launches;
  const int blocks = blocks_for(n);
  uint64_t it = 0;
  int converged = 0;
  double diff_host = 0.0;
  while (true) {
    ppr_prepare_kernel<<<blocks, kThreads, 0, st>>>(n, pr, g.outdeg_l, g.outw_l, contrib, partials);
    ppr_reduce_kernel<<<1, kThreads, 0, st>>>(partials, blocks, scalars);
    launches += 2;
    int rc = launch_gather_phase(g, contrib, &launches, /*heavy_row_sums=*/true, /*weighted=*/g.outw_l != nullptr);
    if (rc) return rc;
    PprRows rows{n, g.n_heavy, g.n_sell, g.heavy_sums, g.sell_sums, pr, p, pr_new, prm.damping_factor, scalars};
    ppr_epilogue_kernel<<<blocks, kThreads, 0, st>>>(rows, partials);
    ppr_reduce_kernel<<<1, kThreads, 0, st>>>(partials, blocks, scalars + 1);
    launches += 2;
    MGB_CUDA(cudaMemcpyAsync(&diff_host, scalars + 1, sizeof(double), cudaMemcpyDeviceToHost, st));
    MGB_CUDA(cudaStreamSynchronize(st));
    std::swap(pr, pr_new);
    ++it;
    if (diff_host < prm.stop_epsilon) {
      converged = 1;
      break;
    }
    if (it >= prm.max_iterations) break;
  }
  ppr_write_kernel<<<blocks_for(n), kThreads, 0, st>>>(n, g.label_of, pr, d_out_original_order);
  ++launches;
  MGB_CUDA(cudaEventRecord(g.ev[3], st));
  MGB_CUDA(cudaStreamSynchronize(st));
  MGB_CUDA(cudaGetLastError());
  float ms = 0.f;
  MGB_CUDA(cudaEventElapsedTime(&ms, g.ev[2], g.ev[3]));
  stats->iterations = it;
  stats->converged = converged;
  stats->last_diff_sum = diff_host;
  stats->iterate_ms = ms;
  stats->kernel_launches = launches;
  return MGB200_OK;
}

}  // namespace mgb200
