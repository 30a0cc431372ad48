// Pieces of the "expand -> stable radix sort by (local row, column) -> run heads" product shared
// by the centroid rows of csrc/hge_jaccard.cu and the candidate rows of
// csrc/hge_device_sampler.cu.  Keys are (local row << 32) | column, sorted ascending, so the runs
// of one row are its distinct columns in ascending order.
#pragma once

#include <algorithm>

#include "hge_common.cuh"

namespace {

constexpr int kExpandBlock = 256;

int grid_for(const hge_ctx* ctx, int64_t work, int per_block = kExpandBlock) {
  const int64_t want = std::max<int64_t>(1, (work + per_block - 1) / per_block);
  return (int)std::min<int64_t>(want, (int64_t)ctx->num_sms * 16);
}

// device buffer released when it goes out of scope (stream-ordered)
template <typename T>
struct DevBuf {
  const hge_ctx* ctx;
  T* p = nullptr;
  explicit DevBuf(const hge_ctx* c) : ctx(c) {}
  ~DevBuf() { hge_dev_free(ctx, p); }
  int alloc(size_t n) {
    hge_dev_free(ctx, p);
    return hge_dev_alloc(ctx, &p, n);
  }
};

template <typename T>
int read_back(hge_ctx* ctx, const T* dev, T* host, size_t n) {
  HGE_CUDA(cudaMemcpyAsync(host, dev, n * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
  HGE_CUDA(cudaStreamSynchronize(ctx->stream));
  return HGE_OK;
}

// head[i] = 1 where a run of equal keys starts
__global__ void k_run_heads(int64_t n, const uint64_t* __restrict__ keys, int64_t* __restrict__ head) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    head[i] = (i == 0 || keys[i] != keys[i - 1]) ? 1 : 0;
}

// start[g0 + k] for k in [0, g1 - g0) (and k = g1 - g0 when last_batch): rows_before + position,
// among the runs of the sorted keys, of the first run of local row k (pos = exclusive scan of
// the run heads, n_runs = number of runs)
__global__ void k_run_starts(int64_t g0, int64_t g1, int64_t n, int64_t n_runs, int64_t rows_before,
                             const uint64_t* __restrict__ keys, const int64_t* __restrict__ pos,
                             int64_t* __restrict__ start, bool last_batch) {
  const int64_t count = g1 - g0 + (last_batch ? 1 : 0);
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < count;
       k += (int64_t)gridDim.x * blockDim.x) {
    const uint64_t want = (uint64_t)k << 32;
    int64_t lo = 0, hi = n;
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (keys[mid] < want) lo = mid + 1; else hi = mid;
    }
    start[g0 + k] = rows_before + (lo < n ? pos[lo] : n_runs);
  }
}

}  // namespace
