// Pieces of the "expand -> stable radix sort by (local row, column) -> run heads" product shared
// by the centroid rows of csrc/hge_jaccard.cu and the candidate rows of
// csrc/hge_device_sampler.cu.  Keys are (local row << 32) | column, sorted ascending, so the runs
// of one row are its distinct columns in ascending order.  Also the grouping of (x, group) pairs
// by group shared by the centroid factors of csrc/hge_jaccard.cu and hge_lp_svm_predict
// (csrc/hge_lp_svm.cu).
#pragma once

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "hge_common.cuh"

namespace {

constexpr int kExpandBlock = 256;

// head[i] = 1 where a run of equal keys starts
__global__ void k_run_heads(int64_t n, const uint64_t* __restrict__ keys, int64_t* __restrict__ head) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    head[i] = (i == 0 || keys[i] != keys[i - 1]) ? 1 : 0;
}

// start[k] for k in [0, L]: position, among the runs of the sorted keys, of the first run of
// local row k (pos = exclusive scan of the run heads, n_runs = number of runs = start[L])
__global__ void k_run_starts(int64_t L, int64_t n, int64_t n_runs, const uint64_t* __restrict__ keys,
                             const int64_t* __restrict__ pos, int64_t* __restrict__ start) {
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k <= L;
       k += (int64_t)gridDim.x * blockDim.x) {
    const uint64_t want = (uint64_t)k << 32;
    int64_t lo = 0, hi = n;
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (keys[mid] < want) lo = mid + 1; else hi = mid;
    }
    start[k] = lo < n ? pos[lo] : n_runs;
  }
}


enum : int { kBadX = 1, kBadGroup = 2 };

// sort input of the pairs: key = group, value = pair index; out-of-range ids are flagged
__global__ void k_pair_keys(int64_t num_pairs, const int32_t* __restrict__ px, int64_t xrows,
                            const int32_t* __restrict__ pg, int64_t groups, uint32_t* __restrict__ key,
                            int32_t* __restrict__ idx, int* __restrict__ status) {
  for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < num_pairs;
       p += (int64_t)gridDim.x * blockDim.x) {
    const int32_t x = px[p], g = pg[p];
    if (x < 0 || x >= xrows) atomicOr(status, kBadX);
    const bool bad_g = g < 0 || g >= groups;
    if (bad_g) atomicOr(status, kBadGroup);
    key[p] = bad_g ? 0u : (uint32_t)g;
    idx[p] = (int32_t)p;
  }
}

// head[i] = 1 where the run of pairs of one group starts (sorted group ids)
__global__ void k_pair_heads(int64_t n, const uint32_t* __restrict__ sg, int32_t* __restrict__ head) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    head[i] = (i == 0 || sg[i] != sg[i - 1]) ? 1 : 0;
}

// named group u = run u of the sorted pairs (u = rank[i] - 1, rank = inclusive scan of the heads):
// ug[u] its group id, ustart[u] its first sorted pair; ustart[U] = n
__global__ void k_named_groups(int64_t n, const uint32_t* __restrict__ sg, const int32_t* __restrict__ head,
                               const int32_t* __restrict__ rank, int32_t* __restrict__ ug,
                               int64_t* __restrict__ ustart) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    if (head[i]) {
      ug[rank[i] - 1] = (int32_t)sg[i];
      ustart[rank[i] - 1] = i;
    }
    if (i == n - 1) ustart[rank[i]] = n;
  }
}

// Pairs (x, group) stably sorted by group, and the groups they name.  After build(): order[i] is
// the pair at sorted position i, rank[i] - 1 its named group, ug[u] the group id of named group u
// (ascending), ustart[u] its first sorted position (ustart[U] = n).  *bad receives kBadX / kBadGroup
// when a pair names an x outside [0, xrows) or a group outside [0, groups); nothing else is built
// then.  n in [1, 2^31).
struct PairGroups {
  DevBuf<uint32_t> key, key2;
  DevBuf<int32_t> idx, idx2, rank, ug;
  DevBuf<int64_t> ustart;
  const int32_t* order = nullptr;
  int64_t U = 0;
  explicit PairGroups(const hge_ctx* c) : key(c), key2(c), idx(c), idx2(c), rank(c), ug(c), ustart(c) {}

  int build(hge_ctx* ctx, int64_t n, const int32_t* px, int64_t xrows, const int32_t* pg, int64_t groups,
            int* bad) {
    DevBuf<int32_t> head(ctx);
    DevBuf<int> status(ctx);
    DevBuf<char> temp(ctx);
    HGE_TRY(key.alloc((size_t)n));
    HGE_TRY(key2.alloc((size_t)n));
    HGE_TRY(idx.alloc((size_t)n));
    HGE_TRY(idx2.alloc((size_t)n));
    HGE_TRY(status.alloc(1));
    HGE_CUDA(cudaMemsetAsync(status.p, 0, sizeof(int), ctx->stream));
    k_pair_keys<<<grid_for(ctx, n), kExpandBlock, 0, ctx->stream>>>(n, px, xrows, pg, groups, key.p, idx.p,
                                                                   status.p);
    HGE_CHECK_LAUNCH(ctx);
    HGE_TRY(read_back(ctx, status.p, bad, 1));
    if (*bad) return HGE_OK;
    int group_bits = 1;
    while ((1ll << group_bits) < groups) ++group_bits;
    cub::DoubleBuffer<uint32_t> dk(key.p, key2.p);
    cub::DoubleBuffer<int32_t> dv(idx.p, idx2.p);
    size_t bytes = 0;
    HGE_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, bytes, dk, dv, n, 0, group_bits, ctx->stream));
    HGE_TRY(temp.alloc(bytes));
    HGE_CUDA(cub::DeviceRadixSort::SortPairs(temp.p, bytes, dk, dv, n, 0, group_bits, ctx->stream));
    ctx->launches++;
    const uint32_t* sg = dk.Current();
    order = dv.Current();
    HGE_TRY(head.alloc((size_t)n));
    HGE_TRY(rank.alloc((size_t)n));
    k_pair_heads<<<grid_for(ctx, n), kExpandBlock, 0, ctx->stream>>>(n, sg, head.p);
    HGE_CHECK_LAUNCH(ctx);
    HGE_CUDA(cub::DeviceScan::InclusiveSum(nullptr, bytes, head.p, rank.p, n, ctx->stream));
    HGE_TRY(temp.alloc(bytes));
    HGE_CUDA(cub::DeviceScan::InclusiveSum(temp.p, bytes, head.p, rank.p, n, ctx->stream));
    ctx->launches++;
    int32_t U32 = 0;
    HGE_TRY(read_back(ctx, rank.p + n - 1, &U32, 1));
    U = U32;
    HGE_TRY(ug.alloc((size_t)U));
    HGE_TRY(ustart.alloc((size_t)U + 1));
    k_named_groups<<<grid_for(ctx, n), kExpandBlock, 0, ctx->stream>>>(n, sg, head.p, rank.p, ug.p, ustart.p);
    HGE_CHECK_LAUNCH(ctx);
    return HGE_OK;
  }
};

}  // namespace
