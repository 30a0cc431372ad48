// Range check of (a, b) index pairs, run by the entry points whose kernels read row pointers at
// the pair indices unchecked (csrc/hge_weighting.cu, csrc/hge_jaccard.cu): every index is checked
// before any of those kernels runs, and a bad one is HGE_ERR_INVALID.
#pragma once

#include "hge_common.cuh"

namespace {

constexpr int kPairCheckBlock = 256;

__global__ void k_check_pairs(int64_t n, const int32_t* __restrict__ a, int64_t rows_a,
                              const int32_t* __restrict__ b, int64_t rows_b, int* __restrict__ bad) {
  for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < n;
       p += (int64_t)gridDim.x * blockDim.x) {
    const int32_t x = __ldcs(a + p), y = __ldcs(b + p);
    if (x < 0 || x >= rows_a || y < 0 || y >= rows_b) *bad = 1;
  }
}

// *ok = every a[p] in [0, rows_a) and every b[p] in [0, rows_b).  Host arrays are scanned on the
// host; device arrays by k_check_pairs, then one flag read-back.
int pairs_in_range(hge_ctx* ctx, int64_t n, const int32_t* a, int64_t rows_a, const int32_t* b,
                   int64_t rows_b, int mem, bool* ok) {
  if (mem != HGE_MEM_DEVICE) {
    bool all = true;
    for (int64_t p = 0; p < n; ++p)
      all &= a[p] >= 0 && a[p] < rows_a && b[p] >= 0 && b[p] < rows_b;
    *ok = all;
    return HGE_OK;
  }
  DevBuf<int> d_bad(ctx);
  HGE_TRY(d_bad.alloc(1));
  HGE_CUDA(cudaMemsetAsync(d_bad.p, 0, sizeof(int), ctx->stream));
  k_check_pairs<<<grid_for(ctx, n, kPairCheckBlock * 8), kPairCheckBlock, 0, ctx->stream>>>(n, a, rows_a, b,
                                                                                          rows_b, d_bad.p);
  HGE_CHECK_LAUNCH(ctx);
  int h_bad = 0;
  HGE_TRY(read_back(ctx, d_bad.p, &h_bad, 1));
  *ok = h_bad == 0;
  return HGE_OK;
}

}  // namespace
