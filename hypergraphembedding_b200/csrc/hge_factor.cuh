// The padded dense factor layout and the incidence product of the factorizations of the node-edge
// incidence: the non-negative factorization (csrc/hge_nmf.cu) and the truncated SVD
// (csrc/hge_svd.cu).  A dense factor is [rows, ld] fp32 row-major, ld = columns rounded up to a
// multiple of 4, the padding columns zero.
#pragma once

#include <algorithm>

#include "hge_common.cuh"

namespace {

constexpr int kFactorBlock = 256;  // threads per block of k_nmf_spmm
constexpr int kSpmmUnroll = 8;     // neighbour rows in flight per sub-warp

inline int factor_ld(int k) { return (k + 3) & ~3; }

// [rows, k] -> [rows, ld] with zero columns k .. ld - 1
__global__ void k_nmf_pad(int64_t rows, int k, int ld, const float* __restrict__ x, float* __restrict__ y) {
  const int64_t total = rows * ld;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / ld;
    const int c = (int)(i - r * ld);
    y[i] = c < k ? x[r * k + c] : 0.f;
  }
}

// P = A Y over a CSR (the node -> edge CSR gives A Y, the edge -> node CSR A^T Y): each row adds
// its neighbours' rows in ascending incidence order, one fp32 add per neighbour from +0 -- scipy's
// order, so P equals scipy's float32 product bit for bit.  A sub-warp of LPR lanes owns a row, a
// lane LPR-strided float4 columns.  Long rows are not split: a split would change the order.
template <int LPR, int S>
__global__ void __launch_bounds__(kFactorBlock) k_nmf_spmm(int32_t rows, const int64_t* __restrict__ ptr,
                                                            const int32_t* __restrict__ idx,
                                                            const float4* __restrict__ y, int ld4,
                                                            float4* __restrict__ p) {
  const int gl = threadIdx.x & (LPR - 1);
  const int64_t sub = ((int64_t)blockIdx.x * kFactorBlock + threadIdx.x) / LPR;
  const int64_t nsub = (int64_t)gridDim.x * kFactorBlock / LPR;
  for (int64_t row = sub; row < rows; row += nsub) {
    const int64_t b = ptr[row], e = ptr[row + 1];
    float4 acc[S];
#pragma unroll
    for (int s = 0; s < S; ++s) acc[s] = hge_f4_zero();
    for (int64_t q = b; q < e; q += kSpmmUnroll) {
      int32_t id[kSpmmUnroll];
#pragma unroll
      for (int u = 0; u < kSpmmUnroll; ++u) id[u] = q + u < e ? __ldg(idx + q + u) : -1;
      float4 v[kSpmmUnroll][S];
#pragma unroll
      for (int u = 0; u < kSpmmUnroll; ++u)
#pragma unroll
        for (int s = 0; s < S; ++s) {
          const int c = s * LPR + gl;
          v[u][s] = (id[u] >= 0 && c < ld4) ? __ldg(y + (size_t)id[u] * ld4 + c) : hge_f4_zero();
        }
#pragma unroll
      for (int u = 0; u < kSpmmUnroll; ++u)
        if (id[u] >= 0)
#pragma unroll
          for (int s = 0; s < S; ++s) hge_f4_add(acc[s], v[u][s]);
    }
#pragma unroll
    for (int s = 0; s < S; ++s) {
      const int c = s * LPR + gl;
      if (c < ld4) p[(size_t)row * ld4 + c] = acc[s];
    }
  }
}

typedef void (*SpmmKernel)(int32_t, const int64_t*, const int32_t*, const float4*, int, float4*);

// sub-warp width: next power of two of ld / 4, at most 32; two column slabs above 128 columns
inline SpmmKernel spmm_kernel(int ld4) {
  if (ld4 <= 1) return k_nmf_spmm<1, 1>;
  if (ld4 <= 2) return k_nmf_spmm<2, 1>;
  if (ld4 <= 4) return k_nmf_spmm<4, 1>;
  if (ld4 <= 8) return k_nmf_spmm<8, 1>;
  if (ld4 <= 16) return k_nmf_spmm<16, 1>;
  if (ld4 <= 32) return k_nmf_spmm<32, 1>;
  return k_nmf_spmm<32, 2>;
}

// Grid of k_nmf_spmm for products of at most `rows` rows: SMs x blocks_per_sm (default 8), fewer
// when the rows need fewer.  The product does not depend on it.
inline int spmm_grid(const hge_ctx* ctx, int64_t rows) {
  const int per_sm = ctx->blocks_per_sm > 0 ? ctx->blocks_per_sm : 8;
  return (int)std::max<int64_t>(1, std::min<int64_t>((rows * 32 + kFactorBlock - 1) / kFactorBlock,
                                                     (int64_t)ctx->num_sms * per_sm));
}

// P [rows of the CSR, ld] = (A or A^T) Y [other rows, ld]
inline int launch_spmm(hge_ctx* ctx, int32_t rows, const int64_t* ptr, const int32_t* idx, const float* y, int ld,
                       float* p, int grid) {
  spmm_kernel(ld / 4)<<<grid, kFactorBlock, 0, ctx->stream>>>(rows, ptr, idx, reinterpret_cast<const float4*>(y),
                                                               ld / 4, reinterpret_cast<float4*>(p));
  HGE_CHECK_LAUNCH(ctx);
  return HGE_OK;
}

}  // namespace
