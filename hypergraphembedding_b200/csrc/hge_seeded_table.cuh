// The seeded dense tables of the library: the hypergraph2vec embedding tables
// (csrc/hge_hg2v_train.cu), the start of the non-negative factorization (csrc/hge_nmf.cu) and the
// start block of the truncated SVD (csrc/hge_svd.cu) and node2vec's input table (csrc/hge_n2v.cu).
#pragma once

#include "hge_philox.cuh"

namespace {

// Seeded dense table [rows, dim]: element (r, c) = offset + scale * ((word c of the stream of row
// r in `phase`) >> 8) * 2^-24, each operation rounded on its own (no contraction), so that the
// float32 numpy restatement gives the same bits.  The hypergraph2vec tables and the
// factorizations' starts are drawn with it.
__global__ void k_init_table(int64_t rows, int dim, uint64_t seed, uint32_t phase, float offset, float scale,
                             float* __restrict__ t) {
  const int blocks = (dim + 3) / 4;
  for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < rows * blocks;
       g += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = g / blocks;
    const int b = (int)(g - r * blocks);
    const HgeWords4 w = hge_philox4x32_10((uint32_t)b, (uint32_t)r, (uint32_t)((uint64_t)r >> 32), phase,
                                          (uint32_t)seed, (uint32_t)(seed >> 32));
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = 4 * b + j;
      if (c < dim) {
        const float u = __fmul_rn(__uint2float_rn(w.v[j] >> 8), 0x1p-24f);
        t[(size_t)r * dim + c] = __fadd_rn(offset, __fmul_rn(scale, u));
      }
    }
  }
}

}  // namespace
