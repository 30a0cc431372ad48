// Truncated SVD of the node-edge incidence on sm_100a: randomized subspace iteration
// (Halko, Martinsson and Tropp, "Finding structure with randomness", 2011) with Rayleigh-Ritz, for
// the 0/1 incidence A [N, E].  The host drives the loop and does the small l x l steps in f64
// (DESIGN.md section 9.11); the device does everything of size N or E:
//
//   start       Omega [E, l] uniform on [-1, 1): k_init_table of csrc/hge_seeded_table.cuh with
//               offset -1 and scale 2 in phase HGE_PHASE_SVD, padded to [E, ld].
//   half        Y = A X (node side, k_nmf_spmm of csrc/hge_factor.cuh over the node -> edge CSR)
//               or Y = A^T X (edge side), then G = Y^T Y in f64 (k_svd_gram): within chunks of
//               kGramChunk consecutive rows each entry is one f64 fma chain in ascending row order
//               from +0, g = fma(Y[i,t], Y[i,r], g) (the product of two floats is exact in f64);
//               k_svd_gram_combine adds the chunk partials in ascending chunk order.  G goes to
//               the host, which computes M = U~ diag(1 / sigma) from eigh(G) and rounds it to fp32.
//   rowmat      out = Y M (k_svd_rowmat): each output entry is one fp32 fma chain over r = 0 .. l-1
//               ascending from +0, out[i,c] = fma(Y[i,r], M[r,c], out[i,c]).
//   flip        scikit-learn's svd_flip on the first k columns: the entry of u_i of largest
//               magnitude (lowest row on a tie) becomes positive; u_i and v_i are negated together.
//   residuals   r_i = || A v_i - sigma_i u_i ||_2 / sigma_1: the product P = A V, then per column
//               d = P[j,i] - sigma_i U[j,i] and s = s + d d in f64, each operation rounded on its
//               own, over chunks of kGramChunk rows in ascending row order, the chunk sums added in
//               ascending chunk order, then sqrt(s) / sigma_1.
// No float atomics: every sum has one order that does not depend on the grid, so every result is
// bit-identical from run to run and for every launch setting.  The flip's column maxima are
// integer atomicMax on (|u| bits, ~row) keys, whose maximum does not depend on the order.
#include <math.h>

#include <algorithm>

#include "hge_factor.cuh"
#include "hge_incidence.cuh"
#include "hge_philox.cuh"
#include "hge_seeded_table.cuh"

namespace {

constexpr int kBlock = 256;
constexpr int kMaxL = 256;
constexpr int kGramChunk = 4096;   // rows per Gram / residual partial
constexpr int kGramTile = 32;      // rows per shared-memory tile of k_svd_gram
constexpr int kGramPer = 8;        // Gram entries per thread
constexpr int kRmRows = 64;        // output rows per block of k_svd_rowmat
constexpr int kRmCols = 64;        // output columns per block of k_svd_rowmat
constexpr int kRmK = 32;           // terms of the chain staged per shared-memory tile

// ---- f64 Gram -------------------------------------------------------------------------------------

// grid (chunks, entry tiles): block (c, j) owns entries j * kBlock * kGramPer + m * kBlock + tid
__global__ void __launch_bounds__(kBlock, 1) k_svd_gram(int64_t rows, int l, int ld, const float* __restrict__ y,
                                                         double* __restrict__ part) {
  extern __shared__ float tile[];   // [kGramTile][ld]
  const int64_t r0 = (int64_t)blockIdx.x * kGramChunk;
  const int64_t r1 = min(rows, r0 + (int64_t)kGramChunk);
  const int ll = l * l;
  int et[kGramPer], er[kGramPer];
  double acc[kGramPer];
#pragma unroll
  for (int m = 0; m < kGramPer; ++m) {
    const int e = (blockIdx.y * kGramPer + m) * kBlock + threadIdx.x;
    et[m] = e < ll ? e / l : 0;
    er[m] = e < ll ? e - (e / l) * l : 0;
    acc[m] = 0.0;
  }
  for (int64_t t0 = r0; t0 < r1; t0 += kGramTile) {
    const int n = (int)min((int64_t)kGramTile, r1 - t0);
    __syncthreads();
    for (int q = threadIdx.x; q < n * ld; q += kBlock) tile[q] = y[t0 * ld + q];
    __syncthreads();
    for (int j = 0; j < n; ++j)
#pragma unroll
      for (int m = 0; m < kGramPer; ++m)
        acc[m] = __fma_rn((double)tile[j * ld + et[m]], (double)tile[j * ld + er[m]], acc[m]);
  }
#pragma unroll
  for (int m = 0; m < kGramPer; ++m) {
    const int e = (blockIdx.y * kGramPer + m) * kBlock + threadIdx.x;
    if (e < ll) part[(size_t)blockIdx.x * ll + e] = acc[m];
  }
}

__global__ void k_svd_gram_combine(int ll, int64_t chunks, const double* __restrict__ part, double* __restrict__ g) {
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < ll; e += gridDim.x * blockDim.x) {
    double s = part[e];
    for (int64_t c = 1; c < chunks; ++c) s = __dadd_rn(s, part[(size_t)c * ll + e]);
    g[e] = s;
  }
}

// ---- row times small matrix -----------------------------------------------------------------------

// out [rows, ld] = y [rows, ld] (columns < l) x m [l, cols]; columns cols .. ld - 1 of out are 0.
// grid (row tiles, column tiles of kRmCols); thread (ty, tx) owns rows ty + 16 a, columns tx + 16 b.
__global__ void __launch_bounds__(kBlock) k_svd_rowmat(int64_t rows, int l, int cols, int ld,
                                                        const float* __restrict__ y, const float* __restrict__ m,
                                                        float* __restrict__ out) {
  __shared__ float ys[kRmRows][kRmK + 1];
  __shared__ float ms[kRmK][kRmCols];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int64_t r0 = (int64_t)blockIdx.x * kRmRows;
  const int c0 = blockIdx.y * kRmCols;
  float acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
  for (int k0 = 0; k0 < l; k0 += kRmK) {
    const int n = min(kRmK, l - k0);
    __syncthreads();
    for (int q = threadIdx.x; q < kRmRows * kRmK; q += kBlock) {
      const int i = q / kRmK, j = q - i * kRmK;
      ys[i][j] = (r0 + i < rows && j < n) ? y[(r0 + i) * ld + k0 + j] : 0.f;
    }
    for (int q = threadIdx.x; q < kRmK * kRmCols; q += kBlock) {
      const int j = q / kRmCols, c = q - j * kRmCols;
      ms[j][c] = (j < n && c0 + c < cols) ? m[(size_t)(k0 + j) * cols + c0 + c] : 0.f;
    }
    __syncthreads();
    for (int j = 0; j < n; ++j) {
      float ya[4], mb[4];
#pragma unroll
      for (int a = 0; a < 4; ++a) ya[a] = ys[ty + 16 * a][j];
#pragma unroll
      for (int b = 0; b < 4; ++b) mb[b] = ms[j][tx + 16 * b];
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = __fmaf_rn(ya[a], mb[b], acc[a][b]);
    }
  }
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    const int64_t r = r0 + ty + 16 * a;
    if (r >= rows) continue;
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int c = c0 + tx + 16 * b;
      if (c < ld) out[r * ld + c] = c < cols ? acc[a][b] : 0.f;
    }
  }
}

// ---- sign flip ------------------------------------------------------------------------------------

// key[c] = max over rows of (bits(|u[r,c]|) << 32) | (0xffffffff - r): the largest magnitude, then
// the lowest row.  One thread per column c < k (blockDim >= k), rows strided over the blocks.
__global__ void k_svd_colmax(int64_t rows, int k, int ld, const float* __restrict__ u,
                             unsigned long long* __restrict__ key) {
  const int c = threadIdx.x;
  if (c >= k) return;
  unsigned long long best = 0;
  for (int64_t r = blockIdx.x; r < rows; r += gridDim.x) {
    const unsigned long long kk = ((unsigned long long)__float_as_uint(fabsf(u[r * ld + c])) << 32) |
                                  (unsigned long long)(0xffffffffu - (uint32_t)r);
    best = kk > best ? kk : best;
  }
  atomicMax(key + c, best);
}

__global__ void k_svd_sign(int k, int ld, const float* __restrict__ u, const unsigned long long* __restrict__ key,
                           int* __restrict__ neg) {
  const int c = threadIdx.x;
  if (c >= k) return;
  const uint32_t r = 0xffffffffu - (uint32_t)(key[c] & 0xffffffffull);
  neg[c] = u[(int64_t)r * ld + c] < 0.f;
}

__global__ void k_svd_negate(int64_t rows, int k, int ld, const int* __restrict__ neg, float* __restrict__ x) {
  const int64_t total = rows * k;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / k;
    const int c = (int)(i - r * k);
    if (neg[c]) x[r * ld + c] = -x[r * ld + c];
  }
}

// ---- residuals ------------------------------------------------------------------------------------

// part[chunk, c] = sum over the chunk's rows in ascending order of d * d, d = p - sigma_c u (f64,
// each operation rounded on its own).  One thread per column c < k.
__global__ void k_svd_resid_part(int64_t rows, int k, int ld, const float* __restrict__ p,
                                 const float* __restrict__ u, const double* __restrict__ sigma,
                                 double* __restrict__ part) {
  const int c = threadIdx.x;
  if (c >= k) return;
  const int64_t r0 = (int64_t)blockIdx.x * kGramChunk;
  const int64_t r1 = min(rows, r0 + (int64_t)kGramChunk);
  const double s = sigma[c];
  double acc = 0.0;
  for (int64_t r = r0; r < r1; ++r) {
    const double d = __dsub_rn((double)p[r * ld + c], __dmul_rn(s, (double)u[r * ld + c]));
    acc = __dadd_rn(acc, __dmul_rn(d, d));
  }
  part[(size_t)blockIdx.x * k + c] = acc;
}

__global__ void k_svd_resid_final(int k, int64_t chunks, const double* __restrict__ part,
                                  const double* __restrict__ sigma, double* __restrict__ resid) {
  const int c = threadIdx.x;
  if (c >= k) return;
  double s = part[c];
  for (int64_t q = 1; q < chunks; ++q) s = __dadd_rn(s, part[(size_t)q * k + c]);
  const double norm = __dsqrt_rn(s);
  resid[c] = sigma[0] > 0.0 ? __ddiv_rn(norm, sigma[0]) : norm;
}

int64_t chunks_of(int64_t rows) { return std::max<int64_t>(1, (rows + kGramChunk - 1) / kGramChunk); }

}  // namespace

extern "C" {

int hge_svd_start(hge_ctx* ctx, int32_t num_edges, int l, uint64_t seed, float* omega, int mem) {
  const char* what = "hge_svd_start";
  HGE_REQUIRE(ctx && omega, "%s: NULL argument", what);
  HGE_REQUIRE(num_edges >= 0, "%s: negative row count", what);
  HGE_REQUIRE(l >= 1 && l <= kMaxL, "%s: l = %d not in [1, %d]", what, l, kMaxL);
  HGE_REQUIRE(mem == HGE_MEM_HOST || mem == HGE_MEM_DEVICE, "%s: bad mem %d", what, mem);
  HGE_CUDA(cudaSetDevice(ctx->device));
  const int ld = factor_ld(l);
  Staged<float> o(ctx);
  HGE_TRY(o.init(omega, (size_t)num_edges * ld, mem, false, true));
  if (num_edges > 0) {
    DevBuf<float> t(ctx);
    HGE_TRY(t.alloc((size_t)num_edges * l));
    k_init_table<<<grid_for(ctx, (int64_t)num_edges * ((l + 3) / 4)), kBlock, 0, ctx->stream>>>(
        num_edges, l, seed, HGE_PHASE_SVD, -1.f, 2.f, t.p);
    HGE_CHECK_LAUNCH(ctx);
    k_nmf_pad<<<grid_for(ctx, (int64_t)num_edges * ld), kBlock, 0, ctx->stream>>>(num_edges, l, ld, t.p, o.dev);
    HGE_CHECK_LAUNCH(ctx);
  }
  HGE_TRY(o.finish());
  if (mem == HGE_MEM_DEVICE) HGE_CUDA(cudaStreamSynchronize(ctx->stream));
  return HGE_OK;
}

int hge_svd_half(hge_ctx* ctx, hge_incidence* inc, int side, int32_t num_nodes, int32_t num_edges, int l,
                 const float* x, float* y, double* gram, int mem, double* phase_ms) {
  const char* what = "hge_svd_half";
  HGE_REQUIRE(ctx && inc && x && y && gram, "%s: NULL argument", what);
  HGE_REQUIRE(!inc->sharded, "%s: needs a whole (not sharded) incidence", what);
  HGE_REQUIRE(side == 0 || side == 1, "%s: side = %d is not 0 (nodes) or 1 (edges)", what, side);
  HGE_REQUIRE(num_nodes == inc->N && num_edges == inc->E,
              "%s: buffers of %d node x %d edge rows for an incidence of %d nodes x %d edges", what, num_nodes,
              num_edges, inc->N, inc->E);
  HGE_REQUIRE(l >= 1 && l <= kMaxL, "%s: l = %d not in [1, %d]", what, l, kMaxL);
  HGE_REQUIRE(x != y, "%s: the output must not alias the input", what);
  HGE_REQUIRE(mem == HGE_MEM_HOST || mem == HGE_MEM_DEVICE, "%s: bad mem %d", what, mem);
  HGE_CUDA(cudaSetDevice(ctx->device));
  const bool nodes = side == 0;
  const int32_t rows = nodes ? inc->N : inc->E;
  const int64_t in_rows = nodes ? inc->E : inc->N;
  const int ld = factor_ld(l);
  const int ll = l * l;
  Staged<float> xs(ctx), ys(ctx);
  HGE_TRY(xs.init(x, (size_t)in_rows * ld, mem, true, false));
  HGE_TRY(ys.init(y, (size_t)rows * ld, mem, false, true));
  DevBuf<double> part(ctx), g(ctx);
  const int64_t chunks = chunks_of(rows);
  HGE_TRY(part.alloc((size_t)chunks * ll));
  HGE_TRY(g.alloc((size_t)ll));
  cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
  struct Events {
    cudaEvent_t* e;
    ~Events() {
      for (int i = 0; i < 3; ++i)
        if (e[i]) cudaEventDestroy(e[i]);
    }
  } own{ev};
  if (phase_ms) {
    for (cudaEvent_t& e : ev) HGE_CUDA(cudaEventCreate(&e));
    HGE_CUDA(cudaEventRecord(ev[0], ctx->stream));
  }
  if (rows > 0)
    HGE_TRY(launch_spmm(ctx, rows, nodes ? inc->n2e_ptr : inc->e2n_ptr, nodes ? inc->n2e_idx : inc->e2n_idx, xs.dev,
                        ld, ys.dev, spmm_grid(ctx, rows)));
  if (phase_ms) HGE_CUDA(cudaEventRecord(ev[1], ctx->stream));
  if (rows == 0) {
    HGE_CUDA(cudaMemsetAsync(g.p, 0, sizeof(double) * ll, ctx->stream));
  } else {
    const dim3 grid((unsigned)chunks, (unsigned)((ll + kBlock * kGramPer - 1) / (kBlock * kGramPer)));
    k_svd_gram<<<grid, kBlock, sizeof(float) * kGramTile * ld, ctx->stream>>>(rows, l, ld, ys.dev, part.p);
    HGE_CHECK_LAUNCH(ctx);
    k_svd_gram_combine<<<(ll + kBlock - 1) / kBlock, kBlock, 0, ctx->stream>>>(ll, chunks, part.p, g.p);
    HGE_CHECK_LAUNCH(ctx);
  }
  if (phase_ms) HGE_CUDA(cudaEventRecord(ev[2], ctx->stream));
  HGE_TRY(read_back(ctx, g.p, gram, (size_t)ll));
  if (phase_ms) {
    float a = 0, b = 0;
    HGE_CUDA(cudaEventElapsedTime(&a, ev[0], ev[1]));
    HGE_CUDA(cudaEventElapsedTime(&b, ev[1], ev[2]));
    phase_ms[0] = a;
    phase_ms[1] = b;
  }
  HGE_TRY(ys.finish());
  return HGE_OK;
}

int hge_svd_rowmat(hge_ctx* ctx, int64_t rows, int l, int cols, const float* y, const float* m, float* out,
                   int mem) {
  const char* what = "hge_svd_rowmat";
  HGE_REQUIRE(ctx && y && m && out, "%s: NULL argument", what);
  HGE_REQUIRE(rows >= 0, "%s: negative row count", what);
  HGE_REQUIRE(l >= 1 && l <= kMaxL, "%s: l = %d not in [1, %d]", what, l, kMaxL);
  HGE_REQUIRE(cols >= 1 && cols <= l, "%s: cols = %d not in [1, l = %d]", what, cols, l);
  HGE_REQUIRE(y != out, "%s: the output must not alias the input", what);
  HGE_REQUIRE(mem == HGE_MEM_HOST || mem == HGE_MEM_DEVICE, "%s: bad mem %d", what, mem);
  HGE_CUDA(cudaSetDevice(ctx->device));
  const int ld = factor_ld(l);
  Staged<float> ys(ctx), os(ctx), ms(ctx);
  HGE_TRY(ys.init(y, (size_t)rows * ld, mem, true, false));
  HGE_TRY(os.init(out, (size_t)rows * ld, mem, false, true));
  HGE_TRY(ms.init(m, (size_t)l * cols, HGE_MEM_HOST, true, false));
  if (rows > 0) {
    const dim3 grid((unsigned)((rows + kRmRows - 1) / kRmRows), (unsigned)((ld + kRmCols - 1) / kRmCols));
    k_svd_rowmat<<<grid, kBlock, 0, ctx->stream>>>(rows, l, cols, ld, ys.dev, ms.dev, os.dev);
    HGE_CHECK_LAUNCH(ctx);
  }
  HGE_TRY(os.finish());
  return HGE_OK;
}

int hge_svd_flip(hge_ctx* ctx, int64_t num_u_rows, int64_t num_v_rows, int l, int k, float* u, float* v, int mem) {
  const char* what = "hge_svd_flip";
  HGE_REQUIRE(ctx && u && v, "%s: NULL argument", what);
  HGE_REQUIRE(num_u_rows >= 1 && num_u_rows <= INT32_MAX && num_v_rows >= 0, "%s: bad row counts", what);
  HGE_REQUIRE(l >= 1 && l <= kMaxL, "%s: l = %d not in [1, %d]", what, l, kMaxL);
  HGE_REQUIRE(k >= 1 && k <= l, "%s: k = %d not in [1, l = %d]", what, k, l);
  HGE_REQUIRE(mem == HGE_MEM_HOST || mem == HGE_MEM_DEVICE, "%s: bad mem %d", what, mem);
  HGE_CUDA(cudaSetDevice(ctx->device));
  const int ld = factor_ld(l);
  Staged<float> us(ctx), vs(ctx);
  HGE_TRY(us.init(u, (size_t)num_u_rows * ld, mem, true, true));
  HGE_TRY(vs.init(v, (size_t)num_v_rows * ld, mem, true, true));
  DevBuf<unsigned long long> key(ctx);
  DevBuf<int> neg(ctx);
  HGE_TRY(key.alloc((size_t)k));
  HGE_TRY(neg.alloc((size_t)k));
  HGE_CUDA(cudaMemsetAsync(key.p, 0, sizeof(unsigned long long) * k, ctx->stream));
  const int threads = (k + 31) & ~31;
  const int blocks = (int)std::min<int64_t>(num_u_rows, (int64_t)ctx->num_sms * 8);
  k_svd_colmax<<<blocks, threads, 0, ctx->stream>>>(num_u_rows, k, ld, us.dev, key.p);
  HGE_CHECK_LAUNCH(ctx);
  k_svd_sign<<<1, threads, 0, ctx->stream>>>(k, ld, us.dev, key.p, neg.p);
  HGE_CHECK_LAUNCH(ctx);
  k_svd_negate<<<grid_for(ctx, num_u_rows * k), kBlock, 0, ctx->stream>>>(num_u_rows, k, ld, neg.p, us.dev);
  HGE_CHECK_LAUNCH(ctx);
  if (num_v_rows > 0) {
    k_svd_negate<<<grid_for(ctx, num_v_rows * k), kBlock, 0, ctx->stream>>>(num_v_rows, k, ld, neg.p, vs.dev);
    HGE_CHECK_LAUNCH(ctx);
  }
  HGE_TRY(us.finish());
  HGE_TRY(vs.finish());
  return HGE_OK;
}

int hge_svd_residuals(hge_ctx* ctx, hge_incidence* inc, int32_t num_nodes, int32_t num_edges, int l, int k,
                      const float* u, const float* v, const double* sigma, double* resid, int mem) {
  const char* what = "hge_svd_residuals";
  HGE_REQUIRE(ctx && inc && u && v && sigma && resid, "%s: NULL argument", what);
  HGE_REQUIRE(!inc->sharded, "%s: needs a whole (not sharded) incidence", what);
  HGE_REQUIRE(num_nodes == inc->N && num_edges == inc->E,
              "%s: buffers of %d node x %d edge rows for an incidence of %d nodes x %d edges", what, num_nodes,
              num_edges, inc->N, inc->E);
  HGE_REQUIRE(l >= 1 && l <= kMaxL, "%s: l = %d not in [1, %d]", what, l, kMaxL);
  HGE_REQUIRE(k >= 1 && k <= l, "%s: k = %d not in [1, l = %d]", what, k, l);
  HGE_REQUIRE(mem == HGE_MEM_HOST || mem == HGE_MEM_DEVICE, "%s: bad mem %d", what, mem);
  HGE_CUDA(cudaSetDevice(ctx->device));
  const int32_t N = inc->N, E = inc->E;
  const int ld = factor_ld(l);
  Staged<float> us(ctx), vs(ctx);
  HGE_TRY(us.init(u, (size_t)N * ld, mem, true, false));
  HGE_TRY(vs.init(v, (size_t)E * ld, mem, true, false));
  Staged<double> sg(ctx);
  HGE_TRY(sg.init(sigma, (size_t)k, HGE_MEM_HOST, true, false));
  const int64_t chunks = chunks_of(N);
  DevBuf<float> p(ctx);
  DevBuf<double> part(ctx), r(ctx);
  HGE_TRY(p.alloc((size_t)N * ld));
  HGE_TRY(part.alloc((size_t)chunks * k));
  HGE_TRY(r.alloc((size_t)k));
  const int threads = (k + 31) & ~31;
  if (N > 0) {
    HGE_TRY(launch_spmm(ctx, N, inc->n2e_ptr, inc->n2e_idx, vs.dev, ld, p.p, spmm_grid(ctx, N)));
    k_svd_resid_part<<<(unsigned)chunks, threads, 0, ctx->stream>>>(N, k, ld, p.p, us.dev, sg.dev, part.p);
    HGE_CHECK_LAUNCH(ctx);
  } else {
    HGE_CUDA(cudaMemsetAsync(part.p, 0, sizeof(double) * k, ctx->stream));
  }
  k_svd_resid_final<<<1, threads, 0, ctx->stream>>>(k, chunks, part.p, sg.dev, r.p);
  HGE_CHECK_LAUNCH(ctx);
  HGE_TRY(read_back(ctx, r.p, resid, (size_t)k));
  return HGE_OK;
}

}  // extern "C"
