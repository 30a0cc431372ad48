// Non-negative factorization of the node-edge incidence on sm_100a: scikit-learn's coordinate
// descent solver (NMF(solver="cd"): _fit_coordinate_descent, _update_cdnmf_fast) with Frobenius
// loss, no regularization and no shuffling, for the 0/1 incidence A [N, E] ~ W [N, k] H [k, E].
//
// One iteration, both halves with the same three steps (W with H^T, then H^T with the new W):
//   k_nmf_spmm  (csrc/hge_factor.cuh, shared with the truncated SVD of csrc/hge_svd.cu)
//               P = A Ht (node rows) or A^T W (edge rows): each row adds its neighbours' rows in
//               ascending incidence order, one fp32 add per neighbour -- scipy's order, so P equals
//               scipy's float32 product bit for bit.  A sub-warp of LPR lanes owns a row, a lane
//               LPR-strided float4 columns (as the gathers of csrc/hge_weighting.cu).  Long rows are
//               not split: a split would change the order of the sum.
//   k_nmf_gram  G = Y^T Y (k x k) in chunks of kGramChunk consecutive rows: within a chunk each
//               entry is one fma chain in ascending row order from +0, g_c = fma(Y[i,t], Y[i,r], g_c);
//               k_nmf_gram_combine adds the chunk partials in ascending chunk order in fp32,
//               G = ((g_0 + g_1) + g_2) + ...
//   k_nmf_cd    one thread per row, kCdRows rows a block, the rows in shared memory.  For t = 0..k-1
//               in sequence (row t of G in shared memory):
//                 grad = fma chain over r = 0..k-1 of G[t,r] * Y[i,r] starting from -P[i,t]
//                 viol += |min(0, grad)| if Y[i,t] == 0 else |grad|          (f64, per thread)
//                 if G[t,t] != 0: Y[i,t] = max(Y[i,t] - grad / G[t,t], 0)    (IEEE division)
//               The block's 64 thread sums are combined by a fixed halving tree (f64) into one
//               partial per block; k_nmf_viol adds the partials of each half in ascending block
//               order and the two halves' sums (W half first).
// No float atomics: every sum has one order that does not depend on the grid, so W and H are
// bit-identical from run to run and for every launch setting.  The host reads the iteration's
// violation (8 bytes) and applies scikit-learn's stop rule.
#include <math.h>

#include <algorithm>

#include "hge_factor.cuh"
#include "hge_incidence.cuh"
#include "hge_philox.cuh"
#include "hge_seeded_table.cuh"

namespace {

constexpr int kBlock = 256;
constexpr int kMaxK = 256;
constexpr int kGramChunk = 4096;   // rows per Gram partial
constexpr int kGramTile = 32;      // rows per shared-memory tile of k_nmf_gram
constexpr int kGramPer = 8;        // Gram entries per thread
constexpr int kCdRows = 64;        // rows (threads) per block of k_nmf_cd

// ---- dense layout (k_nmf_pad and the product k_nmf_spmm are in csrc/hge_factor.cuh) ---------------

__global__ void k_nmf_unpad(int64_t rows, int k, int ld, const float* __restrict__ y, float* __restrict__ x) {
  const int64_t total = rows * k;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / k;
    x[i] = y[r * ld + (i - r * k)];
  }
}

enum : int { kBadValue = 1, kNonzeroW = 2, kNonzeroH = 4 };

// flags: kBadValue for a negative or non-finite entry, `nonzero` when an entry is not zero
__global__ void k_nmf_check(int64_t n, const float* __restrict__ x, int nonzero, int* __restrict__ flags) {
  int f = 0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float v = x[i];
    if (!(v >= 0.f) || !isfinite(v)) f |= kBadValue;
    if (v != 0.f) f |= nonzero;
  }
  f = __reduce_or_sync(0xffffffffu, f);
  if ((threadIdx.x & 31) == 0 && f) atomicOr(flags, f);
}

// ---- Gram -----------------------------------------------------------------------------------------

// grid (chunks, entry tiles): block (c, j) owns entries j * kBlock * kGramPer + m * kBlock + tid
__global__ void __launch_bounds__(kBlock) k_nmf_gram(int64_t rows, int k, int ld, const float* __restrict__ y,
                                                      float* __restrict__ part) {
  extern __shared__ float tile[];   // [kGramTile][ld]
  const int64_t r0 = (int64_t)blockIdx.x * kGramChunk;
  const int64_t r1 = min(rows, r0 + (int64_t)kGramChunk);
  const int kk = k * k;
  int et[kGramPer], er[kGramPer];
  float acc[kGramPer];
#pragma unroll
  for (int m = 0; m < kGramPer; ++m) {
    const int e = (blockIdx.y * kGramPer + m) * kBlock + threadIdx.x;
    et[m] = e < kk ? e / k : 0;
    er[m] = e < kk ? e - (e / k) * k : 0;
    acc[m] = 0.f;
  }
  for (int64_t t0 = r0; t0 < r1; t0 += kGramTile) {
    const int n = (int)min((int64_t)kGramTile, r1 - t0);
    __syncthreads();
    for (int q = threadIdx.x; q < n * ld; q += kBlock) tile[q] = y[t0 * ld + q];
    __syncthreads();
    for (int j = 0; j < n; ++j)
#pragma unroll
      for (int m = 0; m < kGramPer; ++m) acc[m] = __fmaf_rn(tile[j * ld + et[m]], tile[j * ld + er[m]], acc[m]);
  }
#pragma unroll
  for (int m = 0; m < kGramPer; ++m) {
    const int e = (blockIdx.y * kGramPer + m) * kBlock + threadIdx.x;
    if (e < kk) part[(size_t)blockIdx.x * kk + e] = acc[m];
  }
}

__global__ void k_nmf_gram_combine(int kk, int64_t chunks, const float* __restrict__ part, float* __restrict__ g) {
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < kk; e += gridDim.x * blockDim.x) {
    float s = part[e];
    for (int64_t c = 1; c < chunks; ++c) s = __fadd_rn(s, part[(size_t)c * kk + e]);
    g[e] = s;
  }
}

// ---- coordinate descent ---------------------------------------------------------------------------

__global__ void __launch_bounds__(kCdRows) k_nmf_cd(int64_t rows, int k, int ld, const float* __restrict__ g,
                                                     const float* __restrict__ p, float* __restrict__ y,
                                                     double* __restrict__ viol_part) {
  extern __shared__ float sm[];
  const int ks = ld + 1;                 // odd row stride: the threads' rows fall into distinct banks
  float* ys = sm;                        // [kCdRows][ks]
  float* gs = sm + kCdRows * ks;         // row t of G
  __shared__ double vs[kCdRows];
  const int64_t r0 = (int64_t)blockIdx.x * kCdRows;
  const int n = (int)min((int64_t)kCdRows, rows - r0);
  const int i = threadIdx.x;
  for (int q = i; q < n * ld; q += kCdRows) ys[(q / ld) * ks + q % ld] = y[r0 * ld + q];
  float* yi = ys + i * ks;
  const float* pi = p + (r0 + i) * ld;
  double viol = 0.0;
  for (int t = 0; t < k; ++t) {
    __syncthreads();
    for (int r = i; r < k; r += kCdRows) gs[r] = g[(size_t)t * k + r];
    __syncthreads();
    if (i < n) {
      float grad = -pi[t];
      for (int r = 0; r < k; ++r) grad = __fmaf_rn(gs[r], yi[r], grad);
      const float yt = yi[t];
      const float pg = yt == 0.f ? fminf(0.f, grad) : grad;
      viol += fabs((double)pg);
      const float hess = gs[t];
      if (hess != 0.f) yi[t] = fmaxf(__fsub_rn(yt, __fdiv_rn(grad, hess)), 0.f);
    }
  }
  __syncthreads();
  for (int q = i; q < n * ld; q += kCdRows) y[r0 * ld + q] = ys[(q / ld) * ks + q % ld];
  vs[i] = viol;
  __syncthreads();
#pragma unroll
  for (int h = kCdRows / 2; h >= 1; h >>= 1) {
    if (i < h) vs[i] += vs[i + h];
    __syncthreads();
  }
  if (i == 0) viol_part[blockIdx.x] = vs[0];
}

// out = (sum of the W half's block partials) + (sum of the H half's), each in ascending block order
__global__ void k_nmf_viol(int64_t nw, const double* __restrict__ pw, int64_t nh, const double* __restrict__ ph,
                           double* __restrict__ out) {
  double sw = 0.0, sh = 0.0;
  for (int64_t b = 0; b < nw; ++b) sw += pw[b];
  for (int64_t b = 0; b < nh; ++b) sh += ph[b];
  *out = sw + sh;
}

// Workspace and phase timing of one fit.
struct Fit {
  hge_ctx* ctx;
  hge_incidence* inc;
  int k, ld;
  DevBuf<float> w, h, p, part, g;
  DevBuf<double> vpart, viol;
  int64_t blocks_w = 0, blocks_h = 0;
  size_t cd_smem = 0;
  int spmm_grid = 0;
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  explicit Fit(hge_ctx* c, hge_incidence* i, int k_)
      : ctx(c), inc(i), k(k_), ld(factor_ld(k_)), w(c), h(c), p(c), part(c), g(c), vpart(c), viol(c) {}
  ~Fit() {
    for (cudaEvent_t e : ev)
      if (e) cudaEventDestroy(e);
  }

  // one half: P = A_side * other, G = other^T other, CD on `self`; phase times added to ms[3]
  int half(int side, double* vp, double* ms) {
    const bool nodes = side == 0;
    const int32_t rows = nodes ? inc->N : inc->E;
    const int64_t orows = nodes ? inc->E : inc->N;
    float* self = nodes ? w.p : h.p;
    const float* other = nodes ? h.p : w.p;
    if (ms) HGE_CUDA(cudaEventRecord(ev[0], ctx->stream));
    spmm_kernel(ld / 4)<<<spmm_grid, kBlock, 0, ctx->stream>>>(
        rows, nodes ? inc->n2e_ptr : inc->e2n_ptr, nodes ? inc->n2e_idx : inc->e2n_idx,
        reinterpret_cast<const float4*>(other), ld / 4, reinterpret_cast<float4*>(p.p));
    HGE_CHECK_LAUNCH(ctx);
    if (ms) HGE_CUDA(cudaEventRecord(ev[1], ctx->stream));
    const int64_t chunks = std::max<int64_t>(1, (orows + kGramChunk - 1) / kGramChunk);
    if (orows == 0) {
      HGE_CUDA(cudaMemsetAsync(g.p, 0, sizeof(float) * k * k, ctx->stream));
    } else {
      const dim3 grid((unsigned)chunks, (unsigned)((k * k + kBlock * kGramPer - 1) / (kBlock * kGramPer)));
      k_nmf_gram<<<grid, kBlock, sizeof(float) * kGramTile * ld, ctx->stream>>>(orows, k, ld, other, part.p);
      HGE_CHECK_LAUNCH(ctx);
      k_nmf_gram_combine<<<(k * k + kBlock - 1) / kBlock, kBlock, 0, ctx->stream>>>(k * k, chunks, part.p, g.p);
      HGE_CHECK_LAUNCH(ctx);
    }
    if (ms) HGE_CUDA(cudaEventRecord(ev[2], ctx->stream));
    const int64_t blocks = nodes ? blocks_w : blocks_h;
    if (blocks > 0) {
      k_nmf_cd<<<(unsigned)blocks, kCdRows, cd_smem, ctx->stream>>>(rows, k, ld, g.p, p.p, self, vp);
      HGE_CHECK_LAUNCH(ctx);
    }
    if (ms) HGE_CUDA(cudaEventRecord(ev[3], ctx->stream));
    if (ms) {
      HGE_CUDA(cudaEventSynchronize(ev[3]));
      float a = 0, b = 0, c = 0;
      HGE_CUDA(cudaEventElapsedTime(&a, ev[0], ev[1]));
      HGE_CUDA(cudaEventElapsedTime(&b, ev[1], ev[2]));
      HGE_CUDA(cudaEventElapsedTime(&c, ev[2], ev[3]));
      ms[0] += a;
      ms[1] += b;
      ms[2] += c;
    }
    return HGE_OK;
  }
};

}  // namespace

extern "C" {

int hge_nmf_init(hge_ctx* ctx, int32_t num_nodes, int32_t num_edges, int k, uint64_t seed, float scale, float* W,
                 float* Ht, int mem) {
  const char* what = "hge_nmf_init";
  HGE_REQUIRE(ctx && W && Ht, "%s: NULL argument", what);
  HGE_REQUIRE(num_nodes >= 0 && num_edges >= 0, "%s: negative row count", what);
  HGE_REQUIRE(k >= 1 && k <= kMaxK, "%s: k = %d not in [1, %d]", what, k, kMaxK);
  HGE_REQUIRE(scale >= 0.f && isfinite(scale), "%s: scale must be finite and non-negative", what);
  HGE_REQUIRE(mem == HGE_MEM_HOST || mem == HGE_MEM_DEVICE, "%s: bad mem %d", what, mem);
  HGE_CUDA(cudaSetDevice(ctx->device));
  Staged<float> w(ctx), h(ctx);
  HGE_TRY(w.init(W, (size_t)num_nodes * k, mem, false, true));
  HGE_TRY(h.init(Ht, (size_t)num_edges * k, mem, false, true));
  const int blocks = (k + 3) / 4;
  if (num_nodes > 0) {
    k_init_table<<<grid_for(ctx, (int64_t)num_nodes * blocks), kBlock, 0, ctx->stream>>>(
        num_nodes, k, seed, HGE_PHASE_NMF_W, 0.f, scale, w.dev);
    HGE_CHECK_LAUNCH(ctx);
  }
  if (num_edges > 0) {
    k_init_table<<<grid_for(ctx, (int64_t)num_edges * blocks), kBlock, 0, ctx->stream>>>(
        num_edges, k, seed, HGE_PHASE_NMF_H, 0.f, scale, h.dev);
    HGE_CHECK_LAUNCH(ctx);
  }
  HGE_TRY(w.finish());
  HGE_TRY(h.finish());
  return HGE_OK;
}

int hge_nmf_fit(hge_ctx* ctx, hge_incidence* inc, int32_t num_nodes, int32_t num_edges, int k, float* W, float* Ht,
                int max_iter, double tol, int mem, int* n_iter, double* violations, double* phase_ms) {
  const char* what = "hge_nmf_fit";
  HGE_REQUIRE(ctx && inc && W && Ht && n_iter, "%s: NULL argument", what);
  HGE_REQUIRE(!inc->sharded, "%s: needs a whole (not sharded) incidence", what);
  HGE_REQUIRE(num_nodes == inc->N && num_edges == inc->E,
              "%s: factors of %d x %d rows for an incidence of %d nodes x %d edges", what, num_nodes, num_edges,
              inc->N, inc->E);
  HGE_REQUIRE(k >= 1 && k <= kMaxK, "%s: k = %d not in [1, %d]", what, k, kMaxK);
  HGE_REQUIRE(max_iter >= 1, "%s: max_iter = %d must be >= 1", what, max_iter);
  HGE_REQUIRE(tol >= 0.0, "%s: tol must be non-negative (and not NaN)", what);
  HGE_REQUIRE(mem == HGE_MEM_HOST || mem == HGE_MEM_DEVICE, "%s: bad mem %d", what, mem);
  HGE_CUDA(cudaSetDevice(ctx->device));
  const int32_t N = inc->N, E = inc->E;
  Fit f(ctx, inc, k);
  const int ld = f.ld;
  Staged<float> w_in(ctx), h_in(ctx);
  HGE_TRY(w_in.init(W, (size_t)N * k, mem, true, true));
  HGE_TRY(h_in.init(Ht, (size_t)E * k, mem, true, true));

  // the start: finite, non-negative, neither factor all zero (scikit-learn's _check_init)
  {
    DevBuf<int> flags(ctx);
    HGE_TRY(flags.alloc(1));
    HGE_CUDA(cudaMemsetAsync(flags.p, 0, sizeof(int), ctx->stream));
    const int64_t nw = (int64_t)N * k, nh = (int64_t)E * k;
    if (nw > 0) {
      k_nmf_check<<<grid_for(ctx, nw), kBlock, 0, ctx->stream>>>(nw, w_in.dev, kNonzeroW, flags.p);
      HGE_CHECK_LAUNCH(ctx);
    }
    if (nh > 0) {
      k_nmf_check<<<grid_for(ctx, nh), kBlock, 0, ctx->stream>>>(nh, h_in.dev, kNonzeroH, flags.p);
      HGE_CHECK_LAUNCH(ctx);
    }
    int bad = 0;
    HGE_TRY(read_back(ctx, flags.p, &bad, 1));
    HGE_REQUIRE(!(bad & kBadValue), "%s: the start has a negative or non-finite entry", what);
    HGE_REQUIRE(bad & kNonzeroW, "%s: the start W is all zero", what);
    HGE_REQUIRE(bad & kNonzeroH, "%s: the start H is all zero", what);
  }

  const int64_t rmax = std::max<int64_t>(N, E);
  const int64_t chunks_max = std::max<int64_t>(1, (rmax + kGramChunk - 1) / kGramChunk);
  f.blocks_w = ((int64_t)N + kCdRows - 1) / kCdRows;
  f.blocks_h = ((int64_t)E + kCdRows - 1) / kCdRows;
  HGE_TRY(f.w.alloc((size_t)N * ld));
  HGE_TRY(f.h.alloc((size_t)E * ld));
  HGE_TRY(f.p.alloc((size_t)rmax * ld));
  HGE_TRY(f.part.alloc((size_t)chunks_max * k * k));
  HGE_TRY(f.g.alloc((size_t)k * k));
  HGE_TRY(f.vpart.alloc((size_t)(f.blocks_w + f.blocks_h)));
  HGE_TRY(f.viol.alloc((size_t)max_iter));
  f.cd_smem = sizeof(float) * ((size_t)kCdRows * (ld + 1) + k);
  HGE_CUDA(cudaFuncSetAttribute(k_nmf_cd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)f.cd_smem));
  f.spmm_grid = spmm_grid(ctx, rmax);
  if (phase_ms) {
    for (cudaEvent_t& e : f.ev) HGE_CUDA(cudaEventCreate(&e));
    phase_ms[0] = phase_ms[1] = phase_ms[2] = 0.0;
  }
  if (N > 0) {
    k_nmf_pad<<<grid_for(ctx, (int64_t)N * ld), kBlock, 0, ctx->stream>>>(N, k, ld, w_in.dev, f.w.p);
    HGE_CHECK_LAUNCH(ctx);
  }
  if (E > 0) {
    k_nmf_pad<<<grid_for(ctx, (int64_t)E * ld), kBlock, 0, ctx->stream>>>(E, k, ld, h_in.dev, f.h.p);
    HGE_CHECK_LAUNCH(ctx);
  }

  double* slot = static_cast<double*>(hge_ctx_pinned_slot(ctx));
  if (!slot) return HGE_ERR_CUDA;
  double viol0 = 0.0;
  int it = 0;
  while (it < max_iter) {
    ++it;
    HGE_TRY(f.half(0, f.vpart.p, phase_ms));
    HGE_TRY(f.half(1, f.vpart.p + f.blocks_w, phase_ms));
    k_nmf_viol<<<1, 1, 0, ctx->stream>>>(f.blocks_w, f.vpart.p, f.blocks_h, f.vpart.p + f.blocks_w,
                                         f.viol.p + it - 1);
    HGE_CHECK_LAUNCH(ctx);
    HGE_CUDA(cudaMemcpyAsync(slot, f.viol.p + it - 1, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    HGE_CUDA(cudaStreamSynchronize(ctx->stream));
    const double viol = *slot;
    if (violations) violations[it - 1] = viol;
    if (it == 1) viol0 = viol;
    if (viol0 == 0.0) break;
    if (viol / viol0 <= tol) break;
  }
  *n_iter = it;
  if (N > 0) {
    k_nmf_unpad<<<grid_for(ctx, (int64_t)N * k), kBlock, 0, ctx->stream>>>(N, k, ld, f.w.p, w_in.dev);
    HGE_CHECK_LAUNCH(ctx);
  }
  if (E > 0) {
    k_nmf_unpad<<<grid_for(ctx, (int64_t)E * k), kBlock, 0, ctx->stream>>>(E, k, ld, f.h.p, h_in.dev);
    HGE_CHECK_LAUNCH(ctx);
  }
  HGE_TRY(w_in.finish());
  HGE_TRY(h_in.finish());
  if (mem == HGE_MEM_DEVICE) HGE_CUDA(cudaStreamSynchronize(ctx->stream));
  return HGE_OK;
}

}  // extern "C"
