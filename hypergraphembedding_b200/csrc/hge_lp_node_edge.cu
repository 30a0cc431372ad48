// Node-edge link-prediction classifier (LP_NODE_EDGE_CLASSIFIER, evaluation_util.
// NodeEdgeEmbeddingPrediction) on sm_100a: a one-hidden-layer perceptron over [xn[n], xe[e]]
// trained on the incidences (label 1) against as many uniformly drawn non-incidences (label 0).
// The reference trains a Keras model whose architecture is not recorded here; this is a model of
// the usual Keras kind (Dense + relu, Dense + sigmoid, glorot_uniform kernels, zero biases,
// Adagrad, binary cross-entropy), not a port.  oracle/lp_node_edge_ref.py restates the training
// set, the initial weights and the epoch orders bit for bit and trains the same model in float64.
//
//   training set  k_positives (CSR order) + k_negatives (Philox, 64-bit masked rejection over the
//                 S = N E - nnz non-incidences, rank -> (node, edge) through the prefix sum of the
//                 per-node non-member counts and hge_nonmember)
//   epoch order   hge_shuffle_order_phase(HGE_PHASE_LP_NODE_EDGE_SHUFFLE)
//   epoch         k_epoch: ONE launch per epoch of ONE thread-block cluster that walks the batches.
//                 CTA r owns hidden units [r hc, (r + 1) hc): its columns of W1, its entries of b1
//                 and w2 and their Adagrad accumulators stay in shared memory for the epoch.  A
//                 batch is cut into chunks of samples whose rows fit shared memory; per chunk every
//                 CTA gathers the rows itself, computes its hidden units and its part of each
//                 output logit, and the parts are exchanged through distributed shared memory and
//                 added in CTA-rank order, so every CTA derives the same dz.  Every gradient is
//                 local to the CTA that owns the parameter (b2: every CTA keeps the same copy) and
//                 is a per-thread sequential sum in sample order; no float atomics anywhere.
//   predict       k_predict: a warp per link, lane j owns hidden units j, j + 32, ...; each unit a
//                 sequential sum over the 2d inputs, the output a fixed shuffle tree, so a link's
//                 probability depends on its two rows and the model only.
#include <cooperative_groups.h>
#include <cub/device/device_scan.cuh>

#include <chrono>
#include <math.h>
#include <vector>

#include "hge_common.cuh"
#include "hge_incidence.cuh"
#include "hge_pairs.cuh"
#include "hge_philox.cuh"

namespace cg = cooperative_groups;

namespace {

constexpr int kMaxDim = 256;
constexpr int kMaxHidden = 256;
constexpr int kCluster = 8;             // CTAs of the epoch cluster (portable size)
constexpr int kThreads = 512;           // threads of an epoch CTA
constexpr int kMaxChunk = 256;          // samples of a chunk
constexpr int kSmemBudget = 200 << 10;  // dynamic shared memory of an epoch CTA
constexpr int kBlock = 256;
constexpr int kPredictWarps = 8;
constexpr unsigned kFull = 0xffffffffu;

// ---- training set -------------------------------------------------------------------------------

// sample i < nnz: the i-th incidence in CSR order
__global__ void k_positives(int64_t N, int64_t nnz, const int64_t* __restrict__ ptr, const int32_t* __restrict__ idx,
                            int32_t* __restrict__ sn, int32_t* __restrict__ se) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nnz; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t lo = 0, hi = N;   // first row m with ptr[m] > i; the incidence is in row m - 1
    while (lo < hi) {
      const int64_t m = (lo + hi) >> 1;
      if (ptr[m] > i) hi = m; else lo = m + 1;
    }
    sn[i] = (int32_t)(lo - 1);
    se[i] = idx[i];
  }
}

// free[n] = E - deg(n), free[N] = 0 (its exclusive sum is C, C[N] = S)
__global__ void k_free_counts(int64_t N, int64_t E, const int64_t* __restrict__ ptr, int64_t* __restrict__ free) {
  for (int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; n <= N; n += (int64_t)gridDim.x * blockDim.x)
    free[n] = n < N ? E - (ptr[n + 1] - ptr[n]) : 0;
}

// sample nnz + i: r uniform on [0, S) from item i's stream (r = ((w0 << 32) | w1) & mask, redrawn
// while r >= S), then node n with C[n] <= r < C[n + 1] and its (r - C[n])-th non-member edge
__global__ void k_negatives(int64_t nnz, int64_t N, uint64_t seed, uint64_t S, uint64_t mask,
                            const int64_t* __restrict__ C, const int64_t* __restrict__ ptr,
                            const int32_t* __restrict__ idx, int32_t* __restrict__ sn, int32_t* __restrict__ se) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nnz; i += (int64_t)gridDim.x * blockDim.x) {
    HgeStreamRng rng(seed, HGE_PHASE_LP_NODE_EDGE_NEG, (uint64_t)i);
    uint64_t r;
    do {
      const uint64_t w0 = rng.next();
      r = ((w0 << 32) | rng.next()) & mask;
    } while (r >= S);
    int64_t lo = 0, hi = N;   // first m with C[m] > r (C[N] = S > r)
    while (lo < hi) {
      const int64_t m = (lo + hi) >> 1;
      if ((uint64_t)C[m] > r) hi = m; else lo = m + 1;
    }
    const int64_t n = lo - 1;
    sn[nnz + i] = (int32_t)n;
    se[nnz + i] = hge_nonmember(idx + ptr[n], ptr[n + 1] - ptr[n], (int64_t)(r - (uint64_t)C[n]));
  }
}

// ---- initial weights ----------------------------------------------------------------------------

// W1 [in, H] row r = item r, w2 = item in; column j = word j; value -L + (2L) u, u = (w >> 8) 2^-24,
// each operation rounded on its own
__global__ void k_init_weights(int in, int H, uint64_t seed, float L1, float L2, float* __restrict__ W1,
                               float* __restrict__ w2) {
  const int blocks = (H + 3) / 4;
  for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < (int64_t)(in + 1) * blocks;
       g += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(g / blocks), b = (int)(g - (int64_t)r * blocks);
    const HgeWords4 w = hge_philox4x32_10((uint32_t)b, (uint32_t)r, 0u, HGE_PHASE_LP_NODE_EDGE_INIT, (uint32_t)seed,
                                          (uint32_t)(seed >> 32));
    const float L = r < in ? L1 : L2, twoL = __fmul_rn(2.f, L);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = 4 * b + j;
      if (c < H) {
        const float u = __fmul_rn(__uint2float_rn(w.v[j] >> 8), 0x1p-24f);
        (r < in ? W1 + (size_t)r * H : w2)[c] = __fadd_rn(-L, __fmul_rn(twoL, u));
      }
    }
  }
}

// ---- one epoch ----------------------------------------------------------------------------------

struct EpochArgs {
  const int32_t *sn, *se, *order;
  const float *xn, *xe;
  float *W1, *b1, *w2, *b2;       // [in, H], [H], [H], [1]
  float *aW1, *ab1, *aw2, *ab2;   // their Adagrad accumulators
  double* loss;                   // sum of the epoch's sample losses
  int64_t M, nnz;
  int d, H, hc, batch, chunk;
  float lr, eps;
};

__device__ __forceinline__ float adagrad(float w, float g, float& acc, float lr, float eps) {
  acc = __fadd_rn(acc, __fmul_rn(g, g));
  return __fsub_rn(w, __fdiv_rn(__fmul_rn(lr, g), __fadd_rn(__fsqrt_rn(acc), eps)));
}

// ENT: W1 gradient entries per thread (in * hc <= ENT * kThreads)
template <int ENT>
__global__ void __launch_bounds__(kThreads, 1) k_epoch(const EpochArgs a) {
  cg::cluster_group cluster = cg::this_cluster();
  extern __shared__ __align__(16) float smem[];
  __shared__ double red[kThreads];
  __shared__ float s_b2[2];   // b2, its accumulator
  const int t = threadIdx.x;
  const int rank = (int)cluster.block_rank(), C = (int)cluster.num_blocks();
  const int in = 2 * a.d, d = a.d, j0 = rank * a.hc;
  const int hc = min(a.hc, a.H - j0);   // units of this CTA (also the stride of its slices)
  const int ch = a.chunk, xs = in + 1;
  float* sW = smem;                 // [in][hc]
  float* sA = sW + in * a.hc;       // [in][hc]
  float* sb1 = sA + in * a.hc;      // [hc] b1, acc, w2, acc
  float* sab1 = sb1 + a.hc;
  float* sw2 = sab1 + a.hc;
  float* saw2 = sw2 + a.hc;
  float* sX = saw2 + a.hc;          // [ch][xs]
  float* sH = sX + ch * xs;         // [ch][hc] relu(z1)
  float* sD = sH + ch * a.hc;       // [ch][hc] dL / dz1
  float* sDz = sD + ch * a.hc;      // [ch]
  float* sPart = sDz + ch;          // [2][ch] this CTA's part of the output logits
  float* sY = sPart + 2 * ch;       // [ch]
  int32_t* sN = (int32_t*)(sY + ch);
  int32_t* sE = sN + ch;

  for (int e = t; e < in * hc; e += kThreads) {
    const int k = e / hc, jl = e - k * hc;
    sW[e] = a.W1[(size_t)k * a.H + j0 + jl];
    sA[e] = a.aW1[(size_t)k * a.H + j0 + jl];
  }
  for (int jl = t; jl < hc; jl += kThreads) {
    sb1[jl] = a.b1[j0 + jl];
    sab1[jl] = a.ab1[j0 + jl];
    sw2[jl] = a.w2[j0 + jl];
    saw2[jl] = a.aw2[j0 + jl];
  }
  if (t == 0) {
    s_b2[0] = a.b2[0];
    s_b2[1] = a.ab2[0];
  }
  __syncthreads();

  double loss = 0.0;
  float g[ENT];
#pragma unroll
  for (int i = 0; i < ENT; ++i) g[i] = 0.f;
  float gb1 = 0.f, gw2 = 0.f, gb2 = 0.f;
  int buf = 0;
  for (int64_t first = 0; first < a.M; first += a.batch) {
    const int B = (int)min((int64_t)a.batch, a.M - first);
    for (int c0 = 0; c0 < B; c0 += ch) {
      const int bs = min(ch, B - c0);
      // gather the chunk's rows
      for (int s = t; s < bs; s += kThreads) {
        const int32_t id = a.order[first + c0 + s];
        sN[s] = a.sn[id];
        sE[s] = a.se[id];
        sY[s] = id < a.nnz ? 1.f : 0.f;
      }
      __syncthreads();
      for (int e = t; e < bs * in; e += kThreads) {
        const int s = e / in, k = e - s * in;
        sX[s * xs + k] = k < d ? __ldg(a.xn + (size_t)sN[s] * d + k) : __ldg(a.xe + (size_t)sE[s] * d + (k - d));
      }
      __syncthreads();
      // hidden units: z1 = b1 + sum_k x_k W1[k, j], sequential in k
      for (int o = t; o < bs * hc; o += kThreads) {
        const int s = o / hc, jl = o - s * hc;
        const float* x = sX + s * xs;
        float z = sb1[jl];
        for (int k = 0; k < in; ++k) z = fmaf(x[k], sW[k * hc + jl], z);
        sH[o] = fmaxf(z, 0.f);
      }
      __syncthreads();
      // this CTA's part of each logit, sequential in j
      for (int s = t; s < bs; s += kThreads) {
        float p = 0.f;
        for (int jl = 0; jl < hc; ++jl) p = fmaf(sw2[jl], sH[s * hc + jl], p);
        sPart[buf * ch + s] = p;
      }
      cluster.sync();
      // the logits: parts added in rank order, then b2; every CTA gets the same dz
      for (int s = t; s < bs; s += kThreads) {
        float z = 0.f;
        for (int r = 0; r < C; ++r) z = __fadd_rn(z, cluster.map_shared_rank(sPart, r)[buf * ch + s]);
        z = __fadd_rn(z, s_b2[0]);
        const float y = sY[s];
        const float p = __fdiv_rn(1.f, __fadd_rn(1.f, expf(-z)));
        sDz[s] = __fdiv_rn(__fsub_rn(p, y), (float)B);
        if (rank == 0) loss += (double)(fmaxf(z, 0.f) - z * y + log1pf(expf(-fabsf(z))));
      }
      buf ^= 1;
      __syncthreads();
      for (int o = t; o < bs * hc; o += kThreads) {
        const int s = o / hc, jl = o - s * hc;
        sD[o] = sH[o] > 0.f ? __fmul_rn(sDz[s], sw2[jl]) : 0.f;
      }
      __syncthreads();
      // gradients, each a sequential sum over the batch's samples in order
#pragma unroll
      for (int i = 0; i < ENT; ++i) {
        const int e = t + i * kThreads;
        if (e < in * hc) {
          const int k = e / hc, jl = e - k * hc;
          float acc = g[i];
          for (int s = 0; s < bs; ++s) acc = fmaf(sX[s * xs + k], sD[s * hc + jl], acc);
          g[i] = acc;
        }
      }
      if (t < hc) {
        for (int s = 0; s < bs; ++s) {
          gb1 = __fadd_rn(gb1, sD[s * hc + t]);
          gw2 = fmaf(sDz[s], sH[s * hc + t], gw2);
        }
      }
      if (t == kThreads - 1)
        for (int s = 0; s < bs; ++s) gb2 = __fadd_rn(gb2, sDz[s]);
      __syncthreads();
    }
    // Adagrad on the parameters this CTA owns
#pragma unroll
    for (int i = 0; i < ENT; ++i) {
      const int e = t + i * kThreads;
      if (e < in * hc) sW[e] = adagrad(sW[e], g[i], sA[e], a.lr, a.eps);
      g[i] = 0.f;
    }
    if (t < hc) {
      sb1[t] = adagrad(sb1[t], gb1, sab1[t], a.lr, a.eps);
      sw2[t] = adagrad(sw2[t], gw2, saw2[t], a.lr, a.eps);
      gb1 = gw2 = 0.f;
    }
    if (t == kThreads - 1) {
      s_b2[0] = adagrad(s_b2[0], gb2, s_b2[1], a.lr, a.eps);
      gb2 = 0.f;
    }
    __syncthreads();
  }

  for (int e = t; e < in * hc; e += kThreads) {
    const int k = e / hc, jl = e - k * hc;
    a.W1[(size_t)k * a.H + j0 + jl] = sW[e];
    a.aW1[(size_t)k * a.H + j0 + jl] = sA[e];
  }
  for (int jl = t; jl < hc; jl += kThreads) {
    a.b1[j0 + jl] = sb1[jl];
    a.ab1[j0 + jl] = sab1[jl];
    a.w2[j0 + jl] = sw2[jl];
    a.aw2[j0 + jl] = saw2[jl];
  }
  red[t] = loss;
  __syncthreads();
  if (rank == 0 && t == 0) {
    double sum = 0.0;
    for (int i = 0; i < kThreads; ++i) sum += red[i];
    *a.loss = sum;
    a.b2[0] = s_b2[0];
    a.ab2[0] = s_b2[1];
  }
  cluster.sync();   // no CTA leaves while a peer may still read its logit parts
}

// ---- prediction ---------------------------------------------------------------------------------

constexpr int kUnitsPerLane = kMaxHidden / 32;

__global__ void __launch_bounds__(kPredictWarps * 32) k_predict(
    int64_t L, const int32_t* __restrict__ ln, const int32_t* __restrict__ le, const float* __restrict__ xn,
    const float* __restrict__ xe, int d, int H, const float* __restrict__ W1, const float* __restrict__ b1,
    const float* __restrict__ w2, const float* __restrict__ b2, float* __restrict__ prob, uint8_t* __restrict__ keep) {
  __shared__ float sx[kPredictWarps][2 * kMaxDim];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, in = 2 * d;
  float* x = sx[w];
  for (int64_t l = blockIdx.x * (int64_t)kPredictWarps + w; l < L; l += (int64_t)gridDim.x * kPredictWarps) {
    const int64_t n = ln[l], e = le[l];
    for (int k = lane; k < in; k += 32) x[k] = k < d ? xn[n * d + k] : xe[e * d + (k - d)];
    __syncwarp();
    float z[kUnitsPerLane];
#pragma unroll
    for (int i = 0; i < kUnitsPerLane; ++i) z[i] = lane + 32 * i < H ? b1[lane + 32 * i] : 0.f;
    for (int k = 0; k < in; ++k) {
      const float xk = x[k];
      const float* row = W1 + (size_t)k * H;
#pragma unroll
      for (int i = 0; i < kUnitsPerLane; ++i)
        if (lane + 32 * i < H) z[i] = fmaf(xk, row[lane + 32 * i], z[i]);
    }
    float part = 0.f;
#pragma unroll
    for (int i = 0; i < kUnitsPerLane; ++i)
      if (lane + 32 * i < H) part = fmaf(w2[lane + 32 * i], fmaxf(z[i], 0.f), part);
#pragma unroll
    for (int o = 16; o; o >>= 1) part = __fadd_rn(part, __shfl_xor_sync(kFull, part, o));
    if (lane == 0) {
      const float zo = __fadd_rn(part, b2[0]);
      const float p = __fdiv_rn(1.f, __fadd_rn(1.f, expf(-zo)));
      if (prob) prob[l] = p;
      if (keep) keep[l] = p > 0.5f ? 1 : 0;
    }
    __syncwarp();
  }
}

double now_ms() {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// the training set of `inc` into sn / se [2 nnz] (device); *M = 2 nnz
int training_set(hge_ctx* ctx, hge_incidence* inc, uint64_t seed, DevBuf<int32_t>& sn, DevBuf<int32_t>& se,
                 int64_t* M, const char* what) {
  HGE_REQUIRE(!inc->sharded, "%s: needs a whole (not sharded) incidence", what);
  const int64_t N = inc->N, E = inc->E, nnz = hge_incidence_nnz(inc);
  HGE_REQUIRE(nnz > 0, "%s: the graph has no incidences", what);
  HGE_REQUIRE(2 * nnz < ((int64_t)1 << 31), "%s: 2 x %lld incidences are 2^31 or more samples", what,
              (long long)nnz);
  const uint64_t S = (uint64_t)(N * E - nnz);
  HGE_REQUIRE(S > 0, "%s: every (node, edge) pair is an incidence: no negatives to draw", what);
  uint64_t mask = 0;
  while (mask < S - 1) mask = (mask << 1) | 1;
  HGE_TRY(sn.alloc((size_t)(2 * nnz)));
  HGE_TRY(se.alloc((size_t)(2 * nnz)));
  DevBuf<int64_t> nfree(ctx), Cn(ctx);
  DevBuf<char> temp(ctx);
  HGE_TRY(nfree.alloc((size_t)N + 1));
  HGE_TRY(Cn.alloc((size_t)N + 1));
  k_positives<<<grid_for(ctx, nnz), kBlock, 0, ctx->stream>>>(N, nnz, inc->n2e_ptr, inc->n2e_idx, sn.p, se.p);
  HGE_CHECK_LAUNCH(ctx);
  k_free_counts<<<grid_for(ctx, N + 1), kBlock, 0, ctx->stream>>>(N, E, inc->n2e_ptr, nfree.p);
  HGE_CHECK_LAUNCH(ctx);
  size_t bytes = 0;
  HGE_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, bytes, nfree.p, Cn.p, N + 1, ctx->stream));
  HGE_TRY(temp.alloc(bytes));
  HGE_CUDA(cub::DeviceScan::ExclusiveSum(temp.p, bytes, nfree.p, Cn.p, N + 1, ctx->stream));
  ctx->launches++;
  k_negatives<<<grid_for(ctx, nnz), kBlock, 0, ctx->stream>>>(nnz, N, seed, S, mask, Cn.p, inc->n2e_ptr,
                                                               inc->n2e_idx, sn.p, se.p);
  HGE_CHECK_LAUNCH(ctx);
  *M = 2 * nnz;
  return HGE_OK;
}

template <int ENT>
int launch_epoch(hge_ctx* ctx, const EpochArgs& a, int clusters_ctas, size_t smem) {
  HGE_CUDA(cudaFuncSetAttribute(k_epoch<ENT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(clusters_ctas, 1, 1);
  cfg.blockDim = dim3(kThreads, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = ctx->stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = clusters_ctas;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  HGE_CUDA(cudaLaunchKernelEx(&cfg, k_epoch<ENT>, a));
  ctx->launches++;
  return HGE_OK;
}

}  // namespace

extern "C" {

int hge_lp_node_edge_samples(hge_ctx* ctx, hge_incidence* inc, uint64_t seed, int epochs, int32_t* sample_nodes,
                             int32_t* sample_edges, int32_t* orders) {
  const char* what = "hge_lp_node_edge_samples";
  HGE_REQUIRE(ctx && inc && sample_nodes && sample_edges, "%s: NULL argument", what);
  HGE_REQUIRE(epochs >= 0 && (epochs == 0 || orders), "%s: bad epochs / orders", what);
  HGE_CUDA(cudaSetDevice(ctx->device));
  DevBuf<int32_t> sn(ctx), se(ctx);
  int64_t M = 0;
  HGE_TRY(training_set(ctx, inc, seed, sn, se, &M, what));
  HGE_CUDA(cudaMemcpyAsync(sample_nodes, sn.p, (size_t)M * 4, cudaMemcpyDeviceToDevice, ctx->stream));
  HGE_CUDA(cudaMemcpyAsync(sample_edges, se.p, (size_t)M * 4, cudaMemcpyDeviceToDevice, ctx->stream));
  for (int e = 0; e < epochs; ++e)
    HGE_TRY(hge_shuffle_order_phase(ctx, seed, HGE_PHASE_LP_NODE_EDGE_SHUFFLE, (uint32_t)e, M,
                                    orders + (size_t)e * M, HGE_MEM_DEVICE));
  HGE_CUDA(cudaStreamSynchronize(ctx->stream));
  return HGE_OK;
}

int hge_lp_node_edge_train(hge_ctx* ctx, hge_incidence* inc, const float* xn, const float* xe, int d, int hidden,
                           uint64_t seed, int epochs, int batch, float lr, float eps, float* W1, float* b1, float* w2,
                           float* b2, double* epoch_loss, double* phase_ms) {
  const char* what = "hge_lp_node_edge_train";
  HGE_REQUIRE(ctx && inc && xn && xe && W1 && b1 && w2 && b2, "%s: NULL argument", what);
  HGE_REQUIRE(d >= 1 && d <= kMaxDim, "%s: d = %d not in [1, %d]", what, d, kMaxDim);
  HGE_REQUIRE(hidden >= 1 && hidden <= kMaxHidden, "%s: hidden = %d not in [1, %d]", what, hidden, kMaxHidden);
  HGE_REQUIRE(epochs >= 0 && (epochs == 0 || epoch_loss), "%s: bad epochs / epoch_loss", what);
  HGE_REQUIRE(batch >= 1, "%s: batch = %d must be >= 1", what, batch);
  HGE_REQUIRE(lr > 0 && eps > 0 && isfinite(lr) && isfinite(eps), "%s: lr and eps must be positive", what);
  HGE_CUDA(cudaSetDevice(ctx->device));
  double last = now_ms();
  auto mark = [&](int k) -> int {
    if (!phase_ms) return HGE_OK;
    HGE_CUDA(cudaStreamSynchronize(ctx->stream));
    const double t = now_ms();
    phase_ms[k] = t - last;
    last = t;
    return HGE_OK;
  };
  DevBuf<int32_t> sn(ctx), se(ctx), order(ctx);
  int64_t M = 0;
  HGE_TRY(training_set(ctx, inc, seed, sn, se, &M, what));
  const int in = 2 * d, H = hidden;
  const float L1 = (float)sqrt(6.0 / (in + H)), L2 = (float)sqrt(6.0 / (H + 1));
  k_init_weights<<<grid_for(ctx, (int64_t)(in + 1) * ((H + 3) / 4)), kBlock, 0, ctx->stream>>>(in, H, seed, L1, L2,
                                                                                             W1, w2);
  HGE_CHECK_LAUNCH(ctx);
  HGE_CUDA(cudaMemsetAsync(b1, 0, (size_t)H * 4, ctx->stream));
  HGE_CUDA(cudaMemsetAsync(b2, 0, 4, ctx->stream));
  DevBuf<float> acc(ctx);
  DevBuf<double> loss(ctx);
  const size_t nacc = (size_t)in * H + 2 * (size_t)H + 1;
  HGE_TRY(acc.alloc(nacc));
  HGE_TRY(loss.alloc((size_t)epochs));
  HGE_TRY(order.alloc((size_t)M));
  HGE_CUDA(cudaMemsetAsync(acc.p, 0, nacc * 4, ctx->stream));
  HGE_TRY(mark(0));

  // hidden units split over the cluster; the chunk is what shared memory holds next to the slices
  const int hc = (H + std::min(H, kCluster) - 1) / std::min(H, kCluster);
  const int ctas = (H + hc - 1) / hc;
  const int64_t fixed = (2 * (int64_t)in * hc + 4 * hc) * 4;
  const int64_t per_sample = ((int64_t)in + 1 + 2 * hc + 6) * 4;
  const int chunk = (int)std::max<int64_t>(
      1, std::min<int64_t>({(int64_t)kMaxChunk, (int64_t)batch, M, (kSmemBudget - fixed) / per_sample}));
  const size_t smem = (size_t)(fixed + per_sample * chunk);
  const int ent = (in * hc + kThreads - 1) / kThreads;
  EpochArgs a;
  a.sn = sn.p; a.se = se.p; a.order = order.p; a.xn = xn; a.xe = xe;
  a.W1 = W1; a.b1 = b1; a.w2 = w2; a.b2 = b2;
  a.aW1 = acc.p; a.ab1 = acc.p + (size_t)in * H; a.aw2 = a.ab1 + H; a.ab2 = a.aw2 + H;
  a.M = M; a.nnz = M / 2; a.d = d; a.H = H; a.hc = hc; a.batch = batch; a.chunk = chunk;
  a.lr = lr; a.eps = eps;
  for (int e = 0; e < epochs; ++e) {
    HGE_TRY(hge_shuffle_order_phase(ctx, seed, HGE_PHASE_LP_NODE_EDGE_SHUFFLE, (uint32_t)e, M, order.p,
                                    HGE_MEM_DEVICE));
    a.loss = loss.p + e;
    int rc;
    if (ent <= 1) rc = launch_epoch<1>(ctx, a, ctas, smem);
    else if (ent <= 2) rc = launch_epoch<2>(ctx, a, ctas, smem);
    else if (ent <= 4) rc = launch_epoch<4>(ctx, a, ctas, smem);
    else if (ent <= 8) rc = launch_epoch<8>(ctx, a, ctas, smem);
    else if (ent <= 16) rc = launch_epoch<16>(ctx, a, ctas, smem);
    else rc = launch_epoch<32>(ctx, a, ctas, smem);
    HGE_TRY(rc);
    HGE_TRY(mark(1 + e));
  }
  if (epochs > 0) {
    HGE_TRY(read_back(ctx, loss.p, epoch_loss, (size_t)epochs));
    for (int e = 0; e < epochs; ++e) epoch_loss[e] /= (double)M;
  }
  HGE_CUDA(cudaStreamSynchronize(ctx->stream));
  return HGE_OK;
}

int hge_lp_node_edge_predict(hge_ctx* ctx, const float* xn, int64_t num_nodes, const float* xe, int64_t num_edges,
                             int d, int hidden, const float* W1, const float* b1, const float* w2, const float* b2,
                             const int32_t* link_nodes, const int32_t* link_edges, int64_t num_links, float* out_prob,
                             uint8_t* out_keep) {
  const char* what = "hge_lp_node_edge_predict";
  HGE_REQUIRE(ctx && W1 && b1 && w2 && b2, "%s: NULL argument", what);
  HGE_REQUIRE(d >= 1 && d <= kMaxDim, "%s: d = %d not in [1, %d]", what, d, kMaxDim);
  HGE_REQUIRE(hidden >= 1 && hidden <= kMaxHidden, "%s: hidden = %d not in [1, %d]", what, hidden, kMaxHidden);
  HGE_REQUIRE(num_nodes >= 0 && num_edges >= 0, "%s: negative row count", what);
  HGE_REQUIRE(num_links >= 0 && num_links < ((int64_t)1 << 31) &&
                  (num_links == 0 || (xn && xe && link_nodes && link_edges && (out_prob || out_keep))),
              "%s: bad links", what);
  if (num_links == 0) return HGE_OK;
  HGE_CUDA(cudaSetDevice(ctx->device));
  bool ok = false;
  HGE_TRY(pairs_in_range(ctx, num_links, link_nodes, num_nodes, link_edges, num_edges, HGE_MEM_DEVICE, &ok));
  HGE_REQUIRE(ok, "%s: a link names a node outside [0, %lld) or an edge outside [0, %lld)", what,
              (long long)num_nodes, (long long)num_edges);
  k_predict<<<grid_for(ctx, num_links, kPredictWarps), kPredictWarps * 32, 0, ctx->stream>>>(
      num_links, link_nodes, link_edges, xn, xe, d, hidden, W1, b1, w2, b2, out_prob, out_keep);
  HGE_CHECK_LAUNCH(ctx);
  HGE_CUDA(cudaStreamSynchronize(ctx->stream));
  return HGE_OK;
}

}  // extern "C"
