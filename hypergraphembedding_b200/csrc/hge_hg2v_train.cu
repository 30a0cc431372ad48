// hypergraph2vec training on sm_100a: the consumer of the sample columns
// (hg2v_model.py:51-203 BooleanModel / UnweightedFloatModel, fit loop embedding.py:269-305).
//
//   node_node = act(<N[ln], N[rn]>)            edge_edge = act(<E[le], E[re]>)
//   node_edge = mean_i act(<N[nn_i], N[ln]>) * mean_i act(<E[ne_i], E[re]>)
//   loss = sum over the three outputs of the batch mean (KL divergence or squared error),
//   Adagrad (lr 0.01, eps 1e-7, accumulators from 0) on the two embedding tables, whose row 0 is
//   the (trained) padding row every absent index points at.
//
// Mini-batch SGD is sequential in the batches and a batch of 256 samples is ~0.5 MB of gathers,
// so the whole epoch is ONE kernel launch of ONE thread-block cluster (8 CTAs x 32 warps = 256
// warps, a sample per warp) that walks the batches with two hardware cluster barriers each:
//   phase 1  forward + backward of the warp's samples; gradients of duplicated rows are summed
//            with float atomics into dense gradient tables (row 0, which every sample touches
//            several times, is first reduced in shared memory per CTA);
//   phase 2  every warp re-visits the rows its samples touched; the first to claim a row
//            (atomicExch on a per-row batch stamp) applies the Adagrad update and clears the
//            row's gradient.
// Tables, accumulators and gradients are read with ld.global.cg: other SMs rewrite them every
// batch and L1 is not coherent.  A launch per batch would cost ~3 launches x 3 000 batches per
// epoch on the 755 K-sample fixture run; here the per-batch cost is the two barriers.
//
// Batches of more than 256 samples: the same kernel is launched (cooperatively, so that every
// block is resident) as ceil(batch / 256) clusters, up to what the device holds at once (16-18 on
// B200), a sample per warp again, and the two per-batch barriers become cluster barrier ->
// one arrival per cluster on a global counter -> cluster barrier.  The one-cluster launch keeps
// the pure hardware barrier.
//
// The sample buffer can also be filled on the device (hge_hg2v_reserve_samples, then
// hge_hg2v_append_samples per block of sampler output: k_hg2v_append packs and range-checks one
// record per thread), the epoch order drawn on the device (hge_shuffle_order: Philox keys, stable
// radix sort) and the tables initialised on the device (hge_hg2v_create_seeded).
#include <cooperative_groups.h>
#include <cub/device/device_radix_sort.cuh>

#include <algorithm>
#include <cfloat>
#include <new>

#include "hge_common.cuh"
#include "hge_expand.cuh"
#include "hge_philox.cuh"
#include "hge_seeded_table.cuh"

namespace cg = cooperative_groups;

struct hge_hg2v_model {
  hge_ctx* ctx = nullptr;
  int32_t node_rows = 0, edge_rows = 0;
  int dim = 0, k = 0, activation = 0, loss = 0;
  float *N = nullptr, *E = nullptr, *accN = nullptr, *accE = nullptr, *gN = nullptr, *gE = nullptr;
  int32_t *claimN = nullptr, *claimE = nullptr;
  int32_t* feat = nullptr;   // [4 + 2k][M]
  float* target = nullptr;   // [3][M]
  int32_t* order = nullptr;  // [M]
  double* d_loss = nullptr;
  int64_t M = 0;
  int32_t next_batch_id = 0;
  unsigned int* grid_bar = nullptr;   // arrival counter of the inter-cluster batch barrier
  int max_clusters = 0;               // co-resident clusters of k_hg2v_epoch (0: not asked yet)
  int last_clusters = 0;              // clusters of the last epoch's launch
  bool reserved = false;              // feat / target come from hge_hg2v_reserve_samples ...
  int64_t filled = 0;                 // ... and hold this many appended records
  unsigned long long* bad = nullptr;  // first bad (record << 5 | column) of the last append
};

namespace {

constexpr int kCluster = 8;
constexpr int kThreads = 1024;
constexpr int kWarpsPerCta = kThreads / 32;
constexpr unsigned kFull = 0xffffffffu;
constexpr int kMaxDim = 256;

struct TrainArgs {
  float *N, *E, *accN, *accE, *gN, *gE;
  int32_t *claimN, *claimE;
  const int32_t* feat;
  const float* target;
  const int32_t* order;
  double* loss_sum;
  int64_t M;
  int dim, k, batch, activation, loss, batch_id0;
  float lr, eps;
  int clusters;             // clusters of this launch
  unsigned int* grid_bar;   // zero at launch
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int off = 16; off; off >>= 1) v += __shfl_xor_sync(kFull, v, off);
  return v;
}

__device__ __forceinline__ float activate(float z, int kind) {
  return kind == 0 ? 1.0f / (1.0f + __expf(-z)) : fmaxf(z, 0.0f);
}
__device__ __forceinline__ float activate_grad(float z, float p, int kind) {
  return kind == 0 ? p * (1.0f - p) : (z > 0.0f ? 1.0f : 0.0f);
}
// per-sample loss and d loss / d p (hge_hg2v: 0 = KL divergence with clipping, 1 = squared error)
__device__ __forceinline__ float loss_grad(float p, float y, int kind, float* loss) {
  if (kind == 0) {
    const float e = 1e-7f;
    const float yc = fminf(fmaxf(y, e), 1.0f), pc = fminf(fmaxf(p, e), 1.0f);
    *loss = yc * __logf(yc / pc);
    return (p >= e && p <= 1.0f) ? -yc / pc : 0.0f;
  }
  const float d = p - y;
  *loss = d * d;
  return 2.0f * d;
}

// gradient of one table row: row 0 goes to the CTA's shared accumulator, the rest to global
template <int DPL>
__device__ __forceinline__ void add_grad(float* __restrict__ g, float* s_g0, int32_t row, int dim,
                                         int lane, float coef, const float (&v)[DPL]) {
#pragma unroll
  for (int j = 0; j < DPL; ++j) {
    const int c = lane + 32 * j;
    if (c < dim) {
      if (row == 0) atomicAdd(s_g0 + c, coef * v[j]);
      else atomicAdd(g + (size_t)row * dim + c, coef * v[j]);
    }
  }
}

template <int DPL>
__device__ __forceinline__ void load_row(const float* __restrict__ t, int32_t row, int dim, int lane,
                                         float (&v)[DPL]) {
#pragma unroll
  for (int j = 0; j < DPL; ++j) {
    const int c = lane + 32 * j;
    v[j] = c < dim ? __ldcg(t + (size_t)row * dim + c) : 0.0f;
  }
}

template <int DPL>
__device__ __forceinline__ float dot(const float (&a)[DPL], const float (&b)[DPL]) {
  float s = 0.0f;
#pragma unroll
  for (int j = 0; j < DPL; ++j) s = fmaf(a[j], b[j], s);
  return warp_sum(s);
}

template <int DPL>
__global__ void __cluster_dims__(kCluster, 1, 1) __launch_bounds__(kThreads, 1)
    k_hg2v_epoch(const TrainArgs a) {
  cg::cluster_group cluster = cg::this_cluster();
  __shared__ float s_g0[2][kMaxDim];   // gradient of the padding rows N[0], E[0] of this CTA
  const int lane = threadIdx.x & 31;
  const int warp = blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
  const int num_warps = a.clusters * kCluster * kWarpsPerCta;
  // batch barrier: everything every block of the launch wrote (gradient atomics, table updates)
  // is visible to every block after it
  unsigned int bar_target = 0;
  auto batch_barrier = [&]() {
    if (a.clusters == 1) {
      // barrier.cluster arrive.release / wait.acquire: every CTA that touches the tables is in
      // this cluster, so cluster scope orders the gradient atomics before the updates
      cluster.sync();
      return;
    }
    __threadfence();
    cluster.sync();
    bar_target += (unsigned int)a.clusters;
    if (cluster.block_rank() == 0 && threadIdx.x == 0) {
      __threadfence();
      atomicAdd(a.grid_bar, 1u);
      unsigned int seen;
      do {
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(a.grid_bar) : "memory");
      } while (seen < bar_target);
      __threadfence();
    }
    cluster.sync();
  };
  const int dim = a.dim, k = a.k, cols = 4 + 2 * k;
  for (int c = threadIdx.x; c < 2 * kMaxDim; c += kThreads) (&s_g0[0][0])[c] = 0.0f;
  __syncthreads();
  double loss_total = 0.0;
  const int64_t num_batches = (a.M + a.batch - 1) / a.batch;
  // the indices / targets of this warp's first sample of a batch are fetched one batch ahead
  // (during phase 2 of the previous one) and kept for phase 2: two dependent global loads
  // (order -> feature columns) less on the critical path of every phase
  auto fetch = [&](int64_t first, int bs, int s, int32_t* my, float* my_t) {
    *my = 0;
    *my_t = 0.0f;
    if (s < bs) {
      const int64_t sample = a.order[first + s];
      if (lane < cols) *my = a.feat[(size_t)lane * a.M + sample];
      if (lane < 3) *my_t = a.target[(size_t)lane * a.M + sample];
    }
  };
  int32_t my_first, my_next = 0;
  float my_t_first, my_t_next = 0.0f;
  fetch(0, (int)min((int64_t)a.batch, a.M), warp, &my_first, &my_t_first);
  for (int64_t b = 0; b < num_batches; ++b) {
    const int64_t first = b * a.batch;
    const int bs = (int)min((int64_t)a.batch, a.M - first);
    const float inv_bs = 1.0f / (float)bs;
    // ---- phase 1: forward + backward ----------------------------------------------------
    for (int s = warp; s < bs; s += num_warps) {
      int32_t my = my_first;
      float my_t = my_t_first;
      if (s != warp) fetch(first, bs, s, &my, &my_t);
      const int32_t ln = __shfl_sync(kFull, my, 0), le = __shfl_sync(kFull, my, 1);
      const int32_t rn = __shfl_sync(kFull, my, 2), re = __shfl_sync(kFull, my, 3);
      float Ln[DPL], Rn[DPL], Le[DPL], Re[DPL], X[DPL];
      load_row<DPL>(a.N, ln, dim, lane, Ln);
      load_row<DPL>(a.N, rn, dim, lane, Rn);
      load_row<DPL>(a.E, le, dim, lane, Le);
      load_row<DPL>(a.E, re, dim, lane, Re);
      const float z_nn = dot<DPL>(Ln, Rn), z_ee = dot<DPL>(Le, Re);
      const float p_nn = activate(z_nn, a.activation), p_ee = activate(z_ee, a.activation);
      // neighbourhood terms: lane i keeps the pre-activation of neighbour i of either kind.
      // With dim <= 32 and k <= 8 all 2k neighbour rows are loaded up front (one memory latency
      // instead of 2k dependent ones) and stay in registers for the gradient pass.
      constexpr int KM = 8;
      const bool preload = DPL == 1 && k <= KM;
      float nbN[KM], nbE[KM];
      float za_mine = 0.0f, zb_mine = 0.0f;
      if (preload) {
#pragma unroll
        for (int i = 0; i < KM; ++i) {
          const int32_t xn = __shfl_sync(kFull, my, (4 + i) & 31), xe = __shfl_sync(kFull, my, (4 + k + i) & 31);
          nbN[i] = (i < k && lane < dim) ? __ldcg(a.N + (size_t)xn * dim + lane) : 0.0f;
          nbE[i] = (i < k && lane < dim) ? __ldcg(a.E + (size_t)xe * dim + lane) : 0.0f;
        }
#pragma unroll
        for (int i = 0; i < KM; ++i) {
          if (i < k) {
            const float za = warp_sum(nbN[i] * Ln[0]), zb = warp_sum(nbE[i] * Re[0]);
            if (lane == i) {
              za_mine = za;
              zb_mine = zb;
            }
          }
        }
      } else {
        for (int i = 0; i < k; ++i) {
          load_row<DPL>(a.N, __shfl_sync(kFull, my, 4 + i), dim, lane, X);
          const float za = dot<DPL>(X, Ln);
          load_row<DPL>(a.E, __shfl_sync(kFull, my, 4 + k + i), dim, lane, X);
          const float zb = dot<DPL>(X, Re);
          if (lane == i) {
            za_mine = za;
            zb_mine = zb;
          }
        }
      }
      const float a_mine = lane < k ? activate(za_mine, a.activation) : 0.0f;
      const float b_mine = lane < k ? activate(zb_mine, a.activation) : 0.0f;
      const float inv_k = k ? 1.0f / (float)k : 0.0f;
      const float A = warp_sum(a_mine) * inv_k, B = warp_sum(b_mine) * inv_k;
      const float p_ne = A * B;
      float l_nn, l_ee, l_ne;
      const float g_nn = loss_grad(p_nn, __shfl_sync(kFull, my_t, 0), a.loss, &l_nn);
      const float g_ee = loss_grad(p_ee, __shfl_sync(kFull, my_t, 1), a.loss, &l_ee);
      const float g_ne = loss_grad(p_ne, __shfl_sync(kFull, my_t, 2), a.loss, &l_ne);
      if (lane == 0) loss_total += (double)l_nn + (double)l_ee + (double)l_ne;
      const float d_nn = g_nn * inv_bs * activate_grad(z_nn, p_nn, a.activation);
      const float d_ee = g_ee * inv_bs * activate_grad(z_ee, p_ee, a.activation);
      const float da_mine = g_ne * inv_bs * B * inv_k * activate_grad(za_mine, a_mine, a.activation);
      const float db_mine = g_ne * inv_bs * A * inv_k * activate_grad(zb_mine, b_mine, a.activation);
      // gradient of the left node / right edge row: the direct term plus every neighbour term
      float gLn[DPL], gRe[DPL];
#pragma unroll
      for (int j = 0; j < DPL; ++j) {
        gLn[j] = d_nn * Rn[j];
        gRe[j] = d_ee * Le[j];
      }
      if (preload) {
#pragma unroll
        for (int i = 0; i < KM; ++i) {
          if (i < k) {
            const float da = __shfl_sync(kFull, da_mine, i), db = __shfl_sync(kFull, db_mine, i);
            const int32_t xn = __shfl_sync(kFull, my, 4 + i), xe = __shfl_sync(kFull, my, 4 + k + i);
            if (da != 0.0f) {
              gLn[0] = fmaf(da, nbN[i], gLn[0]);
              add_grad<DPL>(a.gN, s_g0[0], xn, dim, lane, da, Ln);
            }
            if (db != 0.0f) {
              gRe[0] = fmaf(db, nbE[i], gRe[0]);
              add_grad<DPL>(a.gE, s_g0[1], xe, dim, lane, db, Re);
            }
          }
        }
      } else {
        for (int i = 0; i < k; ++i) {
          const float da = __shfl_sync(kFull, da_mine, i), db = __shfl_sync(kFull, db_mine, i);
          const int32_t xn = __shfl_sync(kFull, my, 4 + i), xe = __shfl_sync(kFull, my, 4 + k + i);
          if (da != 0.0f) {
            load_row<DPL>(a.N, xn, dim, lane, X);
#pragma unroll
            for (int j = 0; j < DPL; ++j) gLn[j] = fmaf(da, X[j], gLn[j]);
            add_grad<DPL>(a.gN, s_g0[0], xn, dim, lane, da, Ln);
          }
          if (db != 0.0f) {
            load_row<DPL>(a.E, xe, dim, lane, X);
#pragma unroll
            for (int j = 0; j < DPL; ++j) gRe[j] = fmaf(db, X[j], gRe[j]);
            add_grad<DPL>(a.gE, s_g0[1], xe, dim, lane, db, Re);
          }
        }
      }
      add_grad<DPL>(a.gN, s_g0[0], ln, dim, lane, 1.0f, gLn);
      add_grad<DPL>(a.gN, s_g0[0], rn, dim, lane, d_nn, Ln);
      add_grad<DPL>(a.gE, s_g0[1], re, dim, lane, 1.0f, gRe);
      add_grad<DPL>(a.gE, s_g0[1], le, dim, lane, d_ee, Re);
    }
    __syncthreads();
    for (int c = threadIdx.x; c < 2 * dim; c += kThreads) {
      const int t = c / dim, cc = c - t * dim;
      const float v = s_g0[t][cc];
      if (v != 0.0f) atomicAdd((t ? a.gE : a.gN) + cc, v);
      s_g0[t][cc] = 0.0f;
    }
    batch_barrier();
    if (b + 1 < num_batches)
      fetch(first + a.batch, (int)min((int64_t)a.batch, a.M - first - a.batch), warp, &my_next,
            &my_t_next);
    // ---- phase 2: Adagrad on the rows this warp's samples touched ------------------------
    const int32_t stamp = a.batch_id0 + (int32_t)b;
    for (int s = warp; s < bs; s += num_warps) {
      int32_t my = my_first;
      if (s != warp) {
        float unused;
        fetch(first, bs, s, &my, &unused);
      }
      // column c of the sample indexes the node table for c in {0, 2, 4 .. 4+k-1}
      int32_t old = stamp;
      if (lane < cols) {
        const bool node = lane == 0 || lane == 2 || (lane >= 4 && lane < 4 + k);
        old = atomicExch((node ? a.claimN : a.claimE) + my, stamp);
      }
      // the rows this warp owns, four at a time: all loads of a group first, then the updates
      unsigned owned = __ballot_sync(kFull, lane < cols && old != stamp);
      while (owned) {
        int32_t rw[4] = {0, 0, 0, 0};
        unsigned is_node = 0;
        int nr = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (owned) {
            const int c = __ffs(owned) - 1;
            owned &= owned - 1;
            rw[j] = __shfl_sync(kFull, my, c);
            if (c == 0 || c == 2 || (c >= 4 && c < 4 + k)) is_node |= 1u << j;
            nr = j + 1;
          }
        }
        for (int c = lane; c < dim; c += 32) {
          float gv[4], av[4], pv[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const size_t at = (size_t)rw[j] * dim + c;
            const bool node = (is_node >> j) & 1;
            gv[j] = j < nr ? __ldcg((node ? a.gN : a.gE) + at) : 0.0f;
            av[j] = j < nr ? __ldcg((node ? a.accN : a.accE) + at) : 0.0f;
            pv[j] = j < nr ? __ldcg((node ? a.N : a.E) + at) : 0.0f;
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if (j < nr && gv[j] != 0.0f) {
              const size_t at = (size_t)rw[j] * dim + c;
              const bool node = (is_node >> j) & 1;
              const float acc = av[j] + gv[j] * gv[j];
              (node ? a.accN : a.accE)[at] = acc;
              (node ? a.N : a.E)[at] = pv[j] - a.lr * gv[j] / (sqrtf(acc) + a.eps);
              (node ? a.gN : a.gE)[at] = 0.0f;
            }
          }
        }
      }
    }
    batch_barrier();
    my_first = my_next;
    my_t_first = my_t_next;
  }
  if (lane == 0 && loss_total != 0.0) atomicAdd(a.loss_sum, loss_total);
}

template <typename T>
int upload(hge_ctx* ctx, T** dst, const T* src, size_t count, int mem) {
  HGE_TRY(hge_dev_alloc(ctx, dst, count));
  if (count)
    HGE_CUDA(cudaMemcpyAsync(*dst, src, count * sizeof(T),
                             mem == HGE_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice,
                             ctx->stream));
  return HGE_OK;
}

// ---- the sample buffer filled on the device ---------------------------------------------------

struct AppendArgs {
  const int32_t *ln, *le, *rn, *re;    // [count] each, NULL = padding index 0
  const int32_t *nbr_n, *nbr_e;        // [count, k] row-major, NULL = padding index 0
  const float* prob;                   // [count], NULL = prob_value
  int prob_slot;                       // target slot of prob, -1 = none
  float prob_value;
  int64_t count, at, M;
  int k;
  int32_t node_rows, edge_rows;
  int32_t* feat;
  float* target;
  unsigned long long* bad;
};

// np.nan_to_num(x, nan=0.0) in fp32
__device__ __forceinline__ float nan_to_num(float x) {
  if (isnan(x)) return 0.0f;
  if (isinf(x)) return x > 0.0f ? FLT_MAX : -FLT_MAX;
  return x;
}

// _columns_to_model_input(..., weighted=False) for one block of records at record `at` of the
// buffer, one thread per record.  Every index written is checked against its table; the first
// bad one (lowest record, then column) is kept in *bad.
__global__ void k_hg2v_append(const AppendArgs a) {
  const int cols = 4 + 2 * a.k;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < a.count;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t o = a.at + i;
    unsigned long long bad = ~0ull;
    for (int c = 0; c < cols; ++c) {
      const int32_t* src = c == 0 ? a.ln : c == 1 ? a.le : c == 2 ? a.rn : c == 3 ? a.re
                           : c < 4 + a.k ? a.nbr_n : a.nbr_e;
      const int64_t j = c < 4 ? i : i * a.k + (c < 4 + a.k ? c - 4 : c - 4 - a.k);
      const int64_t v = src ? (int64_t)src[j] + 1 : 0;
      const bool node = c == 0 || c == 2 || (c >= 4 && c < 4 + a.k);
      if (v < 0 || v >= (node ? a.node_rows : a.edge_rows))
        bad = min(bad, ((unsigned long long)i << 5) | (unsigned long long)c);
      a.feat[(size_t)c * a.M + o] = (int32_t)v;
    }
    if (bad != ~0ull) atomicMin(a.bad, bad);
    const float p = nan_to_num(a.prob ? a.prob[i] : a.prob_value);
    for (int s = 0; s < 3; ++s) a.target[(size_t)s * a.M + o] = s == a.prob_slot ? p : 0.0f;
  }
}

// ---- seeded epoch order and tables ------------------------------------------------------------

// key of item i in epoch e: words 2e, 2e + 1 of its stream in `phase` (high, low)
__global__ void k_shuffle_keys(int64_t n, uint64_t seed, uint32_t phase, uint32_t epoch,
                               uint64_t* __restrict__ keys, int32_t* __restrict__ idx) {
  const int w = (int)(epoch & 1u) * 2;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    const HgeWords4 r = hge_philox4x32_10(epoch >> 1, (uint32_t)i, (uint32_t)((uint64_t)i >> 32),
                                          phase, (uint32_t)seed, (uint32_t)(seed >> 32));
    keys[i] = ((uint64_t)r.v[w] << 32) | r.v[w + 1];
    idx[i] = (int32_t)i;
  }
}

// hge_hg2v_create and hge_hg2v_create_seeded: tables uploaded from node_init / edge_init, or
// (seed != NULL) drawn on the device
int create_model(hge_ctx* ctx, int32_t node_rows, int32_t edge_rows, int dim, int num_neighbors,
                 int activation, int loss, const float* node_init, const float* edge_init, int mem,
                 const uint64_t* seed, hge_hg2v_model** out, const char* what) {
  HGE_REQUIRE(node_rows >= 1 && edge_rows >= 1, "%s: empty embedding table", what);
  HGE_REQUIRE(dim >= 1 && dim <= kMaxDim, "%s: dimension %d not in [1, %d]", what, dim, kMaxDim);
  HGE_REQUIRE(num_neighbors >= 0 && 4 + 2 * num_neighbors <= 32,
              "%s: num_neighbors %d not in [0, 14]", what, num_neighbors);
  HGE_REQUIRE((activation == 0 || activation == 1) && (loss == 0 || loss == 1),
              "%s: activation / loss must be 0 or 1", what);
  HGE_REQUIRE(mem == HGE_MEM_HOST || mem == HGE_MEM_DEVICE, "%s: bad mem %d", what, mem);
  HGE_CUDA(cudaSetDevice(ctx->device));
  hge_hg2v_model* m = new (std::nothrow) hge_hg2v_model();
  if (!m) return HGE_ERR_NOMEM;
  m->ctx = ctx;
  m->node_rows = node_rows;
  m->edge_rows = edge_rows;
  m->dim = dim;
  m->k = num_neighbors;
  m->activation = activation;
  m->loss = loss;
  const size_t nn = (size_t)node_rows * dim, ne = (size_t)edge_rows * dim;
  int rc = HGE_OK;
  if (seed) {
    rc = hge_dev_alloc(ctx, &m->N, nn);
    if (rc == HGE_OK) rc = hge_dev_alloc(ctx, &m->E, ne);
    if (rc == HGE_OK) {
      const int blocks = (dim + 3) / 4;
      k_init_table<<<grid_for(ctx, (int64_t)node_rows * blocks), kExpandBlock, 0, ctx->stream>>>(
          node_rows, dim, *seed, HGE_PHASE_INIT_NODES, -0.05f, 0.1f, m->N);
      k_init_table<<<grid_for(ctx, (int64_t)edge_rows * blocks), kExpandBlock, 0, ctx->stream>>>(
          edge_rows, dim, *seed, HGE_PHASE_INIT_EDGES, -0.05f, 0.1f, m->E);
      ctx->launches += 2;
      const cudaError_t e = cudaGetLastError();
      if (e != cudaSuccess) {
        hge_set_error("%s: init launch failed: %s", what, cudaGetErrorString(e));
        rc = HGE_ERR_CUDA;
      }
    }
  } else {
    rc = upload(ctx, &m->N, node_init, nn, mem);
    if (rc == HGE_OK) rc = upload(ctx, &m->E, edge_init, ne, mem);
  }
  if (rc == HGE_OK) rc = hge_dev_alloc(ctx, &m->accN, nn);
  if (rc == HGE_OK) rc = hge_dev_alloc(ctx, &m->accE, ne);
  if (rc == HGE_OK) rc = hge_dev_alloc(ctx, &m->gN, nn);
  if (rc == HGE_OK) rc = hge_dev_alloc(ctx, &m->gE, ne);
  if (rc == HGE_OK) rc = hge_dev_alloc(ctx, &m->claimN, (size_t)node_rows);
  if (rc == HGE_OK) rc = hge_dev_alloc(ctx, &m->claimE, (size_t)edge_rows);
  if (rc == HGE_OK) rc = hge_dev_alloc(ctx, &m->d_loss, 1);
  if (rc == HGE_OK) rc = hge_dev_alloc(ctx, &m->grid_bar, 1);
  if (rc == HGE_OK) {
    cudaError_t e = cudaMemsetAsync(m->accN, 0, nn * 4, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(m->accE, 0, ne * 4, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(m->gN, 0, nn * 4, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(m->gE, 0, ne * 4, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(m->claimN, 0xff, (size_t)node_rows * 4, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(m->claimE, 0xff, (size_t)edge_rows * 4, ctx->stream);
    if (e != cudaSuccess) {
      hge_set_error("%s: memset failed: %s", what, cudaGetErrorString(e));
      rc = HGE_ERR_CUDA;
    }
  }
  if (rc != HGE_OK) {
    hge_hg2v_destroy(m);
    return rc;
  }
  *out = m;
  return HGE_OK;
}

}  // namespace

extern "C" {

int hge_hg2v_destroy(hge_hg2v_model* m) {
  if (!m) return HGE_OK;
  const hge_ctx* ctx = m->ctx;
  cudaSetDevice(ctx->device);
  hge_dev_free(ctx, m->N);
  hge_dev_free(ctx, m->E);
  hge_dev_free(ctx, m->accN);
  hge_dev_free(ctx, m->accE);
  hge_dev_free(ctx, m->gN);
  hge_dev_free(ctx, m->gE);
  hge_dev_free(ctx, m->claimN);
  hge_dev_free(ctx, m->claimE);
  hge_dev_free(ctx, m->feat);
  hge_dev_free(ctx, m->target);
  hge_dev_free(ctx, m->order);
  hge_dev_free(ctx, m->d_loss);
  hge_dev_free(ctx, m->grid_bar);
  hge_dev_free(ctx, m->bad);
  delete m;
  return HGE_OK;
}

int hge_hg2v_create(hge_ctx* ctx, int32_t node_rows, int32_t edge_rows, int dim, int num_neighbors,
                    int activation, int loss, const float* node_init, const float* edge_init,
                    int mem, hge_hg2v_model** out) {
  HGE_REQUIRE(ctx && out && node_init && edge_init, "hge_hg2v_create: NULL argument");
  *out = nullptr;
  return create_model(ctx, node_rows, edge_rows, dim, num_neighbors, activation, loss, node_init, edge_init,
                      mem, nullptr, out, "hge_hg2v_create");
}

int hge_hg2v_create_seeded(hge_ctx* ctx, int32_t node_rows, int32_t edge_rows, int dim, int num_neighbors,
                           int activation, int loss, uint64_t seed, hge_hg2v_model** out) {
  HGE_REQUIRE(ctx && out, "hge_hg2v_create_seeded: NULL argument");
  *out = nullptr;
  return create_model(ctx, node_rows, edge_rows, dim, num_neighbors, activation, loss, nullptr, nullptr,
                      HGE_MEM_DEVICE, &seed, out, "hge_hg2v_create_seeded");
}

int hge_hg2v_set_samples(hge_hg2v_model* m, const int32_t* features, const float* targets,
                         int64_t num_samples, int mem) {
  HGE_REQUIRE(m && num_samples >= 0 && (num_samples == 0 || (features && targets)),
              "hge_hg2v_set_samples: bad argument");
  HGE_REQUIRE(mem == HGE_MEM_HOST || mem == HGE_MEM_DEVICE, "hge_hg2v_set_samples: bad mem %d", mem);
  hge_ctx* ctx = m->ctx;
  HGE_CUDA(cudaSetDevice(ctx->device));
  const size_t cols = 4 + 2 * (size_t)m->k;
  // every index must address a table row: check once here instead of in the hot loop, and before
  // the model changes, so that a refused call leaves the samples it had
  if (mem == HGE_MEM_HOST) {
    for (size_t c = 0; c < cols; ++c) {
      const bool node = c == 0 || c == 2 || (c >= 4 && c < 4 + (size_t)m->k);
      const int32_t limit = node ? m->node_rows : m->edge_rows;
      const int32_t* col = features + c * (size_t)num_samples;
      for (int64_t i = 0; i < num_samples; ++i)
        HGE_REQUIRE(col[i] >= 0 && col[i] < limit,
                    "hge_hg2v_set_samples: feature column %zu, sample %lld: index %d outside its "
                    "table of %d rows", c, (long long)i, col[i], limit);
    }
  }
  hge_dev_free(ctx, m->feat);
  hge_dev_free(ctx, m->target);
  hge_dev_free(ctx, m->order);
  m->reserved = false;
  m->M = 0;
  HGE_TRY(upload(ctx, &m->feat, features, cols * (size_t)num_samples, mem));
  HGE_TRY(upload(ctx, &m->target, targets, 3 * (size_t)num_samples, mem));
  HGE_TRY(hge_dev_alloc(ctx, &m->order, (size_t)num_samples));
  m->M = num_samples;
  return HGE_OK;
}

int hge_hg2v_fit_epoch(hge_hg2v_model* m, const int32_t* order, int batch_size, int mem,
                       double* epoch_loss) {
  HGE_REQUIRE(m && epoch_loss && batch_size >= 1, "hge_hg2v_fit_epoch: bad argument");
  HGE_REQUIRE(m->M > 0 && order, "hge_hg2v_fit_epoch: no samples (hge_hg2v_set_samples) or no order");
  HGE_REQUIRE(mem == HGE_MEM_HOST || mem == HGE_MEM_DEVICE, "hge_hg2v_fit_epoch: bad mem %d", mem);
  HGE_REQUIRE(!m->reserved || m->filled == m->M,
              "hge_hg2v_fit_epoch: %lld of the %lld reserved samples are filled (hge_hg2v_append_samples)",
              (long long)m->filled, (long long)m->M);
  hge_ctx* ctx = m->ctx;
  HGE_CUDA(cudaSetDevice(ctx->device));
  if (mem == HGE_MEM_HOST)
    for (int64_t i = 0; i < m->M; ++i)
      HGE_REQUIRE(order[i] >= 0 && order[i] < m->M, "hge_hg2v_fit_epoch: order[%lld] out of range",
                  (long long)i);
  HGE_CUDA(cudaMemcpyAsync(m->order, order, (size_t)m->M * 4,
                           mem == HGE_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice,
                           ctx->stream));
  HGE_CUDA(cudaMemsetAsync(m->d_loss, 0, sizeof(double), ctx->stream));
  const int64_t num_batches = (m->M + batch_size - 1) / batch_size;
  HGE_REQUIRE((int64_t)m->next_batch_id + num_batches < INT32_MAX, "hge_hg2v_fit_epoch: batch counter overflow");
  TrainArgs a;
  a.N = m->N; a.E = m->E; a.accN = m->accN; a.accE = m->accE; a.gN = m->gN; a.gE = m->gE;
  a.claimN = m->claimN; a.claimE = m->claimE;
  a.feat = m->feat; a.target = m->target; a.order = m->order; a.loss_sum = m->d_loss;
  a.M = m->M; a.dim = m->dim; a.k = m->k; a.batch = batch_size;
  a.activation = m->activation; a.loss = m->loss; a.batch_id0 = m->next_batch_id;
  a.lr = 0.01f; a.eps = 1e-7f;   // keras.optimizers.Adagrad defaults
  m->next_batch_id += (int32_t)num_batches;
  const int dpl = (m->dim + 31) / 32;
  void (*kernel)(const TrainArgs) = dpl <= 1 ? k_hg2v_epoch<1> : dpl <= 2 ? k_hg2v_epoch<2>
                                    : dpl <= 4 ? k_hg2v_epoch<4> : k_hg2v_epoch<8>;
  // clusters that can be resident at once (they spin on each other): asked once per model
  if (m->max_clusters == 0) {
    cudaLaunchConfig_t probe = {};
    probe.gridDim = dim3(kCluster * 32, 1, 1);
    probe.blockDim = dim3(kThreads, 1, 1);
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, kernel, &probe) != cudaSuccess || n < 1) {
      cudaGetLastError();
      n = 1;
    }
    m->max_clusters = n;
  }
  const int want = (int)std::min<int64_t>((std::min<int64_t>(batch_size, m->M) + kCluster * kWarpsPerCta - 1) /
                                              (kCluster * kWarpsPerCta), m->max_clusters);
  int clusters = std::max(1, std::min(want, ctx->trainer_max_clusters > 0 ? ctx->trainer_max_clusters : want));
  a.grid_bar = m->grid_bar;
  for (;;) {
    a.clusters = clusters;
    cudaError_t e = cudaSuccess;
    if (clusters == 1) {
      kernel<<<kCluster, kThreads, 0, ctx->stream>>>(a);
      e = cudaGetLastError();
    } else {
      e = cudaMemsetAsync(m->grid_bar, 0, sizeof(unsigned int), ctx->stream);
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(kCluster * clusters, 1, 1);
      cfg.blockDim = dim3(kThreads, 1, 1);
      cfg.stream = ctx->stream;
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeCooperative;   // every block resident, or the launch fails
      attr[0].val.cooperative = 1;
      cfg.attrs = attr;
      cfg.numAttrs = 1;
      if (e == cudaSuccess) e = cudaLaunchKernelEx(&cfg, kernel, a);
    }
    if (e == cudaSuccess) break;
    cudaGetLastError();
    if (clusters == 1) {
      hge_set_error("hge_hg2v_fit_epoch: kernel launch failed: %s", cudaGetErrorString(e));
      return HGE_ERR_CUDA;
    }
    clusters = clusters > 2 ? clusters / 2 : 1;   // fewer clusters fit: same result, more rounds per batch
    m->max_clusters = clusters;
  }
  m->last_clusters = clusters;
  ctx->launches++;
  double total = 0.0;
  HGE_TRY(read_back(ctx, m->d_loss, &total, 1));
  *epoch_loss = total / (double)m->M;
  return HGE_OK;
}

int hge_hg2v_last_clusters(const hge_hg2v_model* m) { return m ? m->last_clusters : 0; }

int hge_hg2v_get_weights(hge_hg2v_model* m, float* node, float* edge, int mem) {
  HGE_REQUIRE(m && node && edge, "hge_hg2v_get_weights: NULL argument");
  HGE_REQUIRE(mem == HGE_MEM_HOST || mem == HGE_MEM_DEVICE, "hge_hg2v_get_weights: bad mem %d", mem);
  hge_ctx* ctx = m->ctx;
  HGE_CUDA(cudaSetDevice(ctx->device));
  const cudaMemcpyKind kind = mem == HGE_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
  HGE_CUDA(cudaMemcpyAsync(node, m->N, (size_t)m->node_rows * m->dim * 4, kind, ctx->stream));
  HGE_CUDA(cudaMemcpyAsync(edge, m->E, (size_t)m->edge_rows * m->dim * 4, kind, ctx->stream));
  HGE_CUDA(cudaStreamSynchronize(ctx->stream));
  return HGE_OK;
}

int hge_hg2v_reserve_samples(hge_hg2v_model* m, int64_t num_samples) {
  HGE_REQUIRE(m, "hge_hg2v_reserve_samples: NULL model");
  HGE_REQUIRE(num_samples >= 0 && num_samples < ((int64_t)1 << 31),
              "hge_hg2v_reserve_samples: %lld samples not in [0, 2^31) (the order is int32)",
              (long long)num_samples);
  hge_ctx* ctx = m->ctx;
  HGE_CUDA(cudaSetDevice(ctx->device));
  hge_dev_free(ctx, m->feat);
  hge_dev_free(ctx, m->target);
  hge_dev_free(ctx, m->order);
  m->M = 0;
  m->reserved = false;
  m->filled = 0;
  const size_t cols = 4 + 2 * (size_t)m->k;
  HGE_TRY(hge_dev_alloc(ctx, &m->feat, cols * (size_t)num_samples));
  HGE_TRY(hge_dev_alloc(ctx, &m->target, 3 * (size_t)num_samples));
  HGE_TRY(hge_dev_alloc(ctx, &m->order, (size_t)num_samples));
  if (!m->bad) HGE_TRY(hge_dev_alloc(ctx, &m->bad, 1));
  m->M = num_samples;
  m->reserved = true;
  return HGE_OK;
}

int hge_hg2v_append_samples(hge_hg2v_model* m, const int32_t* left_node, const int32_t* left_edge,
                            const int32_t* right_node, const int32_t* right_edge, const int32_t* nbr_nodes,
                            const int32_t* nbr_edges, const float* prob, int prob_slot, float prob_value,
                            int64_t count) {
  HGE_REQUIRE(m, "hge_hg2v_append_samples: NULL model");
  HGE_REQUIRE(m->reserved, "hge_hg2v_append_samples: no buffer (hge_hg2v_reserve_samples)");
  HGE_REQUIRE(count >= 0 && count <= m->M - m->filled,
              "hge_hg2v_append_samples: %lld records do not fit: %lld of %lld reserved are filled",
              (long long)count, (long long)m->filled, (long long)m->M);
  HGE_REQUIRE(prob_slot >= -1 && prob_slot <= 2, "hge_hg2v_append_samples: prob_slot %d not in [-1, 2]",
              prob_slot);
  if (count == 0) return HGE_OK;
  hge_ctx* ctx = m->ctx;
  HGE_CUDA(cudaSetDevice(ctx->device));
  AppendArgs a;
  a.ln = left_node; a.le = left_edge; a.rn = right_node; a.re = right_edge;
  a.nbr_n = nbr_nodes; a.nbr_e = nbr_edges;
  a.prob = prob; a.prob_slot = prob_slot; a.prob_value = prob_value;
  a.count = count; a.at = m->filled; a.M = m->M; a.k = m->k;
  a.node_rows = m->node_rows; a.edge_rows = m->edge_rows;
  a.feat = m->feat; a.target = m->target; a.bad = m->bad;
  HGE_CUDA(cudaMemsetAsync(m->bad, 0xff, sizeof(unsigned long long), ctx->stream));
  k_hg2v_append<<<grid_for(ctx, count), kExpandBlock, 0, ctx->stream>>>(a);
  HGE_CHECK_LAUNCH(ctx);
  unsigned long long bad = 0;
  HGE_TRY(read_back(ctx, m->bad, &bad, 1));
  if (bad != ~0ull) {
    const int c = (int)(bad & 31u);
    const bool node = c == 0 || c == 2 || (c >= 4 && c < 4 + m->k);
    hge_set_error("hge_hg2v_append_samples: feature column %d, record %lld of the block: index outside its "
                  "table of %d rows", c, (long long)(bad >> 5), node ? m->node_rows : m->edge_rows);
    return HGE_ERR_INVALID;
  }
  m->filled += count;
  return HGE_OK;
}

int hge_hg2v_get_samples(hge_hg2v_model* m, int32_t* features, float* targets, int mem) {
  HGE_REQUIRE(m && (m->M == 0 || (features && targets)), "hge_hg2v_get_samples: NULL argument");
  HGE_REQUIRE(mem == HGE_MEM_HOST || mem == HGE_MEM_DEVICE, "hge_hg2v_get_samples: bad mem %d", mem);
  if (m->M == 0) return HGE_OK;
  hge_ctx* ctx = m->ctx;
  HGE_CUDA(cudaSetDevice(ctx->device));
  const cudaMemcpyKind kind = mem == HGE_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
  HGE_CUDA(cudaMemcpyAsync(features, m->feat, (4 + 2 * (size_t)m->k) * (size_t)m->M * 4, kind, ctx->stream));
  HGE_CUDA(cudaMemcpyAsync(targets, m->target, 3 * (size_t)m->M * 4, kind, ctx->stream));
  HGE_CUDA(cudaStreamSynchronize(ctx->stream));
  return HGE_OK;
}

}  // extern "C"

int hge_shuffle_order_phase(hge_ctx* ctx, uint64_t seed, uint32_t phase, uint32_t epoch, int64_t n,
                            int32_t* order, int mem) {
  HGE_REQUIRE(ctx, "hge_shuffle_order: NULL context");
  HGE_REQUIRE(n >= 0 && n < ((int64_t)1 << 31), "hge_shuffle_order: n = %lld not in [0, 2^31)", (long long)n);
  HGE_REQUIRE(n == 0 || order, "hge_shuffle_order: NULL order");
  HGE_REQUIRE(mem == HGE_MEM_HOST || mem == HGE_MEM_DEVICE, "hge_shuffle_order: bad mem %d", mem);
  if (n == 0) return HGE_OK;
  HGE_CUDA(cudaSetDevice(ctx->device));
  Staged<int32_t> out(ctx);
  HGE_TRY(out.init(order, (size_t)n, mem, false, true));
  DevBuf<uint64_t> k0(ctx), k1(ctx);
  DevBuf<int32_t> v1(ctx);
  DevBuf<char> temp(ctx);
  HGE_TRY(k0.alloc((size_t)n));
  HGE_TRY(k1.alloc((size_t)n));
  HGE_TRY(v1.alloc((size_t)n));
  cub::DoubleBuffer<uint64_t> keys(k0.p, k1.p);
  cub::DoubleBuffer<int32_t> vals(out.dev, v1.p);
  k_shuffle_keys<<<grid_for(ctx, n), kExpandBlock, 0, ctx->stream>>>(n, seed, phase, epoch, k0.p, out.dev);
  HGE_CHECK_LAUNCH(ctx);
  // LSD radix sort: stable, so equal keys keep ascending item order
  size_t bytes = 0;
  HGE_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, bytes, keys, vals, n, 0, 64, ctx->stream));
  HGE_TRY(temp.alloc(bytes));
  HGE_CUDA(cub::DeviceRadixSort::SortPairs(temp.p, bytes, keys, vals, n, 0, 64, ctx->stream));
  ctx->launches++;
  if (vals.Current() != out.dev)
    HGE_CUDA(cudaMemcpyAsync(out.dev, vals.Current(), (size_t)n * 4, cudaMemcpyDeviceToDevice, ctx->stream));
  return out.finish();
}

extern "C" int hge_shuffle_order(hge_ctx* ctx, uint64_t seed, uint32_t epoch, int64_t n, int32_t* order,
                                 int mem) {
  return hge_shuffle_order_phase(ctx, seed, HGE_PHASE_SHUFFLE, epoch, n, order, mem);
}
