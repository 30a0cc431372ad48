// node2vec on the node-edge bipartite graph of a hypergraph (DESIGN.md section 9.12): seeded
// second-order walks, word2vec's shrunk-window pairs, unigram^0.75 negatives and a deterministic
// mini-batch skip-gram trainer.  oracle/node2vec_ref.py restates every step.
//
// Vertices: compressed node r is vertex r, compressed edge c is vertex N + c (V = N + E).
//
//   walks      walk w (0 <= w < num_walks V) starts at vertex w mod V and reads the Philox stream of
//              item w in HGE_PHASE_N2V_WALK.  First step below(d); then, with t the previous vertex
//              and d = deg(v): d = 1 returns to t without a draw; d >= 2 draws one word u and returns
//              iff (u 2^-32) (q + (d - 1) p) < q in f64, each operation rounded on its own, otherwise
//              j = below(d - 1) picks row[j] (j < pos(t)) or row[j + 1] of v's sorted row.  On a
//              bipartite graph no neighbour of v is adjacent to t, so these two weights (1/p return,
//              1/q elsewhere) are node2vec's whole rule.  A walk from a vertex of degree 0 has one
//              vertex and -1 after it.
//   pairs      token i of a walk (global index g = w L + i) draws b = 1 + below(window) from item g of
//              HGE_PHASE_N2V_WINDOW; its pairs are (token i, token j), j != i, |i - j| <= b, in
//              ascending (g, j) order.  Counted per token, scanned, emitted.
//   negatives  pair i of epoch e reads item e P + i of HGE_PHASE_N2V_NEG: per sample
//              r = ((w0 << 32) | w1) & mask, redrawn while r >= total, then the vertex v with
//              cum[v] <= r < cum[v + 1] (upper-bound search of the cumulative noise table).
//   training   per batch of B pairs (in the epoch order of hge_shuffle_order, phase
//              HGE_PHASE_N2V_SHUFFLE): k_n2v_coef computes every coefficient from the tables as they
//              were at the batch start; k_n2v_delta sums each touched row's contributions in
//              ascending (pair position, slot) order into a delta (one warp per row, segments of a
//              stably sorted plan); k_n2v_apply adds the deltas.  No float atomics anywhere, so the
//              tables and the loss are bit-identical from run to run and for every chunk size.
#include <math.h>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>

#include "hge_common.cuh"
#include "hge_incidence.cuh"
#include "hge_philox.cuh"
#include "hge_seeded_table.cuh"

namespace {

constexpr int kBlock = 256;
constexpr int kWarps = kBlock / 32;
constexpr int kMaxDim = 256;
constexpr int64_t kDefaultPlanBytes = (int64_t)512 << 20;

struct N2vGraph {
  int32_t N;
  const int64_t* nptr;
  const int32_t* nidx;
  const int64_t* eptr;
  const int32_t* eidx;

  // v's sorted neighbour row (ids of the other side), its degree, and the vertex id of entry 0
  __device__ __forceinline__ const int32_t* row(int32_t v, uint32_t& deg, int32_t& base) const {
    if (v < N) {
      const int64_t b = nptr[v];
      deg = (uint32_t)(nptr[v + 1] - b);
      base = N;
      return nidx + b;
    }
    const int64_t b = eptr[v - N];
    deg = (uint32_t)(eptr[v - N + 1] - b);
    base = 0;
    return eidx + b;
  }
};

// ---- walks ----------------------------------------------------------------------------------------

__global__ void k_n2v_walks(N2vGraph g, int64_t walks_total, int32_t V, int L, double p, double q, uint64_t seed,
                            int32_t* __restrict__ walks, unsigned long long* __restrict__ counts) {
  for (int64_t w = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; w < walks_total;
       w += (int64_t)gridDim.x * blockDim.x) {
    int32_t* out = walks + w * L;
    HgeStreamRng rng(seed, HGE_PHASE_N2V_WALK, (uint64_t)w);
    int32_t v = (int32_t)(w % V), t = -1;
    out[0] = v;
    atomicAdd(counts + v, 1ull);
    uint32_t d;
    int32_t base;
    g.row(v, d, base);
    if (d == 0) {
      for (int i = 1; i < L; ++i) out[i] = -1;
      continue;
    }
    for (int i = 1; i < L; ++i) {
      const int32_t* row = g.row(v, d, base);
      int32_t x;
      if (t < 0) {
        x = base + row[rng.below(d)];
      } else if (d == 1) {
        x = t;
      } else {
        const double u = __dmul_rn((double)rng.next(), 0x1p-32);
        const double c = __dadd_rn(q, __dmul_rn((double)(d - 1), p));
        if (__dmul_rn(u, c) < q) {
          x = t;
        } else {
          const uint32_t j = rng.below(d - 1);
          const int32_t key = t - base;
          uint32_t lo = 0, hi = d;   // pos(t): first entry >= t
          while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (row[mid] < key) lo = mid + 1; else hi = mid;
          }
          x = base + row[j < lo ? j : j + 1];
        }
      }
      out[i] = x;
      atomicAdd(counts + x, 1ull);
      t = v;
      v = x;
    }
  }
}

// ---- pairs ----------------------------------------------------------------------------------------

// context range [lo, hi] of token i of a walk, or false for a token past the walk's end
__device__ __forceinline__ bool n2v_window(const int32_t* __restrict__ walk, int L, int i, int window, uint64_t seed,
                                           int64_t g, int& lo, int& hi) {
  if (walk[i] < 0) return false;
  const int len = (L > 1 && walk[1] < 0) ? 1 : L;
  HgeStreamRng rng(seed, HGE_PHASE_N2V_WINDOW, (uint64_t)g);
  const int b = 1 + (int)rng.below((uint32_t)window);
  lo = max(0, i - b);
  hi = min(len - 1, i + b);
  return true;
}

// counts[g] = pairs of token g; counts[tokens] = 0 (the scan's total)
__global__ void k_n2v_pair_counts(const int32_t* __restrict__ walks, int64_t tokens, int L, int window, uint64_t seed,
                                  int64_t* __restrict__ counts) {
  for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g <= tokens;
       g += (int64_t)gridDim.x * blockDim.x) {
    int lo = 0, hi = 0;
    int64_t n = 0;
    if (g < tokens) {
      const int i = (int)(g % L);
      if (n2v_window(walks + (g - i), L, i, window, seed, g, lo, hi)) n = hi - lo;
    }
    counts[g] = n;
  }
}

__global__ void k_n2v_pair_emit(const int32_t* __restrict__ walks, int64_t tokens, int L, int window, uint64_t seed,
                                const int64_t* __restrict__ offsets, int2* __restrict__ pairs) {
  for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < tokens;
       g += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)(g % L);
    const int32_t* walk = walks + (g - i);
    int lo, hi;
    if (!n2v_window(walk, L, i, window, seed, g, lo, hi)) continue;
    int64_t k = offsets[g];
    for (int j = lo; j <= hi; ++j)
      if (j != i) pairs[k++] = make_int2(walk[i], walk[j]);
  }
}

// ---- negatives ------------------------------------------------------------------------------------

struct N2vNoise {
  const int64_t* cum;   // [V + 1], cum[0] = 0, cum[V] = total
  int32_t V;
  uint64_t total, mask;

  __device__ __forceinline__ int32_t draw(HgeStreamRng& rng) const {
    uint64_t r;
    do {
      const uint64_t hi = rng.next();
      r = ((hi << 32) | rng.next()) & mask;
    } while (r >= total);
    int32_t lo = 0, hi = V;   // cum[lo] <= r < cum[hi]
    while (hi - lo > 1) {
      const int32_t mid = lo + ((hi - lo) >> 1);
      if ((uint64_t)cum[mid] <= r) lo = mid; else hi = mid;
    }
    return lo;
  }
};

__global__ void k_n2v_negatives(const N2vNoise noise, int64_t P, int negative, uint64_t seed, uint32_t epoch,
                                int32_t* __restrict__ out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < P; i += (int64_t)gridDim.x * blockDim.x) {
    HgeStreamRng rng(seed, HGE_PHASE_N2V_NEG, (uint64_t)epoch * (uint64_t)P + (uint64_t)i);
    for (int k = 0; k < negative; ++k) out[i * negative + k] = noise.draw(rng);
  }
}

// ---- training plan --------------------------------------------------------------------------------

// The plan of one chunk of whole batches, position p = pair p of the chunk in epoch order:
//   cen[p]          the pair's center
//   cx[p S + s]     slot s's target: the context (s = 0) or negative s - 1, -1 where skipped
//   in_key[p]       (batch of the chunk << 32) | center,  in_val[p] = p
//   out_key[p S + s](batch << 32) | target (V where skipped), out_val = p S + s
// Stable radix sorts of both key arrays then group every batch's contributions to one row in
// ascending (p, s) order; batch b's entries stay at [b B, b B + nb) and [b B S, (b B + nb) S).
__global__ void k_n2v_plan(const int2* __restrict__ pairs, const int32_t* __restrict__ order, int64_t p0, int64_t count,
                           int64_t P, int B, int negative, const N2vNoise noise, uint64_t seed, uint32_t epoch,
                           int32_t* __restrict__ cen, int32_t* __restrict__ cx, uint64_t* __restrict__ in_key,
                           int32_t* __restrict__ in_val, uint64_t* __restrict__ out_key, int32_t* __restrict__ out_val) {
  const int S = negative + 1;
  for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < count; p += (int64_t)gridDim.x * blockDim.x) {
    const int32_t id = order[p0 + p];
    const int2 pr = pairs[id];
    const uint64_t hb = (uint64_t)(p / B) << 32;
    cen[p] = pr.x;
    in_key[p] = hb | (uint32_t)pr.x;
    in_val[p] = (int32_t)p;
    const int64_t o = p * S;
    cx[o] = pr.y;
    out_key[o] = hb | (uint32_t)pr.y;
    out_val[o] = (int32_t)o;
    HgeStreamRng rng(seed, HGE_PHASE_N2V_NEG, (uint64_t)epoch * (uint64_t)P + (uint64_t)id);
    for (int k = 1; k < S; ++k) {
      const int32_t x = noise.draw(rng);
      const bool skip = x == pr.y;
      cx[o + k] = skip ? -1 : x;
      out_key[o + k] = hb | (uint32_t)(skip ? noise.V : x);
      out_val[o + k] = (int32_t)(o + k);
    }
  }
}

// ---- training kernels -----------------------------------------------------------------------------

// row r of a [rows, dim] table as DPL columns per lane: lane + 32 j, 0 beyond dim
template <int DPL>
__device__ __forceinline__ void n2v_load(const float* __restrict__ t, int64_t r, int dim, int lane, float (&v)[DPL]) {
#pragma unroll
  for (int j = 0; j < DPL; ++j) {
    const int c = lane + 32 * j;
    v[j] = c < dim ? t[r * dim + c] : 0.f;
  }
}

__device__ __forceinline__ float n2v_sigmoid(float z) { return __fdiv_rn(1.f, __fadd_rn(1.f, __expf(-z))); }

// one warp per pair p of the batch: G[p S + s] = lr (label - sigmoid(in[c] . out[x])) from the
// batch-start tables, loss[p] = sum over the slots of (double)(-log sigmoid(+-s)) in slot order
template <int DPL>
__global__ void __launch_bounds__(kBlock) k_n2v_coef(int nb, int S, int dim, float lr, const float* __restrict__ tin,
                                                     const float* __restrict__ tout, const int32_t* __restrict__ cen,
                                                     const int32_t* __restrict__ cx, float* __restrict__ G,
                                                     double* __restrict__ loss) {
  const int lane = threadIdx.x & 31;
  const int p = blockIdx.x * kWarps + (threadIdx.x >> 5);
  if (p >= nb) return;
  float a[DPL], b[DPL];
  n2v_load<DPL>(tin, cen[p], dim, lane, a);
  double l = 0.0;
  for (int s = 0; s < S; ++s) {
    const int32_t x = cx[(int64_t)p * S + s];
    if (x < 0) {
      if (lane == 0) G[(int64_t)p * S + s] = 0.f;
      continue;
    }
    n2v_load<DPL>(tout, x, dim, lane, b);
    float z = 0.f;
#pragma unroll
    for (int j = 0; j < DPL; ++j) z = __fmaf_rn(a[j], b[j], z);
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) z = __fadd_rn(z, __shfl_xor_sync(0xffffffffu, z, off));
    const float sg = n2v_sigmoid(z);
    const float label = s == 0 ? 1.f : 0.f;
    const float sy = s == 0 ? sg : n2v_sigmoid(-z);
    l = __dadd_rn(l, (double)(-__logf(sy)));
    if (lane == 0) G[(int64_t)p * S + s] = __fmul_rn(lr, __fsub_rn(label, sg));
  }
  if (lane == 0) loss[p] = l;
}

// One warp per sorted plan entry of the batch: in-side entries [0, nb), out-side [nb, nb + nb S).
// A segment head (first entry of its key) sums the segment's contributions into its delta row:
//   in side:  din[e]  = fma chain of G[p S + s] * out[cx[p S + s]] over the segment's p, then s
//   out side: dout[e] = fma chain of G[v] * in[cen[v / S]] over the segment's v = p S + s
// from +0 in ascending order; hin / hout name the row of a head and are -1 elsewhere.
template <int DPL>
__global__ void __launch_bounds__(kBlock) k_n2v_delta(int nb, int S, int dim, int32_t V, int64_t pb,
                                                      const float* __restrict__ tin, const float* __restrict__ tout,
                                                      const int32_t* __restrict__ cen, const int32_t* __restrict__ cx,
                                                      const float* __restrict__ G, const uint64_t* __restrict__ in_key,
                                                      const int32_t* __restrict__ in_val,
                                                      const uint64_t* __restrict__ out_key,
                                                      const int32_t* __restrict__ out_val, float* __restrict__ din,
                                                      int32_t* __restrict__ hin, float* __restrict__ dout,
                                                      int32_t* __restrict__ hout) {
  const int lane = threadIdx.x & 31;
  const int64_t e = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5);
  const int64_t nin = nb, nout = (int64_t)nb * S;
  if (e >= nin + nout) return;
  const bool in_side = e < nin;
  const int64_t k0 = in_side ? pb + e : pb * S + (e - nin);   // index into the chunk's sorted arrays
  const int64_t end = in_side ? pb + nin : (pb + nb) * (int64_t)S;
  const uint64_t* key = in_side ? in_key : out_key;
  const int64_t first = in_side ? pb : pb * S;
  const uint64_t kk = key[k0];
  const int32_t row = (int32_t)(kk & 0xffffffffu);
  int32_t* head = in_side ? hin + e : hout + (e - nin);
  if ((k0 > first && key[k0 - 1] == kk) || row == V) {
    if (lane == 0) *head = -1;
    return;
  }
  float acc[DPL], b[DPL];
#pragma unroll
  for (int j = 0; j < DPL; ++j) acc[j] = 0.f;
  for (int64_t k = k0; k < end && key[k] == kk; ++k) {
    if (in_side) {
      const int64_t p = in_val[k];
      for (int s = 0; s < S; ++s) {
        const int32_t x = cx[p * S + s];
        if (x < 0) continue;
        const float gv = G[(p - pb) * S + s];
        n2v_load<DPL>(tout, x, dim, lane, b);
#pragma unroll
        for (int j = 0; j < DPL; ++j) acc[j] = __fmaf_rn(gv, b[j], acc[j]);
      }
    } else {
      const int64_t v = out_val[k];
      const float gv = G[v - pb * S];
      n2v_load<DPL>(tin, cen[v / S], dim, lane, b);
#pragma unroll
      for (int j = 0; j < DPL; ++j) acc[j] = __fmaf_rn(gv, b[j], acc[j]);
    }
  }
  float* d = (in_side ? din + e * dim : dout + (e - nin) * dim);
#pragma unroll
  for (int j = 0; j < DPL; ++j) {
    const int c = lane + 32 * j;
    if (c < dim) d[c] = acc[j];
  }
  if (lane == 0) *head = row;
}

// in[hin[e]] += din[e], out[hout[e]] += dout[e]; warp 0 of block 0 first adds the batch loss to
// *epoch_loss: lane l sums loss[l], loss[l + 32], ... in f64, then the xor butterfly 16 .. 1.
__global__ void __launch_bounds__(kBlock) k_n2v_apply(int nb, int S, int dim, float* __restrict__ tin,
                                                      float* __restrict__ tout, const float* __restrict__ din,
                                                      const int32_t* __restrict__ hin, const float* __restrict__ dout,
                                                      const int32_t* __restrict__ hout,
                                                      const double* __restrict__ loss, double* __restrict__ epoch_loss) {
  const int lane = threadIdx.x & 31;
  if (blockIdx.x == 0 && threadIdx.x < 32) {
    double s = 0.0;
    for (int i = lane; i < nb; i += 32) s = __dadd_rn(s, loss[i]);
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) s = __dadd_rn(s, __shfl_xor_sync(0xffffffffu, s, off));
    if (lane == 0) *epoch_loss = __dadd_rn(*epoch_loss, s);
  }
  const int64_t nin = nb, total = nin + (int64_t)nb * S;
  const int64_t warps = (int64_t)gridDim.x * kWarps;
  for (int64_t e = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5); e < total; e += warps) {
    const bool in_side = e < nin;
    const int64_t i = in_side ? e : e - nin;
    const int32_t r = in_side ? hin[i] : hout[i];
    if (r < 0) continue;
    float* t = (in_side ? tin : tout) + (int64_t)r * dim;
    const float* d = (in_side ? din : dout) + i * dim;
    for (int c = lane; c < dim; c += 32) t[c] = __fadd_rn(t[c], d[c]);
  }
}

int lanes_of(int dim) {
  const int dpl = (dim + 31) / 32;
  return dpl <= 1 ? 1 : dpl <= 2 ? 2 : dpl <= 4 ? 4 : 8;
}

template <int DPL>
int train_batch(hge_ctx* ctx, int nb, int S, int dim, int32_t V, int64_t pb, float lr, float* tin, float* tout,
                const int32_t* cen, const int32_t* cx, float* G, double* loss, const uint64_t* in_key,
                const int32_t* in_val, const uint64_t* out_key, const int32_t* out_val, float* din, int32_t* hin,
                float* dout, int32_t* hout, double* epoch_loss) {
  // cen, cx and G are indexed from the batch's first pair: shift by pb
  k_n2v_coef<DPL><<<(nb + kWarps - 1) / kWarps, kBlock, 0, ctx->stream>>>(nb, S, dim, lr, tin, tout, cen + pb,
                                                                          cx + pb * S, G, loss);
  HGE_CHECK_LAUNCH(ctx);
  const int64_t entries = (int64_t)nb * (S + 1);
  k_n2v_delta<DPL><<<(unsigned)((entries + kWarps - 1) / kWarps), kBlock, 0, ctx->stream>>>(
      nb, S, dim, V, pb, tin, tout, cen, cx, G, in_key, in_val, out_key, out_val, din, hin, dout, hout);
  HGE_CHECK_LAUNCH(ctx);
  k_n2v_apply<<<grid_for(ctx, entries * 32), kBlock, 0, ctx->stream>>>(nb, S, dim, tin, tout, din, hin, dout, hout,
                                                                      loss, epoch_loss);
  HGE_CHECK_LAUNCH(ctx);
  return HGE_OK;
}

int noise_of(hge_ctx* ctx, const int64_t* cum, int32_t V, N2vNoise* noise) {
  int64_t total = 0;
  HGE_TRY(read_back(ctx, cum + V, &total, 1));
  HGE_REQUIRE(total >= 1, "node2vec: the noise table's total %lld is not positive", (long long)total);
  uint64_t mask = 0;
  while (mask < (uint64_t)total - 1) mask = (mask << 1) | 1;
  *noise = N2vNoise{cum, V, (uint64_t)total, mask};
  return HGE_OK;
}

}  // namespace

extern "C" {

int hge_n2v_init(hge_ctx* ctx, int32_t num_vertices, int dim, uint64_t seed, float* tin, float* tout) {
  const char* what = "hge_n2v_init";
  HGE_REQUIRE(ctx && tin && tout, "%s: NULL argument", what);
  HGE_REQUIRE(num_vertices >= 1, "%s: %d vertices", what, num_vertices);
  HGE_REQUIRE(dim >= 1 && dim <= kMaxDim, "%s: dimension %d not in [1, %d]", what, dim, kMaxDim);
  HGE_CUDA(cudaSetDevice(ctx->device));
  const float offset = -0.5f / (float)dim, scale = 1.f / (float)dim;
  k_init_table<<<grid_for(ctx, (int64_t)num_vertices * ((dim + 3) / 4)), kBlock, 0, ctx->stream>>>(
      num_vertices, dim, seed, HGE_PHASE_N2V_INIT, offset, scale, tin);
  HGE_CHECK_LAUNCH(ctx);
  HGE_CUDA(cudaMemsetAsync(tout, 0, sizeof(float) * (size_t)num_vertices * dim, ctx->stream));
  return HGE_OK;
}

int hge_n2v_walks(hge_ctx* ctx, hge_incidence* inc, int num_walks, int walk_length, double p, double q,
                  uint64_t seed, int32_t* walks, int64_t* counts) {
  const char* what = "hge_n2v_walks";
  HGE_REQUIRE(ctx && inc && walks && counts, "%s: NULL argument", what);
  HGE_REQUIRE(!inc->sharded, "%s: needs a whole (not sharded) incidence", what);
  HGE_REQUIRE(num_walks >= 1 && walk_length >= 1, "%s: num_walks = %d, walk_length = %d must be >= 1", what,
              num_walks, walk_length);
  HGE_REQUIRE(p > 0 && q > 0 && isfinite(p) && isfinite(q), "%s: p = %g, q = %g must be positive and finite",
              what, p, q);
  const int64_t V = (int64_t)inc->N + inc->E;
  HGE_REQUIRE(V >= 1 && V < ((int64_t)1 << 31), "%s: %lld vertices", what, (long long)V);
  HGE_CUDA(cudaSetDevice(ctx->device));
  const int64_t total = (int64_t)num_walks * V;
  HGE_CUDA(cudaMemsetAsync(counts, 0, sizeof(int64_t) * V, ctx->stream));
  const N2vGraph g{inc->N, inc->n2e_ptr, inc->n2e_idx, inc->e2n_ptr, inc->e2n_idx};
  k_n2v_walks<<<grid_for(ctx, total, 128), 128, 0, ctx->stream>>>(g, total, (int32_t)V, walk_length, p, q, seed,
                                                                   walks,
                                                                   reinterpret_cast<unsigned long long*>(counts));
  HGE_CHECK_LAUNCH(ctx);
  HGE_CUDA(cudaStreamSynchronize(ctx->stream));
  return HGE_OK;
}

int hge_n2v_pairs(hge_ctx* ctx, const int32_t* walks, int64_t num_walk_items, int walk_length, int window,
                  uint64_t seed, int32_t* pairs, int64_t capacity, int64_t* num_pairs) {
  const char* what = "hge_n2v_pairs";
  HGE_REQUIRE(ctx && walks && num_pairs, "%s: NULL argument", what);
  HGE_REQUIRE(num_walk_items >= 0 && walk_length >= 1, "%s: bad walk shape [%lld, %d]", what,
              (long long)num_walk_items, walk_length);
  HGE_REQUIRE(window >= 1, "%s: window = %d must be >= 1", what, window);
  HGE_CUDA(cudaSetDevice(ctx->device));
  const int64_t tokens = num_walk_items * walk_length;
  DevBuf<int64_t> counts(ctx), offsets(ctx);
  DevBuf<char> temp(ctx);
  HGE_TRY(counts.alloc((size_t)tokens + 1));
  HGE_TRY(offsets.alloc((size_t)tokens + 1));
  k_n2v_pair_counts<<<grid_for(ctx, tokens + 1), kBlock, 0, ctx->stream>>>(walks, tokens, walk_length, window, seed,
                                                                          counts.p);
  HGE_CHECK_LAUNCH(ctx);
  size_t bytes = 0;
  HGE_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, bytes, counts.p, offsets.p, tokens + 1, ctx->stream));
  HGE_TRY(temp.alloc(bytes));
  HGE_CUDA(cub::DeviceScan::ExclusiveSum(temp.p, bytes, counts.p, offsets.p, tokens + 1, ctx->stream));
  ctx->launches++;
  int64_t P = 0;
  HGE_TRY(read_back(ctx, offsets.p + tokens, &P, 1));
  *num_pairs = P;
  HGE_REQUIRE(P < ((int64_t)1 << 31), "%s: %lld pairs, at or above the epoch order's limit of 2^31", what,
              (long long)P);
  if (!pairs) return HGE_OK;
  HGE_REQUIRE(capacity >= P, "%s: room for %lld pairs, %lld needed", what, (long long)capacity, (long long)P);
  k_n2v_pair_emit<<<grid_for(ctx, tokens), kBlock, 0, ctx->stream>>>(walks, tokens, walk_length, window, seed,
                                                                    offsets.p, reinterpret_cast<int2*>(pairs));
  HGE_CHECK_LAUNCH(ctx);
  HGE_CUDA(cudaStreamSynchronize(ctx->stream));
  return HGE_OK;
}

int hge_n2v_negatives(hge_ctx* ctx, int64_t num_pairs, const int64_t* cum, int32_t num_vertices, int negative,
                      uint64_t seed, int epoch, int32_t* out) {
  const char* what = "hge_n2v_negatives";
  HGE_REQUIRE(ctx && cum && (out || num_pairs == 0 || negative == 0), "%s: NULL argument", what);
  HGE_REQUIRE(num_pairs >= 0 && num_vertices >= 1 && negative >= 0 && epoch >= 0, "%s: bad arguments", what);
  HGE_CUDA(cudaSetDevice(ctx->device));
  if (num_pairs == 0 || negative == 0) return HGE_OK;
  N2vNoise noise;
  HGE_TRY(noise_of(ctx, cum, num_vertices, &noise));
  k_n2v_negatives<<<grid_for(ctx, num_pairs), kBlock, 0, ctx->stream>>>(noise, num_pairs, negative, seed,
                                                                       (uint32_t)epoch, out);
  HGE_CHECK_LAUNCH(ctx);
  HGE_CUDA(cudaStreamSynchronize(ctx->stream));
  return HGE_OK;
}

int hge_n2v_train_epoch(hge_ctx* ctx, int32_t num_vertices, int dim, float* tin, float* tout, const int32_t* pairs,
                        int64_t num_pairs, const int64_t* cum, int negative, uint64_t seed, int epoch, int epochs,
                        int batch_pairs, double alpha, double min_alpha, int64_t plan_bytes, double* loss) {
  const char* what = "hge_n2v_train_epoch";
  HGE_REQUIRE(ctx && tin && tout && cum && loss && (pairs || num_pairs == 0), "%s: NULL argument", what);
  HGE_REQUIRE(num_vertices >= 1, "%s: %d vertices", what, num_vertices);
  HGE_REQUIRE(dim >= 1 && dim <= kMaxDim, "%s: dimension %d not in [1, %d]", what, dim, kMaxDim);
  HGE_REQUIRE(num_pairs >= 0 && num_pairs < ((int64_t)1 << 31), "%s: %lld pairs not in [0, 2^31)", what,
              (long long)num_pairs);
  HGE_REQUIRE(negative >= 0, "%s: negative = %d", what, negative);
  HGE_REQUIRE(epochs >= 1 && epoch >= 0 && epoch < epochs, "%s: epoch %d of %d", what, epoch, epochs);
  HGE_REQUIRE(batch_pairs >= 1, "%s: batch_pairs = %d", what, batch_pairs);
  HGE_REQUIRE(plan_bytes >= 0, "%s: plan_bytes = %lld", what, (long long)plan_bytes);
  HGE_CUDA(cudaSetDevice(ctx->device));
  *loss = 0.0;
  const int64_t P = num_pairs;
  if (P == 0) return HGE_OK;
  const int S = negative + 1;
  const int B = (int)std::min<int64_t>(batch_pairs, P);
  HGE_REQUIRE((int64_t)B * S < ((int64_t)1 << 31), "%s: %d pairs of %d slots per batch", what, B, S);
  N2vNoise noise;
  HGE_TRY(noise_of(ctx, cum, num_vertices, &noise));
  // chunk of whole batches: per pair 4 + 4 S plan bytes and two (key, value) buffers of 12 (1 + S)
  const int64_t per_pair = 4 + 4 * S + 2 * 12 * (int64_t)(1 + S);
  const int64_t budget = plan_bytes > 0 ? plan_bytes : kDefaultPlanBytes;
  const int64_t nbatches = (P + B - 1) / B;
  int64_t chunk_batches = std::max<int64_t>(1, budget / (per_pair * B));
  chunk_batches = std::min<int64_t>(chunk_batches, nbatches);
  chunk_batches = std::min<int64_t>(chunk_batches, (((int64_t)1 << 31) - 1) / ((int64_t)B * S));
  const int64_t cp = chunk_batches * B;
  int bits = 0;
  while (((int64_t)1 << bits) < chunk_batches) ++bits;
  DevBuf<int32_t> order(ctx), cen(ctx), cx(ctx), in_val(ctx), in_val2(ctx), out_val(ctx), out_val2(ctx), hin(ctx),
      hout(ctx);
  DevBuf<uint64_t> in_key(ctx), in_key2(ctx), out_key(ctx), out_key2(ctx);
  DevBuf<float> G(ctx), din(ctx), dout(ctx);
  DevBuf<double> bl(ctx), el(ctx);
  DevBuf<char> temp(ctx);
  HGE_TRY(order.alloc((size_t)P));
  HGE_TRY(hge_shuffle_order_phase(ctx, seed, HGE_PHASE_N2V_SHUFFLE, (uint32_t)epoch, P, order.p, HGE_MEM_DEVICE));
  HGE_TRY(cen.alloc((size_t)cp));
  HGE_TRY(cx.alloc((size_t)cp * S));
  HGE_TRY(in_key.alloc((size_t)cp));
  HGE_TRY(in_key2.alloc((size_t)cp));
  HGE_TRY(in_val.alloc((size_t)cp));
  HGE_TRY(in_val2.alloc((size_t)cp));
  HGE_TRY(out_key.alloc((size_t)cp * S));
  HGE_TRY(out_key2.alloc((size_t)cp * S));
  HGE_TRY(out_val.alloc((size_t)cp * S));
  HGE_TRY(out_val2.alloc((size_t)cp * S));
  HGE_TRY(G.alloc((size_t)B * S));
  HGE_TRY(bl.alloc((size_t)B));
  HGE_TRY(din.alloc((size_t)B * dim));
  HGE_TRY(dout.alloc((size_t)B * S * dim));
  HGE_TRY(hin.alloc((size_t)B));
  HGE_TRY(hout.alloc((size_t)B * S));
  HGE_TRY(el.alloc(1));
  HGE_CUDA(cudaMemsetAsync(el.p, 0, sizeof(double), ctx->stream));
  size_t tb_in = 0, tb_out = 0;
  {
    cub::DoubleBuffer<uint64_t> k(in_key.p, in_key2.p);
    cub::DoubleBuffer<int32_t> v(in_val.p, in_val2.p);
    HGE_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tb_in, k, v, cp, 0, 32 + bits, ctx->stream));
    cub::DoubleBuffer<uint64_t> k2(out_key.p, out_key2.p);
    cub::DoubleBuffer<int32_t> v2(out_val.p, out_val2.p);
    HGE_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tb_out, k2, v2, cp * S, 0, 32 + bits, ctx->stream));
  }
  HGE_TRY(temp.alloc(std::max(tb_in, tb_out)));
  const int dpl = lanes_of(dim);
  const double T = (double)epochs * (double)nbatches;
  for (int64_t c0 = 0; c0 < P; c0 += cp) {
    const int64_t count = std::min<int64_t>(cp, P - c0);
    const int64_t nbc = (count + B - 1) / B;
    k_n2v_plan<<<grid_for(ctx, count), kBlock, 0, ctx->stream>>>(reinterpret_cast<const int2*>(pairs), order.p, c0,
                                                                 count, P, B, negative, noise, seed, (uint32_t)epoch,
                                                                 cen.p, cx.p, in_key.p, in_val.p, out_key.p,
                                                                 out_val.p);
    HGE_CHECK_LAUNCH(ctx);
    // stable LSD radix sorts: equal keys keep ascending (pair position, slot) order
    cub::DoubleBuffer<uint64_t> ki(in_key.p, in_key2.p), ko(out_key.p, out_key2.p);
    cub::DoubleBuffer<int32_t> vi(in_val.p, in_val2.p), vo(out_val.p, out_val2.p);
    size_t b1 = tb_in, b2 = tb_out;
    HGE_CUDA(cub::DeviceRadixSort::SortPairs(temp.p, b1, ki, vi, count, 0, 32 + bits, ctx->stream));
    HGE_CUDA(cub::DeviceRadixSort::SortPairs(temp.p, b2, ko, vo, count * S, 0, 32 + bits, ctx->stream));
    ctx->launches += 2;
    for (int64_t b = 0; b < nbc; ++b) {
      const int64_t pb = b * B;
      const int nb = (int)std::min<int64_t>(B, count - pb);
      const double t = (double)(epoch * nbatches + c0 / B + b);
      const float lr = (float)(alpha - (alpha - min_alpha) * (t / T));
      int rc;
      switch (dpl) {
#define N2V_BATCH(D)                                                                                              \
  rc = train_batch<D>(ctx, nb, S, dim, num_vertices, pb, lr, tin, tout, cen.p, cx.p, G.p, bl.p, ki.Current(),   \
                      vi.Current(), ko.Current(), vo.Current(), din.p, hin.p, dout.p, hout.p, el.p);
        case 1: N2V_BATCH(1) break;
        case 2: N2V_BATCH(2) break;
        case 4: N2V_BATCH(4) break;
        default: N2V_BATCH(8) break;
#undef N2V_BATCH
      }
      HGE_TRY(rc);
    }
  }
  return read_back(ctx, el.p, loss, 1);
}

}  // extern "C"
