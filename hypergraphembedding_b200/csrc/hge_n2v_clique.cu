// node2vec walks on the weighted clique expansions of a hypergraph (DESIGN.md section 9.13), drawn
// straight from the incidence: the expansion is never built.  tests/n2v_clique_ref.py restates
// the walks; pairs, noise table, negatives, initial table and training are those of csrc/hge_n2v.cu.
//
// Side 0: vertices are the N nodes, w(u, x) = number of edges holding both (u != x).  Side 1: the
// same on the transpose, vertices are the E edges and w(c, y) = number of shared members.  Below,
// "edge" means an incident id of the other side and "member" a vertex of this side.
//
// Proposal from v, S(v) = sum over edges e of v of (|e| - 1): e with probability (|e| - 1) / S(v),
// then a member x != v of e uniformly, so P(x) = w(v, x) / S(v), the weighted first-order step.
// Second order, with t the previous vertex, node2vec's weight alpha(t, x) w(v, x) scaled by p q:
// a' = q (x = t), p q (x shares an edge with t) or p (otherwise), m = max(q, p q, p); a proposal
// is accepted iff (u 2^-32) m < a' in f64, each operation rounded on its own, and the word u is
// drawn only when a' < m (so p = q = 1 draws none).  The first step takes the first proposal.
#include <math.h>

#include <cub/device/device_scan.cuh>

#include "hge_common.cuh"
#include "hge_incidence.cuh"
#include "hge_philox.cuh"

namespace {

// Largest max(q, pq, p) / min(q, pq, p) accepted: the expected number of proposals per step is at
// most this ratio.
constexpr double kMaxWeightRatio = 65536.0;

struct CliqueSide {
  const int64_t* ptr;    // [V + 1] vertex -> its sorted incident edges idx[ptr[v] .. ptr[v + 1])
  const int32_t* idx;
  const int64_t* optr;   // edge -> its sorted members oidx[optr[e] .. optr[e + 1])
  const int32_t* oidx;
  const int64_t* cum;    // [nnz] inclusive prefix of (|e_k| - 1) over the incidences in row order
};

// first position i of the sorted row[0 .. n) with row[i] >= key
__device__ __forceinline__ int64_t lower_bound(const int32_t* __restrict__ row, int64_t lo, int64_t hi, int32_t key) {
  while (lo < hi) {
    const int64_t mid = lo + ((hi - lo) >> 1);
    if (row[mid] < key) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// whether vertices a != b share an edge: each id of the shorter sorted row is searched in the
// longer one, each search starting where the previous one ended
__device__ bool shares_edge(const CliqueSide& g, int32_t a, int32_t b) {
  int64_t sb = g.ptr[a], se = g.ptr[a + 1], lb = g.ptr[b], le = g.ptr[b + 1];
  if (se - sb > le - lb) {
    const int64_t t0 = sb, t1 = se;
    sb = lb, se = le, lb = t0, le = t1;
  }
  for (int64_t k = sb; k < se && lb < le; ++k) {
    const int32_t e = g.idx[k];
    lb = lower_bound(g.idx, lb, le, e);
    if (lb < le && g.idx[lb] == e) return true;
  }
  return false;
}

__global__ void k_clique_weights(const int32_t* __restrict__ idx, const int64_t* __restrict__ optr, int64_t nnz,
                                 int64_t* __restrict__ w) {
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < nnz; k += (int64_t)gridDim.x * blockDim.x) {
    const int32_t e = idx[k];
    w[k] = optr[e + 1] - optr[e] - 1;
  }
}

// Walk w (0 <= w < num_walks V) starts at vertex w mod V and reads item w of
// HGE_PHASE_N2V_CLIQUE_WALK.  Per proposal: r uniform on [0, S(v)) by 64-bit masked rejection (two
// words (hi, lo) per round), e = the first incidence of v whose row prefix exceeds r, then
// below(|e| - 1) over e's sorted members with v's position skipped, then the acceptance word when
// a' < m.  A vertex with S(v) = 0 gives [v, -1, ...].  If S(v) > 0, every neighbour x shares an
// edge of at least two members with v, so S(x) > 0 and a walk never stops after its second
// vertex: n2v_window's length rule (walk[1] < 0 means length 1) holds for these walks too.
__global__ void k_n2v_clique_walks(CliqueSide g, int64_t walks_total, int32_t V, int L, double p, double q,
                                   uint64_t seed, int32_t* __restrict__ walks,
                                   unsigned long long* __restrict__ counts) {
  const double pq = __dmul_rn(p, q);
  const double m = fmax(fmax(q, pq), p);
  const bool adjacency_matters = pq != p;
  for (int64_t w = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; w < walks_total;
       w += (int64_t)gridDim.x * blockDim.x) {
    int32_t* out = walks + w * L;
    HgeStreamRng rng(seed, HGE_PHASE_N2V_CLIQUE_WALK, (uint64_t)w);
    int32_t v = (int32_t)(w % V), t = -1;
    out[0] = v;
    atomicAdd(counts + v, 1ull);
    {
      const int64_t b = g.ptr[v], end = g.ptr[v + 1];
      if (end == b || g.cum[end - 1] == (b > 0 ? g.cum[b - 1] : 0)) {
        for (int i = 1; i < L; ++i) out[i] = -1;
        continue;
      }
    }
    for (int i = 1; i < L; ++i) {
      const int64_t b = g.ptr[v], end = g.ptr[v + 1];
      const int64_t base = b > 0 ? g.cum[b - 1] : 0;
      const uint64_t S = (uint64_t)(g.cum[end - 1] - base);
      const uint64_t mask = S > 1 ? ~0ull >> __clzll((long long)(S - 1)) : 0ull;
      int32_t x;
      for (;;) {
        uint64_t r;
        do {
          const uint64_t hi = rng.next();
          r = ((hi << 32) | rng.next()) & mask;
        } while (r >= S);
        const int64_t key = base + (int64_t)r;
        int64_t lo = b, hi = end - 1;   // first k with cum[k] > key
        while (lo < hi) {
          const int64_t mid = lo + ((hi - lo) >> 1);
          if (g.cum[mid] > key) hi = mid; else lo = mid + 1;
        }
        const int32_t e = g.idx[lo];
        const int64_t eb = g.optr[e];
        const int64_t size = g.optr[e + 1] - eb;
        const int32_t* mem = g.oidx + eb;
        const int64_t j = rng.below((uint32_t)(size - 1));
        const int64_t pos = lower_bound(mem, 0, size, v);
        x = mem[j < pos ? j : j + 1];
        if (t < 0) break;
        double a = p;
        if (x == t) {
          a = q;
        } else if (adjacency_matters) {
          const int64_t pt = lower_bound(mem, 0, size, t);
          if ((pt < size && mem[pt] == t) || shares_edge(g, t, x)) a = pq;
        }
        if (!(a < m)) break;
        const double u = __dmul_rn((double)rng.next(), 0x1p-32);
        if (__dmul_rn(u, m) < a) break;
      }
      out[i] = x;
      atomicAdd(counts + x, 1ull);
      t = v;
      v = x;
    }
  }
}

}  // namespace

extern "C" {

int hge_n2v_clique_walks(hge_ctx* ctx, hge_incidence* inc, int side, int num_walks, int walk_length, double p,
                         double q, uint64_t seed, int32_t* walks, int64_t* counts) {
  const char* what = "hge_n2v_clique_walks";
  HGE_REQUIRE(ctx && inc && walks && counts, "%s: NULL argument", what);
  HGE_REQUIRE(!inc->sharded, "%s: needs a whole (not sharded) incidence", what);
  HGE_REQUIRE(side == 0 || side == 1, "%s: side = %d must be 0 (nodes) or 1 (edges)", what, side);
  HGE_REQUIRE(num_walks >= 1 && walk_length >= 1, "%s: num_walks = %d, walk_length = %d must be >= 1", what,
              num_walks, walk_length);
  HGE_REQUIRE(p > 0 && q > 0 && isfinite(p) && isfinite(q), "%s: p = %g, q = %g must be positive and finite",
              what, p, q);
  const double pq = p * q;
  const double ratio = std::max(std::max(q, pq), p) / std::min(std::min(q, pq), p);
  HGE_REQUIRE(ratio <= kMaxWeightRatio,
              "%s: p = %g, q = %g give max / min of (q, p q, p) = %g, above %g (the expected proposals per step)",
              what, p, q, ratio, kMaxWeightRatio);
  const int32_t V = side == 0 ? inc->N : inc->E;
  HGE_REQUIRE(V >= 1, "%s: %d vertices", what, V);
  HGE_CUDA(cudaSetDevice(ctx->device));
  const CliqueSide g0{inc->n2e_ptr, inc->n2e_idx, inc->e2n_ptr, inc->e2n_idx, nullptr};
  const CliqueSide g1{inc->e2n_ptr, inc->e2n_idx, inc->n2e_ptr, inc->n2e_idx, nullptr};
  CliqueSide g = side == 0 ? g0 : g1;
  int64_t nnz = 0;
  HGE_TRY(read_back(ctx, g.ptr + V, &nnz, 1));
  DevBuf<int64_t> cum(ctx);
  DevBuf<char> temp(ctx);
  HGE_TRY(cum.alloc((size_t)nnz));
  if (nnz > 0) {
    k_clique_weights<<<grid_for(ctx, nnz), 256, 0, ctx->stream>>>(g.idx, g.optr, nnz, cum.p);
    HGE_CHECK_LAUNCH(ctx);
    size_t bytes = 0;
    HGE_CUDA(cub::DeviceScan::InclusiveSum(nullptr, bytes, cum.p, nnz, ctx->stream));
    HGE_TRY(temp.alloc(bytes));
    HGE_CUDA(cub::DeviceScan::InclusiveSum(temp.p, bytes, cum.p, nnz, ctx->stream));
    ctx->launches++;
  }
  g.cum = cum.p;
  const int64_t total = (int64_t)num_walks * V;
  HGE_CUDA(cudaMemsetAsync(counts, 0, sizeof(int64_t) * V, ctx->stream));
  k_n2v_clique_walks<<<grid_for(ctx, total, 128), 128, 0, ctx->stream>>>(
      g, total, V, walk_length, p, q, seed, walks, reinterpret_cast<unsigned long long*>(counts));
  HGE_CHECK_LAUNCH(ctx);
  HGE_CUDA(cudaStreamSynchronize(ctx->stream));
  return HGE_OK;
}

}  // extern "C"
