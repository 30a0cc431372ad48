// Algebraic-distance relaxation on sm_100a.
//
// Reference arithmetic (algebraic_distance.py:34-123), with A the N x E incidence matrix,
// w_E[e] = 1 / deg(e), w_N[n] = 1 / deg(n), s_N = A w_E, s_E = A^T w_N:
//     XN' = (XN + (A  (XE  * w_E)) / s_N) / 2          node half, OLD edge rows
//     XE' = (XE + (A^T (XN' * w_N)) / s_E) / 2          edge half, NEW node rows
//     lo/hi = per-column min/max over XN' and XE' jointly; X <- (X' - lo) / (hi - lo)
//
// Storage ("Y-space").  Rows are kept pre-multiplied by their own weight, Y[r] = X'[r] * w[r],
// fp32 row-major with the row padded to a multiple of 4 floats (ld).  The gather of a
// half-sweep is then a plain sum of neighbour rows (no per-incidence weight lookup), and a
// row's own value is recovered as Y[r] * deg(r).  The rescale is lazy: X' is what is stored,
// and the affine map of sweep t-1, (lo, 1/(hi-lo)), is applied when sweep t reads a row.  It
// commutes with the gather:  sum_b w_b (X'_b - lo) inv / s = inv (acc / s - lo),  so it costs
// two FMAs per row instead of a full read+write pass per sweep.  Per-column min / max of a
// sweep are accumulated by the two half-sweep kernels with warp shuffles, shared memory and
// one atomicMin / atomicMax per column per block on order-preserving int32 encodings.
//
// Every row is updated in place by the one sub-warp (or the last chunk-warp) that owns it, so
// a half-sweep reads each own row once, writes it once, and gathers nnz neighbour rows.
#include <cub/device/device_radix_sort.cuh>

#include <algorithm>
#include <cstring>
#include <new>
#include <vector>

#include "hge_incidence.cuh"
#include "hge_sweep.cuh"

namespace {

constexpr int kBlock = 256;
constexpr int kWarps = kBlock / 32;
constexpr unsigned kFull = 0xffffffffu;

// ----------------------------------------------------------------------------------------
// setup kernels
// ----------------------------------------------------------------------------------------

__global__ void k_row_degree(int32_t rows, const int64_t* __restrict__ ptr,
                             int32_t* __restrict__ deg) {
  for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < rows;
       r += (int64_t)gridDim.x * blockDim.x)
    deg[r] = (int32_t)(ptr[r + 1] - ptr[r]);
}

// ---- edge -> node CSR built on the device from the node -> edge CSR ---------------------------
// (the host-buffer call then uploads one orientation only: 44 of 284 MB less on config 2)

// row id of every stored incidence of a CSR
__global__ void k_expand_rows(int32_t rows, const int64_t* __restrict__ ptr, int32_t* __restrict__ out) {
  const int lane = threadIdx.x & 7;
  const int64_t ng = (int64_t)gridDim.x * (blockDim.x >> 3);
  for (int64_t r = blockIdx.x * (int64_t)(blockDim.x >> 3) + (threadIdx.x >> 3); r < rows; r += ng)
    for (int64_t p = ptr[r] + lane, e = ptr[r + 1]; p < e; p += 8) out[p] = (int32_t)r;
}

// ptr[c] = first position of column c in the sorted column list (ptr[cols] = nnz)
__global__ void k_transpose_ptr(int32_t cols, int64_t nnz, const int32_t* __restrict__ sorted_cols,
                                int64_t* __restrict__ ptr) {
  for (int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; c <= cols;
       c += (int64_t)gridDim.x * blockDim.x) {
    int64_t lo = 0, hi = nnz;
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (sorted_cols[mid] < c) lo = mid + 1; else hi = mid;
    }
    ptr[c] = lo;
  }
}

// wsum[r] = sum_{b in row r} 1 / other_deg[b], accumulated in f64.  Rows up to kWsumLong
// incidences: 8 lanes per row.  Longer rows are only appended to `long_rows` here and summed by
// k_row_wsum_long with one block per row: a 1e5-member edge on 8 lanes was 4.5 of the 7 ms the
// whole incidence set-up took.  Both sums have a fixed shape, so the result is the same on
// every run whatever order the long rows were listed in.
constexpr int kWsumLong = 512;

__global__ void k_row_wsum(int32_t rows, const int64_t* __restrict__ ptr,
                           const int32_t* __restrict__ idx,
                           const int32_t* __restrict__ other_deg, double* __restrict__ wsum,
                           int32_t* __restrict__ long_rows, int32_t* __restrict__ n_long) {
  const int sub = threadIdx.x & 7;
  const int64_t ng = (int64_t)gridDim.x * (blockDim.x >> 3);
  const int64_t g0 = blockIdx.x * (int64_t)(blockDim.x >> 3) + (threadIdx.x >> 3);
  // every lane of a warp runs the same number of outer iterations (full-mask shuffles below)
  for (int64_t base = 0; base < rows; base += ng) {
    const int64_t r = base + g0;
    double s = 0.0;
    bool is_long = false;
    if (r < rows) {
      const int64_t b = ptr[r], e = ptr[r + 1];
      is_long = e - b > kWsumLong;
      if (!is_long)
        for (int64_t p = b + sub; p < e; p += 8) s += 1.0 / (double)other_deg[idx[p]];
    }
#pragma unroll
    for (int off = 4; off; off >>= 1) s += __shfl_xor_sync(kFull, s, off);
    if (r < rows && sub == 0) {
      if (is_long)
        long_rows[atomicAdd(n_long, 1)] = (int32_t)r;
      else
        wsum[r] = s;
    }
  }
}

__global__ void __launch_bounds__(kBlock) k_row_wsum_long(
    const int32_t* __restrict__ long_rows, const int32_t* __restrict__ n_long,
    const int64_t* __restrict__ ptr, const int32_t* __restrict__ idx,
    const int32_t* __restrict__ other_deg, double* __restrict__ wsum) {
  __shared__ double part[kWarps];
  const int n = *n_long;
  for (int i = blockIdx.x; i < n; i += gridDim.x) {
    const int32_t r = long_rows[i];
    const int64_t b = ptr[r], e = ptr[r + 1];
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;     // four independent gathers in flight
    int64_t p = b + threadIdx.x;
    for (; p + 3 * kBlock < e; p += 4 * kBlock) {
      const int32_t d0 = other_deg[idx[p]], d1 = other_deg[idx[p + kBlock]];
      const int32_t d2 = other_deg[idx[p + 2 * kBlock]], d3 = other_deg[idx[p + 3 * kBlock]];
      s0 += 1.0 / (double)d0;
      s1 += 1.0 / (double)d1;
      s2 += 1.0 / (double)d2;
      s3 += 1.0 / (double)d3;
    }
    for (; p < e; p += kBlock) s0 += 1.0 / (double)other_deg[idx[p]];
    double s = (s0 + s1) + (s2 + s3);
#pragma unroll
    for (int off = 16; off; off >>= 1) s += __shfl_xor_sync(kFull, s, off);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0.0;
      for (int w = 0; w < kWarps; ++w) t += part[w];
      wsum[r] = t;
    }
    __syncthreads();
  }
}

__global__ void k_invert(int32_t rows, const double* __restrict__ wsum, float* __restrict__ invs) {
  for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < rows;
       r += (int64_t)gridDim.x * blockDim.x)
    invs[r] = (float)(1.0 / wsum[r]);
}

// pos[t * rows + r] = first incidence of row r whose column id is >= t * tile_cols, for
// t = 0 .. tiles (column ids are sorted inside a row): the sub-range of row r that falls into
// column tile t is [pos[t][r], pos[t + 1][r]).
__global__ void k_tile_offsets(int32_t rows, const int64_t* __restrict__ ptr,
                               const int32_t* __restrict__ idx, int tiles, int32_t tile_cols,
                               int64_t* __restrict__ pos) {
  const int64_t total = (int64_t)rows * (tiles + 1);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int t = (int)(i / rows);
    const int32_t r = (int32_t)(i - (int64_t)t * rows);
    const int64_t b = ptr[r], e = ptr[r + 1];
    int64_t lo = b, hi = e;
    if (t == 0) hi = b;
    else if (t == tiles) lo = e;
    else {
      const int64_t want = (int64_t)t * tile_cols;
      while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (idx[mid] < want) lo = mid + 1; else hi = mid;
      }
    }
    pos[i] = lo;
  }
}

// Number of (row, tile) pairs with at least one incidence (how much per-pair work tiling adds).
__global__ void k_count_tile_pairs(int64_t total, int32_t rows, const int64_t* __restrict__ pos,
                                   unsigned long long* count) {
  unsigned long long c = 0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x)
    c += pos[i + rows] > pos[i];
#pragma unroll
  for (int off = 16; off; off >>= 1) c += __shfl_xor_sync(kFull, c, off);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(count, c);
}

// Reduce-scatter of locally accumulated partial rows [row0, row0 + rows): a row goes to the
// staging block of its owner, slot `rank` (the push the gather kernel does itself when untiled).
__global__ void k_push_rows(int32_t row0, int32_t rows, int ld4, const float4* __restrict__ raw,
                            float4* const* __restrict__ peer_stage, int rank, HgeOwnerMap map) {
  const int64_t total = (int64_t)rows * ld4;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t r = row0 + (int32_t)(i / ld4);
    const int c4 = (int)(i - (int64_t)(r - row0) * ld4);
    int owner;
    int32_t idx;
    map.locate(r, owner, idx);
    peer_stage[owner][((size_t)rank * map.sub_rows + idx) * ld4 + c4] = __ldcs(raw + (size_t)r * ld4 + c4);
  }
}

// Stand-alone joint rescale (_helper_scale_embeddings, algebraic_distance.py:97-123) of dense
// [rows, R] blocks: per-column min / max over both blocks, then x <- (x - min) / (max - min).
__global__ void k_dense_minmax(int64_t rows, int R, const float* __restrict__ x, int32_t* mm) {
  const int64_t total = rows * R;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % R);
    const int v = hge_enc(x[i]);
    atomicMin(mm + c, v);
    atomicMax(mm + R + c, v);
  }
}
__global__ void k_dense_rescale(int64_t rows, int R, float* __restrict__ x,
                                const int32_t* __restrict__ mm) {
  const int64_t total = rows * R;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % R);
    const float lo = hge_dec(mm[c]), hi = hge_dec(mm[R + c]);
    x[i] = (x[i] - lo) / (hi - lo);
  }
}

__global__ void k_fill_minmax(int32_t* mm, int slots, int ld) {
  const int n = slots * 2 * ld;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    mm[i] = ((i / ld) & 1) ? INT32_MIN : INT32_MAX;  // [slot][0]=min, [slot][1]=max
}

// X (dense [rows, R]) -> Y (padded [rows, ld]),  Y = X / deg.
__global__ void k_load_rows(int64_t rows, int R, int ld, const float* __restrict__ x,
                            const int32_t* __restrict__ deg, float* __restrict__ y) {
  const int64_t total = rows * ld;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / ld;
    const int c = (int)(i - r * ld);
    float v = 0.f;
    if (c < R) v = x[r * R + c] * __frcp_rn((float)deg[r]);
    y[i] = v;
  }
}

// Y -> X with the affine map of the last sweep (mm == nullptr: identity).
__global__ void k_store_rows(int64_t rows, int R, int ld, const float* __restrict__ y,
                             const int32_t* __restrict__ deg, const int32_t* __restrict__ mm,
                             float* __restrict__ x) {
  const int64_t total = rows * R;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / R;
    const int c = (int)(i - r * R);
    float v = y[r * ld + c] * (float)deg[r];
    if (mm) {
      const float lo = hge_dec(mm[c]);
      const float hi = hge_dec(mm[ld + c]);
      v = (v - lo) / (hi - lo);
    }
    x[i] = v;
  }
}

// Sharded edge half, second part: the raw sums have been all-reduced over the shards.
__global__ void k_edge_finalize(int64_t row0, int64_t rows, int R, int ld,
                                const float* __restrict__ raw,
                                const int32_t* __restrict__ deg, const float* __restrict__ invs,
                                const int32_t* __restrict__ mm_prev, int32_t* __restrict__ mm_cur,
                                float* __restrict__ y) {
  // one thread per (row, column); columns are the fast index so accesses coalesce
  __shared__ int s_min[1024], s_max[1024];
  for (int c = threadIdx.x; c < ld; c += blockDim.x) {
    s_min[c] = INT32_MAX;
    s_max[c] = INT32_MIN;
  }
  __syncthreads();
  const int64_t total = rows * ld;
  for (int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j < total;
       j += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = row0 * ld + j;
    const int64_t r = i / ld;
    const int c = (int)(i - r * ld);
    if (c >= R) continue;
    const float degf = (float)deg[r];
    float own = y[i] * degf;
    if (mm_prev) {
      const float lo = hge_dec(mm_prev[c]);
      const float inv = 1.0f / (hge_dec(mm_prev[ld + c]) - lo);
      own = fmaf(inv, own, -lo * inv);
    }
    const float x = 0.5f * (own + raw[i] * invs[r]);
    y[i] = x * __frcp_rn(degf);
    atomicMin(&s_min[c], hge_enc(x));
    atomicMax(&s_max[c], hge_enc(x));
  }
  __syncthreads();
  for (int c = threadIdx.x; c < R; c += blockDim.x) {
    if (s_min[c] <= s_max[c]) {
      atomicMin(mm_cur + c, s_min[c]);
      atomicMax(mm_cur + ld + c, s_max[c]);
    }
  }
}

// ----------------------------------------------------------------------------------------
// host side: schedule construction
// ----------------------------------------------------------------------------------------

constexpr int kBlocksPerSm = 32;   // grid cap of the kernels of this file, per multiprocessor

// wsum[r] = sum over the row's neighbours b of 1 / other_deg[b] (f64, device).
// Transposes a CSR whose column ids are sorted inside every row: a stable sort of the
// (column, row) pairs by column keeps the rows of a column in ascending order.
int transpose_csr(hge_ctx* ctx, int32_t rows, int32_t cols, int64_t nnz, const int64_t* d_ptr,
                  const int32_t* d_idx, int64_t* t_ptr, int32_t* t_idx) {
  DevBuf<int32_t> row_of(ctx), cols_sorted(ctx);
  DevBuf<char> temp(ctx);
  HGE_TRY(row_of.alloc((size_t)nnz));
  HGE_TRY(cols_sorted.alloc((size_t)nnz));
  k_expand_rows<<<grid_for(ctx, (int64_t)rows * 8, kBlock, kBlocksPerSm), kBlock, 0, ctx->stream>>>(rows, d_ptr,
                                                                                                 row_of.p);
  HGE_CHECK_LAUNCH(ctx);
  int bits = 1;
  while (bits < 31 && ((int64_t)1 << bits) < cols) ++bits;
  size_t temp_bytes = 0;
  HGE_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, d_idx, cols_sorted.p, row_of.p, t_idx, nnz, 0,
                                           bits, ctx->stream));
  HGE_TRY(temp.alloc(temp_bytes));
  HGE_CUDA(cub::DeviceRadixSort::SortPairs(temp.p, temp_bytes, d_idx, cols_sorted.p, row_of.p, t_idx, nnz, 0,
                                           bits, ctx->stream));
  ctx->launches += 3;
  k_transpose_ptr<<<grid_for(ctx, (int64_t)cols + 1, kBlock, kBlocksPerSm), kBlock, 0, ctx->stream>>>(
      cols, nnz, cols_sorted.p, t_ptr);
  HGE_CHECK_LAUNCH(ctx);
  return HGE_OK;
}

int compute_wsum(hge_ctx* ctx, int32_t rows, const int64_t* d_ptr, const int32_t* d_idx,
                 const int32_t* d_other_deg, DevBuf<double>& wsum) {
  HGE_TRY(wsum.alloc((size_t)rows));
  DevBuf<int32_t> long_rows(ctx);   // [0] = count, [1..] = row ids
  HGE_TRY(long_rows.alloc((size_t)rows + 1));
  HGE_CUDA(cudaMemsetAsync(long_rows.p, 0, sizeof(int32_t), ctx->stream));
  k_row_wsum<<<grid_for(ctx, (int64_t)rows * 8, kBlock, kBlocksPerSm), kBlock, 0, ctx->stream>>>(
      rows, d_ptr, d_idx, d_other_deg, wsum.p, long_rows.p + 1, long_rows.p);
  HGE_CHECK_LAUNCH(ctx);
  k_row_wsum_long<<<ctx->num_sms * 4, kBlock, 0, ctx->stream>>>(long_rows.p + 1, long_rows.p, d_ptr, d_idx,
                                                               d_other_deg, wsum.p);
  HGE_CHECK_LAUNCH(ctx);
  return HGE_OK;
}

// invs = 1 / wsum as fp32 (device).
int invert_wsum(hge_ctx* ctx, int32_t rows, const double* wsum, float** invs) {
  HGE_TRY(hge_dev_alloc(ctx, invs, (size_t)rows));
  k_invert<<<grid_for(ctx, rows, kBlock, kBlocksPerSm), kBlock, 0, ctx->stream>>>(rows, wsum, *invs);
  HGE_CHECK_LAUNCH(ctx);
  return HGE_OK;
}

void free_half_schedule(const hge_ctx* ctx, HgeHalfSchedule* s, bool owns_arrays = true) {
  if (owns_arrays) {
    hge_dev_free(ctx, s->deg);
    hge_dev_free(ctx, s->invs);
  }
  hge_sched_release(ctx, s);
}

}  // namespace

// ----------------------------------------------------------------------------------------
// relaxation state
// ----------------------------------------------------------------------------------------

namespace {

// Blocks of the stream-fed kernel for one schedule: two waves of resident blocks (a warp owns one
// contiguous piece; the second wave evens out what the cost model of the pieces gets wrong:
// 0.399 -> 0.310 ms per sweep on config 2, profiles/r2_half_sweep.md), fewer when there are not
// enough units to go round.
int sweep_blocks(const hge_algdist* st, const HgeHalfSchedule& s, int G) {
  const hge_ctx* ctx = st->ctx;
  const int per_sm = ctx->blocks_per_sm > 0 ? ctx->blocks_per_sm : 2 * st->sweep_resident;
  const int64_t units = (int64_t)s.n_chunks + (s.n_light + G - 1) / G;
  const int64_t want = std::max<int64_t>(1, (units + kWarps - 1) / kWarps);
  return (int)std::min<int64_t>((int64_t)per_sm * ctx->num_sms, want);
}

int run_half_stream(hge_algdist* st, HgeHalfSchedule& s, bool node_half, int sweep, float* raw,
                    const hge_p2p* push, bool accumulate) {
  hge_ctx* ctx = st->ctx;
  const int G = 32 / st->lpr;
  const int mode = push ? kSweepPush : raw ? (accumulate ? kSweepRawAdd : kSweepRaw)
                                           : (node_half ? kSweepNode : kSweepEdge);
  const int with_own = (mode == kSweepNode || mode == kSweepEdge) ? 1 : 0;
  // the stream holds absolute rows of the allocation that starts at the edge rows (ye)
  const int64_t yn_row = (st->yn - st->ye) / st->ld;
  HGE_REQUIRE(st->yn >= st->ye && (st->yn - st->ye) % st->ld == 0 && yn_row + st->inc->N < 0xffffffffll,
              "relaxation tables are not rows of one allocation");
  const uint32_t gather0 = node_half ? 0u : (uint32_t)yn_row;
  const uint32_t own0 = node_half ? (uint32_t)yn_row : 0u;
  const int blocks = sweep_blocks(st, s, G);
  HGE_TRY(hge_sched_stream(ctx, &s, G, with_own, gather0, own0, st->zero_row, blocks * kWarps));
  HgeSweepArgs a = {};
  a.src.stream = s.stream.ids;
  a.src.items = s.stream.items;
  a.src.uoff = s.stream.uoff;
  a.src.piece = s.stream.piece;
  a.src.hrows = s.hrows;
  a.src.chunks = s.chunks;
  a.src.n_chunks = s.n_chunks;
  a.src.n_hrows = s.n_hrows;
  a.src.partials = st->partials;
  a.src.counters = st->counters;
  a.base = reinterpret_cast<const float4*>(st->ye);
  a.own = reinterpret_cast<float4*>(node_half ? st->yn : st->ye);
  a.mm_prev = sweep > 0 ? st->mm + (size_t)(sweep - 1) * 2 * st->ld : nullptr;
  a.mm_cur = st->mm + (size_t)sweep * 2 * st->ld;
  a.raw = reinterpret_cast<float4*>(raw);
  a.push_stage = push ? push->d_peer_stage : nullptr;
  a.push_rank = push ? push->rank : 0;
  a.push_map.sub_rows = push ? push->sub_rows : 1;
  a.R = st->R;
  a.ld4 = st->ld4;
  return hge_sweep_launch(ctx, a, st->lpr, mode, blocks, st->slabs);
}

int run_half(hge_algdist* st, bool node_half, int sweep, float* raw, int slice = -1,
             const hge_p2p* push = nullptr, HgeHalfSchedule* tile = nullptr,
             bool accumulate = false) {
  hge_incidence* inc = st->inc;
  HgeHalfSchedule& s = tile ? *tile
                       : node_half ? inc->node_half
                                   : (slice >= 0 ? inc->edge_slices[(size_t)slice] : inc->edge_half);
  return run_half_stream(st, s, node_half, sweep, raw, push, accumulate);
}

}  // namespace

extern "C" {

static int incidence_finish(hge_incidence* inc);

static int incidence_create_impl(hge_ctx* ctx, int32_t num_nodes, int32_t num_edges,
                                 const int64_t* n2e_ptr, const int32_t* n2e_idx,
                                 const int64_t* e2n_ptr, const int32_t* e2n_idx, bool sharded,
                                 int num_slices, int mem, hge_incidence** out, bool defer_finish = false) {
  const char* fn = sharded ? "hge_incidence_create_sharded" : "hge_incidence_create";
  HGE_REQUIRE(ctx && out, "%s: NULL ctx / out", fn);
  *out = nullptr;
  HGE_REQUIRE(num_nodes > 0 && num_edges > 0, "%s: empty hypergraph (%d nodes, %d edges)", fn,
              num_nodes, num_edges);
  HGE_REQUIRE(n2e_ptr && n2e_idx, "%s: NULL CSR array", fn);
  HGE_REQUIRE((e2n_ptr == nullptr) == (e2n_idx == nullptr), "%s: pass both edge -> node arrays or neither", fn);
  const bool build_e2n = e2n_ptr == nullptr;     // transpose on the device
  HGE_REQUIRE(mem == HGE_MEM_HOST || mem == HGE_MEM_DEVICE, "%s: bad mem %d", fn, mem);
  HGE_REQUIRE(num_slices >= 1 && num_slices <= 64 && num_slices <= num_edges,
              "%s: num_slices %d not in [1, min(64, edges)]", fn, num_slices);
  HGE_CUDA(cudaSetDevice(ctx->device));

  hge_incidence* inc = new (std::nothrow) hge_incidence();
  if (!inc) return HGE_ERR_NOMEM;
  inc->ctx = ctx;
  inc->N = num_nodes;
  inc->E = num_edges;
  inc->sharded = sharded;
  int rc = HGE_OK;
  auto fail = [&](int code) {
    hge_incidence_destroy(inc);
    return code;
  };
  auto cuda_fail = [&](cudaError_t e, const char* what) {
    hge_set_error("%s: %s failed: %s", fn, what, cudaGetErrorString(e));
    return fail(HGE_ERR_CUDA);
  };

  // Order of the queued work: row pointers first (small), then everything that needs only
  // them -- degrees, schedule keys, sort, statistics read-back -- then the column ids (large).
  // The one host wait of the set-up (hge_sched_finish) then overlaps the big upload.
  cudaError_t e = cudaSuccess;
  int64_t nnz_a = 0, nnz_b = 0;
  if (mem == HGE_MEM_HOST) {
    nnz_a = n2e_ptr[num_nodes];
    nnz_b = build_e2n ? nnz_a : e2n_ptr[num_edges];
    if (n2e_ptr[0] != 0 || (!build_e2n && e2n_ptr[0] != 0) || nnz_a < 0 || nnz_b < 0) {
      hge_set_error("%s: row pointers must start at 0 and must not decrease", fn);
      return fail(HGE_ERR_INVALID);
    }
    inc->owns_csr = true;
    if ((rc = hge_dev_alloc(ctx, &inc->n2e_ptr, (size_t)num_nodes + 1)) != HGE_OK) return fail(rc);
    if ((rc = hge_dev_alloc(ctx, &inc->e2n_ptr, (size_t)num_edges + 1)) != HGE_OK) return fail(rc);
    if ((rc = hge_dev_alloc(ctx, &inc->n2e_idx, (size_t)nnz_a)) != HGE_OK) return fail(rc);
    if ((rc = hge_dev_alloc(ctx, &inc->e2n_idx, (size_t)nnz_b)) != HGE_OK) return fail(rc);
    e = cudaMemcpyAsync(inc->n2e_ptr, n2e_ptr, ((size_t)num_nodes + 1) * 8, cudaMemcpyHostToDevice,
                        ctx->stream);
    if (e == cudaSuccess && !build_e2n)
      e = cudaMemcpyAsync(inc->e2n_ptr, e2n_ptr, ((size_t)num_edges + 1) * 8, cudaMemcpyHostToDevice,
                          ctx->stream);
    if (e != cudaSuccess) return cuda_fail(e, "row-pointer upload");
    if (build_e2n) {
      // the transpose needs the column ids first
      if (nnz_a)
        e = cudaMemcpyAsync(inc->n2e_idx, n2e_idx, (size_t)nnz_a * 4, cudaMemcpyHostToDevice, ctx->stream);
      if (e != cudaSuccess) return cuda_fail(e, "column-id upload");
    }
  } else {
    inc->owns_csr = false;
    inc->n2e_ptr = const_cast<int64_t*>(n2e_ptr);
    inc->n2e_idx = const_cast<int32_t*>(n2e_idx);
    if (build_e2n) {
      // only the last row pointer is needed on the host: the number of incidences
      if ((rc = read_back(ctx, n2e_ptr + num_nodes, &nnz_a, 1)) != HGE_OK) return fail(rc);
      inc->owns_e2n = true;
      if ((rc = hge_dev_alloc(ctx, &inc->e2n_ptr, (size_t)num_edges + 1)) != HGE_OK) return fail(rc);
      if ((rc = hge_dev_alloc(ctx, &inc->e2n_idx, (size_t)nnz_a)) != HGE_OK) return fail(rc);
    } else {
      inc->e2n_ptr = const_cast<int64_t*>(e2n_ptr);
      inc->e2n_idx = const_cast<int32_t*>(e2n_idx);
    }
  }
  if (build_e2n) {
    rc = transpose_csr(ctx, num_nodes, num_edges, nnz_a, inc->n2e_ptr, inc->n2e_idx, inc->e2n_ptr, inc->e2n_idx);
    if (rc != HGE_OK) return fail(rc);
  }

  // degrees: a neighbour's weight is 1 / (degree of that neighbour's own row),
  // algebraic_distance.py:47.  In a shard the edge degrees and the edges' weight sums are local
  // partial values until the caller has all-reduced them (hge_incidence_finish_sharded).
  HgeHalfSchedule& nh = inc->node_half;
  HgeHalfSchedule& eh = inc->edge_half;
  nh.ptr = inc->n2e_ptr;
  nh.idx = inc->n2e_idx;
  eh.ptr = inc->e2n_ptr;
  eh.idx = inc->e2n_idx;
  inc->num_slices = num_slices;
  if ((rc = hge_dev_alloc(ctx, &nh.deg, (size_t)num_nodes)) != HGE_OK) return fail(rc);
  if ((rc = hge_dev_alloc(ctx, &eh.deg, (size_t)num_edges)) != HGE_OK) return fail(rc);
  k_row_degree<<<grid_for(ctx, num_nodes, kBlock, kBlocksPerSm), kBlock, 0, ctx->stream>>>(
      num_nodes, inc->n2e_ptr, nh.deg);
  ctx->launches++;
  k_row_degree<<<grid_for(ctx, num_edges, kBlock, kBlocksPerSm), kBlock, 0, ctx->stream>>>(
      num_edges, inc->e2n_ptr, eh.deg);
  ctx->launches++;
  if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail(e, "degree kernel launch");

  // gather schedules, phase 1 (sort by degree + statistics, asynchronous)
  if ((rc = hge_sched_begin(ctx, 0, num_nodes, inc->n2e_ptr, num_edges, &nh)) != HGE_OK) return fail(rc);
  if ((rc = hge_sched_begin(ctx, 0, num_edges, inc->e2n_ptr, num_nodes, &eh)) != HGE_OK) return fail(rc);
  if (sharded) {
    // the sharded edge half runs slice by slice so that the all-reduce of one slice's partial
    // sums overlaps the gather of the next
    inc->edge_slices.resize((size_t)num_slices);
    inc->slice_bounds.resize((size_t)num_slices + 1);
    for (int k = 0; k <= num_slices; ++k)
      inc->slice_bounds[(size_t)k] = (int32_t)((int64_t)num_edges * k / num_slices);
    for (int k = 0; k < num_slices; ++k) {
      rc = hge_sched_begin(ctx, inc->slice_bounds[(size_t)k], inc->slice_bounds[(size_t)k + 1],
                           inc->e2n_ptr, num_nodes, &inc->edge_slices[(size_t)k]);
      if (rc != HGE_OK) return fail(rc);
    }
  }

  if (mem == HGE_MEM_HOST && !build_e2n) {
    if (nnz_a)
      e = cudaMemcpyAsync(inc->n2e_idx, n2e_idx, (size_t)nnz_a * 4, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess && nnz_b)
      e = cudaMemcpyAsync(inc->e2n_idx, e2n_idx, (size_t)nnz_b * 4, cudaMemcpyHostToDevice, ctx->stream);
    if (e != cudaSuccess) return cuda_fail(e, "column-id upload");
  }
  // edge weight sums: sum over (local) members n of 1 / deg(n); node degrees are complete
  DevBuf<double> edge_wsum(ctx);
  rc = compute_wsum(ctx, num_edges, inc->e2n_ptr, inc->e2n_idx, nh.deg, edge_wsum);
  if (rc != HGE_OK) return fail(rc);
  inc->edge_wsum = edge_wsum.release();
  if (!sharded && !defer_finish) {
    rc = incidence_finish(inc);
    if (rc != HGE_OK) return fail(rc);
  }
  *out = inc;
  return HGE_OK;
}

// Second phase: edge degrees / weight sums are final (global).  Builds the inverse weight sums
// and the work items of the gather schedules.
static int incidence_finish(hge_incidence* inc) {
  hge_ctx* ctx = inc->ctx;
  HgeHalfSchedule& nh = inc->node_half;
  HgeHalfSchedule& eh = inc->edge_half;
  DevBuf<double> node_wsum(ctx);
  HGE_TRY(compute_wsum(ctx, inc->N, inc->n2e_ptr, inc->n2e_idx, eh.deg, node_wsum));
  HGE_TRY(invert_wsum(ctx, inc->N, node_wsum.p, &nh.invs));
  node_wsum.reset();
  HGE_TRY(invert_wsum(ctx, inc->E, inc->edge_wsum, &eh.invs));
  HGE_TRY(hge_sched_finish(ctx, "node", &nh));
  HGE_TRY(hge_sched_finish(ctx, "edge", &eh));
  for (HgeHalfSchedule& sl : inc->edge_slices) {
    sl.idx = eh.idx;
    sl.deg = eh.deg;
    sl.invs = eh.invs;
    HGE_TRY(hge_sched_finish(ctx, "edge", &sl));
  }
  inc->finished = true;
  return HGE_OK;
}

int hge_incidence_create(hge_ctx* ctx, int32_t num_nodes, int32_t num_edges,
                         const int64_t* n2e_ptr, const int32_t* n2e_idx,
                         const int64_t* e2n_ptr, const int32_t* e2n_idx, int mem,
                         hge_incidence** out) {
  return incidence_create_impl(ctx, num_nodes, num_edges, n2e_ptr, n2e_idx, e2n_ptr, e2n_idx,
                               false, 1, mem, out);
}

int hge_incidence_create_sharded(hge_ctx* ctx, int32_t num_local_nodes, int32_t num_edges,
                                 const int64_t* n2e_ptr, const int32_t* n2e_idx,
                                 const int64_t* e2n_ptr, const int32_t* e2n_idx, int num_slices,
                                 int mem, hge_incidence** out) {
  return incidence_create_impl(ctx, num_local_nodes, num_edges, n2e_ptr, n2e_idx, e2n_ptr, e2n_idx,
                               true, num_slices, mem, out);
}

int hge_incidence_edge_sums(hge_incidence* inc, int32_t** edge_deg, double** edge_wsum) {
  HGE_REQUIRE(inc && edge_deg && edge_wsum, "hge_incidence_edge_sums: NULL argument");
  HGE_REQUIRE(inc->sharded && !inc->finished,
              "hge_incidence_edge_sums: only valid between create_sharded and finish_sharded");
  *edge_deg = inc->edge_half.deg;
  *edge_wsum = inc->edge_wsum;
  return HGE_OK;
}

int hge_incidence_finish_sharded(hge_incidence* inc) {
  HGE_REQUIRE(inc && inc->sharded && !inc->finished,
              "hge_incidence_finish_sharded: not a pending sharded incidence");
  HGE_CUDA(cudaSetDevice(inc->ctx->device));
  return incidence_finish(inc);
}

int hge_incidence_slice_range(const hge_incidence* inc, int slice, int32_t* row0, int32_t* row1) {
  HGE_REQUIRE(inc && row0 && row1, "hge_incidence_slice_range: NULL argument");
  HGE_REQUIRE(inc->sharded && slice >= 0 && slice < (int)inc->edge_slices.size(),
              "hge_incidence_slice_range: slice %d out of range", slice);
  *row0 = inc->slice_bounds[(size_t)slice];
  *row1 = inc->slice_bounds[(size_t)slice + 1];
  return HGE_OK;
}

int hge_incidence_destroy(hge_incidence* inc) {
  if (!inc) return HGE_OK;
  cudaSetDevice(inc->ctx->device);
  hge_algdist_destroy(inc->cached);
  inc->cached = nullptr;
  const hge_ctx* ctx = inc->ctx;
  free_half_schedule(ctx, &inc->node_half);
  free_half_schedule(ctx, &inc->edge_half);
  for (HgeHalfSchedule& sl : inc->edge_slices) free_half_schedule(ctx, &sl, false);
  inc->edge_slices.clear();
  for (HgeHalfSchedule& tl : inc->edge_tiles) free_half_schedule(ctx, &tl, false);
  inc->edge_tiles.clear();
  hge_dev_free(ctx, inc->tile_pos);
  hge_dev_free(ctx, inc->edge_wsum);
  if (inc->owns_csr) {
    hge_dev_free(ctx, inc->n2e_ptr);
    hge_dev_free(ctx, inc->n2e_idx);
  }
  if (inc->owns_csr || inc->owns_e2n) {
    hge_dev_free(ctx, inc->e2n_ptr);
    hge_dev_free(ctx, inc->e2n_idx);
  }
  delete inc;
  return HGE_OK;
}

int64_t hge_incidence_nnz(const hge_incidence* inc) { return inc ? inc->node_half.nnz : 0; }

// Builds (once per tile height) the node-range tiles of the edge half: per tile a schedule over
// all edges whose rows are the sub-ranges of the member lists that fall into the tile.
static int ensure_edge_tiles(hge_ctx* ctx, hge_incidence* inc, int32_t tile_rows) {
  if (inc->tile_rows == tile_rows && !inc->edge_tiles.empty()) return HGE_OK;
  for (HgeHalfSchedule& tl : inc->edge_tiles) free_half_schedule(ctx, &tl, false);
  inc->edge_tiles.clear();
  hge_dev_free(ctx, inc->tile_pos);
  inc->tile_rows = tile_rows;
  const int tiles = (int)(((int64_t)inc->N + tile_rows - 1) / tile_rows);
  if (tiles <= 1) return HGE_OK;
  const HgeHalfSchedule& eh = inc->edge_half;
  HGE_TRY(hge_dev_alloc(ctx, &inc->tile_pos, (size_t)(tiles + 1) * inc->E));
  k_tile_offsets<<<grid_for(ctx, (int64_t)inc->E * (tiles + 1), kBlock, kBlocksPerSm), kBlock, 0, ctx->stream>>>(
      inc->E, inc->e2n_ptr, inc->e2n_idx, tiles, tile_rows, inc->tile_pos);
  HGE_CHECK_LAUNCH(ctx);
  // Tiling adds work per non-empty (edge, tile) pair (a work item, a read-modify-write of the
  // partial row): it pays when edges are large (config 5: ~180 incidences per pair) and costs
  // more than it saves when they are small (config 2 forced into tiles: ~7 per pair, edge half
  // 0.24 -> 0.45 ms).  Below kMinPerPair incidences per pair the half-sweep stays untiled.
  {
    constexpr double kMinPerPair = 16.0;
    DevBuf<unsigned long long> d_pairs(ctx);
    HGE_TRY(d_pairs.alloc(1));
    HGE_CUDA(cudaMemsetAsync(d_pairs.p, 0, sizeof(unsigned long long), ctx->stream));
    k_count_tile_pairs<<<grid_for(ctx, (int64_t)inc->E * tiles, kBlock, kBlocksPerSm), kBlock, 0, ctx->stream>>>(
        (int64_t)inc->E * tiles, inc->E, inc->tile_pos, d_pairs.p);
    HGE_CHECK_LAUNCH(ctx);
    unsigned long long* h_pairs = static_cast<unsigned long long*>(hge_ctx_pinned_slot(ctx));
    if (!h_pairs) return HGE_ERR_NOMEM;
    HGE_CUDA(cudaMemcpyAsync(h_pairs, d_pairs.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost,
                             ctx->stream));
    HGE_CUDA(cudaStreamSynchronize(ctx->stream));
    d_pairs.reset();
    const double per_pair = *h_pairs ? (double)eh.nnz / (double)*h_pairs : 0.0;
    if (per_pair < kMinPerPair && !ctx->tile_force) {
      hge_dev_free(ctx, inc->tile_pos);
      return HGE_OK;
    }
  }
  inc->edge_tiles.resize((size_t)tiles);
  for (int t = 0; t < tiles; ++t) {
    inc->edge_tiles[(size_t)t].skip_empty = true;
    HGE_TRY(hge_sched_begin_ranges(ctx, 0, inc->E, inc->tile_pos + (size_t)t * inc->E,
                                   inc->tile_pos + (size_t)(t + 1) * inc->E, tile_rows,
                                   &inc->edge_tiles[(size_t)t]));
  }
  for (int t = 0; t < tiles; ++t) {
    HgeHalfSchedule& tl = inc->edge_tiles[(size_t)t];
    tl.idx = eh.idx;
    tl.deg = eh.deg;
    tl.invs = eh.invs;
    HGE_TRY(hge_sched_finish(ctx, "edge tile", &tl));
  }
  return HGE_OK;
}

int hge_algdist_create(hge_ctx* ctx, hge_incidence* inc, int R, int max_iterations,
                       hge_algdist** out) {
  HGE_REQUIRE(ctx && inc && out, "hge_algdist_create: NULL argument");
  *out = nullptr;
  HGE_REQUIRE(R >= 1 && R <= 1024, "hge_algdist_create: dimension %d not in [1, 1024]", R);
  HGE_REQUIRE(max_iterations >= 0, "hge_algdist_create: negative iteration count");
  HGE_REQUIRE(inc->finished, "hge_algdist_create: hge_incidence_finish_sharded has not been called");
  if (inc->node_half.first_empty >= 0 || (!inc->sharded && inc->edge_half.first_empty >= 0)) {
    const bool node = inc->node_half.first_empty >= 0;
    hge_set_error("%s %d has no incidence: the relaxation divides 0/0 there "
                  "(reference: ZeroDivisionError at algebraic_distance.py:49)",
                  node ? "node" : "edge",
                  node ? inc->node_half.first_empty : inc->edge_half.first_empty);
    return HGE_ERR_EMPTY_ROW;
  }
  HGE_CUDA(cudaSetDevice(ctx->device));
  hge_algdist* st = new (std::nothrow) hge_algdist();
  if (!st) return HGE_ERR_NOMEM;
  st->ctx = ctx;
  st->inc = inc;
  st->R = R;
  st->ld = (R + 3) & ~3;
  st->ld4 = st->ld / 4;
  int lpr = 1;
  while (lpr < st->ld4 && lpr < 32) lpr <<= 1;
  st->lpr = lpr;
  st->slabs = (st->ld4 + 31) / 32;
  st->max_iters = max_iterations;
  int rc = HGE_OK;
  auto fail = [&](int code) {
    hge_algdist_destroy(st);
    return code;
  };
  // one block [edge rows | a row of zeros | node rows]: the packed gather stream addresses the
  // gathered rows, a row's own old value and its padding as rows of the same allocation
  if ((rc = hge_dev_alloc(ctx, &st->ybuf, ((size_t)inc->E + 1 + (size_t)inc->N) * st->ld)) != HGE_OK)
    return fail(rc);
  st->ye = st->ybuf;
  st->yn = st->ybuf + ((size_t)inc->E + 1) * st->ld;
  st->zero_row = (uint32_t)inc->E;
  if (cudaMemsetAsync(st->ybuf + (size_t)inc->E * st->ld, 0, (size_t)st->ld * sizeof(float), ctx->stream) !=
      cudaSuccess) {
    hge_set_error("hge_algdist_create: memset failed");
    return fail(HGE_ERR_CUDA);
  }
  if ((rc = hge_dev_alloc(ctx, &st->mm, (size_t)std::max(1, max_iterations) * 2 * st->ld)) != HGE_OK)
    return fail(rc);
  // node rows far beyond what random gathers reach at full rate: tile the edge half (single
  // GPU, and the peer-memory sweep of a shard; the NCCL path of a shard stays untiled)
  if (ctx->tile_mb > 0) {
    const int64_t tile_rows64 = ((int64_t)ctx->tile_mb << 20) / ((int64_t)st->ld * 4);
    const int32_t tile_rows = (int32_t)std::max<int64_t>(1, std::min<int64_t>(tile_rows64, INT32_MAX));
    const int64_t row_bytes = (int64_t)inc->N * st->ld * 4;
    if (row_bytes > ((int64_t)ctx->tile_min_mb << 20) && (int64_t)inc->N > 2 * (int64_t)tile_rows) {
      if ((rc = ensure_edge_tiles(ctx, inc, tile_rows)) != HGE_OK) return fail(rc);
      if (!inc->edge_tiles.empty() &&
          (rc = hge_dev_alloc(ctx, &st->tile_raw, (size_t)inc->E * st->ld)) != HGE_OK)
        return fail(rc);
    }
  }
  size_t n_part = (size_t)std::max(inc->node_half.n_partials, inc->edge_half.n_partials);
  size_t n_cnt = (size_t)std::max(inc->node_half.n_hrows, inc->edge_half.n_hrows);
  if (st->tile_raw)
    for (const HgeHalfSchedule& tl : inc->edge_tiles) {
      n_part = std::max(n_part, (size_t)tl.n_partials);
      n_cnt = std::max(n_cnt, (size_t)tl.n_hrows);
    }
  for (const HgeHalfSchedule& sl : inc->edge_slices) {
    n_part = std::max(n_part, (size_t)sl.n_partials);
    n_cnt = std::max(n_cnt, (size_t)sl.n_hrows);
  }
  n_cnt *= (size_t)st->slabs;
  if ((rc = hge_dev_alloc(ctx, &st->partials, n_part * st->ld4)) != HGE_OK) return fail(rc);
  if ((rc = hge_dev_alloc(ctx, &st->counters, n_cnt)) != HGE_OK) return fail(rc);
  if (cudaMemsetAsync(st->counters, 0, std::max<size_t>(1, n_cnt) * sizeof(int32_t), ctx->stream) !=
      cudaSuccess) {
    hge_set_error("hge_algdist_create: memset failed");
    return fail(HGE_ERR_CUDA);
  }
  if ((rc = hge_sweep_resident_blocks(st->lpr, &st->sweep_resident)) != HGE_OK) return fail(rc);
  *out = st;
  return HGE_OK;
}

int hge_algdist_destroy(hge_algdist* st) {
  if (!st) return HGE_OK;
  cudaSetDevice(st->ctx->device);
  const hge_ctx* ctx = st->ctx;
  hge_dev_free(ctx, st->ybuf);   // (a peer-memory arena owns the rows otherwise)
  hge_dev_free(ctx, st->mm);
  hge_dev_free(ctx, st->partials);
  hge_dev_free(ctx, st->tile_raw);
  hge_dev_free(ctx, st->counters);
  delete st;
  return HGE_OK;
}

int hge_algdist_ld(const hge_algdist* st) { return st ? st->ld : 0; }

// Starts the upload of host vectors into the context's staging block on the copy stream (it runs
// next to whatever is queued on the main stream) and records copy_done.
static int stage_vectors(hge_ctx* ctx, int64_t N, int64_t E, int R, const float* xn, const float* xe) {
  float* stage = nullptr;
  HGE_TRY(hge_ctx_stage(ctx, (size_t)(N + E) * R, &stage));
  HGE_CUDA(cudaStreamWaitEvent(ctx->copy_stream, ctx->stage_idle, 0));
  HGE_CUDA(cudaMemcpyAsync(stage, xn, (size_t)N * R * 4, cudaMemcpyHostToDevice, ctx->copy_stream));
  HGE_CUDA(cudaMemcpyAsync(stage + (size_t)N * R, xe, (size_t)E * R * 4, cudaMemcpyHostToDevice,
                           ctx->copy_stream));
  HGE_CUDA(cudaEventRecord(ctx->copy_done, ctx->copy_stream));
  return HGE_OK;
}

// prestaged: stage_vectors has been called for these vectors already
static int algdist_load_impl(hge_algdist* st, const float* xn, const float* xe, int mem, bool prestaged) {
  HGE_REQUIRE(st && xn && xe, "hge_algdist_load: NULL argument");
  hge_ctx* ctx = st->ctx;
  hge_incidence* inc = st->inc;
  HGE_CUDA(cudaSetDevice(ctx->device));
  const float* dn = xn;
  const float* de = xe;
  if (mem == HGE_MEM_HOST) {
    // upload on the copy stream: it starts now, next to whatever set-up work is still queued
    // on the main stream, which only waits for it right before k_load_rows
    if (!prestaged) HGE_TRY(stage_vectors(ctx, inc->N, inc->E, st->R, xn, xe));
    HGE_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->copy_done, 0));
    dn = ctx->stage;
    de = ctx->stage + (size_t)inc->N * st->R;
  }
  k_fill_minmax<<<grid_for(ctx, (int64_t)std::max(1, st->max_iters) * 2 * st->ld, kBlock, kBlocksPerSm), kBlock, 0,
                  ctx->stream>>>(st->mm, std::max(1, st->max_iters), st->ld);
  HGE_CHECK_LAUNCH(ctx);
  k_load_rows<<<grid_for(ctx, (int64_t)inc->N * st->ld, kBlock, kBlocksPerSm), kBlock, 0, ctx->stream>>>(
      inc->N, st->R, st->ld, dn, inc->node_half.deg, st->yn);
  HGE_CHECK_LAUNCH(ctx);
  k_load_rows<<<grid_for(ctx, (int64_t)inc->E * st->ld, kBlock, kBlocksPerSm), kBlock, 0, ctx->stream>>>(
      inc->E, st->R, st->ld, de, inc->edge_half.deg, st->ye);
  HGE_CHECK_LAUNCH(ctx);
  if (mem == HGE_MEM_HOST) HGE_CUDA(cudaEventRecord(ctx->stage_idle, ctx->stream));
  return HGE_OK;
}

int hge_algdist_load(hge_algdist* st, const float* xn, const float* xe, int mem) {
  return algdist_load_impl(st, xn, xe, mem, false);
}

int hge_algdist_node_half(hge_algdist* st, int sweep) {
  HGE_REQUIRE(st && sweep >= 0 && sweep < st->max_iters, "hge_algdist_node_half: bad sweep %d", sweep);
  HGE_CUDA(cudaSetDevice(st->ctx->device));
  return run_half(st, true, sweep, nullptr);
}

int hge_algdist_edge_half(hge_algdist* st, int sweep) {
  HGE_REQUIRE(st && sweep >= 0 && sweep < st->max_iters, "hge_algdist_edge_half: bad sweep %d", sweep);
  HGE_CUDA(cudaSetDevice(st->ctx->device));
  if (!st->tile_raw || st->inc->sharded) return run_half(st, false, sweep, nullptr);
  // tiled: every tile adds the sums of its node range to tile_raw, then one pass blends,
  // rescales and stores the edge rows (the kernel the sharded path uses after its all-reduce)
  hge_ctx* ctx = st->ctx;
  hge_incidence* inc = st->inc;
  HGE_CUDA(cudaMemsetAsync(st->tile_raw, 0, (size_t)inc->E * st->ld * sizeof(float), ctx->stream));
  for (size_t t = 0; t < inc->edge_tiles.size(); ++t)
    HGE_TRY(run_half(st, false, sweep, st->tile_raw, -1, nullptr, &inc->edge_tiles[t], true));
  HGE_REQUIRE(st->ld <= 1024, "hge_algdist_edge_half: dimension too large for the tiled edge half");
  const int32_t* mm_prev = sweep > 0 ? st->mm + (size_t)(sweep - 1) * 2 * st->ld : nullptr;
  int32_t* mm_cur = st->mm + (size_t)sweep * 2 * st->ld;
  k_edge_finalize<<<grid_for(ctx, (int64_t)inc->E * st->ld, kBlock, kBlocksPerSm), kBlock, 0, ctx->stream>>>(
      0, inc->E, st->R, st->ld, st->tile_raw, inc->edge_half.deg, inc->edge_half.invs, mm_prev, mm_cur,
      st->ye);
  HGE_CHECK_LAUNCH(ctx);
  return HGE_OK;
}

int hge_algdist_edge_partial(hge_algdist* st, int sweep, int slice, float* partial) {
  HGE_REQUIRE(st && partial && sweep >= 0 && sweep < st->max_iters,
              "hge_algdist_edge_partial: bad argument");
  HGE_REQUIRE(st->inc->sharded && slice >= 0 && slice < (int)st->inc->edge_slices.size(),
              "hge_algdist_edge_partial: slice %d out of range (sharded incidence needed)", slice);
  HGE_CUDA(cudaSetDevice(st->ctx->device));
  return run_half(st, false, sweep, partial, slice);
}

int hge_algdist_edge_finalize(hge_algdist* st, int sweep, int slice, const float* partial) {
  HGE_REQUIRE(st && partial && sweep >= 0 && sweep < st->max_iters,
              "hge_algdist_edge_finalize: bad argument");
  HGE_REQUIRE(st->inc->sharded && slice >= 0 && slice < (int)st->inc->edge_slices.size(),
              "hge_algdist_edge_finalize: slice %d out of range (sharded incidence needed)", slice);
  HGE_REQUIRE(st->ld <= 1024, "hge_algdist_edge_finalize: dimension too large");
  hge_ctx* ctx = st->ctx;
  hge_incidence* inc = st->inc;
  HGE_CUDA(cudaSetDevice(ctx->device));
  const int32_t* mm_prev = sweep > 0 ? st->mm + (size_t)(sweep - 1) * 2 * st->ld : nullptr;
  int32_t* mm_cur = st->mm + (size_t)sweep * 2 * st->ld;
  const int64_t row0 = inc->slice_bounds[(size_t)slice];
  const int64_t rows = inc->slice_bounds[(size_t)slice + 1] - row0;
  k_edge_finalize<<<grid_for(ctx, rows * st->ld, kBlock, kBlocksPerSm), kBlock, 0, ctx->stream>>>(
      row0, rows, st->R, st->ld, partial, inc->edge_half.deg, inc->edge_half.invs, mm_prev, mm_cur,
      st->ye);
  HGE_CHECK_LAUNCH(ctx);
  return HGE_OK;
}

// The sharded edge gather with the partial rows pushed to their owners.
int hge_internal_edge_push(hge_algdist* st, int sweep) {
  hge_p2p* p = st->p2p;
  if (!st->tile_raw) return run_half(st, false, sweep, nullptr, -1, p);
  // tiled: the local partial sums are accumulated tile by tile, then pushed to their owners
  hge_ctx* ctx = st->ctx;
  hge_incidence* inc = st->inc;
  HGE_CUDA(cudaMemsetAsync(st->tile_raw, 0, (size_t)inc->E * st->ld * sizeof(float), ctx->stream));
  for (size_t t = 0; t < inc->edge_tiles.size(); ++t)
    HGE_TRY(run_half(st, false, sweep, st->tile_raw, -1, nullptr, &inc->edge_tiles[t], true));
  HgeOwnerMap map;
  map.sub_rows = p->sub_rows;
  k_push_rows<<<grid_for(ctx, (int64_t)inc->E * st->ld4, kBlock, kBlocksPerSm), kBlock, 0, ctx->stream>>>(
      0, inc->E, st->ld4, reinterpret_cast<const float4*>(st->tile_raw), p->d_peer_stage, p->rank, map);
  HGE_CHECK_LAUNCH(ctx);
  return HGE_OK;
}

int hge_algdist_minmax_ptr(hge_algdist* st, int sweep, int32_t** out) {
  HGE_REQUIRE(st && out && sweep >= 0 && sweep < std::max(1, st->max_iters),
              "hge_algdist_minmax_ptr: bad argument");
  *out = st->mm + (size_t)sweep * 2 * st->ld;
  return HGE_OK;
}

int hge_algdist_store(hge_algdist* st, int sweeps_done, float* xn, float* xe, int mem) {
  HGE_REQUIRE(st && xn && xe && sweeps_done >= 0 && sweeps_done <= st->max_iters,
              "hge_algdist_store: bad argument");
  hge_ctx* ctx = st->ctx;
  hge_incidence* inc = st->inc;
  HGE_CUDA(cudaSetDevice(ctx->device));
  const int32_t* mm = sweeps_done > 0 ? st->mm + (size_t)(sweeps_done - 1) * 2 * st->ld : nullptr;
  float* dn = xn;
  float* de = xe;
  if (mem == HGE_MEM_HOST) {
    float* stage = nullptr;
    HGE_TRY(hge_ctx_stage(ctx, (size_t)(inc->N + (int64_t)inc->E) * st->R, &stage));
    dn = stage;
    de = stage + (size_t)inc->N * st->R;
  }
  k_store_rows<<<grid_for(ctx, (int64_t)inc->N * st->R, kBlock, kBlocksPerSm), kBlock, 0, ctx->stream>>>(
      inc->N, st->R, st->ld, st->yn, inc->node_half.deg, mm, dn);
  HGE_CHECK_LAUNCH(ctx);
  k_store_rows<<<grid_for(ctx, (int64_t)inc->E * st->R, kBlock, kBlocksPerSm), kBlock, 0, ctx->stream>>>(
      inc->E, st->R, st->ld, st->ye, inc->edge_half.deg, mm, de);
  HGE_CHECK_LAUNCH(ctx);
  if (mem == HGE_MEM_HOST) {
    HGE_CUDA(cudaMemcpyAsync(xn, dn, (size_t)inc->N * st->R * 4, cudaMemcpyDeviceToHost, ctx->stream));
    HGE_CUDA(cudaMemcpyAsync(xe, de, (size_t)inc->E * st->R * 4, cudaMemcpyDeviceToHost, ctx->stream));
    HGE_CUDA(cudaEventRecord(ctx->stage_idle, ctx->stream));
    HGE_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  return HGE_OK;
}

int hge_column_rescale(hge_ctx* ctx, float* xn, int64_t num_nodes, float* xe, int64_t num_edges,
                       int R, int mem) {
  HGE_REQUIRE(ctx && xn && xe && num_nodes >= 0 && num_edges >= 0 && R >= 1,
              "hge_column_rescale: bad argument");
  HGE_REQUIRE(mem == HGE_MEM_HOST || mem == HGE_MEM_DEVICE, "hge_column_rescale: bad mem %d", mem);
  HGE_CUDA(cudaSetDevice(ctx->device));
  float* dn = xn;
  float* de = xe;
  const size_t nn = (size_t)num_nodes * R, ne = (size_t)num_edges * R;
  if (mem == HGE_MEM_HOST) {
    float* stage = nullptr;
    HGE_TRY(hge_ctx_stage(ctx, nn + ne, &stage));
    dn = stage;
    de = stage + nn;
    HGE_CUDA(cudaMemcpyAsync(dn, xn, nn * 4, cudaMemcpyHostToDevice, ctx->stream));
    HGE_CUDA(cudaMemcpyAsync(de, xe, ne * 4, cudaMemcpyHostToDevice, ctx->stream));
  }
  DevBuf<int32_t> mm(ctx);
  HGE_TRY(mm.alloc((size_t)2 * R));
  k_fill_minmax<<<grid_for(ctx, 2 * R, kBlock, kBlocksPerSm), kBlock, 0, ctx->stream>>>(mm.p, 1, R);
  HGE_CHECK_LAUNCH(ctx);
  k_dense_minmax<<<grid_for(ctx, (int64_t)nn, kBlock, kBlocksPerSm), kBlock, 0, ctx->stream>>>(num_nodes, R, dn, mm.p);
  HGE_CHECK_LAUNCH(ctx);
  k_dense_minmax<<<grid_for(ctx, (int64_t)ne, kBlock, kBlocksPerSm), kBlock, 0, ctx->stream>>>(num_edges, R, de, mm.p);
  HGE_CHECK_LAUNCH(ctx);
  k_dense_rescale<<<grid_for(ctx, (int64_t)nn, kBlock, kBlocksPerSm), kBlock, 0, ctx->stream>>>(num_nodes, R, dn, mm.p);
  HGE_CHECK_LAUNCH(ctx);
  k_dense_rescale<<<grid_for(ctx, (int64_t)ne, kBlock, kBlocksPerSm), kBlock, 0, ctx->stream>>>(num_edges, R, de, mm.p);
  HGE_CHECK_LAUNCH(ctx);
  mm.reset();
  if (mem == HGE_MEM_HOST) {
    HGE_CUDA(cudaMemcpyAsync(xn, dn, nn * 4, cudaMemcpyDeviceToHost, ctx->stream));
    HGE_CUDA(cudaMemcpyAsync(xe, de, ne * 4, cudaMemcpyDeviceToHost, ctx->stream));
    HGE_CUDA(cudaEventRecord(ctx->stage_idle, ctx->stream));
    HGE_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  return HGE_OK;
}

static int algdist_run_impl(hge_ctx* ctx, hge_incidence* inc, float* xn, float* xe, int R, int iterations,
                            int mem, float* lohi, bool prestaged) {
  // the workspace (Y rows, min/max slots, partial sums) is kept with the incidence and re-used
  hge_algdist* st = inc->cached;
  if (!st || st->R != R || st->max_iters < iterations || st->ctx != ctx) {
    hge_algdist_destroy(inc->cached);
    inc->cached = nullptr;
    HGE_TRY(hge_algdist_create(ctx, inc, R, iterations, &st));
    inc->cached = st;
  }
  int rc = algdist_load_impl(st, xn, xe, mem, prestaged);
  for (int t = 0; rc == HGE_OK && t < iterations; ++t) {
    rc = hge_algdist_node_half(st, t);
    if (rc == HGE_OK) rc = hge_algdist_edge_half(st, t);
  }
  if (rc == HGE_OK) rc = hge_algdist_store(st, iterations, xn, xe, mem);
  if (rc == HGE_OK && lohi) {
    std::vector<int32_t> h((size_t)iterations * 2 * st->ld);
    cudaError_t e = cudaMemcpyAsync(h.data(), st->mm, h.size() * 4, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
      hge_set_error("hge_algdist_run: reading min/max failed: %s", cudaGetErrorString(e));
      rc = HGE_ERR_CUDA;
    } else {
      for (int t = 0; t < iterations; ++t)
        for (int k = 0; k < 2; ++k)
          for (int c = 0; c < R; ++c)
            lohi[((size_t)t * 2 + k) * R + c] = hge_dec(h[((size_t)t * 2 + k) * st->ld + c]);
    }
  }
  return rc;
}

int hge_algdist_run(hge_ctx* ctx, hge_incidence* inc, float* xn, float* xe, int R, int iterations,
                    int mem, float* lohi) {
  HGE_REQUIRE(ctx && inc && xn && xe, "hge_algdist_run: NULL argument");
  HGE_REQUIRE(iterations >= 0, "hge_algdist_run: negative iteration count");
  if (iterations == 0) return HGE_OK;  // the initial vectors are the result
  return algdist_run_impl(ctx, inc, xn, xe, R, iterations, mem, lohi, false);
}

// Incidence set-up + relaxation in one call.  With host buffers the upload of the vectors is
// queued (copy stream) right behind the upload of the column ids, BEFORE the set-up's host waits:
// the transpose, the degree sorts and the schedule build then run under the 192 MB of vector
// upload instead of in front of it (hge_incidence_create + hge_algdist_run leave PCIe idle there,
// because the second call is only made when the first has returned).
int hge_algdist_run_csr(hge_ctx* ctx, int32_t num_nodes, int32_t num_edges, const int64_t* n2e_ptr,
                        const int32_t* n2e_idx, const int64_t* e2n_ptr, const int32_t* e2n_idx, float* xn,
                        float* xe, int R, int iterations, int mem, float* lohi) {
  HGE_REQUIRE(ctx && xn && xe, "hge_algdist_run_csr: NULL argument");
  HGE_REQUIRE(iterations >= 0, "hge_algdist_run_csr: negative iteration count");
  HGE_REQUIRE(R >= 1 && R <= 1024, "hge_algdist_run_csr: dimension %d not in [1, 1024]", R);
  hge_incidence* inc = nullptr;
  const bool overlap = mem == HGE_MEM_HOST && iterations > 0;
  HGE_TRY(incidence_create_impl(ctx, num_nodes, num_edges, n2e_ptr, n2e_idx, e2n_ptr, e2n_idx, false, 1, mem,
                                &inc, overlap));
  int rc = HGE_OK;
  if (overlap) {
    rc = stage_vectors(ctx, num_nodes, num_edges, R, xn, xe);
    if (rc == HGE_OK) rc = incidence_finish(inc);
  }
  if (rc == HGE_OK && iterations > 0) rc = algdist_run_impl(ctx, inc, xn, xe, R, iterations, mem, lohi, overlap);
  if (rc != HGE_OK && overlap) {
    // nothing may still be reading the caller's buffers when an error is returned
    cudaStreamSynchronize(ctx->copy_stream);
    cudaStreamSynchronize(ctx->stream);
  }
  hge_incidence_destroy(inc);
  return rc;
}

}  // extern "C"
