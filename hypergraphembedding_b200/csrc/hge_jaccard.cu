// Sparse weighted Jaccard similarities of WeightedJaccardSamples (hg2v_sample.py:250-395) on
// sm_100a, in the reference's own summation order.
//
//   J(x, y) = sum_c min(x_c, y_c) / sum_c max(x_c, y_c)   over the union of the non-zeros,
//   0 when the denominator is 0 (SparseWeightedJaccard, :250-275).
//
// The reference walks the union of the two rows' columns in ascending order and adds the smaller
// value to the numerator and the larger to the denominator ONE BY ONE, in the dtype of the
// features (fp32 for every weighting scheme of hg2v_weighting.py).  On rows with thousands of
// non-zeros that sum is only good to a few 1e-6, so any other order (a warp reduction, the
// identity sum max = sum x + sum y - sum min) misses the 1e-5 bar on a fraction of the records
// even though it is closer to the exact value.  Here a pair is one thread that merges the two
// sorted rows and carries the two fp32 sums in that order: the result is the reference's, bit
// for bit; the parallelism is across the (hundreds of thousands of) sampled pairs.
//
//   same type   (node, node) / (edge, edge): x and y are rows of one feature matrix
//               (SameTypeJaccardSample, :323-340);
//   diff type   (node, edge): x is a feature row, y the CENTROID of a group of feature rows,
//               y = (sum_{t in group} F[t]) / |group|  (CentroidFromRows, :284-299,
//               DiffTypeJaccardSample, :343-392).  The reference materialises the centroid rows
//               with scipy (column sums of F[rows]: the members are added in ascending order,
//               fp32, then one division); so does this file, for the groups the pairs name.
//               centroid_factor, which both centroid entry points call, sorts the pairs by
//               group, then cuts the named groups into batches whose expansion fits a memory
//               budget.  Per batch it expands (group, column, value) triples in member order,
//               stable radix sorts them by (group, column) and sums each run in order -- the
//               classic expand / sort / compress product -- then merges the batch's pairs and
//               frees its rows, so the peak is the budget plus O(pairs).
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <vector>

#include "hge_common.cuh"
#include "hge_expand.cuh"
#include "hge_incidence.cuh"
#include "hge_pairs.cuh"

namespace {

constexpr int kBlock = 256;
constexpr unsigned kFull = 0xffffffffu;

// one step of SparseWeightedJaccard's loop (hg2v_sample.py:264-271)
__device__ __forceinline__ void jaccard_step(float x, float y, float& num, float& den) {
  if (x < y) {
    num = __fadd_rn(num, x);
    den = __fadd_rn(den, y);
  } else {
    num = __fadd_rn(num, y);
    den = __fadd_rn(den, x);
  }
}

// J(A[ra], B[rb]): the union of the two sorted rows walked in ascending column order
__device__ __forceinline__ float jaccard_pair(const int64_t* __restrict__ aptr, const int32_t* __restrict__ aidx,
                                              const float* __restrict__ aval, int64_t ra,
                                              const int64_t* __restrict__ bptr, const int32_t* __restrict__ bidx,
                                              const float* __restrict__ bval, int64_t rb) {
  int64_t i = aptr[ra], j = bptr[rb];
  const int64_t ie = aptr[ra + 1], je = bptr[rb + 1];
  float num = 0.f, den = 0.f;
  int32_t ci = i < ie ? aidx[i] : INT32_MAX, cj = j < je ? bidx[j] : INT32_MAX;
  while (i < ie || j < je) {
    float x = 0.f, y = 0.f;
    const bool take_a = ci <= cj, take_b = cj <= ci;
    if (take_a) {
      x = aval[i];
      ++i;
    }
    if (take_b) {
      y = bval[j];
      ++j;
    }
    if (take_a) ci = i < ie ? aidx[i] : INT32_MAX;
    if (take_b) cj = j < je ? bidx[j] : INT32_MAX;
    jaccard_step(x, y, num, den);
  }
  return den == 0.f ? 0.f : __fdiv_rn(num, den);
}

// out[p] = J(F[pi[p]], F[pj[p]]), one thread per pair
__global__ void __launch_bounds__(kBlock) k_jaccard_merge(
    int64_t num_pairs, const int64_t* __restrict__ ptr, const int32_t* __restrict__ idx,
    const float* __restrict__ val, const int32_t* __restrict__ pi, const int32_t* __restrict__ pj,
    float* __restrict__ out) {
  for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < num_pairs;
       p += (int64_t)gridDim.x * blockDim.x)
    out[p] = jaccard_pair(ptr, idx, val, pi[p], ptr, idx, val, pj[p]);
}

// ---- centroid rows of the named groups, batch by batch ----------------------------------------

// head of a run: the members' values added in member order, then one division by the group size
// (targets2features[rows].sum(axis=0) / len(rows), hg2v_sample.py:293).  Local group l is group
// gid[l] of the group CSR.
__global__ void k_run_sums(int64_t n, const int32_t* __restrict__ gid, const uint64_t* __restrict__ keys,
                           const float* __restrict__ vals, const int64_t* __restrict__ pos,
                           const int64_t* __restrict__ gptr, int32_t* __restrict__ cidx, float* __restrict__ cval) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    const uint64_t key = keys[i];
    if (i > 0 && keys[i - 1] == key) continue;
    float s = 0.f;
    for (int64_t k = i; k < n && keys[k] == key; ++k) s = __fadd_rn(s, vals[k]);
    const int64_t g = gid[key >> 32];
    const int64_t o = pos[i];
    cidx[o] = (int32_t)(uint32_t)key;
    cval[o] = __fdiv_rn(s, (float)(gptr[g + 1] - gptr[g]));
  }
}

struct FeatureMatrix {
  Staged<int64_t> ptr;
  Staged<int32_t> idx;
  Staged<float> val;
  explicit FeatureMatrix(const hge_ctx* c) : ptr(c), idx(c), val(c) {}
  int init(const int64_t* p, const int32_t* i, const float* v, int64_t rows, int64_t nnz, int mem) {
    HGE_TRY(ptr.init(p, (size_t)rows + 1, mem, true, false));
    HGE_TRY(idx.init(i, (size_t)nnz, mem, true, false));
    HGE_TRY(val.init(v, (size_t)nnz, mem, true, false));
    return HGE_OK;
  }
};

// Centroid rows of one batch of L groups from its expansion: keys ((local group << 32) | column)
// and vals, n > 0 entries in member order.  Stable radix sort by key (inside a (group, column) run
// the members stay in ascending order), run heads, then one sequential fp32 sum per run.  Local
// group l is group gid[l] of the group CSR.  The rows go to the CSR (cptr [L + 1], cidx, cval);
// keys / vals are used as sort buffers.
int centroid_batch(hge_ctx* ctx, int64_t n, int64_t L, const int32_t* gid, const int64_t* gptr,
                   DevBuf<uint64_t>& keys, DevBuf<float>& vals, int64_t* cptr, DevBuf<int32_t>& cidx,
                   DevBuf<float>& cval) {
  DevBuf<uint64_t> keys2(ctx);
  DevBuf<float> vals2(ctx);
  DevBuf<int64_t> head(ctx), pos(ctx);
  DevBuf<char> temp(ctx);
  HGE_TRY(keys2.alloc((size_t)n));
  HGE_TRY(vals2.alloc((size_t)n));
  int group_bits = 1;
  while ((1ll << group_bits) < L) ++group_bits;
  cub::DoubleBuffer<uint64_t> dk(keys.p, keys2.p);
  cub::DoubleBuffer<float> dv(vals.p, vals2.p);
  size_t bytes = 0;
  HGE_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, bytes, dk, dv, n, 0, 32 + group_bits, ctx->stream));
  HGE_TRY(temp.alloc(bytes));
  HGE_CUDA(cub::DeviceRadixSort::SortPairs(temp.p, bytes, dk, dv, n, 0, 32 + group_bits, ctx->stream));
  ctx->launches++;
  const uint64_t* sk = dk.Current();
  const float* sv = dv.Current();
  HGE_TRY(head.alloc((size_t)n + 1));
  HGE_TRY(pos.alloc((size_t)n + 1));
  k_run_heads<<<grid_for(ctx, n), kBlock, 0, ctx->stream>>>(n, sk, head.p);
  HGE_CHECK_LAUNCH(ctx);
  HGE_CUDA(cudaMemsetAsync(head.p + n, 0, sizeof(int64_t), ctx->stream));
  HGE_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, bytes, head.p, pos.p, n + 1, ctx->stream));
  HGE_TRY(temp.alloc(bytes));
  HGE_CUDA(cub::DeviceScan::ExclusiveSum(temp.p, bytes, head.p, pos.p, n + 1, ctx->stream));
  ctx->launches++;
  int64_t n_runs = 0;
  HGE_TRY(read_back(ctx, pos.p + n, &n_runs, 1));
  HGE_TRY(cidx.alloc((size_t)std::max<int64_t>(1, n_runs)));
  HGE_TRY(cval.alloc((size_t)std::max<int64_t>(1, n_runs)));
  k_run_sums<<<grid_for(ctx, n), kBlock, 0, ctx->stream>>>(n, gid, sk, sv, pos.p, gptr, cidx.p, cval.p);
  HGE_CHECK_LAUNCH(ctx);
  k_run_starts<<<grid_for(ctx, L + 1), kBlock, 0, ctx->stream>>>(L, n, n_runs, sk, pos.p, cptr);
  HGE_CHECK_LAUNCH(ctx);
  return HGE_OK;
}

constexpr int64_t kDefaultWorkspaceMb = 2048;
// workspace bytes per expanded entry of a batch: keys and their sort buffer (16), values and theirs
// (8), run heads and their scan (16), the centroid entry (8)
constexpr int64_t kBytesPerEntry = 48;

// size[u] = sum over the members m of group ug[u] of nnz(F[m]); size[U] = 0 (one warp per group)
__global__ void __launch_bounds__(kBlock) k_named_sizes(int64_t U, const int32_t* __restrict__ ug,
                                                        const int64_t* __restrict__ gptr,
                                                        const int32_t* __restrict__ gidx,
                                                        const int64_t* __restrict__ fptr, int64_t* __restrict__ size) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = (int64_t)gridDim.x * (kBlock / 32);
  for (int64_t u = blockIdx.x * (int64_t)(kBlock / 32) + (threadIdx.x >> 5); u <= U; u += nw) {
    int64_t s = 0;
    if (u < U) {
      const int32_t g = ug[u];
      for (int64_t t = gptr[g] + lane; t < gptr[g + 1]; t += 32) {
        const int32_t m = gidx[t];
        s += fptr[m + 1] - fptr[m];
      }
    }
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(kFull, s, o);
    if (lane == 0) size[u] = s;
  }
}

// expansion of the named groups [u0, u1): one warp per group, its members in order, 32 at a time
// (a warp scan of their row lengths places them); key = (u - u0) << 32 | column
__global__ void __launch_bounds__(kBlock) k_expand_named(
    int64_t u0, int64_t u1, int64_t base, const int32_t* __restrict__ ug, const int64_t* __restrict__ uoff,
    const int64_t* __restrict__ gptr, const int32_t* __restrict__ gidx, const int64_t* __restrict__ fptr,
    const int32_t* __restrict__ fidx, const float* __restrict__ fval, uint64_t* __restrict__ keys,
    float* __restrict__ vals) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = (int64_t)gridDim.x * (kBlock / 32);
  for (int64_t u = u0 + blockIdx.x * (int64_t)(kBlock / 32) + (threadIdx.x >> 5); u < u1; u += nw) {
    const int32_t g = ug[u];
    const uint64_t hi = (uint64_t)(u - u0) << 32;
    const int64_t t1 = gptr[g + 1];
    int64_t dst = uoff[u] - base;
    for (int64_t tb = gptr[g]; tb < t1; tb += 32) {
      int64_t src = 0, len = 0;
      if (tb + lane < t1) {
        const int32_t m = gidx[tb + lane];
        src = fptr[m];
        len = fptr[m + 1] - src;
      }
      int64_t incl = len;
      for (int o = 1; o < 32; o <<= 1) {
        const int64_t v = __shfl_up_sync(kFull, incl, o);
        if (lane >= o) incl += v;
      }
      const int64_t excl = incl - len;
      const int members = t1 - tb < 32 ? (int)(t1 - tb) : 32;
      for (int j = 0; j < members; ++j) {
        const int64_t s = __shfl_sync(kFull, src, j), l = __shfl_sync(kFull, len, j);
        const int64_t d = dst + __shfl_sync(kFull, excl, j);
        for (int64_t k = lane; k < l; k += 32) {
          keys[d + k] = hi | (uint32_t)fidx[s + k];
          vals[d + k] = fval[s + k];
        }
      }
      dst += __shfl_sync(kFull, incl, 31);
    }
  }
}

// out[order[i]] = J(X[px[order[i]]], centroid row u - u0) for the sorted pairs [i0, i1) of the named
// groups [u0, u1) (u = rank[i] - 1); consecutive threads mostly share a centroid row
__global__ void __launch_bounds__(kBlock) k_merge_named(
    int64_t i0, int64_t i1, int64_t u0, const int32_t* __restrict__ order, const int32_t* __restrict__ rank,
    const int32_t* __restrict__ ug, const int64_t* __restrict__ gptr, const int32_t* __restrict__ px,
    const int64_t* __restrict__ xptr, const int32_t* __restrict__ xidx, const float* __restrict__ xval,
    const int64_t* __restrict__ cptr, const int32_t* __restrict__ cidx, const float* __restrict__ cval,
    float* __restrict__ out) {
  for (int64_t i = i0 + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < i1;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t p = order[i];
    const int64_t u = rank[i] - 1;
    const int32_t g = ug[u];
    out[p] = gptr[g + 1] == gptr[g] ? 0.f   // a group without members has no centroid
                                    : jaccard_pair(xptr, xidx, xval, px[p], cptr, cidx, cval, u - u0);
  }
}

// out[p] = J(X[px[p]], centroid of the members of group pg[p]) for p in [0, n), n in [1, 2^31): the
// groups are the CSR (gptr, gidx) over the rows of F, groups of them (at most 2^31).  Every pointer
// is a device pointer; the centroid rows are built in batches of at most workspace_mb MB.  A pair
// naming a row outside [0, xrows) or a group outside [0, groups) is HGE_ERR_INVALID, reported under
// the entry point's name `who`; nothing is computed then.
int centroid_factor(hge_ctx* ctx, const char* who, const int64_t* gptr, const int32_t* gidx, int64_t groups,
                    const int64_t* xptr, const int32_t* xidx, const float* xval, int64_t xrows,
                    const int64_t* fptr, const int32_t* fidx, const float* fval, const int32_t* px,
                    const int32_t* pg, int64_t n, int64_t workspace_mb, float* out) {
  // 1. pairs stably sorted by group
  PairGroups pg_sorted(ctx);
  int bad = 0;
  HGE_TRY(pg_sorted.build(ctx, n, px, xrows, pg, groups, &bad));
  HGE_REQUIRE(!(bad & kBadX), "%s: a pair names a row outside X's %lld", who, (long long)xrows);
  HGE_REQUIRE(!(bad & kBadGroup), "%s: a pair names a group outside [0, %lld)", who, (long long)groups);
  const int32_t* order = pg_sorted.order;
  const int64_t U = pg_sorted.U;
  DevBuf<int32_t>& ug = pg_sorted.ug;
  DevBuf<int32_t>& rank = pg_sorted.rank;
  DevBuf<int64_t>& ustart = pg_sorted.ustart;

  // 2. the named groups' expansion sizes
  DevBuf<int64_t> usize(ctx), uoff(ctx);
  DevBuf<char> temp(ctx);
  size_t bytes = 0;
  HGE_TRY(usize.alloc((size_t)U + 1));
  HGE_TRY(uoff.alloc((size_t)U + 1));
  k_named_sizes<<<grid_for(ctx, U + 1, kBlock / 32), kBlock, 0, ctx->stream>>>(U, ug.p, gptr, gidx, fptr, usize.p);
  HGE_CHECK_LAUNCH(ctx);
  HGE_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, bytes, usize.p, uoff.p, U + 1, ctx->stream));
  HGE_TRY(temp.alloc(bytes));
  HGE_CUDA(cub::DeviceScan::ExclusiveSum(temp.p, bytes, usize.p, uoff.p, U + 1, ctx->stream));
  ctx->launches++;
  temp.reset();
  usize.reset();
  std::vector<int64_t> h_uoff((size_t)U + 1), h_ustart((size_t)U + 1);
  HGE_TRY(read_back(ctx, uoff.p, h_uoff.data(), (size_t)U + 1));
  HGE_TRY(read_back(ctx, ustart.p, h_ustart.data(), (size_t)U + 1));

  // 3. batches of consecutive named groups whose expansion fits the budget (a single larger group
  //    is its own batch): centroid rows, then the merge of the batch's pairs
  const int64_t budget = std::max<int64_t>(1, (workspace_mb << 20) / kBytesPerEntry);
  for (int64_t u0 = 0; u0 < U;) {
    int64_t u1 = u0 + 1;
    while (u1 < U && h_uoff[(size_t)u1 + 1] - h_uoff[(size_t)u0] <= budget) ++u1;
    const int64_t L = u1 - u0, m = h_uoff[(size_t)u1] - h_uoff[(size_t)u0];
    DevBuf<int64_t> cptr(ctx);
    DevBuf<int32_t> cidx(ctx);
    DevBuf<float> cval(ctx);
    HGE_TRY(cptr.alloc((size_t)L + 1));
    if (m == 0) {   // no member of these groups has a feature: every centroid row is empty
      HGE_CUDA(cudaMemsetAsync(cptr.p, 0, ((size_t)L + 1) * sizeof(int64_t), ctx->stream));
    } else {
      DevBuf<uint64_t> keys(ctx);
      DevBuf<float> vals(ctx);
      int rc = keys.alloc((size_t)m);
      if (rc == HGE_OK) rc = vals.alloc((size_t)m);
      if (rc == HGE_ERR_NOMEM)
        hge_set_error("%s: %lld groups expand to %lld entries, more than the device holds", who, (long long)L,
                      (long long)m);
      HGE_TRY(rc);
      k_expand_named<<<grid_for(ctx, L, kBlock / 32), kBlock, 0, ctx->stream>>>(
          u0, u1, h_uoff[(size_t)u0], ug.p, uoff.p, gptr, gidx, fptr, fidx, fval, keys.p, vals.p);
      HGE_CHECK_LAUNCH(ctx);
      HGE_TRY(centroid_batch(ctx, m, L, ug.p + u0, gptr, keys, vals, cptr.p, cidx, cval));
    }
    const int64_t i0 = h_ustart[(size_t)u0], i1 = h_ustart[(size_t)u1];
    k_merge_named<<<grid_for(ctx, i1 - i0), kBlock, 0, ctx->stream>>>(i0, i1, u0, order, rank.p, ug.p, gptr, px,
                                                                    xptr, xidx, xval, cptr.p, cidx.p, cval.p, out);
    HGE_CHECK_LAUNCH(ctx);
    u0 = u1;
  }
  return HGE_OK;
}

}  // namespace

extern "C" {

int hge_jaccard_rows(hge_ctx* ctx, const int64_t* ptr, const int32_t* idx, const float* val,
                     int64_t rows, int64_t nnz, const int32_t* pi, const int32_t* pj,
                     int64_t num_pairs, float* out, int mem) {
  HGE_REQUIRE(ctx && ptr && (idx || nnz == 0) && (val || nnz == 0) && rows >= 0 && nnz >= 0,
              "hge_jaccard_rows: bad feature matrix");
  HGE_REQUIRE(num_pairs >= 0 && (num_pairs == 0 || (pi && pj && out)), "hge_jaccard_rows: bad pairs");
  HGE_REQUIRE(mem == HGE_MEM_HOST || mem == HGE_MEM_DEVICE, "hge_jaccard_rows: bad mem %d", mem);
  HGE_CUDA(cudaSetDevice(ctx->device));
  if (num_pairs == 0) return HGE_OK;
  bool ok = false;
  HGE_TRY(pairs_in_range(ctx, num_pairs, pi, rows, pj, rows, mem, &ok));
  HGE_REQUIRE(ok, "hge_jaccard_rows: a pair names a row outside [0, %lld)", (long long)rows);
  FeatureMatrix f(ctx);
  Staged<int32_t> s_i(ctx), s_j(ctx);
  Staged<float> s_out(ctx);
  HGE_TRY(f.init(ptr, idx, val, rows, nnz, mem));
  HGE_TRY(s_i.init(pi, (size_t)num_pairs, mem, true, false));
  HGE_TRY(s_j.init(pj, (size_t)num_pairs, mem, true, false));
  HGE_TRY(s_out.init(out, (size_t)num_pairs, mem, false, true));
  k_jaccard_merge<<<grid_for(ctx, num_pairs), kBlock, 0, ctx->stream>>>(num_pairs, f.ptr.dev, f.idx.dev, f.val.dev,
                                                                       s_i.dev, s_j.dev, s_out.dev);
  HGE_CHECK_LAUNCH(ctx);
  return s_out.finish();
}

int hge_jaccard_centroid(hge_ctx* ctx, const int64_t* xptr, const int32_t* xidx, const float* xval,
                         int64_t xrows, int64_t xnnz, const int64_t* gptr, const int32_t* gidx,
                         int64_t grows, int64_t gnnz, const int64_t* fptr, const int32_t* fidx,
                         const float* fval, int64_t frows, int64_t fnnz, const int32_t* px,
                         const int32_t* pg, int64_t num_pairs, float* out, int mem) {
  HGE_REQUIRE(ctx && xptr && gptr && fptr && xrows >= 0 && grows >= 0 && frows >= 0 && xnnz >= 0 &&
                  gnnz >= 0 && fnnz >= 0, "hge_jaccard_centroid: bad matrix");
  HGE_REQUIRE(num_pairs >= 0 && num_pairs < (1ll << 31) && (num_pairs == 0 || (px && pg && out)),
              "hge_jaccard_centroid: bad pairs");
  HGE_REQUIRE(mem == HGE_MEM_HOST || mem == HGE_MEM_DEVICE, "hge_jaccard_centroid: bad mem %d", mem);
  HGE_CUDA(cudaSetDevice(ctx->device));
  if (num_pairs == 0) return HGE_OK;
  FeatureMatrix x(ctx), f(ctx);
  const bool same = xptr == fptr && xidx == fidx && xval == fval;   // usual case: X is F
  Staged<int64_t> s_gptr(ctx);
  Staged<int32_t> s_gidx(ctx), s_px(ctx), s_pg(ctx);
  Staged<float> s_out(ctx);
  HGE_TRY(f.init(fptr, fidx, fval, frows, fnnz, mem));
  if (!same) HGE_TRY(x.init(xptr, xidx, xval, xrows, xnnz, mem));
  HGE_TRY(s_gptr.init(gptr, (size_t)grows + 1, mem, true, false));
  HGE_TRY(s_gidx.init(gidx, (size_t)gnnz, mem, true, false));
  HGE_TRY(s_px.init(px, (size_t)num_pairs, mem, true, false));
  HGE_TRY(s_pg.init(pg, (size_t)num_pairs, mem, true, false));
  HGE_TRY(s_out.init(out, (size_t)num_pairs, mem, false, true));
  const FeatureMatrix& xr = same ? f : x;
  // an int32 pg names no group at or past 2^31, so the clamp keeps the core's range check exact
  HGE_TRY(centroid_factor(ctx, "hge_jaccard_centroid", s_gptr.dev, s_gidx.dev, std::min<int64_t>(grows, 1ll << 31),
                          xr.ptr.dev, xr.idx.dev, xr.val.dev, xrows, f.ptr.dev, f.idx.dev, f.val.dev, s_px.dev,
                          s_pg.dev, num_pairs, kDefaultWorkspaceMb, s_out.dev));
  return s_out.finish();
}

int hge_jaccard_centroid_grouped(hge_ctx* ctx, hge_incidence* inc, int group_side, const int64_t* xptr,
                                 const int32_t* xidx, const float* xval, int64_t xrows, int64_t xnnz,
                                 const int64_t* fptr, const int32_t* fidx, const float* fval, int64_t frows,
                                 int64_t fnnz, const int32_t* px, const int32_t* pg, int64_t num_pairs,
                                 int64_t workspace_mb, float* out) {
  HGE_REQUIRE(ctx && inc, "hge_jaccard_centroid_grouped: NULL argument");
  HGE_REQUIRE(!inc->sharded, "hge_jaccard_centroid_grouped: needs a whole (not sharded) incidence");
  HGE_REQUIRE(group_side == 0 || group_side == 1, "hge_jaccard_centroid_grouped: group_side must be 0 or 1");
  HGE_REQUIRE(xptr && fptr && xrows >= 0 && frows >= 0 && xnnz >= 0 && fnnz >= 0 && (xidx || xnnz == 0) &&
                  (xval || xnnz == 0) && (fidx || fnnz == 0) && (fval || fnnz == 0),
              "hge_jaccard_centroid_grouped: bad matrix");
  // groups are edges with node members (F = node features), or nodes with edge members
  const int64_t groups = group_side == 1 ? inc->E : inc->N, members = group_side == 1 ? inc->N : inc->E;
  HGE_REQUIRE(frows == members, "hge_jaccard_centroid_grouped: F has %lld rows, the members number %lld",
              (long long)frows, (long long)members);
  HGE_REQUIRE(num_pairs >= 0 && num_pairs < (1ll << 31) && (num_pairs == 0 || (px && pg && out)),
              "hge_jaccard_centroid_grouped: bad pairs");
  HGE_REQUIRE(workspace_mb >= 0, "hge_jaccard_centroid_grouped: negative workspace");
  HGE_CUDA(cudaSetDevice(ctx->device));
  if (num_pairs == 0) return HGE_OK;
  return centroid_factor(ctx, "hge_jaccard_centroid_grouped", group_side == 1 ? inc->e2n_ptr : inc->n2e_ptr,
                         group_side == 1 ? inc->e2n_idx : inc->n2e_idx, groups, xptr, xidx, xval, xrows, fptr, fidx,
                         fval, px, pg, num_pairs, workspace_mb ? workspace_mb : kDefaultWorkspaceMb, out);
}

}  // extern "C"
