// FOBE / HOBE pair and neighbour sampling on the device from a seeded counter-based generator
// (hge_sample_pairs_device / hge_sample_neighbors_device, include/hge_b200.h).
//
// The draws have the distribution of _sample_adj_matrix / _sample_neighbors (hg2v_sample.py:49-86)
// but come from Philox word streams (csrc/hge_philox.cuh), one per row or record, instead of
// numpy's sequential MT19937: every row is sampled by its own thread, independently of the others.
// csrc/hge_sampler.cpp keeps the bit-exact replay of the reference's stream.
//
// Candidate rows of a product P = M1 (* M2 (* M3)) are built per batch of rows whose expansion fits
// the workspace budget (a single larger row is its own batch):
//   expand   one warp per row writes (local row << 32 | column) for every member of every factor
//            row it names (k_expand_rows);
//   sort     cub radix sort of the keys;
//   runs     run heads + exclusive scan: the distinct columns of every row, ascending
//            (hge_expand.cuh, shared with the centroid rows of hge_jaccard.cu).
// Three-factor rows expand the DEDUPLICATED two-factor row.  Selection is one thread per row:
// Floyd's algorithm over positions of the row's distinct candidates, marked in a per-row flag
// array, then the marked columns in ascending order.  A row with no more candidates than samples
// emits all of them and draws nothing.  Negatives are one thread per row (k_r draws with
// replacement), neighbour arrays one thread per record.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <vector>

#include "hge_expand.cuh"
#include "hge_incidence.cuh"
#include "hge_philox.cuh"

namespace {

constexpr int kBlock = kExpandBlock;
constexpr int64_t kDefaultWorkspaceMb = 2048;
// workspace bytes per expanded entry: two key buffers, run heads and their scan (8 bytes each),
// one selection flag, and the sort's temporary storage
constexpr int64_t kBytesPerEntry = 40;

enum : int { kBadCount = 1, kEmptyList = 2 };

int exclusive_sum(hge_ctx* ctx, const int64_t* in, int64_t* out, int64_t n) {
  size_t bytes = 0;
  HGE_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, bytes, in, out, n, ctx->stream));
  DevBuf<char> temp(ctx);
  HGE_TRY(temp.alloc(bytes));
  HGE_CUDA(cub::DeviceScan::ExclusiveSum(temp.p, bytes, in, out, n, ctx->stream));
  ctx->launches++;
  return HGE_OK;
}

// size[l] = sum over the members c of source row l of deg_M(c); size[L] = 0 (one warp per row)
__global__ void __launch_bounds__(kBlock) k_expand_sizes(int64_t L, const int64_t* __restrict__ src_ptr,
                                                         const int32_t* __restrict__ src_idx,
                                                         const int64_t* __restrict__ mptr,
                                                         int64_t* __restrict__ size) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = (int64_t)gridDim.x * (kBlock / 32);
  for (int64_t l = blockIdx.x * (int64_t)(kBlock / 32) + (threadIdx.x >> 5); l <= L; l += nw) {
    int64_t s = 0;
    if (l < L)
      for (int64_t t = src_ptr[l] + lane; t < src_ptr[l + 1]; t += 32) {
        const int32_t c = src_idx[t];
        s += mptr[c + 1] - mptr[c];
      }
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) size[l] = s;
  }
}

// keys of source rows [g0, g1): (l - g0) << 32 | column, for every member of every M row that
// source row l names, starting at off[l] - base (one warp per row, factor rows in member order)
__global__ void __launch_bounds__(kBlock) k_expand_rows(int64_t g0, int64_t g1, int64_t base,
                                                        const int64_t* __restrict__ src_ptr,
                                                        const int32_t* __restrict__ src_idx,
                                                        const int64_t* __restrict__ mptr,
                                                        const int32_t* __restrict__ midx,
                                                        const int64_t* __restrict__ off,
                                                        uint64_t* __restrict__ keys) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = (int64_t)gridDim.x * (kBlock / 32);
  for (int64_t l = g0 + blockIdx.x * (int64_t)(kBlock / 32) + (threadIdx.x >> 5); l < g1; l += nw) {
    const uint64_t hi = (uint64_t)(l - g0) << 32;
    int64_t pos = off[l] - base;
    for (int64_t t = src_ptr[l]; t < src_ptr[l + 1]; ++t) {
      const int32_t c = src_idx[t];
      const int64_t s = mptr[c], d = mptr[c + 1] - s;
      for (int64_t k = lane; k < d; k += 32) keys[pos + k] = hi | (uint32_t)midx[s + k];
      pos += d;
    }
  }
}

__global__ void k_run_cols(int64_t n, const uint64_t* __restrict__ keys, const int64_t* __restrict__ pos,
                           int32_t* __restrict__ cols) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    if (i == 0 || keys[i] != keys[i - 1]) cols[pos[i]] = (int32_t)(uint32_t)keys[i];
}

// cnt[l] = records row l emits: min(k_l, n_l) positives, k_l negatives; cnt[L] = 0
__global__ void k_row_counts(int64_t L, const int32_t* __restrict__ k, const int64_t* __restrict__ cptr,
                             bool negative, int64_t* __restrict__ cnt, int* __restrict__ status) {
  for (int64_t l = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; l <= L;
       l += (int64_t)gridDim.x * blockDim.x) {
    if (l == L) {
      cnt[l] = 0;
      continue;
    }
    const int32_t want = k[l];
    if (want < 0) atomicOr(status, kBadCount);
    const int64_t kk = want < 0 ? 0 : want, n = negative ? kk : cptr[l + 1] - cptr[l];
    cnt[l] = kk < n ? kk : n;
  }
}

// Floyd's selection of min(k, n) of the n distinct candidates of every row, emitted ascending.
// cptr / ccol: candidate rows (cptr relative to cbase); flags: one zeroed byte per candidate.
__global__ void k_select(int64_t L, int64_t row_first, const int32_t* __restrict__ k,
                         const int64_t* __restrict__ cptr, int64_t cbase, const int32_t* __restrict__ ccol,
                         const int64_t* __restrict__ out_off, int64_t out_base, uint8_t* __restrict__ flags,
                         uint64_t seed, uint32_t phase, int32_t* __restrict__ out_row,
                         int32_t* __restrict__ out_col) {
  for (int64_t l = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; l < L;
       l += (int64_t)gridDim.x * blockDim.x) {
    const int64_t c0 = cptr[l] - cbase;
    const uint32_t n = (uint32_t)(cptr[l + 1] - cptr[l]);
    const uint32_t want = k[l] < 0 ? 0u : (uint32_t)k[l], kk = want < n ? want : n;
    if (kk == 0) continue;
    const int32_t row = (int32_t)(row_first + l);
    int64_t o = out_base + out_off[l];
    if (kk == n) {
      for (uint32_t p = 0; p < n; ++p, ++o) {
        out_row[o] = row;
        out_col[o] = ccol[c0 + p];
      }
      continue;
    }
    uint8_t* f = flags + c0;
    HgeStreamRng rng(seed, phase, (uint64_t)row);
    for (uint32_t j = n - kk; j < n; ++j) {
      const uint32_t t = rng.below(j + 1);
      if (f[t]) f[j] = 1; else f[t] = 1;
    }
    for (uint32_t p = 0; p < n; ++p)
      if (f[p]) {
        out_row[o] = row;
        out_col[o] = ccol[c0 + p];
        ++o;
      }
  }
}

// k_l draws with replacement, uniform on [0, out_cols), per row
__global__ void k_negatives(int64_t L, int64_t row_first, const int32_t* __restrict__ k, uint32_t out_cols,
                            const int64_t* __restrict__ out_off, int64_t out_base, uint64_t seed, uint32_t phase,
                            int32_t* __restrict__ out_row, int32_t* __restrict__ out_col) {
  for (int64_t l = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; l < L;
       l += (int64_t)gridDim.x * blockDim.x) {
    const int32_t row = (int32_t)(row_first + l);
    HgeStreamRng rng(seed, phase, (uint64_t)row);
    int64_t o = out_base + out_off[l];
    for (int32_t j = 0; j < k[l]; ++j, ++o) {
      out_row[o] = row;
      out_col[o] = (int32_t)rng.below(out_cols);
    }
  }
}

// per record: k draws from the node's edges, then k from the edge's nodes
__global__ void k_neighbors(int64_t count, int k, const int32_t* __restrict__ nodes,
                            const int32_t* __restrict__ edges, const int64_t* __restrict__ n2e_ptr,
                            const int32_t* __restrict__ n2e_idx, const int64_t* __restrict__ e2n_ptr,
                            const int32_t* __restrict__ e2n_idx, uint64_t seed, uint32_t phase,
                            int64_t first_index, int32_t* __restrict__ out_e, int32_t* __restrict__ out_n,
                            int* __restrict__ status) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < count;
       i += (int64_t)gridDim.x * blockDim.x) {
    HgeStreamRng rng(seed, phase, (uint64_t)(first_index + i));
    const int32_t nd = nodes[i], ed = edges[i];
    const int64_t ns = n2e_ptr[nd], es = e2n_ptr[ed];
    const uint32_t ndeg = (uint32_t)(n2e_ptr[nd + 1] - ns), edeg = (uint32_t)(e2n_ptr[ed + 1] - es);
    if (ndeg == 0 || edeg == 0) {
      atomicOr(status, kEmptyList);
      for (int j = 0; j < k; ++j) out_e[i * k + j] = out_n[i * k + j] = -1;
      continue;
    }
    for (int j = 0; j < k; ++j) out_e[i * k + j] = n2e_idx[ns + rng.below(ndeg)];
    for (int j = 0; j < k; ++j) out_n[i * k + j] = e2n_idx[es + rng.below(edeg)];
  }
}

struct DevCsr {
  const int64_t* ptr;
  const int32_t* idx;
};

// One hge_sample_pairs_device call: output cursor, per-row counts and the RNG address.
struct PairSampler {
  hge_ctx* ctx;
  int64_t budget;         // expanded entries per batch
  uint64_t seed;
  uint32_t phase;
  const int32_t* k;       // device, per row of the call's range
  int32_t row0;
  int32_t* out_row;
  int32_t* out_col;
  int64_t capacity;
  int64_t written = 0;
  int* status;

  // selection of rows [l0, l0 + L) of the call from their candidate rows
  int select(int64_t l0, int64_t L, const int64_t* cptr, int64_t cbase, const int32_t* ccol, int64_t ncand) {
    DevBuf<int64_t> cnt(ctx), off(ctx);
    HGE_TRY(cnt.alloc((size_t)L + 1));
    HGE_TRY(off.alloc((size_t)L + 1));
    k_row_counts<<<grid_for(ctx, L + 1), kBlock, 0, ctx->stream>>>(L, k + l0, cptr, false, cnt.p, status);
    HGE_CHECK_LAUNCH(ctx);
    HGE_TRY(exclusive_sum(ctx, cnt.p, off.p, L + 1));
    int64_t total = 0;
    HGE_TRY(read_back(ctx, off.p + L, &total, 1));
    HGE_REQUIRE(written + total <= capacity, "hge_sample_pairs_device: capacity %lld is too small",
                (long long)capacity);
    DevBuf<uint8_t> flags(ctx);
    HGE_TRY(flags.alloc((size_t)ncand));
    HGE_CUDA(cudaMemsetAsync(flags.p, 0, (size_t)std::max<int64_t>(ncand, 1), ctx->stream));
    k_select<<<grid_for(ctx, L), kBlock, 0, ctx->stream>>>(L, row0 + l0, k + l0, cptr, cbase, ccol, off.p, written,
                                                         flags.p, seed, phase, out_row, out_col);
    HGE_CHECK_LAUNCH(ctx);
    written += total;
    return HGE_OK;
  }

  // distinct columns of source rows [g0, g1) of src times M: CSR (uptr [g1 - g0 + 1] from 0, ucol)
  int unique(const int64_t* src_ptr, const int32_t* src_idx, DevCsr m, int64_t g0, int64_t g1,
             const int64_t* off, const std::vector<int64_t>& h_off, DevBuf<int64_t>& uptr,
             DevBuf<int32_t>& ucol, int64_t* n_runs) {
    const int64_t L = g1 - g0, n = h_off[(size_t)g1] - h_off[(size_t)g0];
    DevBuf<uint64_t> keys(ctx), keys2(ctx);
    DevBuf<int64_t> head(ctx), pos(ctx);
    DevBuf<char> temp(ctx);
    int rc = keys.alloc((size_t)n);
    if (rc == HGE_OK) rc = keys2.alloc((size_t)n);
    if (rc == HGE_ERR_NOMEM)
      hge_set_error("hge_sample_pairs_device: %lld rows expand to %lld entries, more than the device holds",
                    (long long)L, (long long)n);
    HGE_TRY(rc);
    k_expand_rows<<<grid_for(ctx, L, kBlock / 32), kBlock, 0, ctx->stream>>>(
        g0, g1, h_off[(size_t)g0], src_ptr, src_idx, m.ptr, m.idx, off, keys.p);
    HGE_CHECK_LAUNCH(ctx);
    int row_bits = 1;
    while ((1ll << row_bits) < L) ++row_bits;
    size_t bytes = 0;
    HGE_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, bytes, keys.p, keys2.p, n, 0, 32 + row_bits, ctx->stream));
    HGE_TRY(temp.alloc(bytes));
    HGE_CUDA(cub::DeviceRadixSort::SortKeys(temp.p, bytes, keys.p, keys2.p, n, 0, 32 + row_bits, ctx->stream));
    ctx->launches++;
    temp.reset();
    keys.reset();
    HGE_TRY(head.alloc((size_t)n + 1));
    HGE_TRY(pos.alloc((size_t)n + 1));
    k_run_heads<<<grid_for(ctx, n), kBlock, 0, ctx->stream>>>(n, keys2.p, head.p);
    HGE_CHECK_LAUNCH(ctx);
    HGE_CUDA(cudaMemsetAsync(head.p + n, 0, sizeof(int64_t), ctx->stream));
    HGE_TRY(exclusive_sum(ctx, head.p, pos.p, n + 1));
    HGE_TRY(read_back(ctx, pos.p + n, n_runs, 1));
    HGE_TRY(ucol.alloc((size_t)*n_runs));
    HGE_TRY(uptr.alloc((size_t)L + 1));
    k_run_cols<<<grid_for(ctx, n), kBlock, 0, ctx->stream>>>(n, keys2.p, pos.p, ucol.p);
    HGE_CHECK_LAUNCH(ctx);
    k_run_starts<<<grid_for(ctx, L + 1), kBlock, 0, ctx->stream>>>(L, n, *n_runs, keys2.p, pos.p, uptr.p);
    HGE_CHECK_LAUNCH(ctx);
    return HGE_OK;
  }

  // per-row expansion sizes of src rows [0, L) times M, their exclusive scan (device) and a host copy
  int sizes(const int64_t* src_ptr, const int32_t* src_idx, DevCsr m, int64_t L, DevBuf<int64_t>& off,
            std::vector<int64_t>& h_off) {
    DevBuf<int64_t> size(ctx);
    HGE_TRY(size.alloc((size_t)L + 1));
    HGE_TRY(off.alloc((size_t)L + 1));
    k_expand_sizes<<<grid_for(ctx, L + 1, kBlock / 32), kBlock, 0, ctx->stream>>>(L, src_ptr, src_idx, m.ptr,
                                                                                   size.p);
    HGE_CHECK_LAUNCH(ctx);
    HGE_TRY(exclusive_sum(ctx, size.p, off.p, L + 1));
    h_off.resize((size_t)L + 1);
    return read_back(ctx, off.p, h_off.data(), (size_t)L + 1);
  }

  // next batch [g0, g1): consecutive rows whose expansion fits the budget, at least one row
  int64_t batch_end(const std::vector<int64_t>& h_off, int64_t g0, int64_t L) const {
    int64_t g1 = g0 + 1;
    while (g1 < L && h_off[(size_t)g1 + 1] - h_off[(size_t)g0] <= budget && g1 - g0 < (1ll << 31) - 1) ++g1;
    return g1;
  }

  int run(int factors, DevCsr m1, DevCsr m2, DevCsr m3, int64_t L) {
    const int64_t* src_ptr = m1.ptr + row0;
    if (factors == 1) {
      int64_t bounds[2];
      HGE_TRY(read_back(ctx, src_ptr, &bounds[0], 1));
      HGE_TRY(read_back(ctx, src_ptr + L, &bounds[1], 1));
      return select(0, L, src_ptr, bounds[0], m1.idx + bounds[0], bounds[1] - bounds[0]);
    }
    DevBuf<int64_t> off2(ctx);
    std::vector<int64_t> h_off2;
    HGE_TRY(sizes(src_ptr, m1.idx, m2, L, off2, h_off2));
    for (int64_t g0 = 0; g0 < L;) {
      const int64_t g1 = batch_end(h_off2, g0, L);
      if (h_off2[(size_t)g1] == h_off2[(size_t)g0]) {   // no candidates in these rows
        g0 = g1;
        continue;
      }
      DevBuf<int64_t> uptr(ctx);
      DevBuf<int32_t> ucol(ctx);
      int64_t nu = 0;
      HGE_TRY(unique(src_ptr, m1.idx, m2, g0, g1, off2.p, h_off2, uptr, ucol, &nu));
      if (factors == 2) {
        HGE_TRY(select(g0, g1 - g0, uptr.p, 0, ucol.p, nu));
      } else {
        // third factor over the deduplicated two-factor rows, in sub-batches of its own
        const int64_t L2 = g1 - g0;
        DevBuf<int64_t> off3(ctx);
        std::vector<int64_t> h_off3;
        HGE_TRY(sizes(uptr.p, ucol.p, m3, L2, off3, h_off3));
        for (int64_t s0 = 0; s0 < L2;) {
          const int64_t s1 = batch_end(h_off3, s0, L2);
          if (h_off3[(size_t)s1] != h_off3[(size_t)s0]) {
            DevBuf<int64_t> vptr(ctx);
            DevBuf<int32_t> vcol(ctx);
            int64_t nv = 0;
            HGE_TRY(unique(uptr.p, ucol.p, m3, s0, s1, off3.p, h_off3, vptr, vcol, &nv));
            HGE_TRY(select(g0 + s0, s1 - s0, vptr.p, 0, vcol.p, nv));
          }
          s0 = s1;
        }
      }
      g0 = g1;
    }
    return HGE_OK;
  }

  int negatives(int64_t L, uint32_t out_cols) {
    DevBuf<int64_t> cnt(ctx), off(ctx);
    HGE_TRY(cnt.alloc((size_t)L + 1));
    HGE_TRY(off.alloc((size_t)L + 1));
    k_row_counts<<<grid_for(ctx, L + 1), kBlock, 0, ctx->stream>>>(L, k, nullptr, true, cnt.p, status);
    HGE_CHECK_LAUNCH(ctx);
    HGE_TRY(exclusive_sum(ctx, cnt.p, off.p, L + 1));
    int64_t total = 0;
    HGE_TRY(read_back(ctx, off.p + L, &total, 1));
    HGE_REQUIRE(written + total <= capacity, "hge_sample_pairs_device: capacity %lld is too small",
                (long long)capacity);
    k_negatives<<<grid_for(ctx, L), kBlock, 0, ctx->stream>>>(L, row0, k, out_cols, off.p, written, seed, phase,
                                                            out_row, out_col);
    HGE_CHECK_LAUNCH(ctx);
    written += total;
    return HGE_OK;
  }
};

int check_status(hge_ctx* ctx, const int* d_status, const char* what) {
  int status = 0;
  HGE_TRY(read_back(ctx, d_status, &status, 1));
  HGE_REQUIRE(!(status & kBadCount), "%s: negative sample count", what);
  HGE_REQUIRE(!(status & kEmptyList), "%s: 'a' cannot be empty unless no samples are taken", what);
  return HGE_OK;
}

}  // namespace

extern "C" {

int hge_sample_pairs_device(hge_ctx* ctx, hge_incidence* inc, int side, int factors, int32_t row0,
                            int32_t row1, const int32_t* samples_per_row, int negative, uint64_t seed,
                            uint32_t phase, int64_t workspace_mb, int32_t* out_row, int32_t* out_col,
                            int64_t capacity, int64_t* out_count, int mem) {
  HGE_REQUIRE(ctx && inc && out_count, "hge_sample_pairs_device: NULL argument");
  HGE_REQUIRE(!inc->sharded, "hge_sample_pairs_device: needs a whole (not sharded) incidence");
  HGE_REQUIRE(side == 0 || side == 1, "hge_sample_pairs_device: side must be 0 or 1");
  HGE_REQUIRE(factors >= 1 && factors <= 3, "hge_sample_pairs_device: factors must be 1, 2 or 3");
  const int32_t rows = side == 0 ? inc->N : inc->E;
  HGE_REQUIRE(0 <= row0 && row0 <= row1 && row1 <= rows, "hge_sample_pairs_device: bad row range [%d, %d)",
              row0, row1);
  HGE_REQUIRE(row0 == row1 || samples_per_row, "hge_sample_pairs_device: NULL samples_per_row");
  HGE_REQUIRE(capacity >= 0 && (capacity == 0 || (out_row && out_col)), "hge_sample_pairs_device: bad outputs");
  HGE_REQUIRE(workspace_mb >= 0, "hge_sample_pairs_device: negative workspace");
  HGE_REQUIRE(mem == HGE_MEM_HOST || mem == HGE_MEM_DEVICE, "hge_sample_pairs_device: bad mem %d", mem);
  HGE_CUDA(cudaSetDevice(ctx->device));
  *out_count = 0;
  const int64_t L = row1 - row0;
  if (L == 0) return HGE_OK;
  const DevCsr n2e = {inc->n2e_ptr, inc->n2e_idx}, e2n = {inc->e2n_ptr, inc->e2n_idx};
  const DevCsr m1 = side == 0 ? n2e : e2n, m2 = side == 0 ? e2n : n2e;
  // columns of M1 (M1 * M2 (* M3)): E / N alternate with the number of factors
  const uint32_t out_cols = (uint32_t)(((side == 0) == (factors != 2)) ? inc->E : inc->N);
  Staged<int32_t> s_k(ctx), s_row(ctx), s_col(ctx);
  HGE_TRY(s_k.init(samples_per_row, (size_t)L, mem, true, false));
  HGE_TRY(s_row.init(out_row, (size_t)capacity, mem, false, true));
  HGE_TRY(s_col.init(out_col, (size_t)capacity, mem, false, true));
  DevBuf<int> status(ctx);
  HGE_TRY(status.alloc(1));
  HGE_CUDA(cudaMemsetAsync(status.p, 0, sizeof(int), ctx->stream));
  const int64_t mb = workspace_mb ? workspace_mb : kDefaultWorkspaceMb;
  PairSampler s{ctx, std::max<int64_t>(1, (mb << 20) / kBytesPerEntry), seed, phase, s_k.dev, row0,
                s_row.dev, s_col.dev, capacity};
  s.status = status.p;
  HGE_TRY(negative ? s.negatives(L, out_cols) : s.run(factors, m1, m2, m1, L));
  HGE_TRY(check_status(ctx, status.p, "hge_sample_pairs_device"));
  *out_count = s.written;
  s_row.count = s_col.count = (size_t)s.written;
  HGE_TRY(s_row.finish());
  return s_col.finish();
}

int hge_sample_neighbors_device(hge_ctx* ctx, hge_incidence* inc, const int32_t* nodes, const int32_t* edges,
                                int64_t count, int k, uint64_t seed, uint32_t phase, int64_t first_index,
                                int32_t* out_nbr_edges, int32_t* out_nbr_nodes, int mem) {
  HGE_REQUIRE(ctx && inc, "hge_sample_neighbors_device: NULL argument");
  HGE_REQUIRE(!inc->sharded, "hge_sample_neighbors_device: needs a whole (not sharded) incidence");
  HGE_REQUIRE(count >= 0 && k >= 0 && first_index >= 0, "hge_sample_neighbors_device: bad counts");
  HGE_REQUIRE(count == 0 || (nodes && edges), "hge_sample_neighbors_device: NULL records");
  HGE_REQUIRE(count == 0 || k == 0 || (out_nbr_edges && out_nbr_nodes),
              "hge_sample_neighbors_device: NULL outputs");
  HGE_REQUIRE(mem == HGE_MEM_HOST || mem == HGE_MEM_DEVICE, "hge_sample_neighbors_device: bad mem %d", mem);
  HGE_CUDA(cudaSetDevice(ctx->device));
  if (count == 0 || k == 0) return HGE_OK;
  Staged<int32_t> s_n(ctx), s_e(ctx), s_oe(ctx), s_on(ctx);
  HGE_TRY(s_n.init(nodes, (size_t)count, mem, true, false));
  HGE_TRY(s_e.init(edges, (size_t)count, mem, true, false));
  HGE_TRY(s_oe.init(out_nbr_edges, (size_t)count * k, mem, false, true));
  HGE_TRY(s_on.init(out_nbr_nodes, (size_t)count * k, mem, false, true));
  DevBuf<int> status(ctx);
  HGE_TRY(status.alloc(1));
  HGE_CUDA(cudaMemsetAsync(status.p, 0, sizeof(int), ctx->stream));
  k_neighbors<<<grid_for(ctx, count), kBlock, 0, ctx->stream>>>(count, k, s_n.dev, s_e.dev, inc->n2e_ptr,
                                                              inc->n2e_idx, inc->e2n_ptr, inc->e2n_idx, seed,
                                                              phase, first_index, s_oe.dev, s_on.dev, status.p);
  HGE_CHECK_LAUNCH(ctx);
  HGE_TRY(check_status(ctx, status.p, "hge_sample_neighbors_device"));
  HGE_TRY(s_oe.finish());
  return s_on.finish();
}

}  // extern "C"
