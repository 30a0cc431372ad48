// Degree-binned gather schedule of one half-sweep, built on the device.
//
// The rows of a CSR are ordered by descending degree (stable, so equal degrees stay in
// ascending row order): rows longer than light_max_deg come first and are cut into chunks of
// `chunk` incidences, the rest become 16-byte light items.  Building this on the host cost two
// passes over every row pointer plus a 24 MB upload per call (6 ms of the 8.6 ms incidence
// creation on the 1M-node / 500K-edge workload, and 0.3 s at 65M rows); here it is one key
// kernel, one radix sort and three small kernels that only need the row pointers.
//
// Two phases, so that the one host wait overlaps the upload of the column ids:
//   hge_sched_begin   keys + statistics + sort, statistics copied to pinned memory, event
//                     recorded (needs only the row pointers on the device)
//   hge_sched_finish  waits for the event, sizes the arrays, writes the work items (needs the
//                     inverse weight sums `invs` of the rows)
// The sort and the prefix sums are cub device primitives (set-up, not the hot path).
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>

#include "hge_incidence.cuh"

namespace {

constexpr int kBlock = 256;

enum { kHeavy = 0, kChunks, kPartials, kMaxDeg, kFirstEmpty, kBadRow, kNnz, kFirstPtr, kEmpty, kStatWords };
static_assert(kStatWords * sizeof(long long) <= 128, "statistics must fit one pinned slot");

__global__ void k_sched_init(long long* stats) {
  if (threadIdx.x < kStatWords)
    stats[threadIdx.x] = (threadIdx.x == kFirstEmpty || threadIdx.x == kBadRow) ? LLONG_MAX : 0;
}

// key = key_max - degree (ascending key = descending degree), value = row id; statistics of
// the row range by block reduction + one atomic per block.
__global__ void k_sched_keys(int32_t row0, int32_t rows, const int64_t* __restrict__ rb,
                             const int64_t* __restrict__ re, int light_max, int chunk,
                             uint32_t key_max,
                             uint32_t* __restrict__ keys, int32_t* __restrict__ vals,
                             long long* stats) {
  long long heavy = 0, chunks = 0, partials = 0, max_deg = 0, nnz = 0, empty = 0;
  long long first_empty = LLONG_MAX, bad = LLONG_MAX;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < rows;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t r = row0 + (int32_t)i;
    const int64_t d = re[r] - rb[r];
    if (d < 0 || d > (int64_t)key_max) {
      bad = min(bad, (long long)r);
      keys[i] = key_max;
      vals[i] = r;
      continue;
    }
    if (d == 0) {
      first_empty = min(first_empty, (long long)r);
      empty += 1;
    }
    max_deg = max(max_deg, (long long)d);
    nnz += d;
    if (d > light_max) {
      const long long nch = (d + chunk - 1) / chunk;
      heavy += 1;
      chunks += nch;
      partials += nch > 1 ? nch : 0;
    }
    keys[i] = key_max - (uint32_t)d;
    vals[i] = r;
  }
#pragma unroll
  for (int off = 16; off; off >>= 1) {
    heavy += __shfl_xor_sync(0xffffffffu, heavy, off);
    chunks += __shfl_xor_sync(0xffffffffu, chunks, off);
    partials += __shfl_xor_sync(0xffffffffu, partials, off);
    nnz += __shfl_xor_sync(0xffffffffu, nnz, off);
    empty += __shfl_xor_sync(0xffffffffu, empty, off);
    max_deg = max(max_deg, __shfl_xor_sync(0xffffffffu, max_deg, off));
    first_empty = min(first_empty, __shfl_xor_sync(0xffffffffu, first_empty, off));
    bad = min(bad, __shfl_xor_sync(0xffffffffu, bad, off));
  }
  if ((threadIdx.x & 31) == 0) {
    if (heavy) atomicAdd(reinterpret_cast<unsigned long long*>(stats + kHeavy), (unsigned long long)heavy);
    if (chunks) atomicAdd(reinterpret_cast<unsigned long long*>(stats + kChunks), (unsigned long long)chunks);
    if (partials)
      atomicAdd(reinterpret_cast<unsigned long long*>(stats + kPartials), (unsigned long long)partials);
    if (nnz) atomicAdd(reinterpret_cast<unsigned long long*>(stats + kNnz), (unsigned long long)nnz);
    if (empty) atomicAdd(reinterpret_cast<unsigned long long*>(stats + kEmpty), (unsigned long long)empty);
    if (max_deg) atomicMax(stats + kMaxDeg, max_deg);
    if (first_empty != LLONG_MAX) atomicMin(stats + kFirstEmpty, first_empty);
    if (bad != LLONG_MAX) atomicMin(stats + kBadRow, bad);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) stats[kFirstPtr] = rb[row0];
}

__global__ void k_sched_light(int64_t n_light, const int32_t* __restrict__ sorted_rows,
                              const int64_t* __restrict__ rb, const int64_t* __restrict__ re,
                              const float* __restrict__ invs, HgeLightItem* __restrict__ items) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_light;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t r = sorted_rows[i];
    const int64_t b = rb[r], d = re[r] - b;
    HgeLightItem it;
    it.row = r;
    it.deg_hi = (uint32_t)d | (uint32_t)((b >> 32) << 8);
    it.start_lo = (uint32_t)(b & 0xffffffffll);
    it.invs = invs[r];
    items[i] = it;
  }
}

__global__ void k_sched_heavy_counts(int32_t n_heavy, const int32_t* __restrict__ sorted_rows,
                                     const int64_t* __restrict__ rb,
                                     const int64_t* __restrict__ re, int chunk,
                                     int32_t* __restrict__ nch, int32_t* __restrict__ npart) {
  for (int32_t h = blockIdx.x * blockDim.x + threadIdx.x; h < n_heavy; h += gridDim.x * blockDim.x) {
    const int32_t r = sorted_rows[h];
    const int64_t d = re[r] - rb[r];
    const int32_t c = (int32_t)((d + chunk - 1) / chunk);
    nch[h] = c;
    npart[h] = c > 1 ? c : 0;
  }
}

// One warp per long row: its descriptor and its (row, chunk) work items; the chunks of the
// longest rows come first, so their reductions finish early.
__global__ void k_sched_heavy_write(int32_t n_heavy, const int32_t* __restrict__ sorted_rows,
                                    const int64_t* __restrict__ rb, const int64_t* __restrict__ re,
                                    const float* __restrict__ invs,
                                    int chunk, const int32_t* __restrict__ chunk_off,
                                    const int32_t* __restrict__ part_off,
                                    HgeHeavyRow* __restrict__ hrows, int2* __restrict__ chunks) {
  const int lane = threadIdx.x & 31;
  const int32_t warps = gridDim.x * (blockDim.x >> 5);
  for (int32_t h = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); h < n_heavy; h += warps) {
    const int32_t r = sorted_rows[h];
    const int64_t b = rb[r], d = re[r] - b;
    const int32_t nch = (int32_t)((d + chunk - 1) / chunk);
    if (lane == 0) {
      HgeHeavyRow hr;
      hr.row = r;
      hr.deg = (int32_t)d;
      hr.start = b;
      hr.nchunks = nch;
      hr.partial_base = nch > 1 ? part_off[h] : 0;
      hr.invs = invs[r];
      hr.pad = 0;
      hrows[h] = hr;
    }
    const int32_t base = chunk_off[h];
    for (int32_t k = lane; k < nch; k += 32) chunks[base + k] = make_int2(h, k);
  }
}

// ---- packed gather stream (HgeStream) ---------------------------------------------------

// steps[u] of every unit (chunks of long rows first, then groups of G short rows); steps[n_units] = 0
__global__ void k_unit_steps(int32_t n_units, int32_t n_chunks, int64_t n_light, int G, int with_own,
                             int chunk, const int2* __restrict__ chunks,
                             const HgeHeavyRow* __restrict__ hrows,
                             const HgeLightItem* __restrict__ light, uint32_t* __restrict__ steps) {
  for (int64_t u = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; u <= n_units;
       u += (int64_t)gridDim.x * blockDim.x) {
    uint32_t st = 0;
    if (u < n_chunks) {
      const int2 ch = chunks[u];
      const int cnt = min(chunk, hrows[ch.x].deg - ch.y * chunk);
      st = (uint32_t)((cnt + 4 * G - 1) / (4 * G));
      st = (st + kStreamStepAlign - 1) / kStreamStepAlign * kStreamStepAlign;
    } else if (u < n_units) {
      // rows are sorted by descending degree: the first row of the group is its longest
      const int64_t first = (u - n_chunks) * G;
      const int d = first < n_light ? (int)(light[first].deg_hi & 0xffu) : 0;
      st = (uint32_t)max(1, (d + with_own + 3) / 4);
    }
    steps[u] = st;
  }
}

// one block per chunk of a long row: its column ids in storage order, padded with the zero row
__global__ void k_stream_heavy(int32_t n_chunks, int G, int chunk, uint32_t gather0, uint32_t zero,
                               const int2* __restrict__ chunks, const HgeHeavyRow* __restrict__ hrows,
                               const int32_t* __restrict__ idx, const uint32_t* __restrict__ uoff,
                               int32_t* __restrict__ ids) {
  for (int32_t u = blockIdx.x; u < n_chunks; u += gridDim.x) {
    const int2 ch = chunks[u];
    const HgeHeavyRow hr = hrows[ch.x];
    const int cnt = min(chunk, hr.deg - ch.y * chunk);
    const int32_t* src = idx + hr.start + (int64_t)ch.y * chunk;
    const uint32_t pos = uoff[u];
    const int total = (int)(uoff[u + 1] - pos) * 4 * G;
    int32_t* dst = ids + (size_t)pos * 4 * G;
    for (int j = threadIdx.x; j < total; j += blockDim.x)
      dst[j] = j < cnt ? (int32_t)(gather0 + (uint32_t)src[j]) : (int32_t)zero;
  }
}

// one warp per group of G short rows: slot (step s, group g, j) holds incidence 4 s + j of row g,
// the zero row beyond the row's degree, and (with_own) the row itself in the group's last slot
__global__ void k_stream_light(int32_t n_quads, int32_t n_chunks, int64_t n_light, int G, int with_own,
                               uint32_t gather0, uint32_t own0, uint32_t zero,
                               const HgeLightItem* __restrict__ light, const int32_t* __restrict__ idx,
                               const uint32_t* __restrict__ uoff, int32_t* __restrict__ ids,
                               int4* __restrict__ items) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t q = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5); q < n_quads; q += warps) {
    const uint32_t pos = uoff[n_chunks + q];
    const int steps = (int)(uoff[n_chunks + q + 1] - pos);
    if (lane < G) {
      const int64_t i = q * G + lane;
      int4 it = make_int4(-1, 0, steps, 0);
      if (i < n_light) {
        const HgeLightItem li = light[i];
        it.x = li.row;
        it.y = (int)(li.deg_hi & 0xffu);
        it.w = __float_as_int(li.invs);
      }
      items[i] = it;
    }
    const int total = steps * 4 * G;
    int32_t* dst = ids + (size_t)pos * 4 * G;
    for (int f = lane; f < total; f += 32) {
      const int g = (f >> 2) % G;
      const int k = (f / (4 * G)) * 4 + (f & 3);
      const int64_t i = q * G + g;
      int32_t v = (int32_t)zero;
      if (i < n_light) {
        const HgeLightItem li = light[i];
        const int d = (int)(li.deg_hi & 0xffu);
        if (k < d) {
          const int64_t start = ((int64_t)(li.deg_hi >> 8) << 32) | (int64_t)li.start_lo;
          v = (int32_t)(gather0 + (uint32_t)idx[start + k]);
        } else if (with_own && k == steps * 4 - 1) {
          v = (int32_t)(own0 + (uint32_t)li.row);
        }
      }
      dst[f] = v;
    }
  }
}

// what k_sweep reads past the end: zero-row ids for its id look-ahead, descriptors that never
// finish for its descriptor ring
__global__ void k_stream_slack(int n, uint32_t zero, int32_t* __restrict__ dst, int4* __restrict__ items) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    dst[i] = (int32_t)zero;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < kStreamSlackItems; i += gridDim.x * blockDim.x)
    items[i] = make_int4(-1, 0, 0x7fffffff, 0);
}

// piece[p] = first unit whose cost prefix (steps before it + 1 per unit before it) reaches
// p / pieces of the total
__global__ void k_piece_bounds(int pieces, int32_t n_units, const uint32_t* __restrict__ uoff,
                               int32_t* __restrict__ piece) {
  const unsigned long long total = (unsigned long long)uoff[n_units] + (unsigned long long)n_units;
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p <= pieces; p += gridDim.x * blockDim.x) {
    if (p == pieces) {
      piece[p] = n_units;
      continue;
    }
    const unsigned long long want = total * (unsigned long long)p / (unsigned long long)pieces;
    int32_t lo = 0, hi = n_units;
    while (lo < hi) {
      const int32_t mid = lo + ((hi - lo) >> 1);
      const unsigned long long c = (unsigned long long)uoff[mid] + (unsigned long long)mid;
      if (c < want) lo = mid + 1; else hi = mid;
    }
    piece[p] = lo;
  }
}

}  // namespace

int hge_sched_begin(hge_ctx* ctx, int32_t row0, int32_t row1, const int64_t* d_ptr,
                    int64_t max_degree_possible, HgeHalfSchedule* s) {
  return hge_sched_begin_ranges(ctx, row0, row1, d_ptr, d_ptr + 1, max_degree_possible, s);
}

int hge_sched_begin_ranges(hge_ctx* ctx, int32_t row0, int32_t row1, const int64_t* row_begin,
                           const int64_t* row_end, int64_t max_degree_possible,
                           HgeHalfSchedule* s) {
  const int32_t rows = row1 - row0;
  s->rows = rows;
  s->row0 = row0;
  s->chunk_sz = ctx->chunk;
  s->ptr = row_begin;
  s->row_end = row_end;
  s->ranges = row_end != row_begin + 1;
  int bits = 1;
  while (bits < 31 && ((int64_t)1 << bits) <= max_degree_possible) ++bits;
  const uint32_t key_max = (uint32_t)(((int64_t)1 << bits) - 1);
  DevBuf<uint32_t> keys_in(ctx), keys_out(ctx);
  DevBuf<int32_t> vals_in(ctx);
  DevBuf<char> temp(ctx);
  HGE_TRY(keys_in.alloc((size_t)rows));
  HGE_TRY(keys_out.alloc((size_t)rows));
  HGE_TRY(vals_in.alloc((size_t)rows));
  HGE_TRY(hge_dev_alloc(ctx, &s->sorted_rows, (size_t)rows));
  HGE_TRY(hge_dev_alloc(ctx, &s->d_stats, (size_t)kStatWords));
  s->h_stats = static_cast<long long*>(hge_ctx_pinned_slot(ctx));
  if (!s->h_stats) return HGE_ERR_NOMEM;
  k_sched_init<<<1, 32, 0, ctx->stream>>>(s->d_stats);
  HGE_CHECK_LAUNCH(ctx);
  k_sched_keys<<<grid_for(ctx, rows, kBlock), kBlock, 0, ctx->stream>>>(
      row0, rows, row_begin, row_end, ctx->light_max_deg, ctx->chunk, key_max, keys_in.p, vals_in.p,
      s->d_stats);
  HGE_CHECK_LAUNCH(ctx);
  size_t temp_bytes = 0;
  HGE_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, keys_in.p, keys_out.p, vals_in.p,
                                           s->sorted_rows, (int64_t)rows, 0, bits, ctx->stream));
  HGE_TRY(temp.alloc(temp_bytes));
  HGE_CUDA(cub::DeviceRadixSort::SortPairs(temp.p, temp_bytes, keys_in.p, keys_out.p, vals_in.p,
                                           s->sorted_rows, (int64_t)rows, 0, bits, ctx->stream));
  ctx->launches += 3;   // histogram + onesweep passes (library kernels, counted approximately)
  HGE_CUDA(cudaMemcpyAsync(s->h_stats, s->d_stats, kStatWords * sizeof(long long),
                           cudaMemcpyDeviceToHost, ctx->stream));
  if (!s->stats_ready) HGE_CUDA(cudaEventCreateWithFlags(&s->stats_ready, cudaEventDisableTiming));
  HGE_CUDA(cudaEventRecord(s->stats_ready, ctx->stream));
  return HGE_OK;
}

int hge_sched_finish(hge_ctx* ctx, const char* what, HgeHalfSchedule* s) {
  HGE_CUDA(cudaEventSynchronize(s->stats_ready));
  const long long* st = s->h_stats;
  if (st[kBadRow] != LLONG_MAX) {
    hge_set_error("%s %lld: row pointers decrease, or the row has more than 2^31-1 incidences", what,
                  st[kBadRow]);
    return HGE_ERR_INVALID;
  }
  if (s->row0 == 0 && !s->ranges && st[kFirstPtr] != 0) {
    hge_set_error("%s row pointers must start at 0", what);
    return HGE_ERR_INVALID;
  }
  if (st[kChunks] > INT32_MAX) {
    hge_set_error("%s schedule needs more than 2^31-1 chunks", what);
    return HGE_ERR_UNSUPPORTED;
  }
  s->nnz = st[kNnz];
  s->max_deg = (int32_t)st[kMaxDeg];
  s->first_empty = st[kFirstEmpty] == LLONG_MAX ? -1 : (int32_t)st[kFirstEmpty];
  s->n_hrows = (int32_t)st[kHeavy];
  s->n_light = (int64_t)s->rows - s->n_hrows;
  // rows are sorted by descending degree, so the empty ones are the tail of the light items; a
  // tile of the edge half leaves them out (it adds nothing to their sums)
  if (s->skip_empty) s->n_light -= st[kEmpty];
  s->n_chunks = (int32_t)st[kChunks];
  s->n_partials = (int32_t)st[kPartials];
  HGE_TRY(hge_dev_alloc(ctx, &s->light, (size_t)s->n_light));
  HGE_TRY(hge_dev_alloc(ctx, &s->hrows, (size_t)s->n_hrows));
  HGE_TRY(hge_dev_alloc(ctx, &s->chunks, (size_t)s->n_chunks));
  if (s->n_light) {
    k_sched_light<<<grid_for(ctx, s->n_light, kBlock), kBlock, 0, ctx->stream>>>(
        s->n_light, s->sorted_rows + s->n_hrows, s->ptr, s->row_end, s->invs, s->light);
    HGE_CHECK_LAUNCH(ctx);
  }
  if (s->n_hrows) {
    const int32_t nh = s->n_hrows;
    DevBuf<int32_t> nch(ctx), npart(ctx), coff(ctx), poff(ctx);
    DevBuf<char> temp(ctx);
    HGE_TRY(nch.alloc((size_t)nh));
    HGE_TRY(npart.alloc((size_t)nh));
    HGE_TRY(coff.alloc((size_t)nh));
    HGE_TRY(poff.alloc((size_t)nh));
    k_sched_heavy_counts<<<grid_for(ctx, nh, kBlock), kBlock, 0, ctx->stream>>>(
        nh, s->sorted_rows, s->ptr, s->row_end, s->chunk_sz, nch.p, npart.p);
    HGE_CHECK_LAUNCH(ctx);
    size_t temp_bytes = 0;
    HGE_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, temp_bytes, nch.p, coff.p, nh, ctx->stream));
    HGE_TRY(temp.alloc(temp_bytes));
    HGE_CUDA(cub::DeviceScan::ExclusiveSum(temp.p, temp_bytes, nch.p, coff.p, nh, ctx->stream));
    HGE_CUDA(cub::DeviceScan::ExclusiveSum(temp.p, temp_bytes, npart.p, poff.p, nh, ctx->stream));
    ctx->launches += 2;
    k_sched_heavy_write<<<grid_for(ctx, nh, kBlock / 32), kBlock, 0, ctx->stream>>>(
        nh, s->sorted_rows, s->ptr, s->row_end, s->invs, s->chunk_sz, coff.p, poff.p, s->hrows, s->chunks);
    HGE_CHECK_LAUNCH(ctx);
  }
  hge_dev_free(ctx, s->sorted_rows);
  hge_dev_free(ctx, s->d_stats);
  return HGE_OK;
}

static void stream_release(const hge_ctx* ctx, HgeStream* t) {
  hge_dev_free(ctx, t->ids);
  hge_dev_free(ctx, t->items);
  hge_dev_free(ctx, t->uoff);
  hge_dev_free(ctx, t->piece);
  *t = HgeStream();
}

int hge_sched_stream(hge_ctx* ctx, HgeHalfSchedule* s, int G, int with_own, uint32_t gather0,
                     uint32_t own0, uint32_t zero, int pieces) {
  HgeStream& t = s->stream;
  if (t.ids && t.G == G && t.with_own == with_own && t.gather0 == gather0 && t.own0 == own0 &&
      t.zero == zero && t.pieces == pieces)
    return HGE_OK;
  stream_release(ctx, &t);
  HGE_REQUIRE(G >= 1 && G <= 32 && pieces >= 1, "hge_sched_stream: bad group count / piece count");
  const int64_t n_quads = (s->n_light + G - 1) / G;
  const int64_t n_units = (int64_t)s->n_chunks + n_quads;
  if (n_units >= INT32_MAX) {
    hge_set_error("gather stream needs more than 2^31-1 units");
    return HGE_ERR_UNSUPPORTED;
  }
  t.G = G;
  t.with_own = with_own;
  t.gather0 = gather0;
  t.own0 = own0;
  t.zero = zero;
  t.pieces = pieces;
  t.n_units = (int32_t)n_units;
  t.n_quads = (int32_t)n_quads;
  DevBuf<uint32_t> steps(ctx);
  DevBuf<char> temp(ctx);
  HGE_TRY(steps.alloc((size_t)n_units + 1));
  HGE_TRY(hge_dev_alloc(ctx, &t.uoff, (size_t)n_units + 1));
  k_unit_steps<<<grid_for(ctx, n_units + 1, kBlock), kBlock, 0, ctx->stream>>>(
      t.n_units, s->n_chunks, s->n_light, G, with_own, s->chunk_sz, s->chunks, s->hrows, s->light, steps.p);
  HGE_CHECK_LAUNCH(ctx);
  size_t temp_bytes = 0;
  HGE_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, temp_bytes, steps.p, t.uoff, n_units + 1, ctx->stream));
  HGE_TRY(temp.alloc(temp_bytes));
  HGE_CUDA(cub::DeviceScan::ExclusiveSum(temp.p, temp_bytes, steps.p, t.uoff, n_units + 1, ctx->stream));
  ctx->launches += 1;
  temp.reset();
  steps.reset();
  // the one host wait: the stream's length (a 32-bit sum that wrapped shows as a mismatch with
  // the 64-bit bound below)
  uint32_t* h_total = static_cast<uint32_t*>(hge_ctx_pinned_slot(ctx));
  if (!h_total) return HGE_ERR_NOMEM;
  HGE_CUDA(cudaMemcpyAsync(h_total, t.uoff + n_units, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  HGE_CUDA(cudaStreamSynchronize(ctx->stream));
  t.total_steps = *h_total;
  const double bound = (double)s->nnz / 4.0 + 2.0 * (double)n_units + 64.0 * 256.0;
  if (bound > 4.0e9) {
    hge_set_error("gather stream of %.3g steps does not fit 32-bit step offsets", bound);
    return HGE_ERR_UNSUPPORTED;
  }
  const size_t n_ids = ((size_t)t.total_steps + kStreamSlackSteps) * 4 * G;
  HGE_TRY(hge_dev_alloc(ctx, &t.ids, n_ids));
  HGE_TRY(hge_dev_alloc(ctx, &t.items, (size_t)n_quads * G + kStreamSlackItems));
  HGE_TRY(hge_dev_alloc(ctx, &t.piece, (size_t)pieces + 1));
  if (s->n_chunks) {
    k_stream_heavy<<<(int)std::min<int64_t>(s->n_chunks, (int64_t)ctx->num_sms * 16), kBlock, 0, ctx->stream>>>(
        s->n_chunks, G, s->chunk_sz, gather0, zero, s->chunks, s->hrows, s->idx, t.uoff, t.ids);
    HGE_CHECK_LAUNCH(ctx);
  }
  if (n_quads) {
    k_stream_light<<<grid_for(ctx, n_quads, kBlock / 32), kBlock, 0, ctx->stream>>>(
        t.n_quads, s->n_chunks, s->n_light, G, with_own, gather0, own0, zero, s->light, s->idx, t.uoff,
        t.ids, t.items);
    HGE_CHECK_LAUNCH(ctx);
  }
  k_stream_slack<<<1, kBlock, 0, ctx->stream>>>(kStreamSlackSteps * 4 * G, zero,
                                                t.ids + (size_t)t.total_steps * 4 * G,
                                                t.items + (size_t)n_quads * G);
  HGE_CHECK_LAUNCH(ctx);
  k_piece_bounds<<<grid_for(ctx, pieces + 1, kBlock), kBlock, 0, ctx->stream>>>(pieces, t.n_units, t.uoff,
                                                                              t.piece);
  HGE_CHECK_LAUNCH(ctx);
  return HGE_OK;
}

void hge_sched_release(const hge_ctx* ctx, HgeHalfSchedule* s) {
  stream_release(ctx, &s->stream);
  hge_dev_free(ctx, s->sorted_rows);
  hge_dev_free(ctx, s->d_stats);
  if (s->stats_ready) cudaEventDestroy(s->stats_ready);
  s->stats_ready = nullptr;
  hge_dev_free(ctx, s->light);
  hge_dev_free(ctx, s->hrows);
  hge_dev_free(ctx, s->chunks);
}
