// Distances, weight transforms, spans and HOBE probabilities on sm_100a
// (hg2v_weighting.py:34-103, 214-233, 301-333; hg2v_sample.py:527-629).
//
// Everything here is a gather: a pair of R-float rows per unit of work, one fp32 result.  Rows
// are read as float4 by sub-warps of LPR lanes (LPR = next power of two of ceil(R / 4), at
// most 32), several pairs in flight per lane; dense inputs whose rows are not 16-byte aligned
// (R % 4 != 0) are first copied into a zero-padded buffer.
#include <cub/device/device_scan.cuh>
#include <math.h>

#include <algorithm>
#include <new>

#include "hge_incidence.cuh"
#include "hge_staged.cuh"

namespace {

constexpr int kBlock = 256;
constexpr unsigned kFull = 0xffffffffu;

int grid_for(const hge_ctx* ctx, int64_t work_items, int items_per_block) {
  int64_t want = (work_items + items_per_block - 1) / items_per_block;
  if (want < 1) want = 1;
  return (int)std::min<int64_t>(want, (int64_t)ctx->num_sms * 16);
}

int lanes_per_row(int ld4) {
  int lpr = 1;
  while (lpr < ld4 && lpr < 32) lpr <<= 1;
  return lpr;
}

__global__ void k_pad_rows(int64_t rows, int R, int ld, const float* __restrict__ x,
                           float* __restrict__ y) {
  const int64_t total = rows * ld;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / ld;
    const int c = (int)(i - r * ld);
    y[i] = c < R ? x[r * R + c] : 0.f;
  }
}

// Dense [rows, R] rows as float4-addressable [rows, ld]: the input itself when R % 4 == 0.
struct PaddedRows {
  const hge_ctx* ctx = nullptr;
  const float4* rows4 = nullptr;
  float* owned = nullptr;
  int init(hge_ctx* c, const float* x, int64_t rows, int R) {
    ctx = c;
    if (R % 4 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0) {
      rows4 = reinterpret_cast<const float4*>(x);
      return HGE_OK;
    }
    const int ld = (R + 3) & ~3;
    HGE_TRY(hge_dev_alloc(ctx, &owned, (size_t)rows * ld));
    k_pad_rows<<<grid_for(c, rows * ld, kBlock), kBlock, 0, c->stream>>>(rows, R, ld, x, owned);
    HGE_CHECK_LAUNCH(c);
    rows4 = reinterpret_cast<const float4*>(owned);
    return HGE_OK;
  }
  ~PaddedRows() {
    if (owned) hge_dev_free(ctx, owned);
  }
};

__device__ __forceinline__ float sq_diff(const float4& a, const float4& b) {
  const float dx = a.x - b.x, dy = a.y - b.y, dz = a.z - b.z, dw = a.w - b.w;
  return fmaf(dx, dx, fmaf(dy, dy, fmaf(dz, dz, dw * dw)));
}

template <int LPR>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int off = LPR >> 1; off; off >>= 1) v += __shfl_xor_sync(kFull, v, off);
  return v;
}

// ---- per-incidence distance -------------------------------------------------------------
// One warp walks a row's incidences 32 at a time (coalesced column ids); each of its G = 32/LPR
// sub-warps takes every G-th incidence, 4 of them in flight.  Rows are distributed over warps
// in blocks of `rows_per_warp`, long rows are split into segments by the host.
struct Segment {        // a run of incidences of one row
  int32_t row;
  int32_t count;
  int64_t start;
};

template <int LPR>
__global__ void __launch_bounds__(kBlock) k_incidence_l2(
    int64_t num_segments, const Segment* __restrict__ segs, const int32_t* __restrict__ idx,
    const float4* __restrict__ x_self, const float4* __restrict__ x_other, int ld4, float max_dist,
    int as_weight, float* __restrict__ out) {
  constexpr int G = 32 / LPR;
  constexpr int U = 4;
  const int lane = threadIdx.x & 31, gl = lane & (LPR - 1), g = lane / LPR;
  const int64_t gw = (int64_t)blockIdx.x * (kBlock / 32) + (threadIdx.x >> 5);
  const int64_t nw = (int64_t)gridDim.x * (kBlock / 32);
  for (int64_t s = gw; s < num_segments; s += nw) {
    const Segment sg = segs[s];
    float4 self[(LPR == 32) ? 8 : 1];
    constexpr int S = (LPR == 32) ? 8 : 1;   // column slabs of 32 float4 (R <= 1024)
#pragma unroll
    for (int k = 0; k < S; ++k)
      self[k] = (k * LPR + gl) < ld4 ? __ldg(x_self + (size_t)sg.row * ld4 + k * LPR + gl)
                                     : hge_f4_zero();
    for (int base = 0; base < sg.count; base += 32) {
      const int my = (base + lane < sg.count) ? __ldcs(idx + sg.start + base + lane) : -1;
      for (int r0 = 0; r0 < LPR; r0 += U) {
        float acc[U];
        int col[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int t = (r0 + u) * G + g;
          col[u] = (r0 + u < LPR) ? __shfl_sync(kFull, my, t & 31) : -1;
          acc[u] = 0.f;
        }
#pragma unroll
        for (int k = 0; k < S; ++k) {
          float4 v[U];
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const bool on = col[u] >= 0 && (k * LPR + gl) < ld4;
            v[u] = on ? __ldg(x_other + (size_t)col[u] * ld4 + k * LPR + gl) : self[k];
          }
#pragma unroll
          for (int u = 0; u < U; ++u) acc[u] += sq_diff(self[k], v[u]);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const float d = sqrtf(group_sum<LPR>(acc[u]));
          const int t = (r0 + u) * G + g;
          if (gl == 0 && col[u] >= 0)
            out[sg.start + base + t] = as_weight ? (max_dist - d) / max_dist : d;
        }
      }
    }
  }
}

// ---- arbitrary pairs ---------------------------------------------------------------------
template <int LPR>
__global__ void __launch_bounds__(kBlock) k_pair_l2(int64_t num_pairs,
                                                    const int32_t* __restrict__ ia,
                                                    const int32_t* __restrict__ ib,
                                                    const float4* __restrict__ xa,
                                                    const float4* __restrict__ xb, int ld4,
                                                    float* __restrict__ out) {
  constexpr int G = 32 / LPR;
  constexpr int U = 4;
  constexpr int S = (LPR == 32) ? 8 : 1;
  const int lane = threadIdx.x & 31, gl = lane & (LPR - 1), g = lane / LPR;
  const int64_t gw = (int64_t)blockIdx.x * (kBlock / 32) + (threadIdx.x >> 5);
  const int64_t nw = (int64_t)gridDim.x * (kBlock / 32);
  for (int64_t base = gw * 32; base < num_pairs; base += nw * 32) {
    const bool have = base + lane < num_pairs;
    const int my_a = have ? __ldcs(ia + base + lane) : -1;
    const int my_b = have ? __ldcs(ib + base + lane) : -1;
    for (int r0 = 0; r0 < LPR; r0 += U) {
      float acc[U];
      int a[U], b[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int t = ((r0 + u) * G + g) & 31;
        a[u] = __shfl_sync(kFull, my_a, t);
        b[u] = __shfl_sync(kFull, my_b, t);
        if (r0 + u >= LPR) a[u] = -1;
        acc[u] = 0.f;
      }
#pragma unroll
      for (int k = 0; k < S; ++k) {
        float4 va[U], vb[U];
        const bool col_on = (k * LPR + gl) < ld4;
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const bool on = a[u] >= 0 && col_on;
          va[u] = on ? __ldg(xa + (size_t)a[u] * ld4 + k * LPR + gl) : hge_f4_zero();
          vb[u] = on ? __ldg(xb + (size_t)b[u] * ld4 + k * LPR + gl) : hge_f4_zero();
        }
#pragma unroll
        for (int u = 0; u < U; ++u) acc[u] += sq_diff(va[u], vb[u]);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const float d = sqrtf(group_sum<LPR>(acc[u]));
        const int t = (r0 + u) * G + g;
        if (gl == 0 && a[u] >= 0) out[base + t] = d;
      }
    }
  }
}

// ---- min / max and the weight transform -----------------------------------------------------
__global__ void k_minmax_init(int32_t* mm) {
  mm[0] = INT32_MAX;
  mm[1] = INT32_MIN;
}

__global__ void k_minmax(int64_t n, const float* __restrict__ v, int32_t* mm) {
  const float inf = __int_as_float(0x7f800000);
  float lo = inf, hi = -inf;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    const float x = __ldcs(v + i);
    lo = fminf(lo, x);
    hi = fmaxf(hi, x);
  }
#pragma unroll
  for (int off = 16; off; off >>= 1) {
    lo = fminf(lo, __shfl_xor_sync(kFull, lo, off));
    hi = fmaxf(hi, __shfl_xor_sync(kFull, hi, off));
  }
  __shared__ float slo[kBlock / 32], shi[kBlock / 32];
  if ((threadIdx.x & 31) == 0) {
    slo[threadIdx.x >> 5] = lo;
    shi[threadIdx.x >> 5] = hi;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < kBlock / 32; ++w) {
      lo = fminf(lo, slo[w]);
      hi = fmaxf(hi, shi[w]);
    }
    if (lo <= hi) {
      atomicMin(mm, hge_enc(lo));
      atomicMax(mm + 1, hge_enc(hi));
    }
  }
}

// v <- alpha + (1 - alpha) * (1 - (v - min) / delta), each step rounded to fp32 exactly as the
// reference's numpy float32 scalars are (no FMA contraction).
__global__ void k_scale_transform(int64_t n, float* __restrict__ v, const int32_t* __restrict__ mm,
                                  float alpha, float one_minus_alpha) {
  const float lo = hge_dec(mm[0]);
  const float delta = __fsub_rn(hge_dec(mm[1]), lo);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    const float scaled = (delta == 0.f) ? 1.f : __fdiv_rn(__fsub_rn(v[i], lo), delta);
    const float flipped = __fsub_rn(1.f, scaled);
    v[i] = __fadd_rn(alpha, __fmul_rn(one_minus_alpha, flipped));
  }
}

// ---- spans --------------------------------------------------------------------------------
template <int LPR>
__global__ void __launch_bounds__(kBlock) k_row_span(int32_t rows, const int64_t* __restrict__ ptr,
                                                     const int32_t* __restrict__ idx,
                                                     const float4* __restrict__ x_self,
                                                     const float4* __restrict__ x_other, int ld4,
                                                     int R, float* __restrict__ span) {
  constexpr int G = 32 / LPR;
  constexpr int S = (LPR == 32) ? 8 : 1;
  const int lane = threadIdx.x & 31, gl = lane & (LPR - 1), g = lane / LPR;
  const int64_t gw = (int64_t)blockIdx.x * (kBlock / 32) + (threadIdx.x >> 5);
  const int64_t nw = (int64_t)gridDim.x * (kBlock / 32);
  for (int64_t r = gw; r < rows; r += nw) {
    const int64_t b = ptr[r], e = ptr[r + 1];
    float lo = 0.f, hi = 0.f;
#pragma unroll
    for (int k = 0; k < S; ++k) {
      const int c4 = k * LPR + gl;
      if (c4 >= ld4) continue;
      const float4 self = __ldg(x_self + (size_t)r * ld4 + c4);
      const int c0 = c4 * 4;
      for (int64_t p = b + g; p < e; p += G) {
        const float4 o = __ldg(x_other + (size_t)idx[p] * ld4 + c4);
        const float d0 = o.x - self.x, d1 = o.y - self.y, d2 = o.z - self.z, d3 = o.w - self.w;
        if (c0 + 0 < R) { lo = fminf(lo, d0); hi = fmaxf(hi, d0); }
        if (c0 + 1 < R) { lo = fminf(lo, d1); hi = fmaxf(hi, d1); }
        if (c0 + 2 < R) { lo = fminf(lo, d2); hi = fmaxf(hi, d2); }
        if (c0 + 3 < R) { lo = fminf(lo, d3); hi = fmaxf(hi, d3); }
      }
    }
#pragma unroll
    for (int off = 16; off; off >>= 1) {
      lo = fminf(lo, __shfl_xor_sync(kFull, lo, off));
      hi = fmaxf(hi, __shfl_xor_sync(kFull, hi, off));
    }
    if (lane == 0) span[r] = hi - lo;
  }
}

// ---- HOBE probabilities ---------------------------------------------------------------------
// max over the intersection of two sorted rows of min(w_a, w_b); the lanes of the calling group
// (GP lanes, lane id `gl`) stride over the shorter row and binary-search the longer one.
template <int GP>
__device__ __forceinline__ float intersect_max_min(const int32_t* __restrict__ idx,
                                                   const float* __restrict__ w, int64_t sa, int da,
                                                   int64_t sb, int db, int gl) {
  if (da > db) {
    const int64_t ts = sa; sa = sb; sb = ts;
    const int td = da; da = db; db = td;
  }
  float best = 0.f;
  for (int t = gl; t < da; t += GP) {
    const int c = __ldg(idx + sa + t);
    int lo = 0, hi = db;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (__ldg(idx + sb + mid) < c) lo = mid + 1; else hi = mid;
    }
    if (lo < db && __ldg(idx + sb + lo) == c)
      best = fmaxf(best, fminf(__ldg(w + sa + t), __ldg(w + sb + lo)));
  }
  return best;
}

template <int GP>
__global__ void __launch_bounds__(kBlock) k_same_type_prob(int64_t num_pairs,
                                                           const int64_t* __restrict__ ptr,
                                                           const int32_t* __restrict__ idx,
                                                           const float* __restrict__ w,
                                                           const int32_t* __restrict__ pi,
                                                           const int32_t* __restrict__ pj,
                                                           float* __restrict__ prob) {
  const int gl = threadIdx.x & (GP - 1);
  const int64_t gid = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / GP;
  const int64_t ng = (int64_t)gridDim.x * blockDim.x / GP;
  for (int64_t p0 = gid; p0 < ((num_pairs + ng - 1) / ng) * ng; p0 += ng) {
    const bool on = p0 < num_pairs;   // keep whole warps in the shuffles below
    float best = 0.f;
    if (on) {
      const int i = pi[p0], j = pj[p0];
      const int64_t si = ptr[i], sj = ptr[j];
      best = intersect_max_min<GP>(idx, w, si, (int)(ptr[i + 1] - si), sj, (int)(ptr[j + 1] - sj), gl);
    }
#pragma unroll
    for (int off = GP >> 1; off; off >>= 1) best = fmaxf(best, __shfl_xor_sync(kFull, best, off));
    if (on && gl == 0) prob[p0] = best;
  }
}

__global__ void __launch_bounds__(kBlock) k_diff_type_prob(
    int64_t num_pairs, const int64_t* __restrict__ n2e_ptr, const int32_t* __restrict__ n2e_idx,
    const int64_t* __restrict__ e2n_ptr, const int32_t* __restrict__ e2n_idx,
    const float* __restrict__ w_e2n, const int32_t* __restrict__ pn, const int32_t* __restrict__ pe,
    float* __restrict__ prob) {
  const int lane = threadIdx.x & 31;
  const int64_t gw = (int64_t)blockIdx.x * (kBlock / 32) + (threadIdx.x >> 5);
  const int64_t nw = (int64_t)gridDim.x * (kBlock / 32);
  for (int64_t p = gw; p < num_pairs; p += nw) {
    const int n = pn[p], e = pe[p];
    const int64_t se = e2n_ptr[e];
    const int de = (int)(e2n_ptr[e + 1] - se);
    float best = 0.f;
    for (int64_t q = n2e_ptr[n]; q < n2e_ptr[n + 1]; ++q) {
      const int other = n2e_idx[q];
      const int64_t so = e2n_ptr[other];
      best = fmaxf(best, intersect_max_min<32>(e2n_idx, w_e2n, se, de, so,
                                               (int)(e2n_ptr[other + 1] - so), lane));
    }
#pragma unroll
    for (int off = 16; off; off >>= 1) best = fmaxf(best, __shfl_xor_sync(kFull, best, off));
    if (lane == 0) prob[p] = best;
  }
}

// ---- pair index range checks ------------------------------------------------------------------
// The kernels above trust their pair indices: k_same_type_prob and k_diff_type_prob read row
// pointers at them, k_pair_l2 skips a negative one and leaves its output unwritten.  The entry
// points therefore check every index before any of those kernels runs.
__global__ void k_check_pairs(int64_t n, const int32_t* __restrict__ a, int64_t rows_a,
                              const int32_t* __restrict__ b, int64_t rows_b, int* __restrict__ bad) {
  for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < n;
       p += (int64_t)gridDim.x * blockDim.x) {
    const int32_t x = __ldcs(a + p), y = __ldcs(b + p);
    if (x < 0 || x >= rows_a || y < 0 || y >= rows_b) *bad = 1;
  }
}

// *ok = every a[p] in [0, rows_a) and every b[p] in [0, rows_b).  Host arrays are scanned on the
// host; device arrays by k_check_pairs, then one flag read-back.
int pairs_in_range(hge_ctx* ctx, int64_t n, const int32_t* a, int64_t rows_a, const int32_t* b,
                   int64_t rows_b, int mem, bool* ok) {
  if (mem != HGE_MEM_DEVICE) {
    bool all = true;
    for (int64_t p = 0; p < n; ++p)
      all &= a[p] >= 0 && a[p] < rows_a && b[p] >= 0 && b[p] < rows_b;
    *ok = all;
    return HGE_OK;
  }
  int* d_bad = nullptr;
  HGE_TRY(hge_dev_alloc(ctx, &d_bad, 1));
  int h_bad = 0;
  cudaError_t e = cudaMemsetAsync(d_bad, 0, sizeof(int), ctx->stream);
  if (e == cudaSuccess) {
    k_check_pairs<<<grid_for(ctx, n, kBlock * 8), kBlock, 0, ctx->stream>>>(n, a, rows_a, b, rows_b,
                                                                          d_bad);
    ctx->launches++;
    e = cudaGetLastError();
  }
  if (e == cudaSuccess)
    e = cudaMemcpyAsync(&h_bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);   // h_bad is on this stack frame
  hge_dev_free(ctx, d_bad);
  if (e != cudaSuccess) {
    hge_set_error("pair index check: %s", cudaGetErrorString(e));
    return HGE_ERR_CUDA;
  }
  *ok = h_bad == 0;
  return HGE_OK;
}

// rows -> segments of at most kSegment incidences, on the device: per row ceil(deg / kSegment)
// segments, an exclusive prefix sum for their positions (cub; set-up), one thread per row writes
// them.  (A host loop over the row pointers did this before: two passes over 1.5 M rows, a 24 MB
// upload and a stream drain per call on the 1M-node workload.)
constexpr int kSegment = 2048;

__global__ void k_segment_counts(int32_t rows, const int64_t* __restrict__ ptr,
                                 int64_t* __restrict__ counts) {
  for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < rows;
       r += (int64_t)gridDim.x * blockDim.x)
    counts[r] = (ptr[r + 1] - ptr[r] + kSegment - 1) / kSegment;
}

__global__ void k_segment_write(int32_t rows, const int64_t* __restrict__ ptr,
                                const int64_t* __restrict__ offset, Segment* __restrict__ segs) {
  for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < rows;
       r += (int64_t)gridDim.x * blockDim.x) {
    int64_t at = offset[r];
    for (int64_t s = ptr[r]; s < ptr[r + 1]; s += kSegment) {
      Segment sg;
      sg.row = (int32_t)r;
      sg.start = s;
      sg.count = (int32_t)min((int64_t)kSegment, ptr[r + 1] - s);
      segs[at++] = sg;
    }
  }
}

int build_segments(hge_ctx* ctx, int32_t rows, const int64_t* d_ptr, int64_t nnz, Segment** d_segs,
                   int64_t* count) {
  *d_segs = nullptr;
  *count = 0;
  if (rows <= 0) return HGE_OK;
  int64_t *counts = nullptr, *offset = nullptr;
  HGE_TRY(hge_dev_alloc(ctx, &counts, (size_t)rows + 1));
  HGE_TRY(hge_dev_alloc(ctx, &offset, (size_t)rows + 1));
  HGE_CUDA(cudaMemsetAsync(counts + rows, 0, sizeof(int64_t), ctx->stream));
  const int grid = grid_for(ctx, rows, kBlock);
  k_segment_counts<<<grid, kBlock, 0, ctx->stream>>>(rows, d_ptr, counts);
  HGE_CHECK_LAUNCH(ctx);
  size_t temp_bytes = 0;
  HGE_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, temp_bytes, counts, offset, rows + 1, ctx->stream));
  char* temp = nullptr;
  HGE_TRY(hge_dev_alloc(ctx, &temp, temp_bytes));
  HGE_CUDA(cub::DeviceScan::ExclusiveSum(temp, temp_bytes, counts, offset, rows + 1, ctx->stream));
  ctx->launches += 1;
  // the segment count is bounded without a read-back: every row adds at most one partial segment
  const int64_t bound = nnz / kSegment + rows;
  HGE_TRY(hge_dev_alloc(ctx, d_segs, (size_t)bound));
  k_segment_write<<<grid, kBlock, 0, ctx->stream>>>(rows, d_ptr, offset, *d_segs);
  HGE_CHECK_LAUNCH(ctx);
  int64_t total = 0;
  HGE_CUDA(cudaMemcpyAsync(&total, offset + rows, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
  HGE_CUDA(cudaStreamSynchronize(ctx->stream));
  hge_dev_free(ctx, temp);
  hge_dev_free(ctx, counts);
  hge_dev_free(ctx, offset);
  *count = total;
  return HGE_OK;
}

#define HGE_DISPATCH_LPR(lpr, CALL) \
  switch (lpr) {                    \
    case 1: { constexpr int L = 1; CALL; } break;   \
    case 2: { constexpr int L = 2; CALL; } break;   \
    case 4: { constexpr int L = 4; CALL; } break;   \
    case 8: { constexpr int L = 8; CALL; } break;   \
    case 16: { constexpr int L = 16; CALL; } break; \
    default: { constexpr int L = 32; CALL; } break; \
  }

}  // namespace

extern "C" {

int hge_incidence_l2(hge_ctx* ctx, hge_incidence* inc, const float* xn, const float* xe, int R,
                     int order, int as_weight, float* dist, int mem) {
  HGE_REQUIRE(ctx && inc && xn && xe && dist, "hge_incidence_l2: NULL argument");
  HGE_REQUIRE(R >= 1 && R <= 1024, "hge_incidence_l2: dimension %d not in [1, 1024]", R);
  HGE_REQUIRE(order == 0 || order == 1, "hge_incidence_l2: order must be 0 or 1");
  HGE_CUDA(cudaSetDevice(ctx->device));
  const HgeHalfSchedule& half = order == 0 ? inc->node_half : inc->edge_half;
  Staged<float> s_xn, s_xe, s_out;
  HGE_TRY(s_xn.init(ctx, xn, (size_t)inc->N * R, mem, true, false));
  HGE_TRY(s_xe.init(ctx, xe, (size_t)inc->E * R, mem, true, false));
  HGE_TRY(s_out.init(ctx, dist, (size_t)half.nnz, mem, false, true));
  PaddedRows pn, pe;
  HGE_TRY(pn.init(ctx, s_xn.dev, inc->N, R));
  HGE_TRY(pe.init(ctx, s_xe.dev, inc->E, R));
  Segment* segs = nullptr;
  int64_t nseg = 0;
  HGE_TRY(build_segments(ctx, half.rows, half.ptr, half.nnz, &segs, &nseg));
  const int ld4 = ((R + 3) & ~3) / 4;
  const float max_dist = (float)sqrt((double)R);
  const float4* self = order == 0 ? pn.rows4 : pe.rows4;
  const float4* other = order == 0 ? pe.rows4 : pn.rows4;
  const int grid = grid_for(ctx, nseg, kBlock / 32);
  HGE_DISPATCH_LPR(lanes_per_row(ld4),
                   (k_incidence_l2<L><<<grid, kBlock, 0, ctx->stream>>>(
                       nseg, segs, half.idx, self, other, ld4, max_dist, as_weight, s_out.dev)));
  ctx->launches++;
  cudaError_t e = cudaGetLastError();
  hge_dev_free(ctx, segs);
  if (e != cudaSuccess) {
    hge_set_error("hge_incidence_l2: launch failed: %s", cudaGetErrorString(e));
    return HGE_ERR_CUDA;
  }
  return s_out.finish();
}

int hge_pair_l2(hge_ctx* ctx, const float* xa, int64_t rows_a, const float* xb, int64_t rows_b,
                int R, const int32_t* ia, const int32_t* ib, int64_t num_pairs, float* dist,
                int mem) {
  HGE_REQUIRE(ctx && xa && xb && dist, "hge_pair_l2: NULL argument");
  HGE_REQUIRE(num_pairs >= 0 && (num_pairs == 0 || (ia && ib)), "hge_pair_l2: bad pair arrays");
  HGE_REQUIRE(R >= 1 && R <= 1024, "hge_pair_l2: dimension %d not in [1, 1024]", R);
  if (num_pairs == 0) return HGE_OK;
  HGE_CUDA(cudaSetDevice(ctx->device));
  bool ok = false;
  HGE_TRY(pairs_in_range(ctx, num_pairs, ia, rows_a, ib, rows_b, mem, &ok));
  HGE_REQUIRE(ok, "hge_pair_l2: a pair names a row outside [0, %lld) x [0, %lld)", (long long)rows_a,
              (long long)rows_b);
  Staged<float> s_xa, s_xb, s_out;
  Staged<int32_t> s_ia, s_ib;
  HGE_TRY(s_xa.init(ctx, xa, (size_t)rows_a * R, mem, true, false));
  if (xb == xa) {
    s_xb.ctx = ctx;
    s_xb.dev = s_xa.dev;
  } else {
    HGE_TRY(s_xb.init(ctx, xb, (size_t)rows_b * R, mem, true, false));
  }
  HGE_TRY(s_ia.init(ctx, ia, (size_t)num_pairs, mem, true, false));
  HGE_TRY(s_ib.init(ctx, ib, (size_t)num_pairs, mem, true, false));
  HGE_TRY(s_out.init(ctx, dist, (size_t)num_pairs, mem, false, true));
  PaddedRows pa, pb;
  HGE_TRY(pa.init(ctx, s_xa.dev, rows_a, R));
  if (s_xb.dev == s_xa.dev) {
    pb.ctx = ctx;
    pb.rows4 = pa.rows4;
  } else {
    HGE_TRY(pb.init(ctx, s_xb.dev, rows_b, R));
  }
  const int ld4 = ((R + 3) & ~3) / 4;
  const int grid = grid_for(ctx, (num_pairs + 31) / 32, kBlock / 32);
  HGE_DISPATCH_LPR(lanes_per_row(ld4),
                   (k_pair_l2<L><<<grid, kBlock, 0, ctx->stream>>>(
                       num_pairs, s_ia.dev, s_ib.dev, pa.rows4, pb.rows4, ld4, s_out.dev)));
  HGE_CHECK_LAUNCH(ctx);
  return s_out.finish();
}

int hge_scale_transform(hge_ctx* ctx, float* values, int64_t n, double alpha, float* minmax,
                        int mem) {
  HGE_REQUIRE(ctx && (values || n == 0), "hge_scale_transform: NULL argument");
  HGE_REQUIRE(alpha >= 0.0, "hge_scale_transform: alpha %g < 0 (hg2v_weighting.py:331)", alpha);
  HGE_REQUIRE(alpha <= 1.0, "hge_scale_transform: alpha %g > 1 (hg2v_weighting.py:332)", alpha);
  HGE_REQUIRE(n >= 0, "hge_scale_transform: negative count");
  if (n == 0) return HGE_OK;   // ZeroOneScaleValues({}) == {}
  HGE_CUDA(cudaSetDevice(ctx->device));
  Staged<float> s_v;
  HGE_TRY(s_v.init(ctx, values, (size_t)n, mem, true, true));
  int32_t* mm = nullptr;
  HGE_TRY(hge_dev_alloc(ctx, &mm, 2));
  k_minmax_init<<<1, 1, 0, ctx->stream>>>(mm);
  ctx->launches++;
  const int grid = grid_for(ctx, n, kBlock * 8);
  k_minmax<<<grid, kBlock, 0, ctx->stream>>>(n, s_v.dev, mm);
  ctx->launches++;
  k_scale_transform<<<grid, kBlock, 0, ctx->stream>>>(n, s_v.dev, mm, (float)alpha,
                                                      (float)(1.0 - alpha));
  ctx->launches++;
  cudaError_t e = cudaGetLastError();
  int rc = HGE_OK;
  if (e != cudaSuccess) {
    hge_set_error("hge_scale_transform: launch failed: %s", cudaGetErrorString(e));
    rc = HGE_ERR_CUDA;
  }
  if (rc == HGE_OK && minmax) {
    int32_t h[2];
    e = cudaMemcpyAsync(h, mm, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
      hge_set_error("hge_scale_transform: reading min/max failed: %s", cudaGetErrorString(e));
      rc = HGE_ERR_CUDA;
    } else {
      minmax[0] = hge_dec(h[0]);
      minmax[1] = hge_dec(h[1]);
    }
  }
  hge_dev_free(ctx, mm);
  if (rc != HGE_OK) return rc;
  return s_v.finish();
}

// The two halves of hge_scale_transform for values that are spread over several GPUs: every rank
// reduces its own values, the caller all-reduces (min, max) over the ranks, every rank applies.
int hge_scale_minmax(hge_ctx* ctx, const float* values, int64_t n, float* minmax, int mem) {
  HGE_REQUIRE(ctx && minmax && (values || n == 0) && n >= 0, "hge_scale_minmax: bad argument");
  HGE_CUDA(cudaSetDevice(ctx->device));
  minmax[0] = INFINITY;
  minmax[1] = -INFINITY;
  if (n == 0) return HGE_OK;
  Staged<float> s_v;
  HGE_TRY(s_v.init(ctx, values, (size_t)n, mem, true, false));
  int32_t* mm = nullptr;
  HGE_TRY(hge_dev_alloc(ctx, &mm, 2));
  k_minmax_init<<<1, 1, 0, ctx->stream>>>(mm);
  ctx->launches++;
  k_minmax<<<grid_for(ctx, n, kBlock * 8), kBlock, 0, ctx->stream>>>(n, s_v.dev, mm);
  ctx->launches++;
  int32_t h[2];
  cudaError_t e = cudaMemcpyAsync(h, mm, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  hge_dev_free(ctx, mm);
  if (e != cudaSuccess) {
    hge_set_error("hge_scale_minmax: %s", cudaGetErrorString(e));
    return HGE_ERR_CUDA;
  }
  minmax[0] = hge_dec(h[0]);
  minmax[1] = hge_dec(h[1]);
  return HGE_OK;
}

int hge_scale_apply(hge_ctx* ctx, float* values, int64_t n, double alpha, float lo, float hi,
                    int mem) {
  HGE_REQUIRE(ctx && (values || n == 0) && n >= 0, "hge_scale_apply: bad argument");
  HGE_REQUIRE(alpha >= 0.0 && alpha <= 1.0, "hge_scale_apply: alpha %g not in [0, 1] "
              "(hg2v_weighting.py:331-332)", alpha);
  HGE_REQUIRE(lo <= hi, "hge_scale_apply: min %g > max %g", lo, hi);
  if (n == 0) return HGE_OK;
  HGE_CUDA(cudaSetDevice(ctx->device));
  Staged<float> s_v;
  HGE_TRY(s_v.init(ctx, values, (size_t)n, mem, true, true));
  int32_t* mm = nullptr;
  HGE_TRY(hge_dev_alloc(ctx, &mm, 2));
  const int32_t h[2] = {hge_enc(lo), hge_enc(hi)};
  cudaError_t e = cudaMemcpyAsync(mm, h, sizeof(h), cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) {
    k_scale_transform<<<grid_for(ctx, n, kBlock * 8), kBlock, 0, ctx->stream>>>(
        n, s_v.dev, mm, (float)alpha, (float)(1.0 - alpha));
    ctx->launches++;
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);   // h is on this stack frame
  hge_dev_free(ctx, mm);
  if (e != cudaSuccess) {
    hge_set_error("hge_scale_apply: %s", cudaGetErrorString(e));
    return HGE_ERR_CUDA;
  }
  return s_v.finish();
}

int hge_row_span(hge_ctx* ctx, hge_incidence* inc, const float* xn, const float* xe, int R,
                 int side, float* span, int mem) {
  HGE_REQUIRE(ctx && inc && xn && xe && span, "hge_row_span: NULL argument");
  HGE_REQUIRE(R >= 1 && R <= 1024, "hge_row_span: dimension %d not in [1, 1024]", R);
  HGE_REQUIRE(side == 0 || side == 1, "hge_row_span: side must be 0 or 1");
  HGE_CUDA(cudaSetDevice(ctx->device));
  const HgeHalfSchedule& half = side == 0 ? inc->node_half : inc->edge_half;
  Staged<float> s_xn, s_xe, s_out;
  HGE_TRY(s_xn.init(ctx, xn, (size_t)inc->N * R, mem, true, false));
  HGE_TRY(s_xe.init(ctx, xe, (size_t)inc->E * R, mem, true, false));
  HGE_TRY(s_out.init(ctx, span, (size_t)half.rows, mem, false, true));
  PaddedRows pn, pe;
  HGE_TRY(pn.init(ctx, s_xn.dev, inc->N, R));
  HGE_TRY(pe.init(ctx, s_xe.dev, inc->E, R));
  const int ld4 = ((R + 3) & ~3) / 4;
  const float4* self = side == 0 ? pn.rows4 : pe.rows4;
  const float4* other = side == 0 ? pe.rows4 : pn.rows4;
  const int grid = grid_for(ctx, half.rows, kBlock / 32);
  HGE_DISPATCH_LPR(lanes_per_row(ld4),
                   (k_row_span<L><<<grid, kBlock, 0, ctx->stream>>>(half.rows, half.ptr, half.idx, self,
                                                                  other, ld4, R, s_out.dev)));
  HGE_CHECK_LAUNCH(ctx);
  return s_out.finish();
}

int hge_same_type_prob(hge_ctx* ctx, hge_incidence* inc, int side, const float* w,
                       const int32_t* pi, const int32_t* pj, int64_t num_pairs, float* prob,
                       int mem) {
  HGE_REQUIRE(ctx && inc && w && prob, "hge_same_type_prob: NULL argument");
  HGE_REQUIRE(side == 0 || side == 1, "hge_same_type_prob: side must be 0 or 1");
  HGE_REQUIRE(num_pairs >= 0 && (num_pairs == 0 || (pi && pj)), "hge_same_type_prob: bad pairs");
  if (num_pairs == 0) return HGE_OK;
  HGE_CUDA(cudaSetDevice(ctx->device));
  const HgeHalfSchedule& half = side == 0 ? inc->node_half : inc->edge_half;
  bool ok = false;
  HGE_TRY(pairs_in_range(ctx, num_pairs, pi, half.rows, pj, half.rows, mem, &ok));
  HGE_REQUIRE(ok, "hge_same_type_prob: a pair names a row outside [0, %d)", half.rows);
  Staged<float> s_w, s_out;
  Staged<int32_t> s_i, s_j;
  HGE_TRY(s_w.init(ctx, w, (size_t)half.nnz, mem, true, false));
  HGE_TRY(s_i.init(ctx, pi, (size_t)num_pairs, mem, true, false));
  HGE_TRY(s_j.init(ctx, pj, (size_t)num_pairs, mem, true, false));
  HGE_TRY(s_out.init(ctx, prob, (size_t)num_pairs, mem, false, true));
  const double mean_deg = (double)half.nnz / std::max(1, half.rows);
  if (mean_deg <= 24.0) {
    const int grid = grid_for(ctx, num_pairs, kBlock / 8);
    k_same_type_prob<8><<<grid, kBlock, 0, ctx->stream>>>(num_pairs, half.ptr, half.idx, s_w.dev,
                                                         s_i.dev, s_j.dev, s_out.dev);
  } else {
    const int grid = grid_for(ctx, num_pairs, kBlock / 32);
    k_same_type_prob<32><<<grid, kBlock, 0, ctx->stream>>>(num_pairs, half.ptr, half.idx, s_w.dev,
                                                          s_i.dev, s_j.dev, s_out.dev);
  }
  HGE_CHECK_LAUNCH(ctx);
  return s_out.finish();
}

int hge_diff_type_prob(hge_ctx* ctx, hge_incidence* inc, const float* w_e2n, const int32_t* pn,
                       const int32_t* pe, int64_t num_pairs, float* prob, int mem) {
  HGE_REQUIRE(ctx && inc && w_e2n && prob, "hge_diff_type_prob: NULL argument");
  HGE_REQUIRE(num_pairs >= 0 && (num_pairs == 0 || (pn && pe)), "hge_diff_type_prob: bad pairs");
  if (num_pairs == 0) return HGE_OK;
  HGE_CUDA(cudaSetDevice(ctx->device));
  bool ok = false;
  HGE_TRY(pairs_in_range(ctx, num_pairs, pn, inc->N, pe, inc->E, mem, &ok));
  HGE_REQUIRE(ok, "hge_diff_type_prob: a pair names a node outside [0, %d) or an edge outside [0, %d)",
              inc->N, inc->E);
  Staged<float> s_w, s_out;
  Staged<int32_t> s_n, s_e;
  HGE_TRY(s_w.init(ctx, w_e2n, (size_t)inc->edge_half.nnz, mem, true, false));
  HGE_TRY(s_n.init(ctx, pn, (size_t)num_pairs, mem, true, false));
  HGE_TRY(s_e.init(ctx, pe, (size_t)num_pairs, mem, true, false));
  HGE_TRY(s_out.init(ctx, prob, (size_t)num_pairs, mem, false, true));
  const int grid = grid_for(ctx, num_pairs, kBlock / 32);
  k_diff_type_prob<<<grid, kBlock, 0, ctx->stream>>>(num_pairs, inc->n2e_ptr, inc->n2e_idx,
                                                     inc->e2n_ptr, inc->e2n_idx, s_w.dev, s_n.dev,
                                                     s_e.dev, s_out.dev);
  HGE_CHECK_LAUNCH(ctx);
  return s_out.finish();
}

}  // extern "C"
