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
#include "hge_pairs.cuh"

namespace {

constexpr int kBlock = 256;
constexpr unsigned kFull = 0xffffffffu;

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
  DevBuf<float> padded;
  const float4* rows4 = nullptr;
  explicit PaddedRows(const hge_ctx* c) : padded(c) {}
  int init(hge_ctx* ctx, const float* x, int64_t rows, int R) {
    if (R % 4 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0) {
      rows4 = reinterpret_cast<const float4*>(x);
      return HGE_OK;
    }
    const int ld = (R + 3) & ~3;
    HGE_TRY(padded.alloc((size_t)rows * ld));
    k_pad_rows<<<grid_for(ctx, rows * ld, kBlock), kBlock, 0, ctx->stream>>>(rows, R, ld, x, padded.p);
    HGE_CHECK_LAUNCH(ctx);
    rows4 = reinterpret_cast<const float4*>(padded.p);
    return HGE_OK;
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

// The kernels above trust their pair indices: k_same_type_prob and k_diff_type_prob read row
// pointers at them, k_pair_l2 skips a negative one and leaves its output unwritten.  The entry
// points therefore check every index with pairs_in_range (hge_pairs.cuh) first.

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

int build_segments(hge_ctx* ctx, int32_t rows, const int64_t* d_ptr, int64_t nnz, DevBuf<Segment>& segs,
                   int64_t* count) {
  *count = 0;
  if (rows <= 0) return HGE_OK;
  DevBuf<int64_t> counts(ctx), offset(ctx);
  DevBuf<char> temp(ctx);
  HGE_TRY(counts.alloc((size_t)rows + 1));
  HGE_TRY(offset.alloc((size_t)rows + 1));
  HGE_CUDA(cudaMemsetAsync(counts.p + rows, 0, sizeof(int64_t), ctx->stream));
  const int grid = grid_for(ctx, rows, kBlock);
  k_segment_counts<<<grid, kBlock, 0, ctx->stream>>>(rows, d_ptr, counts.p);
  HGE_CHECK_LAUNCH(ctx);
  size_t temp_bytes = 0;
  HGE_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, temp_bytes, counts.p, offset.p, rows + 1, ctx->stream));
  HGE_TRY(temp.alloc(temp_bytes));
  HGE_CUDA(cub::DeviceScan::ExclusiveSum(temp.p, temp_bytes, counts.p, offset.p, rows + 1, ctx->stream));
  ctx->launches += 1;
  // the segment count is bounded without a read-back: every row adds at most one partial segment
  const int64_t bound = nnz / kSegment + rows;
  HGE_TRY(segs.alloc((size_t)bound));
  k_segment_write<<<grid, kBlock, 0, ctx->stream>>>(rows, d_ptr, offset.p, segs.p);
  HGE_CHECK_LAUNCH(ctx);
  return read_back(ctx, offset.p + rows, count, 1);
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
  Staged<float> s_xn(ctx), s_xe(ctx), s_out(ctx);
  HGE_TRY(s_xn.init(xn, (size_t)inc->N * R, mem, true, false));
  HGE_TRY(s_xe.init(xe, (size_t)inc->E * R, mem, true, false));
  HGE_TRY(s_out.init(dist, (size_t)half.nnz, mem, false, true));
  PaddedRows pn(ctx), pe(ctx);
  HGE_TRY(pn.init(ctx, s_xn.dev, inc->N, R));
  HGE_TRY(pe.init(ctx, s_xe.dev, inc->E, R));
  DevBuf<Segment> segs(ctx);
  int64_t nseg = 0;
  HGE_TRY(build_segments(ctx, half.rows, half.ptr, half.nnz, segs, &nseg));
  const int ld4 = ((R + 3) & ~3) / 4;
  const float max_dist = (float)sqrt((double)R);
  const float4* self = order == 0 ? pn.rows4 : pe.rows4;
  const float4* other = order == 0 ? pe.rows4 : pn.rows4;
  const int grid = grid_for(ctx, nseg, kBlock / 32);
  HGE_DISPATCH_LPR(lanes_per_row(ld4),
                   (k_incidence_l2<L><<<grid, kBlock, 0, ctx->stream>>>(
                       nseg, segs.p, half.idx, self, other, ld4, max_dist, as_weight, s_out.dev)));
  HGE_CHECK_LAUNCH(ctx);
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
  // xb == xa (distances inside one table) is staged and padded once
  const bool same = xb == xa;
  Staged<float> s_xa(ctx), s_xb(ctx), s_out(ctx);
  Staged<int32_t> s_ia(ctx), s_ib(ctx);
  HGE_TRY(s_xa.init(xa, (size_t)rows_a * R, mem, true, false));
  if (!same) HGE_TRY(s_xb.init(xb, (size_t)rows_b * R, mem, true, false));
  HGE_TRY(s_ia.init(ia, (size_t)num_pairs, mem, true, false));
  HGE_TRY(s_ib.init(ib, (size_t)num_pairs, mem, true, false));
  HGE_TRY(s_out.init(dist, (size_t)num_pairs, mem, false, true));
  PaddedRows pa(ctx), pb(ctx);
  HGE_TRY(pa.init(ctx, s_xa.dev, rows_a, R));
  if (!same) HGE_TRY(pb.init(ctx, s_xb.dev, rows_b, R));
  const float4* rows_b4 = same ? pa.rows4 : pb.rows4;
  const int ld4 = ((R + 3) & ~3) / 4;
  const int grid = grid_for(ctx, (num_pairs + 31) / 32, kBlock / 32);
  HGE_DISPATCH_LPR(lanes_per_row(ld4),
                   (k_pair_l2<L><<<grid, kBlock, 0, ctx->stream>>>(
                       num_pairs, s_ia.dev, s_ib.dev, pa.rows4, rows_b4, ld4, s_out.dev)));
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
  Staged<float> s_v(ctx);
  HGE_TRY(s_v.init(values, (size_t)n, mem, true, true));
  DevBuf<int32_t> mm(ctx);
  HGE_TRY(mm.alloc(2));
  k_minmax_init<<<1, 1, 0, ctx->stream>>>(mm.p);
  ctx->launches++;
  const int grid = grid_for(ctx, n, kBlock * 8);
  k_minmax<<<grid, kBlock, 0, ctx->stream>>>(n, s_v.dev, mm.p);
  ctx->launches++;
  k_scale_transform<<<grid, kBlock, 0, ctx->stream>>>(n, s_v.dev, mm.p, (float)alpha,
                                                      (float)(1.0 - alpha));
  HGE_CHECK_LAUNCH(ctx);
  if (minmax) {
    int32_t h[2];
    HGE_TRY(read_back(ctx, mm.p, h, 2));
    minmax[0] = hge_dec(h[0]);
    minmax[1] = hge_dec(h[1]);
  }
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
  Staged<float> s_v(ctx);
  HGE_TRY(s_v.init(values, (size_t)n, mem, true, false));
  DevBuf<int32_t> mm(ctx);
  HGE_TRY(mm.alloc(2));
  k_minmax_init<<<1, 1, 0, ctx->stream>>>(mm.p);
  ctx->launches++;
  k_minmax<<<grid_for(ctx, n, kBlock * 8), kBlock, 0, ctx->stream>>>(n, s_v.dev, mm.p);
  HGE_CHECK_LAUNCH(ctx);
  int32_t h[2];
  HGE_TRY(read_back(ctx, mm.p, h, 2));
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
  Staged<float> s_v(ctx);
  HGE_TRY(s_v.init(values, (size_t)n, mem, true, true));
  DevBuf<int32_t> mm(ctx);
  HGE_TRY(mm.alloc(2));
  const int32_t h[2] = {hge_enc(lo), hge_enc(hi)};
  HGE_CUDA(cudaMemcpyAsync(mm.p, h, sizeof(h), cudaMemcpyHostToDevice, ctx->stream));
  k_scale_transform<<<grid_for(ctx, n, kBlock * 8), kBlock, 0, ctx->stream>>>(
      n, s_v.dev, mm.p, (float)alpha, (float)(1.0 - alpha));
  HGE_CHECK_LAUNCH(ctx);
  HGE_CUDA(cudaStreamSynchronize(ctx->stream));   // h is on this stack frame
  return s_v.finish();
}

int hge_row_span(hge_ctx* ctx, hge_incidence* inc, const float* xn, const float* xe, int R,
                 int side, float* span, int mem) {
  HGE_REQUIRE(ctx && inc && xn && xe && span, "hge_row_span: NULL argument");
  HGE_REQUIRE(R >= 1 && R <= 1024, "hge_row_span: dimension %d not in [1, 1024]", R);
  HGE_REQUIRE(side == 0 || side == 1, "hge_row_span: side must be 0 or 1");
  HGE_CUDA(cudaSetDevice(ctx->device));
  const HgeHalfSchedule& half = side == 0 ? inc->node_half : inc->edge_half;
  Staged<float> s_xn(ctx), s_xe(ctx), s_out(ctx);
  HGE_TRY(s_xn.init(xn, (size_t)inc->N * R, mem, true, false));
  HGE_TRY(s_xe.init(xe, (size_t)inc->E * R, mem, true, false));
  HGE_TRY(s_out.init(span, (size_t)half.rows, mem, false, true));
  PaddedRows pn(ctx), pe(ctx);
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
  Staged<float> s_w(ctx), s_out(ctx);
  Staged<int32_t> s_i(ctx), s_j(ctx);
  HGE_TRY(s_w.init(w, (size_t)half.nnz, mem, true, false));
  HGE_TRY(s_i.init(pi, (size_t)num_pairs, mem, true, false));
  HGE_TRY(s_j.init(pj, (size_t)num_pairs, mem, true, false));
  HGE_TRY(s_out.init(prob, (size_t)num_pairs, mem, false, true));
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
  Staged<float> s_w(ctx), s_out(ctx);
  Staged<int32_t> s_n(ctx), s_e(ctx);
  HGE_TRY(s_w.init(w_e2n, (size_t)inc->edge_half.nnz, mem, true, false));
  HGE_TRY(s_n.init(pn, (size_t)num_pairs, mem, true, false));
  HGE_TRY(s_e.init(pe, (size_t)num_pairs, mem, true, false));
  HGE_TRY(s_out.init(prob, (size_t)num_pairs, mem, false, true));
  const int grid = grid_for(ctx, num_pairs, kBlock / 32);
  k_diff_type_prob<<<grid, kBlock, 0, ctx->stream>>>(num_pairs, inc->n2e_ptr, inc->n2e_idx,
                                                     inc->e2n_ptr, inc->e2n_idx, s_w.dev, s_n.dev,
                                                     s_e.dev, s_out.dev);
  HGE_CHECK_LAUNCH(ctx);
  return s_out.finish();
}

}  // extern "C"
