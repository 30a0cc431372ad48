// k_sweep: one half-sweep of the algebraic-distance relaxation over a packed gather stream.
//
// Reference arithmetic (algebraic_distance.py:34-51): row a <- (x_a + sum_b w_b x_b / sum_b w_b) / 2
// with w_b = 1 / deg(b); storage, lazy rescale and fused min / max as described at the top of
// hge_algdist.cu.  What this kernel changes against the first-generation k_half_sweep is how a
// warp is fed (ncu source page of that kernel, profiles/r2_half_sweep.md: 256 issued
// instructions per 8 gathered rows per lane, 26 % of the stall samples waiting for the column
// ids of the next rows, gathers drained to zero at the end of every group of rows):
//
//   * the column ids are read from a stream that hge_sched_stream laid out in exactly the order
//     the warp consumes them (HgeStream, hge_incidence.cuh): one coalesced 16 G-byte load per
//     step of 4 gathers per lane, addresses that depend on nothing but a counter, so the ids are
//     loaded 6 steps ahead of their use and never wait for a row descriptor;
//   * slots hold absolute row indices of one allocation, padding is a row of zeros: a gather is
//     one multiply-add, one 128-bit load and two packed adds (FADD2), no predicate, no select;
//   * a row's own old value is the last slot of its last step, so it arrives through the same
//     pipeline instead of a dependent load per row;
//   * a warp issues two steps (8 rows per lane) back to back and only then adds them up; a group
//     of rows may end after either step, and the loads never sit inside a branch;
//   * every warp owns one contiguous, cost-balanced piece of the unit list, two waves of blocks.
#include <algorithm>

#include "hge_incidence.cuh"
#include "hge_sweep.cuh"

namespace {

constexpr int kBlock = 256;
constexpr int kWarps = kBlock / 32;
constexpr unsigned kFull = 0xffffffffu;
constexpr int kMinBlocks = 4;          // resident blocks per SM the register budget is cut for
constexpr int kPrefetchSteps = 24;     // distance, in steps, of the L2 prefetch of the id stream

// A gathered float4 is one 128-bit virtual register from the load to the add.  ptxas gives such
// a register an aligned quad, so the software-pipelined (loop-carried) slots are loaded in place;
// with four 32-bit or two 64-bit registers per slot it homed the slots in unaligned registers,
// loaded into an aligned temporary and copied -- and the copy waits for the load it follows,
// which serialises the very gathers the pipeline is there to overlap.  The accumulator is two
// 64-bit pairs: FADD2 adds both halves of a pair in one issue slot.
typedef unsigned __int128 quad;
struct pair4 {
  unsigned long long x, y;
};
__device__ __forceinline__ quad ldg_quad(const void* p) {
  quad v;
  // volatile: the compiler must not sink a load into the branch that consumes it
  asm volatile("ld.global.nc.b128 %0, [%1];" : "=q"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ void f4_acc(pair4& a, const quad& v) {
  asm("{\n\t.reg .b64 lo, hi;\n\tmov.b128 {lo, hi}, %2;\n\tadd.rn.f32x2 %0, %0, lo;\n\tadd.rn.f32x2 %1, %1, hi;\n\t}"
      : "+l"(a.x), "+l"(a.y)
      : "q"(v));
}
__device__ __forceinline__ float4 unpack4(const pair4& p) {
  float4 f;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(f.x), "=f"(f.y) : "l"(p.x));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(f.z), "=f"(f.w) : "l"(p.y));
  return f;
}
__device__ __forceinline__ float4 unpack4(const quad& v) {
  pair4 p;
  asm("mov.b128 {%0, %1}, %2;" : "=l"(p.x), "=l"(p.y) : "q"(v));
  return unpack4(p);
}
__device__ __forceinline__ pair4 pair4_zero() {
  pair4 p;
  p.x = 0ull;
  p.y = 0ull;
  return p;
}

// 16-byte asynchronous copy global -> shared (LDGSTS): no staging register, so nothing waits for it
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem)),
               "l"(gmem)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

__device__ __forceinline__ void kahan_add4(float4& s, float4& c, const float4& v) {
  float y, t;
  y = v.x - c.x; t = s.x + y; c.x = (t - s.x) - y; s.x = t;
  y = v.y - c.y; t = s.y + y; c.y = (t - s.y) - y; s.y = t;
  y = v.z - c.z; t = s.z + y; c.z = (t - s.z) - y; s.z = t;
  y = v.w - c.w; t = s.w + y; c.w = (t - s.w) - y; s.w = t;
}

template <int LPR, int MODE>
__global__ void __launch_bounds__(kBlock, kMinBlocks) k_sweep(const HgeSweepArgs a) {
  constexpr int G = 32 / LPR;                      // lane groups (rows in flight) per warp
  constexpr int K = LPR >= 4 ? 1 : 4 / LPR;        // id registers per lane and step
  constexpr int D = kStreamStepAlign;              // id look-ahead ring = unroll, in steps
  constexpr bool kOwn = MODE == kSweepNode || MODE == kSweepEdge;

  // per-thread constants of the lazily applied affine map and the running min / max of the rows
  // this thread produced: shared memory instead of 16 registers (touched once per finished row;
  // 64 registers do not hold them without spills)
  __shared__ float4 s_state[kOwn ? 4 * kBlock + 1 : 1];
  __shared__ float4 s_min[kOwn ? kWarps : 1][LPR];
  __shared__ float4 s_max[kOwn ? kWarps : 1][LPR];
  // row descriptors of the short rows, two halves of 32 per warp, filled by asynchronous copies
  // 32 / G .. 64 / G groups of rows ahead of their use
  __shared__ int4 s_items[kWarps][2][32];
  float4* const sst = s_state + threadIdx.x;

  const int lane = threadIdx.x & 31;
  const int gl = lane & (LPR - 1);
  const int g = lane / LPR;
  const int warp = threadIdx.x >> 5;
  const int slab = blockIdx.y;                     // column slab of 32 float4 (R > 128 only)
  const int ld4 = a.ld4;
  const int c4 = slab * LPR + gl;                  // this lane's float4 column
  const bool active = c4 < ld4;                    // lanes beyond the row gather a valid column
  const int c4c = active ? c4 : ld4 - 1;           // and store nothing
  const char* const basel = reinterpret_cast<const char*>(a.base + c4c);
  const uint32_t row_bytes = (uint32_t)ld4 * 16u;

  if (kOwn) {
    float lo[4] = {0.f, 0.f, 0.f, 0.f}, inv[4] = {1.f, 1.f, 1.f, 1.f};
    if (a.mm_prev && active) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int col = c4 * 4 + j;
        if (col < a.R) {
          lo[j] = hge_dec(a.mm_prev[col]);
          inv[j] = 1.0f / (hge_dec(a.mm_prev[ld4 * 4 + col]) - lo[j]);
        }
      }
    }
    // x' = c1 y + (c2 acc - c3):  c1 = inv deg / 2;  node half (the gathered rows carry the map
    // too): c2 = inv invs / 2, c3 = inv lo;  edge half: c2 = invs / 2, c3 = inv lo / 2
    const float h = MODE == kSweepNode ? 1.0f : 0.5f;
    sst[0] = make_float4(inv[0], inv[1], inv[2], inv[3]);
    sst[kBlock] = make_float4(h * (lo[0] * inv[0]), h * (lo[1] * inv[1]), h * (lo[2] * inv[2]), h * (lo[3] * inv[3]));
    const float inf = __int_as_float(0x7f800000);
    sst[2 * kBlock] = make_float4(inf, inf, inf, inf);
    sst[3 * kBlock] = make_float4(-inf, -inf, -inf, -inf);
  }

  // ---- feeding ----------------------------------------------------------------------------
  auto issue_one = [&](quad& v, const int (&r)[K], const int j) {
    const int c = __shfl_sync(kFull, r[K == 1 ? 0 : j / LPR], K == 1 ? j : j % LPR, LPR);
    v = ldg_quad(basel + (size_t)(uint32_t)c * row_bytes);
  };
  auto issue = [&](quad (&v)[4], const int (&r)[K]) {
#pragma unroll
    for (int j = 0; j < 4; ++j) issue_one(v[j], r, j);
  };
  // ---- finishing ----------------------------------------------------------------------------
  // called by the lanes that own (row, c4); acc is the full gathered sum of the row
  auto finish_row = [&](int row, float degf, float invs, const float4& yown, const float4& acc) {
    const size_t off = (size_t)row * ld4 + c4;
    if (MODE == kSweepPush) {
      // fused reduce-scatter: the partial row goes straight into the owning GPU's staging block
      int owner;
      int32_t idx;
      a.push_map.locate(row, owner, idx);
      float4* dst = a.push_stage[owner] + ((size_t)a.push_rank * a.push_map.sub_rows + idx) * ld4 + c4;
      *dst = acc;
    } else if (MODE == kSweepRawAdd) {
      float4 prev = a.raw[off];
      prev.x += acc.x; prev.y += acc.y; prev.z += acc.z; prev.w += acc.w;
      a.raw[off] = prev;
    } else if (MODE == kSweepRaw) {
      a.raw[off] = acc;
    } else {
      const float4 inv = sst[0], c3 = sst[kBlock];
      const float hd = 0.5f * degf, hs = 0.5f * invs;
      float4 x;
      if (MODE == kSweepNode) {
        x.x = fmaf(inv.x * hd, yown.x, fmaf(inv.x * hs, acc.x, -c3.x));
        x.y = fmaf(inv.y * hd, yown.y, fmaf(inv.y * hs, acc.y, -c3.y));
        x.z = fmaf(inv.z * hd, yown.z, fmaf(inv.z * hs, acc.z, -c3.z));
        x.w = fmaf(inv.w * hd, yown.w, fmaf(inv.w * hs, acc.w, -c3.w));
      } else {
        x.x = fmaf(inv.x * hd, yown.x, fmaf(hs, acc.x, -c3.x));
        x.y = fmaf(inv.y * hd, yown.y, fmaf(hs, acc.y, -c3.y));
        x.z = fmaf(inv.z * hd, yown.z, fmaf(hs, acc.z, -c3.z));
        x.w = fmaf(inv.w * hd, yown.w, fmaf(hs, acc.w, -c3.w));
      }
      const float w = __frcp_rn(degf);
      const float4 y = make_float4(x.x * w, x.y * w, x.z * w, x.w * w);
      // streaming (evict-first) store: the rows a half writes compete for L2 with the table it
      // gathers from (config 2, profiles/r2_half_sweep.md: 0.3069 -> 0.3042 ms per sweep)
      __stcs(a.own + off, y);
      // padding columns (>= R) stay 0 and are not published, so no per-column mask here
      float4 lo4 = sst[2 * kBlock], hi4 = sst[3 * kBlock];
      lo4.x = fminf(lo4.x, x.x); hi4.x = fmaxf(hi4.x, x.x);
      lo4.y = fminf(lo4.y, x.y); hi4.y = fmaxf(hi4.y, x.y);
      lo4.z = fminf(lo4.z, x.z); hi4.z = fmaxf(hi4.z, x.z);
      lo4.w = fminf(lo4.w, x.w); hi4.w = fmaxf(hi4.w, x.w);
      sst[2 * kBlock] = lo4;
      sst[3 * kBlock] = hi4;
    }
  };
  auto reduce_groups = [&](float4& v) {
#pragma unroll
    for (int off = LPR; off < 32; off <<= 1) {
      v.x += __shfl_xor_sync(kFull, v.x, off);
      v.y += __shfl_xor_sync(kFull, v.y, off);
      v.z += __shfl_xor_sync(kFull, v.z, off);
      v.w += __shfl_xor_sync(kFull, v.w, off);
    }
  };
  auto load_own = [&](int row) -> float4 {
    return __ldcs(a.own + (size_t)row * ld4 + c4);
  };

  // ---- one piece of one schedule ----------------------------------------------------------------
  // (kept as a lambda: unwrapped, the same code gets a different register and stack-slot
  // allocation in every instantiation)
  auto run_piece = [&](const HgeSweepSrc& src, const int pi) {
  const int32_t* const stream0 = src.stream;
  const int32_t* const sp = stream0 + g * 4 + (K == 1 ? (gl & 3) : gl);   // this lane's column of the id stream
  auto load_ids = [&](uint32_t step, int (&r)[K]) {
#pragma unroll
    for (int k = 0; k < K; ++k) r[k] = __ldcs(sp + (size_t)step * (4 * G) + LPR * k);
  };
  // the id stream is read once, front to back: one lane per warp asks L2 for the line a few
  // steps ahead, so the register ring above only has to cover an L2 hit
  auto prefetch_ids = [&](uint32_t step) {
    if (lane == 0)
      asm volatile("prefetch.global.L2 [%0];" ::"l"(stream0 + (size_t)(step + kPrefetchSteps) * (4 * G)));
  };
  const int32_t u0 = src.piece[pi], u1 = src.piece[pi + 1];

  // ---- chunks of long rows: the G groups share the chunk ------------------------------------
  for (int32_t u = u0; u < min(u1, src.n_chunks); ++u) {
    const int2 ch = src.chunks[u];
    const HgeHeavyRow hr = src.hrows[ch.x];
    const uint32_t pos = src.uoff[u];
    const uint32_t total = src.uoff[u + 1] - pos;
    int r[D][K];
#pragma unroll
    for (int d = 0; d < D; ++d) load_ids(pos + d, r[d]);
    pair4 accp = pair4_zero();
    for (uint32_t i = 0; i < total; i += D) {
#pragma unroll
      for (int d = 0; d < D; d += 2) {
        // one round: two steps issued back to back, then added up.  Loads and adds sit in one
        // basic block (no branch between them, nothing carried around the loop), so every
        // gathered quad is added from the registers it was loaded into.  A chunk's steps are
        // padded with the zero row to a multiple of the unroll, so nothing needs a guard.
        quad va[4], vb[4];
        issue(va, r[d]);
        issue(vb, r[d + 1]);
        load_ids(pos + i + d + D, r[d]);
        load_ids(pos + i + d + 1 + D, r[d + 1]);
        if (d == 0) prefetch_ids(pos + i);
        f4_acc(accp, va[0]);
        f4_acc(accp, va[1]);
        f4_acc(accp, va[2]);
        f4_acc(accp, va[3]);
        f4_acc(accp, vb[0]);
        f4_acc(accp, vb[1]);
        f4_acc(accp, vb[2]);
        f4_acc(accp, vb[3]);
      }
    }
    float4 acc = unpack4(accp);
    // single-chunk rows are finished here; multi-chunk rows park the chunk sum, and the last
    // chunk of the row to arrive adds the parked sums in chunk order (deterministic)
    reduce_groups(acc);
    if (hr.nchunks == 1) {
      if (g == 0 && active) {
        float4 yown = hge_f4_zero();
        if (kOwn) yown = load_own(hr.row);
        finish_row(hr.row, (float)hr.deg, hr.invs, yown, acc);
      }
      continue;
    }
    if (g == 0 && active) __stcg(src.partials + (size_t)(hr.partial_base + ch.y) * ld4 + c4, acc);
    __threadfence();
    __syncwarp();
    int prev = 0;
    if (lane == 0) prev = atomicAdd(src.counters + (size_t)slab * src.n_hrows + ch.x, 1);
    prev = __shfl_sync(kFull, prev, 0);
    if (prev != hr.nchunks - 1) continue;
    __threadfence();
    float4 yown = hge_f4_zero();
    if (kOwn && g == 0 && active) yown = load_own(hr.row);
    float4 tot = hge_f4_zero(), tcomp = hge_f4_zero();
    for (int k = g; k < hr.nchunks; k += G)
      if (active) kahan_add4(tot, tcomp, __ldcg(src.partials + (size_t)(hr.partial_base + k) * ld4 + c4));
    tot = make_float4(tot.x - tcomp.x, tot.y - tcomp.y, tot.z - tcomp.z, tot.w - tcomp.w);
    reduce_groups(tot);
    if (g == 0 && active) finish_row(hr.row, (float)hr.deg, hr.invs, yown, tot);
    if (lane == 0) src.counters[(size_t)slab * src.n_hrows + ch.x] = 0;   // ready for the next launch
  }

  // ---- groups of G short rows: group g gathers row g ------------------------------------------
  const int32_t q0 = max(u0, src.n_chunks);
  if (q0 < u1) {
    const uint32_t pos = src.uoff[q0];
    const uint32_t total = src.uoff[u1] - pos;
    // descriptor ring: lane l copies item (32 blk + l) of the piece into half (blk & 1)
    int4(*ring)[32] = s_items[warp];
    const int4* const ibase = src.items + (size_t)(q0 - src.n_chunks) * G + lane;
    cp_async16(&ring[0][lane], ibase);
    cp_async_commit();
    cp_async16(&ring[1][lane], ibase + 32);
    cp_async_commit();
    int blk_next = 2;
    int slot = g;                                  // this group's item of the current rows, 0 .. 63
    int r[D][K];
#pragma unroll
    for (int d = 0; d < D; ++d) load_ids(pos + d, r[d]);
    cp_async_wait<1>();
    __syncwarp();
    // A row's own old value is the one load of a round that always comes from DRAM (every row is
    // read once per launch), and a round lasts as long as its slowest load.  The descriptors sit
    // in the ring ahead of their use, so each lane asks L2 for the row of one descriptor half a
    // ring (16 / G .. 48 / G groups of rows) before it is gathered.
    auto prefetch_own = [&](int half) {
      if (kOwn) {
        const int row = ring[half][lane].x;
        if (row >= 0)
          asm volatile("prefetch.global.L2 [%0];" ::"l"(a.own + (size_t)row * ld4 + slab * LPR));
      }
    };
    prefetch_own(0);
    pair4 acc = pair4_zero();
    int left = ring[0][slot].z;
    int groups = u1 - q0;                          // groups of rows left in this piece
    // a group of rows is complete: update / store its rows, move to the next descriptor
    auto finish_group = [&](const quad& own_slot) {
      const int4 it = ring[slot >> 5][slot & 31];
      if (it.x >= 0 && active)
        finish_row(it.x, (float)it.y, __int_as_float(it.w), unpack4(own_slot), unpack4(acc));
      acc = pair4_zero();
      slot += G;
      if ((slot & 31) == g) {
        // entered the other half: its copy was issued at least 32 / G groups ago; the half
        // just left is refilled
        cp_async_wait<0>();
        __syncwarp();
        cp_async16(&ring[((slot >> 5) & 1) ^ 1][lane], ibase + 32 * blk_next);
        cp_async_commit();
        ++blk_next;
        slot &= 63;
      }
      if (kOwn && G <= 16 && (slot & 31) == 16 + g) {
        // half way through this half of the ring: the other half (requested when this one was
        // entered) has landed by now -- ask L2 for the rows it describes
        cp_async_wait<0>();
        __syncwarp();
        prefetch_own(((slot >> 5) & 1) ^ 1);
      }
      left = --groups == 0 ? 0x7fffffff : ring[slot >> 5][slot & 31].z;
    };
    for (uint32_t i = 0; i < total; i += D) {
#pragma unroll
      for (int d = 0; d < D; d += 2) {
        // one round: two steps issued back to back (8 rows per lane in flight), then added up.
        // Nothing is guarded: a piece ends at a group boundary, after its last group `left`
        // never reaches zero again, so the up to D - 1 steps past the end (the next piece's rows
        // or the zero row) are added to an accumulator nobody reads.
        quad va[4], vb[4];
        issue(va, r[d]);
        issue(vb, r[d + 1]);
        load_ids(pos + i + d + D, r[d]);
        load_ids(pos + i + d + 1 + D, r[d + 1]);
        if (d == 0) prefetch_ids(pos + i);
        f4_acc(acc, va[0]);
        f4_acc(acc, va[1]);
        f4_acc(acc, va[2]);
        // the row's own old value rides in the last slot of its last step (kOwn)
        if (--left == 0) {
          if (!kOwn) f4_acc(acc, va[3]);
          finish_group(va[3]);
        } else {
          f4_acc(acc, va[3]);
        }
        f4_acc(acc, vb[0]);
        f4_acc(acc, vb[1]);
        f4_acc(acc, vb[2]);
        if (--left == 0) {
          if (!kOwn) f4_acc(acc, vb[3]);
          finish_group(vb[3]);
        } else {
          f4_acc(acc, vb[3]);
        }
      }
    }
    cp_async_wait<0>();
  }
  };   // run_piece

  run_piece(a.src, blockIdx.x * kWarps + warp);

  // ---- per-column min / max of the rows this block produced -------------------------------------
  if (kOwn) {
    float4 lo4 = sst[2 * kBlock], hi4 = sst[3 * kBlock];
#pragma unroll
    for (int off = LPR; off < 32; off <<= 1) {
      lo4.x = fminf(lo4.x, __shfl_xor_sync(kFull, lo4.x, off));
      lo4.y = fminf(lo4.y, __shfl_xor_sync(kFull, lo4.y, off));
      lo4.z = fminf(lo4.z, __shfl_xor_sync(kFull, lo4.z, off));
      lo4.w = fminf(lo4.w, __shfl_xor_sync(kFull, lo4.w, off));
      hi4.x = fmaxf(hi4.x, __shfl_xor_sync(kFull, hi4.x, off));
      hi4.y = fmaxf(hi4.y, __shfl_xor_sync(kFull, hi4.y, off));
      hi4.z = fmaxf(hi4.z, __shfl_xor_sync(kFull, hi4.z, off));
      hi4.w = fmaxf(hi4.w, __shfl_xor_sync(kFull, hi4.w, off));
    }
    if (g == 0) {
      s_min[warp][gl] = lo4;
      s_max[warp][gl] = hi4;
    }
    __syncthreads();
    if (threadIdx.x < LPR * 4) {
      const int l = threadIdx.x >> 2, j = threadIdx.x & 3;
      const int col = (slab * LPR + l) * 4 + j;
      if (col < a.R) {
        const float inf = __int_as_float(0x7f800000);
        float lo = inf, hi = -inf;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) {
          lo = fminf(lo, reinterpret_cast<const float*>(&s_min[w][l])[j]);
          hi = fmaxf(hi, reinterpret_cast<const float*>(&s_max[w][l])[j]);
        }
        if (lo <= hi) {  // this block produced at least one row
          atomicMin(a.mm_cur + col, hge_enc(lo));
          atomicMax(a.mm_cur + ld4 * 4 + col, hge_enc(hi));
        }
      }
    }
  }
}

template <int LPR>
int launch_mode(const HgeSweepArgs& a, int mode, dim3 grid, cudaStream_t stream) {
  switch (mode) {
    case kSweepNode: k_sweep<LPR, kSweepNode><<<grid, kBlock, 0, stream>>>(a); break;
    case kSweepEdge: k_sweep<LPR, kSweepEdge><<<grid, kBlock, 0, stream>>>(a); break;
    case kSweepRaw: k_sweep<LPR, kSweepRaw><<<grid, kBlock, 0, stream>>>(a); break;
    case kSweepRawAdd: k_sweep<LPR, kSweepRawAdd><<<grid, kBlock, 0, stream>>>(a); break;
    default: k_sweep<LPR, kSweepPush><<<grid, kBlock, 0, stream>>>(a); break;
  }
  return HGE_OK;
}

template <int LPR>
int resident_blocks(int* out) {
  int per_sm = 0;
  HGE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_sweep<LPR, kSweepNode>, kBlock, 0));
  *out = per_sm < 1 ? 1 : per_sm;
  return HGE_OK;
}

}  // namespace

int hge_sweep_resident_blocks(int lpr, int* out) {
  switch (lpr) {
    case 1: return resident_blocks<1>(out);
    case 2: return resident_blocks<2>(out);
    case 4: return resident_blocks<4>(out);
    case 8: return resident_blocks<8>(out);
    case 16: return resident_blocks<16>(out);
    default: return resident_blocks<32>(out);
  }
}

int hge_sweep_launch(hge_ctx* ctx, const HgeSweepArgs& a, int lpr, int mode, int blocks, int slabs) {
  dim3 grid(blocks, slabs);
  switch (lpr) {
    case 1: launch_mode<1>(a, mode, grid, ctx->stream); break;
    case 2: launch_mode<2>(a, mode, grid, ctx->stream); break;
    case 4: launch_mode<4>(a, mode, grid, ctx->stream); break;
    case 8: launch_mode<8>(a, mode, grid, ctx->stream); break;
    case 16: launch_mode<16>(a, mode, grid, ctx->stream); break;
    default: launch_mode<32>(a, mode, grid, ctx->stream); break;
  }
  HGE_CHECK_LAUNCH(ctx);
  return HGE_OK;
}
