// Peer-memory exchange for the row-partitioned relaxation: the collectives of the sharded edge
// half are done by the kernels themselves over NVLink, with no NCCL kernel competing for SMs.
//
//   gather (k_sweep, push mode)        every rank stores the raw partial sum of edge e straight
//                                      into the staging block of e's OWNER  -> reduce-scatter
//   barrier A                          flags in peer memory
//   k_edge_reduce_push                 the owner adds the `world` staged rows in rank order
//                                      (deterministic), blends / rescales the edge row and
//                                      stores the new row into EVERY rank's edge block
//                                                                             -> all-gather
//   barrier B (+ min/max)              every rank pushes its 2 x ld encoded bounds to all
//                                      peers, signals, waits, and reduces them locally
//                                                                   -> all-reduce(min / max)
//
// Rank o owns the edge rows [o sub_rows, (o + 1) sub_rows) (HgeOwnerMap).  Each phase is one
// launch on the context's stream.  Overlapping the owner-side reduce with the gather was tried
// and was slower (profiles/r2_multi_gpu.md, section 4).
//
// Each rank owns one cudaMalloc arena [edge rows | row of zeros | staging | bounds | flags |
// error | local node rows] that the other ranks of the node map through CUDA IPC (the node rows
// are never touched by a peer; they live here so that the packed gather stream of k_sweep can
// address gathered rows, own rows and padding as rows of one allocation).  Barriers are
// sequence-numbered flags: rank r writes seq into flags[r] of every peer (release, system scope)
// and spins on its own flags
// (acquire, system scope) with a wall-clock timeout that raises an error flag instead of
// hanging.  One process per GPU: the spinning kernels of different ranks run on different
// devices.
#include <algorithm>
#include <new>

#include "hge_incidence.cuh"

namespace {

constexpr int kBlock = 256;
constexpr unsigned kFull = 0xffffffffu;
constexpr int kFlagStride = 32;                       // one 128-byte line per flag
constexpr unsigned long long kTimeoutNs = 20ull * 1000 * 1000 * 1000;

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// Barrier over the ranks, optionally carrying the all-reduce(min / max) of this sweep's bounds.
// One block.  mm_cur == nullptr: plain barrier.
__global__ void k_exchange(int rank, int world, uint32_t seq, uint32_t* const* peer_flags,
                           uint32_t* my_flags, int32_t* const* peer_mmx, int32_t* my_mmx,
                           int parity, int ld, int32_t* mm_cur, int* err) {
  const int tid = threadIdx.x;
  const int words = 2 * ld;
  if (mm_cur) {
    // slot layout: mmx[parity][src rank][2][ld]
    for (int i = tid; i < words; i += blockDim.x) {
      const int32_t v = mm_cur[i];
      for (int p = 0; p < world; ++p)
        peer_mmx[p][((size_t)parity * world + rank) * words + i] = v;
    }
  }
  __threadfence_system();
  __syncthreads();
  if (tid < world) st_release_sys(peer_flags[tid] + (size_t)rank * kFlagStride, seq);
  if (tid < world) {
    const unsigned long long t0 = global_ns();
    // sequence numbers only grow; a peer can be at most one barrier ahead
    while ((int32_t)(ld_acquire_sys(my_flags + (size_t)tid * kFlagStride) - seq) < 0) {
      if (global_ns() - t0 > kTimeoutNs) {
        *err = 1;
        break;
      }
    }
  }
  __syncthreads();
  if (mm_cur) {
    for (int i = tid; i < words; i += blockDim.x) {
      const bool is_max = i >= ld;
      int32_t r = is_max ? INT32_MIN : INT32_MAX;
      for (int p = 0; p < world; ++p) {
        const int32_t v = my_mmx[((size_t)parity * world + p) * words + i];
        r = is_max ? max(r, v) : min(r, v);
      }
      mm_cur[i] = r;
    }
  }
}

// Owner-side reduce of the staged partial rows + row update + push of the new row to all ranks.
// row0 = first edge row of this rank's run; every source rank's block of the staging area holds
// sub_rows rows.
template <int LPR>
__global__ void __launch_bounds__(kBlock) k_edge_reduce_push(
    int rank, int world, int32_t row0, int32_t rows, int32_t sub_rows, int R, int ld4,
    const float4* __restrict__ stage, const float4* __restrict__ ye_local,
    float4* const* __restrict__ peer_ye, const int32_t* __restrict__ deg,
    const float* __restrict__ invs, const int32_t* __restrict__ mm_prev, int32_t* mm_cur) {
  constexpr int G = 32 / LPR;
  const int lane = threadIdx.x & 31, gl = lane & (LPR - 1), g = lane / LPR;
  const int warp = threadIdx.x >> 5;
  const int slab = blockIdx.y;
  const int c4 = slab * LPR + gl;
  const bool active = c4 < ld4;
  const int col0 = c4 * 4;
  float lo[4] = {0.f, 0.f, 0.f, 0.f}, inv[4] = {1.f, 1.f, 1.f, 1.f};
  if (mm_prev && active) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (col0 + j < R) {
        lo[j] = hge_dec(mm_prev[col0 + j]);
        inv[j] = 1.0f / (hge_dec(mm_prev[ld4 * 4 + col0 + j]) - lo[j]);
      }
  }
  const float inf = __int_as_float(0x7f800000);
  float vmin[4] = {inf, inf, inf, inf}, vmax[4] = {-inf, -inf, -inf, -inf};
  const int64_t gq = ((int64_t)blockIdx.x * (kBlock / 32) + warp) * G + g;
  const int64_t nq = (int64_t)gridDim.x * (kBlock / 32) * G;
  for (int64_t i = gq; i < rows; i += nq) {
    if (!active) continue;
    const int32_t row = row0 + (int32_t)i;
    float4 acc = hge_f4_zero();
    for (int p = 0; p < world; ++p)     // rank order: the sum is the same on every run
      hge_f4_add(acc, __ldcs(stage + ((size_t)p * sub_rows + i) * ld4 + c4));
    const float4 y = __ldcs(ye_local + (size_t)row * ld4 + c4);
    const float degf = (float)deg[row];
    const float hd = 0.5f * degf, hs = 0.5f * invs[row];
    const float a4[4] = {acc.x, acc.y, acc.z, acc.w}, y4[4] = {y.x, y.y, y.z, y.w};
    float x[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      // same two-FMA update as the single-GPU edge half (finalize_value, gather_affine = false)
      x[j] = fmaf(inv[j] * hd, y4[j], fmaf(hs, a4[j], -0.5f * (lo[j] * inv[j])));
      if (col0 + j < R) {
        vmin[j] = fminf(vmin[j], x[j]);
        vmax[j] = fmaxf(vmax[j], x[j]);
      }
    }
    const float w = __frcp_rn(degf);
    const float4 out = make_float4(x[0] * w, x[1] * w, x[2] * w, x[3] * w);
    for (int p = 0; p < world; ++p) peer_ye[p][(size_t)row * ld4 + c4] = out;
  }
  // block-level min / max, one atomic per column
  __shared__ float smin[kBlock / 32][32 * 4], smax[kBlock / 32][32 * 4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
#pragma unroll
    for (int off = LPR; off < 32; off <<= 1) {
      vmin[j] = fminf(vmin[j], __shfl_xor_sync(kFull, vmin[j], off));
      vmax[j] = fmaxf(vmax[j], __shfl_xor_sync(kFull, vmax[j], off));
    }
    if (g == 0) {
      smin[warp][gl * 4 + j] = vmin[j];
      smax[warp][gl * 4 + j] = vmax[j];
    }
  }
  __syncthreads();
  if (threadIdx.x < LPR * 4) {
    const int col = slab * LPR * 4 + threadIdx.x;
    if (col < R) {
      float l = inf, h = -inf;
      for (int w = 0; w < kBlock / 32; ++w) {
        l = fminf(l, smin[w][threadIdx.x]);
        h = fmaxf(h, smax[w][threadIdx.x]);
      }
      if (l <= h) {
        atomicMin(mm_cur + col, hge_enc(l));
        atomicMax(mm_cur + ld4 * 4 + col, hge_enc(h));
      }
    }
  }
}

int launch_exchange(hge_algdist* st, int sweep_for_mm) {
  hge_p2p* p = st->p2p;
  hge_ctx* ctx = st->ctx;
  p->seq += 1;
  const bool with_mm = sweep_for_mm >= 0;
  int32_t* mm_cur = with_mm ? st->mm + (size_t)sweep_for_mm * 2 * st->ld : nullptr;
  k_exchange<<<1, 128, 0, ctx->stream>>>(
      p->rank, p->world, p->seq, p->d_peer_flags, reinterpret_cast<uint32_t*>(p->base + p->off_flags),
      p->d_peer_mmx, reinterpret_cast<int32_t*>(p->base + p->off_mmx), with_mm ? (sweep_for_mm & 1) : 0,
      st->ld, mm_cur, reinterpret_cast<int*>(p->base + p->off_err));
  HGE_CHECK_LAUNCH(ctx);
  return HGE_OK;
}

}  // namespace

extern "C" {

int hge_p2p_create(hge_ctx* ctx, int rank, int world, int32_t num_local_nodes, int32_t num_edges,
                   int ld, hge_p2p** out) {
  HGE_REQUIRE(ctx && out, "hge_p2p_create: NULL argument");
  *out = nullptr;
  HGE_REQUIRE(num_local_nodes >= 0, "hge_p2p_create: negative node count");
  HGE_REQUIRE(world >= 1 && world <= 16 && rank >= 0 && rank < world,
              "hge_p2p_create: rank %d / world %d not supported (world <= 16)", rank, world);
  HGE_REQUIRE(num_edges > 0 && ld > 0 && ld % 4 == 0, "hge_p2p_create: bad shape");
  HGE_CUDA(cudaSetDevice(ctx->device));
  hge_p2p* p = new (std::nothrow) hge_p2p();
  if (!p) return HGE_ERR_NOMEM;
  p->ctx = ctx;
  p->rank = rank;
  p->world = world;
  p->E = num_edges;
  p->N = num_local_nodes;
  p->ld = ld;
  p->sub_rows = (num_edges + world - 1) / world;
  size_t off = 0;
  p->off_ye = off;
  off = align_up(off + ((size_t)num_edges + 1) * ld * 4, 256);   // + the row of zeros
  p->off_stage = off;
  off = align_up(off + (size_t)world * p->sub_rows * ld * 4, 256);
  p->off_mmx = off;
  off = align_up(off + (size_t)2 * world * 2 * ld * 4, 256);
  p->off_flags = off;
  off = align_up(off + (size_t)world * kFlagStride * 4, 256);
  p->off_err = off;
  off = align_up(off + 256, 256);
  // offsets above are the same on every rank (peers address them); the node rows differ in size
  off = align_up(off, (size_t)ld * 4);
  p->off_yn = off;
  off = align_up(off + (size_t)num_local_nodes * ld * 4, 256);
  p->bytes = off;
  // IPC-exportable memory must come from cudaMalloc, not from the stream-ordered pool
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&p->base), p->bytes);
  if (e != cudaSuccess) {
    hge_set_error("hge_p2p_create: cudaMalloc of %zu bytes failed: %s", p->bytes, cudaGetErrorString(e));
    delete p;
    return HGE_ERR_NOMEM;
  }
  e = cudaMemsetAsync(p->base, 0, p->bytes, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess) {
    hge_set_error("hge_p2p_create: memset failed: %s", cudaGetErrorString(e));
    cudaFree(p->base);
    delete p;
    return HGE_ERR_CUDA;
  }
  p->peer_base[rank] = p->base;
  *out = p;
  return HGE_OK;
}

int hge_p2p_export(hge_p2p* p, void* handle64) {
  HGE_REQUIRE(p && handle64, "hge_p2p_export: NULL argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  HGE_CUDA(cudaSetDevice(p->ctx->device));
  cudaIpcMemHandle_t h;
  HGE_CUDA(cudaIpcGetMemHandle(&h, p->base));
  memcpy(handle64, &h, 64);
  return HGE_OK;
}

int hge_p2p_open_peers(hge_p2p* p, const void* handles) {
  HGE_REQUIRE(p && (handles || p->world == 1), "hge_p2p_open_peers: NULL argument");
  HGE_REQUIRE(!p->peers_open, "hge_p2p_open_peers: already open");
  hge_ctx* ctx = p->ctx;
  HGE_CUDA(cudaSetDevice(ctx->device));
  for (int r = 0; r < p->world; ++r) {
    if (r == p->rank) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, static_cast<const char*>(handles) + (size_t)r * 64, 64);
    void* ptr = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      hge_set_error("hge_p2p_open_peers: cudaIpcOpenMemHandle(rank %d) failed: %s", r,
                    cudaGetErrorString(e));
      cudaGetLastError();
      return HGE_ERR_CUDA;
    }
    p->peer_base[r] = static_cast<char*>(ptr);
  }
  void* tables[4][16];
  for (int r = 0; r < p->world; ++r) {
    tables[0][r] = p->peer_base[r] + p->off_stage;
    tables[1][r] = p->peer_base[r] + p->off_ye;
    tables[2][r] = p->peer_base[r] + p->off_mmx;
    tables[3][r] = p->peer_base[r] + p->off_flags;
  }
  DevBuf<void*> dev[4] = {DevBuf<void*>(ctx), DevBuf<void*>(ctx), DevBuf<void*>(ctx), DevBuf<void*>(ctx)};
  for (int k = 0; k < 4; ++k) {
    HGE_TRY(dev[k].alloc((size_t)p->world));
    HGE_CUDA(cudaMemcpyAsync(dev[k].p, tables[k], sizeof(void*) * p->world, cudaMemcpyHostToDevice,
                             ctx->stream));
  }
  HGE_CUDA(cudaStreamSynchronize(ctx->stream));
  p->d_peer_stage = reinterpret_cast<float4**>(dev[0].release());
  p->d_peer_ye = reinterpret_cast<float4**>(dev[1].release());
  p->d_peer_mmx = reinterpret_cast<int32_t**>(dev[2].release());
  p->d_peer_flags = reinterpret_cast<uint32_t**>(dev[3].release());
  p->peers_open = true;
  return HGE_OK;
}

// Unmaps the peers' arenas.  Every rank must have called this (and a host-level barrier must
// have passed) before any rank destroys its own arena.
int hge_p2p_close_peers(hge_p2p* p) {
  if (!p) return HGE_OK;
  cudaSetDevice(p->ctx->device);
  cudaStreamSynchronize(p->ctx->stream);
  for (int r = 0; r < p->world; ++r)
    if (r != p->rank && p->peer_base[r]) {
      cudaIpcCloseMemHandle(p->peer_base[r]);
      p->peer_base[r] = nullptr;
    }
  return HGE_OK;
}

int hge_p2p_destroy(hge_p2p* p) {
  if (!p) return HGE_OK;
  hge_ctx* ctx = p->ctx;
  hge_p2p_close_peers(p);
  for (cudaEvent_t e : p->marks) cudaEventDestroy(e);
  hge_dev_free(ctx, p->d_peer_stage);
  hge_dev_free(ctx, p->d_peer_ye);
  hge_dev_free(ctx, p->d_peer_mmx);
  hge_dev_free(ctx, p->d_peer_flags);
  cudaFree(p->base);
  delete p;
  return HGE_OK;
}

int hge_algdist_attach_p2p(hge_algdist* st, hge_p2p* p) {
  HGE_REQUIRE(st && p, "hge_algdist_attach_p2p: NULL argument");
  HGE_REQUIRE(st->inc->sharded, "hge_algdist_attach_p2p: the incidence is not a shard");
  HGE_REQUIRE(p->peers_open, "hge_algdist_attach_p2p: hge_p2p_open_peers has not been called");
  HGE_REQUIRE(p->E == st->inc->E && p->N == st->inc->N && p->ld == st->ld && p->ctx == st->ctx,
              "hge_algdist_attach_p2p: arena shape does not match the relaxation state");
  hge_dev_free(st->ctx, st->ybuf);
  st->ye = reinterpret_cast<float*>(p->base + p->off_ye);
  st->yn = reinterpret_cast<float*>(p->base + p->off_yn);
  st->zero_row = (uint32_t)p->E;
  st->p2p = p;
  return HGE_OK;
}

// Owner-side reduce of this rank's run of edge rows.
static int launch_reduce_push(hge_algdist* st, int sweep) {
  hge_p2p* p = st->p2p;
  hge_ctx* ctx = st->ctx;
  hge_incidence* inc = st->inc;
  const int32_t* mm_prev = sweep > 0 ? st->mm + (size_t)(sweep - 1) * 2 * st->ld : nullptr;
  int32_t* mm_cur = st->mm + (size_t)sweep * 2 * st->ld;
  const float4* stage = reinterpret_cast<const float4*>(p->base + p->off_stage);
  const float4* ye = reinterpret_cast<const float4*>(st->ye);
  // rows [rank sub_rows, + sub_rows), clipped at E
  const int64_t r0 = std::min<int64_t>((int64_t)p->rank * p->sub_rows, p->E);
  const int32_t rows = (int32_t)(std::min<int64_t>(r0 + p->sub_rows, p->E) - r0);
  if (rows <= 0) return HGE_OK;
  const int G = 32 / st->lpr;
  int blocks = (int)std::min<int64_t>(((int64_t)rows + (kBlock / 32) * G - 1) / ((kBlock / 32) * G),
                                      (int64_t)ctx->num_sms * 8);
  dim3 grid(std::max(1, blocks), st->slabs);
#define HGE_LAUNCH_RP(L)                                                                              \
  k_edge_reduce_push<L><<<grid, kBlock, 0, ctx->stream>>>(p->rank, p->world, (int32_t)r0, rows, p->sub_rows, \
                                                          st->R, st->ld4, stage, ye, p->d_peer_ye,            \
                                                          inc->edge_half.deg, inc->edge_half.invs, mm_prev, mm_cur)
  switch (st->lpr) {
    case 1: HGE_LAUNCH_RP(1); break;
    case 2: HGE_LAUNCH_RP(2); break;
    case 4: HGE_LAUNCH_RP(4); break;
    case 8: HGE_LAUNCH_RP(8); break;
    case 16: HGE_LAUNCH_RP(16); break;
    default: HGE_LAUNCH_RP(32); break;
  }
#undef HGE_LAUNCH_RP
  HGE_CHECK_LAUNCH(ctx);
  return HGE_OK;
}

// One sweep of the sharded relaxation with the exchange fused into the kernels.
int hge_algdist_sweep_p2p(hge_algdist* st, int sweep) {
  HGE_REQUIRE(st && st->p2p && sweep >= 0 && sweep < st->max_iters,
              "hge_algdist_sweep_p2p: bad argument (attach a peer arena first)");
  hge_p2p* p = st->p2p;
  hge_ctx* ctx = st->ctx;
  HGE_CUDA(cudaSetDevice(ctx->device));
  // phase marks (hge_p2p_set_timing): 6 events per sweep, up to 256 sweeps between two read-outs
  const bool timed = p->timing && p->marks.size() < 6 * 256;
  size_t mark0 = p->marks.size();
  auto mark = [&]() {
    if (!timed) return;
    cudaEvent_t e = nullptr;
    if (cudaEventCreate(&e) == cudaSuccess) {
      cudaEventRecord(e, ctx->stream);
      p->marks.push_back(e);
    }
  };
  mark();
  HGE_TRY(hge_algdist_node_half(st, sweep));
  mark();
  HGE_TRY(hge_internal_edge_push(st, sweep));             // gather + reduce-scatter (peer stores)
  mark();
  HGE_TRY(launch_exchange(st, -1));                       // barrier A
  mark();
  HGE_TRY(launch_reduce_push(st, sweep));                 // owner reduce + all-gather
  mark();
  HGE_TRY(launch_exchange(st, sweep));                    // barrier B + all-reduce(min / max)
  mark();
  if (timed && p->marks.size() != mark0 + 6) {            // an event could not be created: drop the sweep
    while (p->marks.size() > mark0) {
      cudaEventDestroy(p->marks.back());
      p->marks.pop_back();
    }
  }
  return HGE_OK;
}

int hge_p2p_set_timing(hge_p2p* p, int on) {
  HGE_REQUIRE(p, "hge_p2p_set_timing: NULL argument");
  p->timing = on != 0;
  return HGE_OK;
}

// Mean milliseconds per sweep of the five phases recorded since the last call (hge_p2p_set_timing):
// node half, edge gather with the partial rows pushed to their owners, barrier A, owner-side
// reduce + all-gather, barrier B with the min / max exchange.  *sweeps = sweeps averaged over.
int hge_p2p_phase_ms(hge_p2p* p, double* out5, int* sweeps) {
  HGE_REQUIRE(p && out5 && sweeps, "hge_p2p_phase_ms: NULL argument");
  HGE_CUDA(cudaSetDevice(p->ctx->device));
  HGE_CUDA(cudaStreamSynchronize(p->ctx->stream));
  // the first recorded sweep waits for the slowest rank to arrive at all (tens of ms of skew that
  // belong to whatever ran before): it is left out when there are others
  const size_t total = p->marks.size() / 6;
  const size_t first = total > 1 ? 1 : 0;
  const size_t n = total - first;
  for (int k = 0; k < 5; ++k) out5[k] = 0.0;
  for (size_t i = first; i < total; ++i)
    for (int k = 0; k < 5; ++k) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, p->marks[6 * i + k], p->marks[6 * i + k + 1]);
      out5[k] += ms / (double)n;
    }
  for (cudaEvent_t e : p->marks) cudaEventDestroy(e);
  p->marks.clear();
  *sweeps = (int)n;
  return HGE_OK;
}

// 0 = no barrier has timed out so far (synchronises the stream).
int hge_p2p_check(hge_p2p* p) {
  HGE_REQUIRE(p, "hge_p2p_check: NULL argument");
  HGE_CUDA(cudaSetDevice(p->ctx->device));
  int err = 0;
  HGE_CUDA(cudaMemcpyAsync(&err, p->base + p->off_err, sizeof(int), cudaMemcpyDeviceToHost,
                           p->ctx->stream));
  HGE_CUDA(cudaStreamSynchronize(p->ctx->stream));
  if (err) {
    hge_set_error("hge_p2p_check: a peer-memory barrier timed out (a rank is missing or stalled)");
    return HGE_ERR_CUDA;
  }
  return HGE_OK;
}

}  // extern "C"
