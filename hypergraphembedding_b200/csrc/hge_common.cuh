// Shared internals of libhge_b200.so: error reporting, the context object, small device
// helpers.  Not part of the public ABI (see include/hge_b200.h).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>

#include "../../include/hge_b200.h"

void hge_set_error(const char* fmt, ...);

#define HGE_CUDA(call)                                                              \
  do {                                                                              \
    cudaError_t e_ = (call);                                                        \
    if (e_ != cudaSuccess) {                                                        \
      hge_set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #call,              \
                    cudaGetErrorString(e_));                                        \
      return HGE_ERR_CUDA;                                                          \
    }                                                                               \
  } while (0)

#define HGE_CHECK_LAUNCH(ctx)                                                       \
  do {                                                                              \
    (ctx)->launches++;                                                              \
    HGE_CUDA(cudaGetLastError());                                                   \
  } while (0)

#define HGE_REQUIRE(cond, ...)                                                      \
  do {                                                                              \
    if (!(cond)) {                                                                  \
      hge_set_error(__VA_ARGS__);                                                   \
      return HGE_ERR_INVALID;                                                       \
    }                                                                               \
  } while (0)

#define HGE_TRY(call)                                                               \
  do {                                                                              \
    int rc_ = (call);                                                               \
    if (rc_ != HGE_OK) return rc_;                                                  \
  } while (0)

struct hge_ctx {
  int device;
  cudaStream_t stream;
  bool own_stream;
  int num_sms;
  // schedule tuning (hge_ctx_set_tuning)
  int light_max_deg;
  int chunk;
  int blocks_per_sm;
  int trainer_max_clusters;  // cap on the clusters of one hg2v training launch (0: what fits)
  int tile_mb;           // node-range tile of the single-GPU edge half in MB of rows (0 = off)
  int tile_min_mb;       // ... used when the node rows exceed this many MB
  int tile_force;        // min_rows_mb == 0 (tests): tile whatever the edge sizes are
  int64_t launches;
  // ring of 128-byte pinned host slots for small device -> host read-backs (schedule statistics)
  char* pinned_ring;
  int pinned_next;
  // host-buffer calls: dense staging block on the device (grow-only) and a copy stream, so the
  // upload of the initial vectors overlaps the set-up kernels still queued on `stream`
  float* stage;
  size_t stage_floats;
  cudaStream_t copy_stream;
  cudaEvent_t copy_done;    // recorded on copy_stream after an upload into `stage`
  cudaEvent_t stage_idle;   // recorded on `stream` after the last reader / writer of `stage`
  // HGE_FAIL_ALLOC_AT = n > 0: the n-th device allocation after the last tuning reset fails with
  // HGE_ERR_NOMEM, so that the error paths of every entry point can be exercised (0: off)
  int64_t fail_alloc_at;
  mutable int64_t allocs;
};

// Staging block of at least `floats` floats (contents undefined).  Growing it drains the stream.
int hge_ctx_stage(hge_ctx* ctx, size_t floats, float** out);

// One 128-byte pinned host slot; slots are handed out round-robin from a ring of 256, so a slot
// stays untouched until 255 later requests on the same context.  nullptr on failure.
void* hge_ctx_pinned_slot(hge_ctx* ctx);

// hge_shuffle_order (csrc/hge_hg2v_train.cu) with the keys read from the streams of `phase`: the
// epoch orders of every trainer that shuffles its samples.
int hge_shuffle_order_phase(hge_ctx* ctx, uint64_t seed, uint32_t phase, uint32_t epoch, int64_t n,
                            int32_t* order, int mem);

// Device buffers come from the device's stream-ordered memory pool (cudaMallocAsync on the
// context's stream; hge_ctx_create raises the pool's release threshold so freed blocks are
// reused instead of being returned to the driver).  Everything is released explicitly by the
// owning object; all work of a context is queued on one stream, so stream order is enough.
template <typename T>
[[nodiscard]] static inline int hge_dev_alloc(const hge_ctx* ctx, T** p, size_t count) {
  *p = nullptr;
  if (count == 0) count = 1;
  if (ctx->fail_alloc_at > 0 && ++ctx->allocs == ctx->fail_alloc_at) {
    hge_set_error("device allocation %lld failed (HGE_FAIL_ALLOC_AT)", (long long)ctx->allocs);
    return HGE_ERR_NOMEM;
  }
  cudaError_t e = cudaMallocAsync(reinterpret_cast<void**>(p), count * sizeof(T), ctx->stream);
  if (e != cudaSuccess) {
    hge_set_error("cudaMallocAsync of %zu bytes failed: %s", count * sizeof(T),
                  cudaGetErrorString(e));
    cudaGetLastError();
    return e == cudaErrorMemoryAllocation ? HGE_ERR_NOMEM : HGE_ERR_CUDA;
  }
  return HGE_OK;
}

template <typename T>
static inline void hge_dev_free(const hge_ctx* ctx, T*& p) {
  if (p) cudaFreeAsync(p, ctx->stream);
  p = nullptr;
}

// Owner of a device buffer that lives for one call: freed (stream-ordered) when the owner goes
// out of scope or at reset(), or handed with release() to an object that frees it itself.
template <typename T>
struct DevBuf {
  const hge_ctx* ctx;
  T* p = nullptr;
  explicit DevBuf(const hge_ctx* c) : ctx(c) {}
  DevBuf(DevBuf&& o) noexcept : ctx(o.ctx), p(o.release()) {}
  DevBuf& operator=(DevBuf&& o) {
    reset();
    p = o.release();
    return *this;
  }
  ~DevBuf() { reset(); }
  [[nodiscard]] int alloc(size_t n) {
    reset();
    return hge_dev_alloc(ctx, &p, n);
  }
  void reset() { hge_dev_free(ctx, p); }
  [[nodiscard]] T* release() {
    T* q = p;
    p = nullptr;
    return q;
  }
};

// n elements device -> host, waited for
template <typename T>
int read_back(const hge_ctx* ctx, const T* dev, T* host, size_t n) {
  HGE_CUDA(cudaMemcpyAsync(host, dev, n * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
  HGE_CUDA(cudaStreamSynchronize(ctx->stream));
  return HGE_OK;
}

// Host <-> device staging for the HGE_MEM_HOST flavour of the entry points: `dev` is the
// caller's array for HGE_MEM_DEVICE, otherwise a device copy, uploaded by init() when `in` and
// copied back by finish() when `out`.
template <typename T>
struct Staged {
  DevBuf<T> copy;
  T* dev = nullptr;
  T* host = nullptr;
  size_t count = 0;
  bool copy_out = false;
  explicit Staged(const hge_ctx* c) : copy(c) {}

  int init(const T* p, size_t n, int mem, bool in, bool out) {
    count = n;
    copy_out = out && mem == HGE_MEM_HOST;
    host = const_cast<T*>(p);
    if (mem == HGE_MEM_DEVICE || p == nullptr) {
      dev = const_cast<T*>(p);
      return HGE_OK;
    }
    HGE_TRY(copy.alloc(n));
    dev = copy.p;
    if (in && n)
      HGE_CUDA(cudaMemcpyAsync(dev, p, n * sizeof(T), cudaMemcpyHostToDevice, copy.ctx->stream));
    return HGE_OK;
  }
  int finish() { return copy_out && count ? read_back(copy.ctx, dev, host, count) : HGE_OK; }
};

// Blocks of a grid-stride launch over `work` items, `per_block` a block: at least one, at most
// `per_sm` a multiprocessor.
static inline int grid_for(const hge_ctx* ctx, int64_t work, int per_block = 256, int per_sm = 16) {
  const int64_t want = std::max<int64_t>(1, (work + per_block - 1) / per_block);
  return (int)std::min<int64_t>(want, (int64_t)ctx->num_sms * per_sm);
}

#ifdef __CUDACC__
// Order-preserving float <-> int32 map: a < b  <=>  enc(a) < enc(b) as signed ints, so the
// joint per-column min / max of the rescale step can be kept with atomicMin / atomicMax.
__host__ __device__ static inline int hge_enc(float f) {
#ifdef __CUDA_ARCH__
  int i = __float_as_int(f);
#else
  int i;
  memcpy(&i, &f, 4);
#endif
  return i ^ ((i >> 31) & 0x7fffffff);
}
__host__ __device__ static inline float hge_dec(int i) {
  i = i ^ ((i >> 31) & 0x7fffffff);
#ifdef __CUDA_ARCH__
  return __int_as_float(i);
#else
  float f;
  memcpy(&f, &i, 4);
  return f;
#endif
}

__device__ __forceinline__ float4 hge_ld_stream(const float4* p) { return __ldcs(p); }
__device__ __forceinline__ float4 hge_f4_zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ void hge_f4_add(float4& a, const float4& b) {
  a.x += b.x;
  a.y += b.y;
  a.z += b.z;
  a.w += b.w;
}
#endif
