// Context, error reporting and versioning of libhge_b200.so.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <new>

#include "hge_common.cuh"

static thread_local char g_err[1024] = "";

void hge_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

void* hge_ctx_pinned_slot(hge_ctx* ctx) {
  if (!ctx->pinned_ring) {
    void* p = nullptr;
    if (cudaMallocHost(&p, 256 * 128) != cudaSuccess) {
      cudaGetLastError();
      hge_set_error("cudaMallocHost of the pinned slot ring failed");
      return nullptr;
    }
    ctx->pinned_ring = static_cast<char*>(p);
    ctx->pinned_next = 0;
  }
  char* slot = ctx->pinned_ring + (size_t)(ctx->pinned_next & 255) * 128;
  ctx->pinned_next++;
  return slot;
}

int hge_ctx_stage(hge_ctx* ctx, size_t floats, float** out) {
  if (!ctx->copy_stream) {
    HGE_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    HGE_CUDA(cudaEventCreateWithFlags(&ctx->copy_done, cudaEventDisableTiming));
    HGE_CUDA(cudaEventCreateWithFlags(&ctx->stage_idle, cudaEventDisableTiming));
  }
  if (ctx->stage_floats < floats) {
    HGE_CUDA(cudaStreamSynchronize(ctx->stream));
    HGE_CUDA(cudaStreamSynchronize(ctx->copy_stream));
    if (ctx->stage) cudaFree(ctx->stage);
    ctx->stage = nullptr;
    ctx->stage_floats = 0;
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&ctx->stage), floats * sizeof(float));
    if (e != cudaSuccess) {
      cudaGetLastError();
      hge_set_error("cudaMalloc of the %zu-byte staging block failed: %s", floats * sizeof(float),
                    cudaGetErrorString(e));
      return HGE_ERR_NOMEM;
    }
    ctx->stage_floats = floats;
  }
  *out = ctx->stage;
  return HGE_OK;
}

// Schedule / kernel defaults (hge_ctx_create, hge_ctx_reset_tuning).  The API setters change
// them; the only environment variable read is the allocation-failure countdown of the tests,
// re-read on every reset.
static void set_default_tuning(hge_ctx* ctx) {
  // schedule defaults from the sweep in profiles/r1_half_sweep_experiments.md (config 2, 4-block
  // kernel): sub-warp rows up to degree 128, chunks of 1024
  ctx->light_max_deg = 128;
  ctx->chunk = 1024;
  ctx->blocks_per_sm = 0;  // 0: 2 x what the occupancy calculator says is resident
  ctx->trainer_max_clusters = 0;
  // random 128-byte gathers over 8 GB of rows run at a third of the rate they reach inside 1 GB;
  // the edge half over more than 512 MB of node rows is tiled by node range into L2-sized tiles
  // when the edges are large enough for that to pay (profiles/r1_tiled_edge_half.md)
  ctx->tile_mb = 64;
  ctx->tile_min_mb = 512;
  ctx->tile_force = 0;
  ctx->fail_alloc_at = 0;
  if (const char* env = getenv("HGE_FAIL_ALLOC_AT")) ctx->fail_alloc_at = std::max(0ll, atoll(env));
  ctx->allocs = 0;
}

extern "C" {

int hge_version(void) { return 100; }

const char* hge_last_error(void) { return g_err; }

int hge_ctx_create(int device, void* stream, hge_ctx** out) {
  HGE_REQUIRE(out != nullptr, "hge_ctx_create: out is NULL");
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    hge_set_error("hge_ctx_create: no CUDA device is usable (%s); this library has no CPU path",
                  e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    return HGE_ERR_CUDA;
  }
  HGE_REQUIRE(device >= 0 && device < count, "hge_ctx_create: device %d out of range [0, %d)",
              device, count);
  HGE_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  HGE_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) {
    hge_set_error("hge_ctx_create: device %d is sm_%d%d; this library is built for sm_100a only",
                  device, prop.major, prop.minor);
    return HGE_ERR_UNSUPPORTED;
  }
  hge_ctx* ctx = new (std::nothrow) hge_ctx();
  if (!ctx) return HGE_ERR_NOMEM;
  ctx->device = device;
  ctx->num_sms = prop.multiProcessorCount;
  ctx->own_stream = false;
  set_default_tuning(ctx);
  ctx->launches = 0;
  ctx->pinned_ring = nullptr;
  ctx->pinned_next = 0;
  ctx->stage = nullptr;
  ctx->stage_floats = 0;
  ctx->copy_stream = nullptr;
  ctx->copy_done = nullptr;
  ctx->stage_idle = nullptr;
  // NULL selects the legacy default stream, which is also torch's default stream, so work
  // queued by the caller on that stream is ordered with ours.
  ctx->stream = reinterpret_cast<cudaStream_t>(stream);
  // keep freed blocks in the stream-ordered pool: the per-call workspaces are re-used
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
    uint64_t threshold = UINT64_MAX;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &threshold);
  }
  cudaGetLastError();
  *out = ctx;
  return HGE_OK;
}

int hge_ctx_destroy(hge_ctx* ctx) {
  if (!ctx) return HGE_OK;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (ctx->pinned_ring) cudaFreeHost(ctx->pinned_ring);
  if (ctx->copy_stream) {
    cudaStreamSynchronize(ctx->copy_stream);
    cudaStreamDestroy(ctx->copy_stream);
    cudaEventDestroy(ctx->copy_done);
    cudaEventDestroy(ctx->stage_idle);
  }
  if (ctx->stage) cudaFree(ctx->stage);
  if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
  return HGE_OK;
}

int hge_ctx_set_stream(hge_ctx* ctx, void* stream) {
  HGE_REQUIRE(ctx != nullptr, "hge_ctx_set_stream: ctx is NULL");
  cudaStream_t next = reinterpret_cast<cudaStream_t>(stream);
  if (next != ctx->stream) {
    // allocations and frees are ordered on the context's stream: drain it before switching
    HGE_CUDA(cudaSetDevice(ctx->device));
    HGE_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  ctx->stream = next;
  return HGE_OK;
}

int hge_ctx_sync(hge_ctx* ctx) {
  HGE_REQUIRE(ctx != nullptr, "hge_ctx_sync: ctx is NULL");
  HGE_CUDA(cudaSetDevice(ctx->device));
  HGE_CUDA(cudaStreamSynchronize(ctx->stream));
  return HGE_OK;
}

int hge_ctx_set_tuning(hge_ctx* ctx, int light_max_deg, int chunk, int blocks_per_sm) {
  HGE_REQUIRE(ctx != nullptr, "hge_ctx_set_tuning: ctx is NULL");
  HGE_REQUIRE(light_max_deg >= 0 && light_max_deg <= 255,
              "hge_ctx_set_tuning: light_max_deg %d not in [0, 255]", light_max_deg);
  HGE_REQUIRE(chunk >= 0 && (chunk == 0 || chunk % 32 == 0),
              "hge_ctx_set_tuning: chunk %d must be a multiple of 32", chunk);
  HGE_REQUIRE(blocks_per_sm >= 0 && blocks_per_sm <= 32,
              "hge_ctx_set_tuning: blocks_per_sm %d not in [0, 32]", blocks_per_sm);
  if (light_max_deg) ctx->light_max_deg = light_max_deg;
  if (chunk) ctx->chunk = chunk;
  ctx->blocks_per_sm = blocks_per_sm;
  return HGE_OK;
}

int hge_ctx_set_tile_mb(hge_ctx* ctx, int tile_mb, int min_rows_mb) {
  HGE_REQUIRE(ctx != nullptr, "hge_ctx_set_tile_mb: ctx is NULL");
  HGE_REQUIRE(tile_mb >= 0 && tile_mb <= (1 << 20) && min_rows_mb >= 0 && min_rows_mb <= (1 << 20),
              "hge_ctx_set_tile_mb: %d / %d MB not in [0, 2^20]", tile_mb, min_rows_mb);
  ctx->tile_mb = tile_mb;
  ctx->tile_min_mb = min_rows_mb;
  ctx->tile_force = min_rows_mb == 0;
  return HGE_OK;
}

int hge_ctx_set_trainer_clusters(hge_ctx* ctx, int max_clusters) {
  HGE_REQUIRE(ctx != nullptr, "hge_ctx_set_trainer_clusters: ctx is NULL");
  HGE_REQUIRE(max_clusters >= 0 && max_clusters <= 64, "hge_ctx_set_trainer_clusters: %d not in [0, 64]",
              max_clusters);
  ctx->trainer_max_clusters = max_clusters;
  return HGE_OK;
}

int hge_ctx_reset_tuning(hge_ctx* ctx) {
  HGE_REQUIRE(ctx != nullptr, "hge_ctx_reset_tuning: ctx is NULL");
  set_default_tuning(ctx);
  return HGE_OK;
}

int64_t hge_ctx_launch_count(const hge_ctx* ctx) { return ctx ? ctx->launches : 0; }

}  // extern "C"
