// Interface between the relaxation driver (hge_algdist.cu) and the stream-fed half-sweep
// kernel (hge_sweep.cu).
#pragma once

#include "hge_incidence.cuh"

enum {
  kSweepNode = 0,    // node half: update the owned rows, the gathered rows carry the previous affine map
  kSweepEdge = 1,    // edge half on one GPU: update the owned rows from this sweep's node rows
  kSweepRaw = 2,     // store the raw gathered sums to raw[rows, ld4] (sharded edge half, NCCL path)
  kSweepRawAdd = 3,  // add them to raw (node-range tiles of the edge half)
  kSweepPush = 4,    // store them into the owning rank's staging block (peer-memory sweep)
};

// One schedule's gather stream as the kernel reads it.
struct HgeSweepSrc {
  const int32_t* stream;       // HgeStream::ids
  const int4* items;           // HgeStream::items
  const uint32_t* uoff;        // HgeStream::uoff
  const int32_t* piece;        // HgeStream::piece
  const HgeHeavyRow* hrows;
  const int2* chunks;
  int32_t n_chunks;
  int32_t n_hrows;
  float4* partials;            // [n_partials, ld4] parked chunk sums of multi-chunk rows
  int32_t* counters;           // [slabs, n_hrows]
};

struct HgeSweepArgs {
  HgeSweepSrc src;             // a warp runs piece blockIdx.x * warps + warp of this schedule
  const float4* base;          // row 0 of the allocation the stream's row indices refer to
  float4* own;                 // owned rows [rows, ld4]
  const int32_t* mm_prev;      // affine map of the previous sweep, or nullptr (identity)
  int32_t* mm_cur;             // min / max slots of this sweep
  float4* raw;
  float4* const* push_stage;   // kSweepPush: staging blocks of all ranks
  int32_t push_rank;
  HgeOwnerMap push_map;        //   edge row -> (owner, row inside the owner's block)
  int32_t R;
  int32_t ld4;
};

// resident blocks per SM of k_sweep<lpr, .> (occupancy calculator)
int hge_sweep_resident_blocks(int lpr, int* out);
// one half-sweep: `blocks` x `slabs` blocks of 8 warps; the stream must have been built for
// blocks * 8 pieces
int hge_sweep_launch(hge_ctx* ctx, const HgeSweepArgs& a, int lpr, int mode, int blocks, int slabs);
