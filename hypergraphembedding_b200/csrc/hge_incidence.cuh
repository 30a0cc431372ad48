// Internal layout of the incidence object and its degree-binned gather schedule.
//
// One "half schedule" describes how the rows of one CSR (node->edge for the node half-sweep,
// edge->node for the edge half-sweep) are handed to warps:
//   * light rows (degree <= light_max_deg): one sub-warp of LPR lanes per row, rows sorted by
//     descending degree so the sub-warps of a warp run the same trip count;
//   * longer rows: cut into chunks of `chunk` incidences, one warp per chunk; a row with
//     several chunks parks per-chunk partial sums and the last chunk to finish adds them in
//     chunk order (deterministic) and finalises the row.
#pragma once

#include <vector>

#include "hge_common.cuh"

struct HgeLightItem {   // 16 B, read as one int4
  int32_t row;
  uint32_t deg_hi;      // bits 0..7 degree, bits 8..31 high bits of the CSR offset
  uint32_t start_lo;    // low 32 bits of the CSR offset
  float invs;           // 1 / sum of the neighbours' weights
};

struct HgeHeavyRow {    // 32 B
  int32_t row;
  int32_t deg;
  int64_t start;
  int32_t nchunks;
  int32_t partial_base;  // first slot in the partial buffer (multi-chunk rows only)
  float invs;
  int32_t pad;
};

// Packed gather stream of a half schedule, built for one group count G = 32 / (lanes per row)
// by hge_sched_stream (csrc/hge_schedule.cu) and read by k_sweep (csrc/hge_sweep.cu).
//
// A "step" is 4 gathered rows for each of the G lane groups of a warp: 4 G row indices, stored
// group-major ([g][4]) so a warp reads one contiguous block per step.  A "unit" is either one
// chunk of a long row (the groups share the chunk's incidences) or one group of
// G consecutive short rows of the degree-sorted order (group g gathers row g); its steps are
// consecutive in the stream and the units themselves are laid out back to back, long-row
// chunks first.  Row indices are absolute rows of the ONE allocation that holds the gathered
// and the owned table (gather0 / own0 = first row of either, zero = a row of zeros used as
// padding), so a slot costs one multiply-add and one load, with no predicate.  With with_own
// the last slot of a short row's last step is the row itself: its old value arrives through
// the same pipeline as the neighbours'.  `piece` cuts the unit list into `pieces` contiguous
// runs of equal cost (steps + 1 per unit), one per warp of the grid.
struct HgeStream {
  int G = 0;
  int with_own = 0;
  uint32_t gather0 = 0, own0 = 0, zero = 0;
  int pieces = 0;
  int32_t* ids = nullptr;        // [(total_steps + kStreamSlackSteps) * 4 G]
  int4* items = nullptr;         // [n_quads * G + kStreamSlackItems]: {row (-1: none), degree, steps of the unit, 1 / weight sum}
  uint32_t* uoff = nullptr;      // [n_units + 1] first step of every unit
  int32_t* piece = nullptr;      // [pieces + 1] first unit of every piece
  int32_t n_units = 0;
  int32_t n_quads = 0;
  uint32_t total_steps = 0;
};
constexpr int kStreamStepAlign = 4;     // k_sweep's unroll: the steps of a long-row chunk are padded to it
constexpr int kStreamSlackSteps = 12;  // the id look-ahead of k_sweep reads past the last step
constexpr int kStreamSlackItems = 128; // ... and its descriptor ring past the last descriptor

struct HgeHalfSchedule {
  int32_t rows = 0;
  int64_t nnz = 0;
  const int64_t* ptr = nullptr;   // device CSR row pointers [rows + 1] (= first incidence per row)
  const int64_t* row_end = nullptr;  // one past the last incidence per row (ptr + 1 for a plain CSR)
  bool ranges = false;            // rows are sub-ranges of CSR rows (node-range tiles)
  bool skip_empty = false;        // leave rows without incidences out of the work items
  const int32_t* idx = nullptr;   // device CSR column ids [nnz]
  int32_t* deg = nullptr;         // device, weight degree of each row (global degree if sharded)
  float* invs = nullptr;          // device, 1 / sum_b (1 / deg_other[b]) per row
  HgeLightItem* light = nullptr;
  int64_t n_light = 0;
  HgeHeavyRow* hrows = nullptr;
  int32_t n_hrows = 0;
  int2* chunks = nullptr;         // (heavy row index, chunk index)
  int32_t n_chunks = 0;
  int32_t n_partials = 0;
  int32_t chunk_sz = 0;
  int32_t max_deg = 0;
  int32_t first_empty = -1;       // first row without incidences, or -1
  HgeStream stream;               // packed form of the work items for k_sweep (built on first use)
  // transient, between hge_sched_begin and hge_sched_finish (csrc/hge_schedule.cu)
  int32_t row0 = 0;
  int32_t* sorted_rows = nullptr; // device: row ids by descending degree
  long long* d_stats = nullptr;
  long long* h_stats = nullptr;   // pinned slot
  cudaEvent_t stats_ready = nullptr;
};

// Device-side construction of a half schedule for rows [row0, row1) of a CSR whose row pointers
// are on the device.  begin: sort + statistics (asynchronous); finish: one event wait, then
// the work items (needs s->invs).  release frees everything the two allocated.
int hge_sched_begin(hge_ctx* ctx, int32_t row0, int32_t row1, const int64_t* d_ptr,
                    int64_t max_degree_possible, HgeHalfSchedule* s);
// The same for rows given as [row_begin[r], row_end[r]) ranges of a column-id array (sub-ranges
// of CSR rows: the node-range tiles of the edge half).
int hge_sched_begin_ranges(hge_ctx* ctx, int32_t row0, int32_t row1, const int64_t* row_begin,
                           const int64_t* row_end, int64_t max_degree_possible,
                           HgeHalfSchedule* s);
int hge_sched_finish(hge_ctx* ctx, const char* what, HgeHalfSchedule* s);
// Builds (or keeps, when the parameters match) the packed gather stream of a finished schedule.
int hge_sched_stream(hge_ctx* ctx, HgeHalfSchedule* s, int G, int with_own, uint32_t gather0,
                     uint32_t own0, uint32_t zero, int pieces);
void hge_sched_release(const hge_ctx* ctx, HgeHalfSchedule* s);

struct hge_incidence {
  hge_ctx* ctx = nullptr;
  int32_t N = 0, E = 0;
  bool owns_csr = false;
  bool owns_e2n = false;           // borrowed node -> edge arrays, edge -> node built by the library
  int64_t* n2e_ptr = nullptr;
  int32_t* n2e_idx = nullptr;
  int64_t* e2n_ptr = nullptr;
  int32_t* e2n_idx = nullptr;
  HgeHalfSchedule node_half, edge_half;
  // shard of a row-partitioned hypergraph (hge_incidence_create_sharded): local node rows, all
  // edges; the edge half is additionally cut into slices of consecutive edges
  bool sharded = false;
  bool finished = false;           // schedules built (a shard needs the all-reduced edge sums first)
  int num_slices = 1;
  double* edge_wsum = nullptr;     // device [E]: sum over members n of 1 / deg(n)
  std::vector<HgeHalfSchedule> edge_slices;
  std::vector<int32_t> slice_bounds;
  hge_algdist* cached = nullptr;   // workspace of the last hge_algdist_run, re-used across calls
  // Node-range tiles of the edge half (single GPU, node rows beyond the TLB reach of random
  // gathers): tile t gathers only the members in [t * tile_rows, (t + 1) * tile_rows) of every
  // edge.  Built on first use by hge_algdist_create (the tile height depends on R).
  std::vector<HgeHalfSchedule> edge_tiles;
  int64_t* tile_pos = nullptr;     // device [(tiles + 1) x E] incidence offsets
  int32_t tile_rows = 0;
};

// Peer-memory exchange arena of one shard (csrc/hge_p2p.cu): one cudaMalloc block, exported to
// the other ranks of the node through CUDA IPC.
struct hge_p2p {
  hge_ctx* ctx = nullptr;
  int rank = 0, world = 1;
  int32_t E = 0, N = 0, ld = 0;                // N = local node rows
  // Ownership of the edge rows: rank o owns the sub_rows consecutive rows from o * sub_rows on
  // (HgeOwnerMap), clipped at E (the last runs may be short or empty)
  int32_t sub_rows = 0;
  char* base = nullptr;                      // local arena
  size_t off_ye = 0, off_stage = 0, off_mmx = 0, off_flags = 0, off_err = 0, off_yn = 0, bytes = 0;
  char* peer_base[16] = {nullptr};           // peer arenas (own slot = base)
  // device-side pointer tables [world]
  float4** d_peer_stage = nullptr;
  float4** d_peer_ye = nullptr;
  int32_t** d_peer_mmx = nullptr;
  uint32_t** d_peer_flags = nullptr;
  uint32_t seq = 0;                          // barrier sequence number (same on every rank)
  bool peers_open = false;
  // hge_p2p_set_timing: events around the phases of every sweep (node half, gather + push,
  // barrier A, owner reduce + all-gather, barrier B), read by hge_p2p_phase_ms
  bool timing = false;
  std::vector<cudaEvent_t> marks;            // 6 per recorded sweep
};

// (owner rank, row inside the owner's block) of an edge row -- shared by the kernels that push
// partial rows to their owners and by the owner-side reduce
struct HgeOwnerMap {
  int32_t sub_rows;   // rows owned per rank (= rows per source rank in a staging block)
  __host__ __device__ void locate(int32_t row, int& owner, int32_t& idx) const {
    owner = row / sub_rows;
    idx = row - owner * sub_rows;
  }
};

// Relaxation state (csrc/hge_algdist.cu).
struct hge_algdist {
  hge_ctx* ctx = nullptr;
  hge_incidence* inc = nullptr;
  int R = 0, ld = 0, ld4 = 0, lpr = 0, slabs = 1;
  int max_iters = 0;
  float* ybuf = nullptr;        // [E + 1 + N, ld]: edge rows, a row of zeros, node rows (nullptr: the
                                // rows live in a peer-memory arena with the same order)
  float* yn = nullptr;
  float* ye = nullptr;
  uint32_t zero_row = 0;        // row of zeros, counted from ye
  int sweep_resident = 1;       // resident blocks per SM of k_sweep
  int32_t* mm = nullptr;        // [max_iters][2][ld]
  float* tile_raw = nullptr;    // [E, ld] un-normalised edge sums accumulated over the tiles
  float4* partials = nullptr;   // max over the two halves
  int32_t* counters = nullptr;
  int grid = 0;
  hge_p2p* p2p = nullptr;
};

// id of position p of the ascending non-member list of the sorted member row mem[0 .. m)
__device__ __forceinline__ int32_t hge_nonmember(const int32_t* __restrict__ mem, int64_t m, int64_t p) {
  int64_t lo = 0, hi = m;   // first c with mem[c] - c > p
  while (lo < hi) {
    const int64_t c = (lo + hi) >> 1;
    if (mem[c] - c > p) hi = c; else lo = c + 1;
  }
  return (int32_t)(p + lo);
}

// internal: the sharded edge gather with the partial rows pushed to their owners
extern "C" int hge_internal_edge_push(hge_algdist* st, int sweep);
