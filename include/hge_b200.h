/*
 * hge_b200.h -- C ABI of the B200-native HOBE hot path (libhge_b200.so).
 *
 * The reference (JSybrandt/HypergraphEmbedding) is pure Python and has no FFI of its own
 * (SURVEY.md section 8b): its boundary is a set of Python callables.  This header is the
 * C-level boundary those callables bind to in this build; every entry point names the
 * reference function (file:line, relative to the reference tree) whose arithmetic it
 * replaces.  The Python mirror of the reference interface lives in
 * hypergraphembedding_b200/{algebraic_distance,hg2v_weighting,hg2v_sample}.py and calls
 * these symbols through ctypes (INTEGRATION.md shows the stub).
 *
 * Conventions
 *   - Every function returns int: 0 = HGE_OK, < 0 = error.  hge_last_error() returns a
 *     thread-local message for the last failing call.  Nothing throws across the boundary.
 *   - Pointers are plain C pointers.  "mem" arguments say where they live:
 *     HGE_MEM_HOST (the library stages through its own device buffers, copies included) or
 *     HGE_MEM_DEVICE (borrowed device pointers, e.g. torch tensor storage; the caller keeps
 *     them alive until hge_ctx_sync()).
 *   - Row pointers are int64, column ids int32, values fp32, row-major.
 *   - One context per device; calls on one context are not re-entrant.
 *   - There is no CPU fallback: without a usable CUDA device every compute entry point
 *     fails with HGE_ERR_CUDA.
 */
#ifndef HGE_B200_H_
#define HGE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HGE_OK 0
#define HGE_ERR_INVALID (-1)     /* bad argument (the reference would assert)            */
#define HGE_ERR_CUDA (-2)        /* CUDA runtime / launch failure, or no device          */
#define HGE_ERR_EMPTY_ROW (-3)   /* a node or edge without incidences: the reference     */
                                 /* divides 0/0 there (algebraic_distance.py:49)         */
#define HGE_ERR_NOMEM (-4)
#define HGE_ERR_UNSUPPORTED (-5)

#define HGE_MEM_HOST 0
#define HGE_MEM_DEVICE 1

typedef struct hge_ctx hge_ctx;
typedef struct hge_incidence hge_incidence;
typedef struct hge_algdist hge_algdist;

/* ---- library / context ------------------------------------------------------------ */

int hge_version(void);
const char* hge_last_error(void);

/* stream: the cudaStream_t every launch and copy of this context is queued on (e.g. torch's
 * current stream); NULL is the legacy default stream.  The caller owns the stream. */
int hge_ctx_create(int device, void* stream, hge_ctx** out);
int hge_ctx_destroy(hge_ctx* ctx);
int hge_ctx_set_stream(hge_ctx* ctx, void* stream);
int hge_ctx_sync(hge_ctx* ctx);
/* Tuning knobs of the relaxation schedule (0 keeps the default):
 *   light_max_deg  rows up to this degree are gathered by one sub-warp (<= 255; default 128)
 *   chunk          incidences per warp work item for longer rows (default 1024)
 *   blocks_per_sm  grid size = SMs * blocks_per_sm (default: 4 x the resident blocks) */
int hge_ctx_set_tuning(hge_ctx* ctx, int light_max_deg, int chunk, int blocks_per_sm);
/* Edge half over node rows that exceed what random 128-byte gathers reach at full rate
 * (measured on config 5: 1.9 TB/s over 8.3 GB of rows, 4.9 TB/s inside 1 GB, 6.3 TB/s inside an
 * L2-sized block): when the (local) node rows exceed min_rows_mb megabytes the half-sweep runs
 * in node-range tiles of tile_mb megabytes of rows -- tile t gathers only the members of every
 * edge that fall into its range and adds their sum to an E x R buffer, one more pass finishes
 * the rows (single GPU) or pushes them to their owners (peer-memory sweep of a shard).
 * Defaults 64 / 512; tile_mb 0 disables; min_rows_mb 0 forces tiles even when the edges are too
 * small for them to pay (< 16 incidences per non-empty (edge, tile) pair, where the per-pair
 * work dominates and the half-sweep otherwise stays untiled).  Config 5: 122 -> 37 ms per edge
 * half on one GPU, 200 -> 159 ms per step on 8.  Results differ from the untiled half-sweep only
 * by fp32 summation order. */
int hge_ctx_set_tile_mb(hge_ctx* ctx, int tile_mb, int min_rows_mb);
/* hypergraph2vec training: at most this many 8-block clusters per epoch launch (0, the default:
 * one per 256 samples of a batch, up to what the device holds at once). */
int hge_ctx_set_trainer_clusters(hge_ctx* ctx, int max_clusters);
/* Back to the defaults of hge_ctx_create for every knob above (tuning, kernel, tiles). */
int hge_ctx_reset_tuning(hge_ctx* ctx);
/* Number of kernels this context has launched so far (bench.py's gpu_launches). */
int64_t hge_ctx_launch_count(const hge_ctx* ctx);

/* ---- incidence storage ------------------------------------------------------------
 * Replaces ToCsrMatrix / ToEdgeCsrMatrix (hypergraph_util.py:96-135): the node->edge
 * incidence as int32 CSR (n2e) and the edge->node incidence as int32 CSR (e2n, i.e. the
 * CSC of the same matrix when the hypergraph is consistent).  Column ids must be sorted
 * and unique inside a row, as scipy's canonical CSR is.  Builds the degree-binned gather
 * schedule and the inverse neighbour-weight sums used by the relaxation.
 * Rows without incidences are accepted here (the weighting entry points work on sparse id
 * ranges); the relaxation refuses them with HGE_ERR_EMPTY_ROW (hge_algdist_create / _run).
 * e2n_ptr == e2n_idx == NULL: the edge -> node orientation is built on the device from the
 * node -> edge one (a stable radix sort of the (edge, node) pairs), so a host-buffer caller
 * uploads one orientation only. */
int hge_incidence_create(hge_ctx* ctx, int32_t num_nodes, int32_t num_edges,
                         const int64_t* n2e_ptr, const int32_t* n2e_idx,
                         const int64_t* e2n_ptr, const int32_t* e2n_idx, int mem,
                         hge_incidence** out);
/* One shard of a hypergraph whose NODES are row-partitioned over several GPUs (DESIGN.md
 * "Multi-GPU"): n2e holds the num_local_nodes local node rows (global edge ids), e2n holds for
 * every edge its LOCAL member nodes (local node ids; may be empty).  Creation is two-phase:
 *   1. hge_incidence_create_sharded uploads the arrays and computes, on the device, the local
 *      edge degrees (int32 [E]) and the local edge weight sums  sum_{n local} 1 / deg(n)
 *      (f64 [E]);
 *   2. the caller all-reduces (SUM) both arrays in place through the device pointers returned
 *      by hge_incidence_edge_sums -- the one set-up exchange of the path --
 *   3. hge_incidence_finish_sharded builds the inverse weight sums and the gather schedules.
 * The edge half-sweep of a shard runs in num_slices slices of consecutive edges. */
int hge_incidence_create_sharded(hge_ctx* ctx, int32_t num_local_nodes, int32_t num_edges,
                                 const int64_t* n2e_ptr, const int32_t* n2e_idx,
                                 const int64_t* e2n_ptr, const int32_t* e2n_idx, int num_slices,
                                 int mem, hge_incidence** out);
int hge_incidence_edge_sums(hge_incidence* inc, int32_t** edge_deg, double** edge_wsum);
int hge_incidence_finish_sharded(hge_incidence* inc);
int hge_incidence_slice_range(const hge_incidence* inc, int slice, int32_t* row0, int32_t* row1);
int hge_incidence_destroy(hge_incidence* inc);
int64_t hge_incidence_nnz(const hge_incidence* inc);

/* ---- algebraic-distance relaxation --------------------------------------------------
 * Replaces the loop of EmbedAlgebraicDistance (algebraic_distance.py:149-164):
 * `iterations` x { node half (_update_alg_dist, :34-51, old edge rows), edge half (new node
 * rows), joint per-column min/max rescale (_helper_scale_embeddings, :97-123) }.
 * xn [N, R] and xe [E, R] hold the initial vectors on entry (algebraic_distance.py:140-141,
 * drawn by the caller) and the rescaled result on return, fp32 row-major, dense.
 * lohi (optional, host, [iterations][2][R]) receives each sweep's per-column (min, max). */
int hge_algdist_run(hge_ctx* ctx, hge_incidence* inc, float* xn, float* xe, int R,
                    int iterations, int mem, float* lohi);
/* The same relaxation straight from the CSR arrays: hge_incidence_create + hge_algdist_run +
 * hge_incidence_destroy in one call -- what EmbedAlgebraicDistance (algebraic_distance.py:126-175)
 * does per call.  With host buffers the vectors' upload is queued behind the column ids' and the
 * set-up kernels (transpose, schedules) run under it.  e2n_ptr / e2n_idx may be NULL (the
 * edge -> node orientation is then built on the device). */
int hge_algdist_run_csr(hge_ctx* ctx, int32_t num_nodes, int32_t num_edges, const int64_t* n2e_ptr,
                        const int32_t* n2e_idx, const int64_t* e2n_ptr, const int32_t* e2n_idx, float* xn,
                        float* xe, int R, int iterations, int mem, float* lohi);

/* _helper_scale_embeddings (algebraic_distance.py:97-123) on its own: joint per-column min / max
 * of the two dense blocks, x <- (x - min) / (max - min), in place.  (hge_algdist_run fuses this
 * into the half-sweeps; the stand-alone form exists for callers that drive the sweeps
 * themselves.) */
int hge_column_rescale(hge_ctx* ctx, float* xn, int64_t num_nodes, float* xe, int64_t num_edges,
                       int R, int mem);

/* Stepwise form of the same loop, used when the node rows are sharded over several GPUs
 * and the host interleaves collectives (DESIGN.md "Multi-GPU").  All pointers are device
 * pointers. */
int hge_algdist_create(hge_ctx* ctx, hge_incidence* inc, int R, int max_iterations,
                       hge_algdist** out);
int hge_algdist_destroy(hge_algdist* st);
int hge_algdist_load(hge_algdist* st, const float* xn, const float* xe, int mem);
int hge_algdist_node_half(hge_algdist* st, int sweep);
int hge_algdist_edge_half(hge_algdist* st, int sweep);
/* Sharded edge half, per slice of edges: the first call writes the un-normalised local sums
 * sum_{n local} w_n * xn'[n]  of the slice's edges into their rows of partial [E, ld]; after
 * the caller's all-reduce(sum) of those rows the second call blends, rescales and stores the
 * slice's edge rows (every shard redundantly).  ld = hge_algdist_ld(). */
int hge_algdist_edge_partial(hge_algdist* st, int sweep, int slice, float* partial);
int hge_algdist_edge_finalize(hge_algdist* st, int sweep, int slice, const float* partial);
/* Device pointer to this sweep's order-preserving int32 encoded (min[ld], max[ld]) slots,
 * for an all-reduce(MIN) / (MAX) across shards. */
int hge_algdist_minmax_ptr(hge_algdist* st, int sweep, int32_t** out);
int hge_algdist_ld(const hge_algdist* st);
int hge_algdist_store(hge_algdist* st, int sweeps_done, float* xn, float* xe, int mem);

/* ---- peer-memory exchange for the sharded relaxation (single node, NVLink) ---------------
 * The collectives of the sharded edge half done by the kernels themselves: partial rows are
 * stored into the owning GPU's staging block from inside the gather kernel (reduce-scatter),
 * the owner reduces them in rank order, updates the edge rows and stores them into every
 * rank's edge block (all-gather); barriers and the min / max exchange are flags and 2R-word
 * slots in peer memory.  One arena per rank, shared through CUDA IPC: create, export the
 * 64-byte handle, exchange the handles between the ranks (any transport), open the peers'
 * arenas, attach to the relaxation state; then hge_algdist_sweep_p2p replaces
 * node_half / edge_partial / all-reduce / edge_finalize / min-max all-reduce.  All ranks must
 * call the same sequence of sweeps; each rank must drive its own GPU.  A barrier that is not
 * met within 20 s raises an error flag (hge_p2p_check) instead of hanging. */
typedef struct hge_p2p hge_p2p;
/* num_local_nodes: this rank's node rows (they live in the arena next to the edge rows, though no
 * peer touches them). */
int hge_p2p_create(hge_ctx* ctx, int rank, int world, int32_t num_local_nodes, int32_t num_edges,
                   int ld, hge_p2p** out);
int hge_p2p_export(hge_p2p* p, void* handle64);
int hge_p2p_open_peers(hge_p2p* p, const void* handles /* world x 64 bytes */);
int hge_p2p_check(hge_p2p* p);
/* Phase timing of the peer-memory sweep (off by default, switched by hge_p2p_set_timing): CUDA
 * events around the five phases of every sweep.
 * hge_p2p_phase_ms returns the mean ms per sweep of each since the last call -- node half, edge
 * gather + push, barrier A, owner reduce + all-gather, barrier B + min/max -- and the number of
 * sweeps averaged over (0: nothing recorded). */
int hge_p2p_set_timing(hge_p2p* p, int on);
int hge_p2p_phase_ms(hge_p2p* p, double* out5, int* sweeps);
int hge_p2p_close_peers(hge_p2p* p);   /* all ranks, then a host barrier, then destroy */
int hge_p2p_destroy(hge_p2p* p);
int hge_algdist_attach_p2p(hge_algdist* st, hge_p2p* p);
int hge_algdist_sweep_p2p(hge_algdist* st, int sweep);

/* ---- distances and HOBE / FOBE weights ------------------------------------------------
 * All vectors are dense fp32 [rows, R]; outputs are fp32.  `mem` applies to every array
 * argument of a call. */

/* dist[p] = || xn[n] - xe[e] ||_2 for every stored incidence p, in the storage order of the
 * node->edge CSR (order == 0) or of the edge->node CSR (order == 1).  Replaces the per-pair
 * np.linalg.norm of WeightByDistance (hg2v_weighting.py:86-91) and of _same_type_dist_calc
 * (hg2v_sample.py:540-541).  With as_weight != 0 the HOBE incidence weight
 * (sqrt(R) - d) / sqrt(R) is stored instead (hg2v_sample.py:537-541). */
int hge_incidence_l2(hge_ctx* ctx, hge_incidence* inc, const float* xn, const float* xe, int R,
                     int order, int as_weight, float* dist, int mem);

/* dist[p] = || xa[ia[p]] - xb[ib[p]] ||_2 for arbitrary (node,node), (node,edge) or
 * (edge,edge) sample pairs: the distance part of WeightBySameTypeDistance
 * (hg2v_weighting.py:37-45) and of the 100M-pair weighting of BASELINE.json configs[2].
 * An index outside [0, rows_a) / [0, rows_b) is HGE_ERR_INVALID; nothing is computed then. */
int hge_pair_l2(hge_ctx* ctx, const float* xa, int64_t rows_a, const float* xb, int64_t rows_b,
                int R, const int32_t* ia, const int32_t* ib, int64_t num_pairs, float* dist,
                int mem);

/* In place: v <- alpha + (1 - alpha) * (1 - (v - min) / (max - min)), min / max over all n
 * values; a zero range maps every value to alpha + (1 - alpha) * 0.  This is
 * AlphaScaleValues(OneMinusValues(ZeroOneScaleValues(.))) (hg2v_weighting.py:301-333) with the
 * reference's fp32 operation order, so equal inputs give bit-equal outputs.  minmax (optional,
 * host, 2 floats) receives (min, max).  alpha outside [0, 1] is HGE_ERR_INVALID. */
int hge_scale_transform(hge_ctx* ctx, float* values, int64_t n, double alpha, float* minmax,
                        int mem);

/* The same transform in two steps, for values spread over several GPUs (pairs are sharded over
 * the ranks, SURVEY.md section 8e): each rank reduces its own values to (min, max), the caller
 * all-reduces them (MIN / MAX), each rank applies the transform with the global pair. */
int hge_scale_minmax(hge_ctx* ctx, const float* values, int64_t n, float* minmax, int mem);
int hge_scale_apply(hge_ctx* ctx, float* values, int64_t n, double alpha, float lo, float hi,
                    int mem);

/* span[r] = max(0, max over neighbours b and components c of (x_other[b][c] - x_self[r][c]))
 *         - min(0, min over the same set), for the rows of the node->edge CSR (side == 0,
 * x_self = xn) or of the edge->node CSR (side == 1, x_self = xe): _compute_span
 * (hg2v_weighting.py:214-233). */
int hge_row_span(hge_ctx* ctx, hge_incidence* inc, const float* xn, const float* xe, int R,
                 int side, float* span, int mem);

/* HOBE same-type probability (hg2v_sample.py:527-543) for num_pairs pairs (i, j) of rows of
 * the node->edge CSR (side == 0) or of the edge->node CSR (side == 1):
 *     prob = max over shared columns k of min(w(i,k), w(j,k)),  0 without a shared column,
 * with w the incidence weights in that CSR's storage order (hge_incidence_l2, as_weight).  An index
 * outside the side's rows is HGE_ERR_INVALID; nothing is computed then. */
int hge_same_type_prob(hge_ctx* ctx, hge_incidence* inc, int side, const float* w,
                       const int32_t* pi, const int32_t* pj, int64_t num_pairs, float* prob,
                       int mem);

/* HOBE node-edge probability (hg2v_sample.py:606-629) for pairs (node n, edge e):
 *     prob = max(0, max over the node's edges e' of same_type_prob_edges(e, e')),
 * w_e2n = incidence weights in edge->node storage order.  A node outside [0, N) or an edge outside
 * [0, E) is HGE_ERR_INVALID; nothing is computed then. */
int hge_diff_type_prob(hge_ctx* ctx, hge_incidence* inc, const float* w_e2n, const int32_t* pn,
                       const int32_t* pe, int64_t num_pairs, float* prob, int mem);

/* ---- sparse weighted Jaccard (WeightedJaccardSamples, hg2v_sample.py:250-510) -----------
 * Feature matrices are CSR with int64 row pointers, sorted int32 column ids and fp32 values.
 * J(x, y) = sum min / sum max over the union of the non-zeros, 0 when the denominator is 0
 * (SparseWeightedJaccard, :250-275).  Both sums are carried in fp32 in the reference's own order
 * (ascending column, one value at a time), so the result equals the reference's bit for bit on
 * fp32 features. */

/* out[p] = J(F[pi[p]], F[pj[p]]): SameTypeJaccardSample (:323-340).  An index outside [0, rows) is
 * HGE_ERR_INVALID; nothing is computed then. */
int hge_jaccard_rows(hge_ctx* ctx, const int64_t* ptr, const int32_t* idx, const float* val,
                     int64_t rows, int64_t nnz, const int32_t* pi, const int32_t* pj,
                     int64_t num_pairs, float* out, int mem);

/* out[p] = J(X[px[p]], mean_{t in G[pg[p]]} F[t]): one factor of DiffTypeJaccardSample
 * (:343-392).  The centroid rows of the groups the pairs name are materialised on the device the
 * way CentroidFromRows (:284-299) computes them (members added in ascending order in fp32, one
 * division by the group size).  G is a boolean CSR (group -> member rows of F); X and F have the
 * same number of columns (X may be F itself).  An empty group gives 0.  The pairs are stably sorted
 * by group and the centroid rows built in batches of consecutive named groups whose expansion fits
 * 2048 MB (48 bytes per expanded entry), each batch freed after the merge of its pairs; besides that
 * budget the call holds at most 52 bytes per pair and, for HGE_MEM_HOST, the device copies of its
 * inputs.  A pair index outside [0, xrows) or outside [0, grows) is HGE_ERR_INVALID, and so is
 * num_pairs >= 2^31 (refused before any array is read); nothing is computed then. */
int hge_jaccard_centroid(hge_ctx* ctx, const int64_t* xptr, const int32_t* xidx, const float* xval,
                         int64_t xrows, int64_t xnnz, const int64_t* gptr, const int32_t* gidx,
                         int64_t grows, int64_t gnnz, const int64_t* fptr, const int32_t* fidx,
                         const float* fval, int64_t frows, int64_t fnnz, const int32_t* px,
                         const int32_t* pg, int64_t num_pairs, float* out, int mem);

/* The same factor with the groups taken from the incidence's own CSR, for pairs held on the
 * device: group_side 1 = groups are edges with their member nodes (edge -> node CSR, F = node
 * features, frows = nodes), group_side 0 = groups are nodes with their edges (node -> edge CSR,
 * F = edge features, frows = edges).  All pointers are device pointers.  The pairs are stably
 * sorted by group; the centroid rows of the named groups are built once per call, in batches of
 * consecutive named groups whose expansion fits workspace_mb megabytes (0 = 2048, 48 bytes per
 * expanded entry), each batch freed after the merge of its pairs.  A single group larger than the
 * budget is its own batch; one the device cannot hold is HGE_ERR_NOMEM.  Besides the budget the
 * call holds at most 52 bytes per pair.  Both centroid entry points run the same code, so the
 * result equals hge_jaccard_centroid's bit for bit on the same inputs, for every workspace_mb.  A
 * pair index outside X or outside the groups is HGE_ERR_INVALID, and so is num_pairs >= 2^31;
 * nothing is computed then. */
int hge_jaccard_centroid_grouped(hge_ctx* ctx, hge_incidence* inc, int group_side, const int64_t* xptr,
                                 const int32_t* xidx, const float* xval, int64_t xrows, int64_t xnnz,
                                 const int64_t* fptr, const int32_t* fidx, const float* fval, int64_t frows,
                                 int64_t fnnz, const int32_t* px, const int32_t* pg, int64_t num_pairs,
                                 int64_t workspace_mb, float* out);

/* ---- candidate rows and bit-exact sampling (host code; all pointers are host pointers) ---
 * The reference draws every sample from numpy's process-global legacy MT19937, sequentially
 * and with data-dependent rejection, so this part of the path runs on the host; the drawn
 * pairs are then weighted on the GPU.  state625 = the 624 key words of
 * np.random.get_state() followed by its `pos`; it is advanced in place. */

/* Next n raw 32-bit outputs / n bounded integers in [0, max_inclusive] (numpy rk_interval:
 * masked rejection; max 0 consumes nothing).  Test hooks for the stream replay. */
int hge_mt19937_random_raw(uint32_t* state625, int64_t n, uint32_t* out);
int hge_mt19937_interval(uint32_t* state625, uint32_t max_inclusive, int64_t n, uint32_t* out);

/* Rows of M1 (kind 0), M1*M2 (kind 1) or (M1*M2)*M3 (kind 2) as boolean CSR, for the listed
 * rows, in the column order scipy's csr_matmat stores them (reverse first-discovery order;
 * this is the candidate order of _sample_adj_matrix, hg2v_sample.py:77) or sorted
 * (sorted != 0: the nonzero pattern used by WeightBySameTypeDistance, hg2v_weighting.py:56-61).
 * mid_cols / out_cols = column counts of M1*M2 and of the final product.  With out_idx == NULL
 * only out_ptr (num_rows + 1 entries) is filled, so the caller can size out_idx. */
int hge_spgemm_rows(int kind, const int64_t* p1, const int32_t* i1, const int64_t* p2,
                    const int32_t* i2, const int64_t* p3, const int32_t* i3, int32_t mid_cols,
                    int32_t out_cols, const int32_t* rows, int64_t num_rows, int sorted,
                    int64_t* out_ptr, int32_t* out_idx, int64_t capacity);

/* _sample_adj_matrix (hg2v_sample.py:53-86) over the same three kinds of matrix: for each
 * listed row, in order, either `samples_per_row` uniform columns in [0, out_cols) (negative),
 * or a draw without / with replacement from the row's candidates (np.random.choice; at most
 * len(candidates) without replacement; rows without candidates are skipped).  Emits (row, col)
 * pairs; capacity must be >= sum(samples_per_row). */
int hge_sample_adj_rows(int kind, const int64_t* p1, const int32_t* i1, const int64_t* p2,
                        const int32_t* i2, const int64_t* p3, const int32_t* i3, int32_t mid_cols,
                        int32_t out_cols, const int32_t* rows, int64_t num_rows,
                        const int32_t* samples_per_row, int replace, int negative,
                        uint32_t* state625, int32_t* out_row, int32_t* out_col, int64_t capacity,
                        int64_t* out_count);

/* Worker threads around the (sequential) draw loop of hge_sample_adj_rows: they build the
 * candidate rows ahead of it and turn its draws into samples behind it.  0 = automatic (inline
 * below 512 product rows, else up to 4 workers; HGE_SAMPLER_THREADS overrides), 1 = everything
 * inline.  Results do not depend on it. */
int hge_sampler_set_threads(int threads);

/* _sample_neighbors (hg2v_sample.py:49-51) for a list of (node, edge) samples: per sample k
 * draws with replacement from the node's edges, then k from the edge's nodes
 * (hg2v_sample.py:184-187, 604-605).  Outputs are [num_samples, k]. */
int hge_sample_neighbors(const int64_t* n2e_ptr, const int32_t* n2e_idx, const int64_t* e2n_ptr,
                         const int32_t* e2n_idx, const int32_t* nodes, const int32_t* edges,
                         int64_t num_samples, int k, uint32_t* state625, int32_t* out_nbr_edges,
                         int32_t* out_nbr_nodes);

/* ---- device sampling from a seeded counter-based generator -------------------------------
 * The distribution of _sample_adj_matrix / _sample_neighbors (hg2v_sample.py:49-86), drawn on the
 * GPU from Philox4x32-10 word streams instead of numpy's MT19937 (csrc/hge_philox.cuh documents the
 * key / counter layout and the phase constants; oracle/device_sampler_ref.py restates it).  Every
 * row (pairs) and every record (neighbours) owns its stream, so results do not depend on how a
 * caller splits rows or records into calls, nor on the workspace budget.  The bit-exact replay
 * of the reference's stream is hge_sample_adj_rows above.  `mem` applies to every array argument.
 *
 * Pairs: rows [row0, row1) of P = M1 (factors 1), M1 * M2 (2) or (M1 * M2) * M3 (3), with
 * M1 = M3 = the node -> edge CSR and M2 = the edge -> node CSR for side 0 (node rows), the other
 * way round for side 1 (edge rows).  Positive (negative == 0): row r emits min(k_r, n_r) distinct
 * columns, uniform among the subsets of that size of its n_r distinct candidates, ascending; rows
 * without candidates emit nothing.  Negative: row r emits k_r columns uniform on [0, columns of
 * P), with replacement, in draw order.  Rows come out in ascending order as (out_row, out_col);
 * samples_per_row holds k_r for the row1 - row0 rows; capacity >= sum(k_r) always suffices.
 * Candidate rows are built in batches of rows whose expansion fits workspace_mb megabytes
 * (0 = 2048); a row that needs more than the device holds is HGE_ERR_NOMEM.  A negative k_r is
 * HGE_ERR_INVALID.  Needs an incidence made by hge_incidence_create (not a shard). */
int hge_sample_pairs_device(hge_ctx* ctx, hge_incidence* inc, int side, int factors, int32_t row0,
                            int32_t row1, const int32_t* samples_per_row, int negative, uint64_t seed,
                            uint32_t phase, int64_t workspace_mb, int32_t* out_row, int32_t* out_col,
                            int64_t capacity, int64_t* out_count, int mem);

/* Neighbour arrays of `count` (node, edge) records, record i being number first_index + i of its
 * block: k draws with replacement from the node's edges, then k from the edge's nodes.  Outputs
 * are [count, k].  A draw from an empty list is HGE_ERR_INVALID ("cannot be empty"). */
int hge_sample_neighbors_device(hge_ctx* ctx, hge_incidence* inc, const int32_t* nodes,
                                const int32_t* edges, int64_t count, int k, uint64_t seed,
                                uint32_t phase, int64_t first_index, int32_t* out_nbr_edges,
                                int32_t* out_nbr_nodes, int mem);

/* ---- hypergraph2vec training (hg2v_model.py:51-203, fit loop embedding.py:269-305) ---------
 * The consumer of the sample columns.  Two embedding tables [rows, dim] fp32 whose row 0 is the
 * trained padding row (Embedding(input_dim = max id + 2)); outputs
 *   node_node = act(<N[ln], N[rn]>), edge_edge = act(<E[le], E[re]>),
 *   node_edge = mean_i act(<N[nn_i], N[ln]>) * mean_i act(<E[ne_i], E[re]>);
 * activation 0 = sigmoid (BooleanModel), 1 = relu (UnweightedFloatModel); loss 0 = Keras
 * kullback_leibler_divergence, 1 = mean_squared_error, summed over the three outputs; optimizer =
 * Keras Adagrad defaults (lr 0.01, epsilon 1e-7).  One call of hge_hg2v_fit_epoch is one epoch:
 * consecutive batches of `batch_size` samples taken in the given order, one kernel launch of one
 * thread-block cluster per 256 samples of a batch (a sample per warp; several clusters are
 * launched cooperatively and meet at a global barrier twice per batch). */
typedef struct hge_hg2v_model hge_hg2v_model;
int hge_hg2v_create(hge_ctx* ctx, int32_t node_rows, int32_t edge_rows, int dim, int num_neighbors,
                    int activation, int loss, const float* node_init, const float* edge_init,
                    int mem, hge_hg2v_model** out);
int hge_hg2v_destroy(hge_hg2v_model* m);
/* features: int32 [4 + 2 * num_neighbors][num_samples], the columns of SamplesToModelInput
 * (hg2v_sample.py:751-797, weighted = False): left node, left edge, right node, right edge,
 * nodes_in_edge_0.., edges_containing_node_0.. (0 = padding row); targets: fp32
 * [3][num_samples] = node_node, edge_edge, node_edge probabilities. */
int hge_hg2v_set_samples(hge_hg2v_model* m, const int32_t* features, const float* targets,
                         int64_t num_samples, int mem);
/* order: int32 [num_samples] permutation (Keras: np.random.shuffle per epoch).  *epoch_loss =
 * sample-weighted mean of the batch losses (what EarlyStopping(monitor="loss") watches). */
int hge_hg2v_fit_epoch(hge_hg2v_model* m, const int32_t* order, int batch_size, int mem,
                       double* epoch_loss);
/* Clusters the last hge_hg2v_fit_epoch launched (0 before the first). */
int hge_hg2v_last_clusters(const hge_hg2v_model* m);
int hge_hg2v_get_weights(hge_hg2v_model* m, float* node, float* edge, int mem);

/* Seeded sample -> train pipeline on the device (Hg2vModel.seeded / fit_device).
 *
 * hge_hg2v_create_seeded: hge_hg2v_create with the tables drawn on the device from U(-0.05, 0.05),
 * the range of Keras' 'uniform' initializer (hg2v_model.py:75-84): element (r, c) =
 * -0.05 + 0.1 * ((w >> 8) * 2^-24) in fp32, each operation rounded on its own, w = word c of the
 * Philox stream of item r (csrc/hge_philox.cuh), phase HGE_PHASE_INIT_NODES (13) for the node
 * table and HGE_PHASE_INIT_EDGES (14) for the edge table. */
int hge_hg2v_create_seeded(hge_ctx* ctx, int32_t node_rows, int32_t edge_rows, int dim, int num_neighbors,
                           int activation, int loss, uint64_t seed, hge_hg2v_model** out);
/* Allocates the model's own sample buffer (features [4 + 2k][num_samples] int32, targets
 * [3][num_samples] fp32) and sets its append cursor to 0; num_samples < 2^31.  Until every
 * record is appended hge_hg2v_fit_epoch refuses the model. */
int hge_hg2v_reserve_samples(hge_hg2v_model* m, int64_t num_samples);
/* Writes `count` records of sampler output at the cursor, as SamplesToModelInput(..., weighted =
 * False) (hg2v_sample.py:751-797) packs them: indices + 1, a NULL column is the padding index 0,
 * nbr_nodes / nbr_edges are [count, k] row-major and go to the k neighbour-node then the k
 * neighbour-edge columns; target slot prob_slot (0 node-node, 1 edge-edge, 2 node-edge) is prob[i]
 * (NaN -> 0), or prob_value when prob is NULL, every other slot 0 (prob_slot = -1: all three 0).
 * All pointers are device pointers.  Every index written is checked against its table on the
 * device; a bad one, or records past the reservation, is HGE_ERR_INVALID and leaves the cursor. */
int hge_hg2v_append_samples(hge_hg2v_model* m, const int32_t* left_node, const int32_t* left_edge,
                            const int32_t* right_node, const int32_t* right_edge, const int32_t* nbr_nodes,
                            const int32_t* nbr_edges, const float* prob, int prob_slot, float prob_value,
                            int64_t count);
/* Copies the sample buffer out, in the layout of hge_hg2v_set_samples. */
int hge_hg2v_get_samples(hge_hg2v_model* m, int32_t* features, float* targets, int mem);
/* A uniform random permutation of [0, n), n < 2^31, for epoch `epoch` (Keras: np.random.shuffle
 * per epoch, training_arrays.py).  Item i's 64-bit key is (word 2e << 32) | word 2e + 1 of its
 * Philox stream in phase HGE_PHASE_SHUFFLE (12); items are stably sorted by key, so ties go by
 * index.  The result is hge_hg2v_fit_epoch's order. */
int hge_shuffle_order(hge_ctx* ctx, uint64_t seed, uint32_t epoch, int64_t n, int32_t* order, int mem);

/* Personalized link-prediction classifiers (csrc/hge_lp_svm.cu): one RBF C-SVC per owner named by
 * a link (item, owner), as LP_EDGE_CLASSIFIERS / LP_NODE_CLASSIFIERS train them.  owner_side 1:
 * owners are edges, their members their nodes (edge -> node CSR), items the nodes; owner_side 0:
 * owners are nodes, members their edges, items the edges.  item_vectors: fp32 [items, d], d >= 1.
 * An owner with M members among N items trains on M (label +1, ascending) and k = min(N - M, 2M)
 * distinct non-members (label -1, ascending) chosen uniformly by Floyd's algorithm over the
 * positions of its ascending non-member list, from the Philox stream (csrc/hge_philox.cuh) of item =
 * owner row, phase HGE_PHASE_LP_EDGE_OWNERS (15) / HGE_PHASE_LP_NODE_OWNERS (16); k = N - M takes
 * them all and draws nothing.  The dual is libsvm's (Solver, WSS3, no shrinking) with K(x, z) =
 * exp(-gamma ||x - z||^2) in fp32, gradient and alpha in fp64, stop at tol, at most
 * max(10^7, 100 n) iterations.  out_keep[l] = 1 iff sum_i alpha_i y_i K(x_i, x_item) - rho > 0
 * (out_decision, optional, receives that value).  An owner without members rejects its links
 * (rho = +inf), one whose members are every item keeps them (rho = -inf); neither has points.
 * Owners of more than 32 points are solved in batches whose workspace fits workspace_mb megabytes
 * (0 = 2048; 24 + 4 d bytes a point); a single larger owner is its own batch, one the device cannot
 * hold is HGE_ERR_NOMEM.  Besides that the call holds 16 bytes a training point and 24 a
 * link.  Everything is bit-identical for every workspace_mb and from run to run.
 * All array pointers are device pointers except out_counts and phase_ms (host, optional):
 *   out_counts[3] = { named owners U, training points T, owners that hit the iteration cap };
 *   phase_ms[4]   = milliseconds of grouping, negatives, solve and predict, each ended by a
 *                   stream synchronise (only when phase_ms is given).
 * Optional model outputs, named owners in ascending owner id: owner_ids [U], owner_rho [U],
 * owner_iters [U], owner_offset [U + 1] (first training point of each owner); point_ids [T] and
 * point_coef [T] (alpha_i y_i) in training order, T <= point_capacity (U <= num_links).  A link
 * naming an item or owner out of range, or a bad owner_side, is HGE_ERR_INVALID and nothing is
 * written. */
int hge_lp_svm_predict(hge_ctx* ctx, hge_incidence* inc, int owner_side, const float* item_vectors, int d,
                       const int32_t* link_items, const int32_t* link_owners, int64_t num_links, uint64_t seed,
                       double C, double gamma, double tol, int64_t workspace_mb, uint8_t* out_keep,
                       double* out_decision, int64_t* out_counts, int32_t* owner_ids, double* owner_rho,
                       int64_t* owner_iters, int64_t* owner_offset, int32_t* point_ids, double* point_coef,
                       int64_t point_capacity, double* phase_ms);

/* Node-edge link-prediction classifier (csrc/hge_lp_node_edge.cu), the GPU form of the classifier
 * LP_NODE_EDGE_CLASSIFIER passes to NodeEdgeEmbeddingPrediction.  Not a port of the reference's
 * Keras model (its architecture is not recorded): a model of the usual Keras kind,
 *   x = [xn[n], xe[e]] (2d), h = relu(W1^T x + b1) (W1 [2d, hidden]), p = sigmoid(w2 . h + b2),
 * 1 <= d <= 256, 1 <= hidden <= 256.
 *
 * hge_lp_node_edge_train: training set, initialisation and `epochs` epochs on the device.
 *   Samples 0 .. nnz - 1 (label 1) are the incidences of `inc` in CSR order; sample nnz + i
 *   (label 0) is a non-incidence drawn uniformly, with replacement, from the S = N E - nnz of them:
 *   r = ((w0 << 32) | w1) & mask from the Philox stream (csrc/hge_philox.cuh) of item i, phase
 *   HGE_PHASE_LP_NODE_EDGE_NEG (17), redrawn while r >= S (mask = smallest 2^k - 1 >= S - 1); node n
 *   with C[n] <= r < C[n + 1] (C = exclusive prefix sum of E - deg(n)), edge = the (r - C[n])-th
 *   edge id not in n's row.  nnz = 0, S = 0 or 2 nnz >= 2^31 is HGE_ERR_INVALID.
 *   Weights: Keras glorot_uniform kernels, zero biases.  Row i of W1 is item i, w2 item 2d of
 *   phase HGE_PHASE_LP_NODE_EDGE_INIT (19), word j for column j; value -L + (2L) u with
 *   u = (w >> 8) 2^-24, each fp32 operation rounded on its own, L1 = fp32(sqrt(6 / (2d + hidden)))
 *   for W1, L2 = fp32(sqrt(6 / (hidden + 1))) for w2.
 *   Epoch e visits the samples in hge_shuffle_order's order with the keys of phase
 *   HGE_PHASE_LP_NODE_EDGE_SHUFFLE (18), in batches of `batch` (the last one ragged); loss per
 *   sample max(z, 0) - z y + log1p(exp(-|z|)) of the logit z, batch mean; Adagrad
 *   (acc += g^2, w -= lr g / (sqrt(acc) + eps), accumulators from 0) on every parameter after each
 *   batch.  epoch_loss[e] (host) = sum of the epoch's sample losses / 2 nnz.  Every sum has one
 *   fixed order, so weights and losses are bit-identical from run to run.
 *   W1 [2d, hidden] row-major, b1 [hidden], w2 [hidden], b2 [1]: caller-owned device arrays,
 *   written with the trained weights (epochs = 0: the initial ones).  xn fp32 [N, d], xe fp32
 *   [E, d] device.  phase_ms (host, optional) [1 + epochs]: milliseconds of the set-up (training
 *   set, initialisation), then of each epoch, each phase ended by a stream synchronise.  Besides
 *   the weights the call holds 8 bytes a sample for the training set, 4 for the epoch order (plus
 *   the sort's 20), and the accumulators.
 *
 * hge_lp_node_edge_samples: what hge_lp_node_edge_train trains on, for inspection: the training
 *   set (sample_nodes, sample_edges: device int32 [2 nnz]) and the orders of epochs 0 .. epochs - 1
 *   (orders: device int32 [epochs][2 nnz], may be NULL when epochs = 0).
 *
 * hge_lp_node_edge_predict: p of each link (link_nodes[l], link_edges[l]) into out_prob (fp32,
 *   optional) and out_keep[l] = p > 0.5 (optional); p depends on the model and the link's two rows
 *   only, never on the other links.  All array pointers are device pointers.  A link naming a node
 *   outside [0, num_nodes) or an edge outside [0, num_edges) is HGE_ERR_INVALID and nothing is
 *   written. */
int hge_lp_node_edge_train(hge_ctx* ctx, hge_incidence* inc, const float* xn, const float* xe, int d, int hidden,
                           uint64_t seed, int epochs, int batch, float lr, float eps, float* W1, float* b1, float* w2,
                           float* b2, double* epoch_loss, double* phase_ms);
int hge_lp_node_edge_samples(hge_ctx* ctx, hge_incidence* inc, uint64_t seed, int epochs, int32_t* sample_nodes,
                             int32_t* sample_edges, int32_t* orders);
int hge_lp_node_edge_predict(hge_ctx* ctx, const float* xn, int64_t num_nodes, const float* xe, int64_t num_edges,
                             int d, int hidden, const float* W1, const float* b1, const float* w2, const float* b2,
                             const int32_t* link_nodes, const int32_t* link_edges, int64_t num_links, float* out_prob,
                             uint8_t* out_keep);

/* ---- non-negative factorization of the incidence (csrc/hge_nmf.cu) -------------------------
 * The NMF baseline embedder (embedding.py:110-261 of the reference runs scikit-learn's NMF):
 * A [N, E] (the 0/1 incidence of `inc`) ~ W [N, k] H [k, E], 1 <= k <= 256, by scikit-learn's
 * coordinate descent (solver "cd", Frobenius loss, no regularization, no shuffling).  W and
 * Ht = H^T [E, k] are dense fp32 row-major; `mem` applies to both.
 *
 * hge_nmf_init: a seeded start in the style of scikit-learn's init="random": element (r, c) =
 *   scale * ((w >> 8) * 2^-24) in fp32, each operation rounded on its own, w = word c of the Philox
 *   stream (csrc/hge_philox.cuh) of item r, phase HGE_PHASE_NMF_W (20) for W and HGE_PHASE_NMF_H
 *   (21) for Ht.  NonNegativeFactorizationDevice passes scale = 2 fp32(sqrt(nnz / (N E k))).
 *
 * hge_nmf_fit: W and Ht hold the start on entry and the factors on return.  Iteration it updates
 *   every row of W from P = A Ht and G = Ht^T Ht, then every row of Ht from P = A^T W and
 *   G = W^T W (with the new W), and sums the projected-gradient violations of both; it stops after
 *   the first iteration when that sum is 0, when violation / violation of iteration 1 <= tol, or
 *   after max_iter.  *n_iter receives the iterations done, violations (host, optional,
 *   [max_iter]) each iteration's violation, phase_ms (host, optional, [3]) the milliseconds spent
 *   in the products, the Gram matrices and the coordinate-descent passes, summed over the
 *   iterations (CUDA events; each half then ends with an event wait).  Every sum has one fixed
 *   order (DESIGN.md section 9.10), so the result is bit-identical from run to run.  k outside
 *   [1, 256], max_iter < 1, tol negative or NaN, num_nodes / num_edges different from the
 *   incidence's, a start with a negative or non-finite entry, or a W or Ht that is all zero is
 *   HGE_ERR_INVALID; nothing is written then.  Besides the staged copies of host arguments the
 *   call holds 4 ld (N + E + max(N, E)) bytes (ld = k rounded up to a multiple of 4), one k x k
 *   partial per 4096 rows and 8 bytes per 64 rows. */
int hge_nmf_init(hge_ctx* ctx, int32_t num_nodes, int32_t num_edges, int k, uint64_t seed, float scale, float* W,
                 float* Ht, int mem);
int hge_nmf_fit(hge_ctx* ctx, hge_incidence* inc, int32_t num_nodes, int32_t num_edges, int k, float* W, float* Ht,
                int max_iter, double tol, int mem, int* n_iter, double* violations, double* phase_ms);

/* ---- truncated SVD of the incidence (csrc/hge_svd.cu) ---------------------------------------
 * The SVD baseline embedder (embedding.py:110-261 of the reference): A [N, E] (the 0/1 incidence
 * of `inc`) ~ U diag(s) V^T by randomized subspace iteration with Rayleigh-Ritz (DESIGN.md section
 * 9.11).  The host drives the loop and does the l x l steps in f64; these entry points do the
 * work of size N or E.  Every dense array is fp32 row-major [rows, ld], ld = l rounded up to a
 * multiple of 4, with columns l .. ld - 1 zero; 1 <= l <= 256.  `mem` applies to the dense arrays;
 * gram, m, sigma and resid are host arrays.  Every sum has one fixed order, so every result is
 * bit-identical from run to run and for every launch setting.  The host loop, per iteration:
 *   hge_svd_half(side 0, X = Omega -> Y), M from eigh(G), hge_svd_rowmat(Y, M -> Q),
 *   hge_svd_half(side 1, Q -> Z),         M from eigh(G), hge_svd_rowmat(Z, M -> Omega)
 * with M = U~ diag(1 / sigma) (1 / sigma = 0 where sigma <= 1e-6 sigma_1), rounded to fp32.
 *
 * hge_svd_start: omega [num_edges, ld], element (r, c < l) = -1 + 2 ((w >> 8) 2^-24) in fp32, each
 *   operation rounded on its own, w = word c of the Philox stream (csrc/hge_philox.cuh) of item r
 *   in phase HGE_PHASE_SVD (22).
 * hge_svd_half: side 0: y [N, ld] = A x (x [E, ld]); side 1: y [E, ld] = A^T x (x [N, ld]); then
 *   gram [l, l] (f64) = y^T y over the first l columns: per entry an f64 fma chain in ascending row
 *   order within chunks of 4096 rows, the chunk partials added in ascending order.  phase_ms
 *   (optional, [2]): milliseconds of the product and of the Gram matrix (CUDA events).
 * hge_svd_rowmat: out [rows, ld] = y [rows, ld] (first l columns) times m [l, cols] (fp32, host),
 *   1 <= cols <= l; each entry one fp32 fma chain over r = 0 .. l - 1 ascending from +0; columns
 *   cols .. ld - 1 of out are 0.  out must not alias y.
 * hge_svd_flip: scikit-learn's svd_flip on the first k <= l columns of u [num_u_rows, ld] and
 *   v [num_v_rows, ld]: where the entry of largest magnitude of column i of u (lowest row on a
 *   tie) is negative, columns i of u and of v are negated.
 * hge_svd_residuals: resid[i] = || A v_i - sigma_i u_i ||_2 / sigma_0 for i < k (sigma [k], f64),
 *   with u [N, ld], v [E, ld]: the product A v, then per column d = (A v)[j,i] - sigma_i u[j,i] and
 *   sum d d in f64, each operation rounded on its own, in ascending row order within chunks of
 *   4096 rows, the chunk sums in ascending order; sigma_0 = 0 gives the unscaled norm.
 * Refused with HGE_ERR_INVALID before anything is written: l outside [1, 256], k or cols outside
 * [1, l], a sharded incidence, num_nodes / num_edges different from the incidence's, y == out. */
int hge_svd_start(hge_ctx* ctx, int32_t num_edges, int l, uint64_t seed, float* omega, int mem);
int hge_svd_half(hge_ctx* ctx, hge_incidence* inc, int side, int32_t num_nodes, int32_t num_edges, int l,
                 const float* x, float* y, double* gram, int mem, double* phase_ms);
int hge_svd_rowmat(hge_ctx* ctx, int64_t rows, int l, int cols, const float* y, const float* m, float* out,
                   int mem);
int hge_svd_flip(hge_ctx* ctx, int64_t num_u_rows, int64_t num_v_rows, int l, int k, float* u, float* v, int mem);
int hge_svd_residuals(hge_ctx* ctx, hge_incidence* inc, int32_t num_nodes, int32_t num_edges, int l, int k,
                      const float* u, const float* v, const double* sigma, double* resid, int mem);

/* ---- node2vec on the node-edge bipartite graph (csrc/hge_n2v.cu) ----------------------------
 * The node2vec baseline embedder (embedding.py:110-261 of the reference) on the bipartite graph of
 * V = N + E vertices (node r is vertex r, edge c is vertex N + c); DESIGN.md section 9.12.  Every
 * array argument is a DEVICE pointer.  The host loop:
 *   hge_n2v_walks -> walks, counts; hge_n2v_pairs twice (count, then emit); noise table cum from
 *   counts^0.75 (host); hge_n2v_init; hge_n2v_train_epoch for epoch = 0 .. epochs - 1.
 *
 * hge_n2v_walks: walks [num_walks V, walk_length] int32 (walk w starts at vertex w mod V; a walk
 *   from a vertex of degree 0 is that vertex followed by -1), counts [V] int64 the occurrences of
 *   every vertex in the walks.  Draws from Philox phase HGE_PHASE_N2V_WALK (23), item = walk.
 * hge_n2v_pairs: (center, context) int32 pairs [*num_pairs, 2] of word2vec's shrunk windows (phase
 *   HGE_PHASE_N2V_WINDOW (24), item = token), in ascending (token, context position) order.
 *   pairs = NULL only counts.  2^31 pairs or more, or capacity < the count, is HGE_ERR_INVALID
 *   (*num_pairs still receives the count).
 * hge_n2v_negatives: out [num_pairs, negative] int32, the negatives pair i draws in `epoch`
 *   (phase HGE_PHASE_N2V_NEG (26), item = epoch num_pairs + i) from the cumulative noise table cum
 *   [num_vertices + 1] int64 (cum[0] = 0, cum[V] > 0): vertex v with cum[v] <= r < cum[v + 1] for
 *   r uniform on [0, cum[V]).  Draws equal to the pair's context are included (training skips them).
 * hge_n2v_init: tin [V, dim] uniform on [-0.5 / dim, 0.5 / dim) (phase HGE_PHASE_N2V_INIT (27)),
 *   tout [V, dim] zero; 1 <= dim <= 256.
 * hge_n2v_train_epoch: one epoch of mini-batch skip-gram with negative sampling over pairs [num_pairs,
 *   2] in the order of hge_shuffle_order in phase HGE_PHASE_N2V_SHUFFLE (25), batches of
 *   batch_pairs pairs.  Within a batch every coefficient g = lr (label - sigmoid(in[c] . out[x])) is
 *   computed from the tables at the batch start; then in[c] += sum g out[x] and out[x] += sum g in[c]
 *   over each row's contributions in ascending (pair position, slot) order.  lr of global batch t of
 *   T = epochs ceil(num_pairs / batch_pairs) is (float)(alpha - (alpha - min_alpha) (t / T)) in f64.
 *   *loss receives the epoch's sum of -log sigmoid(s+) - sum log sigmoid(-s-), in a fixed f64
 *   order.  plan_bytes bounds the per-chunk plan (0: 512 MiB); results do not depend on it.  The
 *   tables, *loss and the launch sequence are bit-identical from run to run.  Per epoch:
 *   1 + (radix passes) launches for the order, 3 per chunk (plan, two sorts) and 3 per batch. */
int hge_n2v_walks(hge_ctx* ctx, hge_incidence* inc, int num_walks, int walk_length, double p, double q,
                  uint64_t seed, int32_t* walks, int64_t* counts);
int hge_n2v_pairs(hge_ctx* ctx, const int32_t* walks, int64_t num_walk_items, int walk_length, int window,
                  uint64_t seed, int32_t* pairs, int64_t capacity, int64_t* num_pairs);
int hge_n2v_negatives(hge_ctx* ctx, int64_t num_pairs, const int64_t* cum, int32_t num_vertices, int negative,
                      uint64_t seed, int epoch, int32_t* out);
int hge_n2v_init(hge_ctx* ctx, int32_t num_vertices, int dim, uint64_t seed, float* tin, float* tout);
int hge_n2v_train_epoch(hge_ctx* ctx, int32_t num_vertices, int dim, float* tin, float* tout, const int32_t* pairs,
                        int64_t num_pairs, const int64_t* cum, int negative, uint64_t seed, int epoch, int epochs,
                        int batch_pairs, double alpha, double min_alpha, int64_t plan_bytes, double* loss);

/* ---- node2vec on a weighted clique expansion (csrc/hge_n2v_clique.cu) -----------------------
 * Walks of node2vec on one weighted clique expansion of the incidence, drawn from the incidence
 * without building the expansion; DESIGN.md section 9.13.  side 0: V = N node vertices, w(u, x) =
 * number of edges holding both; side 1: V = E edge vertices, w(c, y) = number of shared members
 * (the side convention of hge_row_span).  Every array argument is a DEVICE pointer, with the
 * contract of hge_n2v_walks: walks [num_walks V, walk_length] int32, walk w starting at vertex
 * w mod V; a vertex with S(v) = sum over its edges e of (|e| - 1) = 0 gives that vertex followed
 * by -1; counts [V] int64 the occurrences of every vertex.  Draws from Philox phase
 * HGE_PHASE_N2V_CLIQUE_WALK (28), item = walk.  One int64 per incidence of the side is allocated
 * for the call.  The pairs, noise table and training of the bipartite walker apply unchanged
 * (hge_n2v_pairs, hge_n2v_init, hge_n2v_train_epoch with num_vertices = V).
 * Refused with HGE_ERR_INVALID before anything runs: NULL pointers, a sharded incidence, side not
 * 0 or 1, num_walks or walk_length < 1, p or q not positive and finite, max / min of (q, p q, p)
 * above 65536 (the bound on the expected proposals per step), a side without vertices. */
int hge_n2v_clique_walks(hge_ctx* ctx, hge_incidence* inc, int side, int num_walks, int walk_length, double p,
                         double q, uint64_t seed, int32_t* walks, int64_t* counts);

/* ---- hypergraph.proto wire format (host code; all pointers are host pointers) --------------
 * The data formats either side of the path: a serialized Hypergraph (hypergraph.proto:6-23) is
 * read straight into arrays, replacing the per-incidence Python loops of ToCsrMatrix /
 * ToEdgeCsrMatrix (hypergraph_util.py:96-135) and CompressRange / Relabel (:198-244); the result
 * of EmbedAlgebraicDistance is written as a serialized HypergraphEmbedding (:26-35), replacing
 * the per-row packing loop (algebraic_distance.py:169-174).  Map entries are reported in wire
 * order (the producing serializer's order, which need not be its map iteration order);
 * duplicate keys: the last entry wins. */
typedef struct hge_hypergraph hge_hypergraph;
typedef struct hge_embedding hge_embedding;

int hge_hypergraph_parse(const void* buf, size_t len, hge_hypergraph** out);
int hge_hypergraph_destroy(hge_hypergraph* hg);
/* sizes4 = { node entries, edge entries, sum len(node.edges), sum len(edge.nodes) } */
int hge_hypergraph_sizes(const hge_hypergraph* hg, int64_t* sizes4);
/* Per side: ids [entries], row pointers [entries + 1], members in stored order (duplicates
 * kept), weights (default 1).  Any output may be NULL. */
int hge_hypergraph_arrays(const hge_hypergraph* hg, int32_t* node_ids, int64_t* node_ptr,
                          int32_t* node_edges, float* node_weight, int32_t* edge_ids,
                          int64_t* edge_ptr, int32_t* edge_nodes, float* edge_weight);
/* CompressRange + ToCsrMatrix + transpose in one pass (algebraic_distance.py:133-146): ids are
 * replaced by their rank among the sorted keys, connections come from node.edges only, column
 * ids are sorted and duplicates collapse.  sorted_*_ids are the inverse maps.  n2e_idx / e2n_idx
 * need room for sum len(node.edges) entries; *nnz_out is the number stored.  An edge id that is
 * not a key of the edge map is HGE_ERR_INVALID (Relabel asserts, hypergraph_util.py:207). */
int hge_hypergraph_compress(const hge_hypergraph* hg, int32_t* sorted_node_ids,
                            int32_t* sorted_edge_ids, int64_t* n2e_ptr, int32_t* n2e_idx,
                            int64_t* e2n_ptr, int32_t* e2n_idx, int64_t* nnz_out);

/* Serialized HypergraphEmbedding from dense fp32 [num_nodes, R] / [num_edges, R] rows keyed by
 * strictly ascending ids, plus dim and method_name (NULL: absent): field for field the bytes
 * the protobuf runtime emits for the message the reference builds (proto2: floats unpacked),
 * with the map entries in ascending key order. */
int hge_embedding_wire_size(const int32_t* node_ids, int64_t num_nodes, const int32_t* edge_ids,
                            int64_t num_edges, int32_t R, int32_t dim, const char* method_name,
                            size_t* out);
int hge_embedding_write(const int32_t* node_ids, int64_t num_nodes, const float* xn,
                        const int32_t* edge_ids, int64_t num_edges, const float* xe, int32_t R,
                        int32_t dim, const char* method_name, void* out, size_t capacity,
                        size_t* written);
/* The reverse (input of AlgebraicDistanceSamples / WeightByDistance): ids in wire order, row
 * pointers into the value arrays (rows may be ragged), *dim = -1 when the field is absent. */
int hge_embedding_parse(const void* buf, size_t len, hge_embedding** out);
int hge_embedding_destroy(hge_embedding* emb);
int hge_embedding_sizes(const hge_embedding* emb, int64_t* sizes4, int32_t* dim);
int hge_embedding_arrays(const hge_embedding* emb, int32_t* node_ids, int64_t* node_ptr,
                         float* node_values, int32_t* edge_ids, int64_t* edge_ptr,
                         float* edge_values);

#ifdef __cplusplus
}
#endif
#endif /* HGE_B200_H_ */
