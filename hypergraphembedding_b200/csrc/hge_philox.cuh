// Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC'11) and the
// word-stream layout of the device sampler (csrc/hge_device_sampler.cu).  oracle/
// device_sampler_ref.py restates everything in this file in numpy; oracle/seeded_training_ref.py
// restates the training phases (epoch order, initial tables), oracle/lp_svm_ref.py the negatives of
// the link-prediction classifiers, oracle/lp_node_edge_ref.py the training set, epoch orders and
// initial weights of the node-edge classifier, oracle/nmf_ref.py the factorization's start, oracle/svd_ref.py
// the truncated SVD's start, oracle/node2vec_ref.py the walks, windows, negatives, epoch orders and
// initial table of node2vec, tests/n2v_clique_ref.py node2vec's walks on a clique expansion.
//
// Layout.  Every item owns one stream of 32-bit words:
//   key     = { (uint32)seed, (uint32)(seed >> 32) }
//   counter = { block, (uint32)item, (uint32)(item >> 32), phase }
// block 0 gives words 0..3 (x, y, z, w of the Philox output), block 1 words 4..7, and so on.
// `item` is the row id for pair draws and the record's index inside its block for neighbour
// draws; `phase` names the block (HgePhase below), so no two blocks of one sampler call share a
// stream.  A result therefore depends only on (seed, phase, item) and the graph, never on how
// rows are batched or chunked.
//
// Bounded draws U[0, s) use Lemire's multiply-shift with rejection ("Fast random integer
// generation in an interval", 2019), exactly unbiased:
//   m = x * s (64 bit); if low32(m) < s: while low32(m) < (2^32 - s) mod s: redraw x, m = x * s
//   result = m >> 32
#pragma once

#include <stdint.h>

// Phases of the record blocks, in the order the samplers emit them.  The negative edge-edge block
// appears twice, as in the reference (hg2v_sample.py:215-221).
enum HgePhase : uint32_t {
  HGE_PHASE_NN = 1,            // node-node pairs, rows of A * A^T
  HGE_PHASE_EE = 2,            // edge-edge pairs, rows of B * B^T
  HGE_PHASE_NE = 3,            // node-edge pairs, node rows (A, or (A * A^T) * A for HOBE)
  HGE_PHASE_EN = 4,            // edge-node pairs, edge rows (B, or (B * B^T) * B for HOBE)
  HGE_PHASE_NEIGHBORS = 5,     // neighbour arrays of the NE + EN records
  HGE_PHASE_NEG_NN = 6,
  HGE_PHASE_NEG_EE = 7,
  HGE_PHASE_NEG_EE_AGAIN = 8,
  HGE_PHASE_NEG_NE = 9,
  HGE_PHASE_NEG_EN = 10,
  HGE_PHASE_NEG_NEIGHBORS = 11,
  // hypergraph2vec training (csrc/hge_hg2v_train.cu): item = sample index, epoch e reads words
  // 2e and 2e + 1 as its 64-bit sort key
  HGE_PHASE_SHUFFLE = 12,
  // initial embedding tables: item = row, word c is column c
  HGE_PHASE_INIT_NODES = 13,
  HGE_PHASE_INIT_EDGES = 14,
  // negatives of the personalized link-prediction classifiers (csrc/hge_lp_svm.cu): item = owner
  // row, Floyd's selection over the owner's non-members
  HGE_PHASE_LP_EDGE_OWNERS = 15,
  HGE_PHASE_LP_NODE_OWNERS = 16,
  // node-edge link-prediction classifier (csrc/hge_lp_node_edge.cu): negative i of the training
  // set (item = i, 64-bit masked rejection over the non-incidences), the epoch orders (item =
  // sample index, as HGE_PHASE_SHUFFLE), the initial weights (item = row of W1, item 2d = w2;
  // word j is column j)
  HGE_PHASE_LP_NODE_EDGE_NEG = 17,
  HGE_PHASE_LP_NODE_EDGE_SHUFFLE = 18,
  HGE_PHASE_LP_NODE_EDGE_INIT = 19,
  // seeded start of the non-negative factorization (csrc/hge_nmf.cu): item = row of W (node) or
  // of H^T (edge), word c is column c
  HGE_PHASE_NMF_W = 20,
  HGE_PHASE_NMF_H = 21,
  // seeded start of the truncated SVD (csrc/hge_svd.cu): item = row of the start block Omega
  // (edge), word c is column c
  HGE_PHASE_SVD = 22,
  // node2vec (csrc/hge_n2v.cu): walk w (item = w) reads its words in step order, one below(d) for
  // the first step, then per step of a vertex of degree >= 2 one Bernoulli word and, when it does
  // not return, below(d - 1); token g = w L + i of the walks draws its window (item = g, one
  // below(window)); the epoch orders (item = pair index, as HGE_PHASE_SHUFFLE); negatives of pair i
  // in epoch e (item = e P + i, per sample two words (high, low) per 64-bit rejection round); the
  // initial input table (item = vertex, word c is column c)
  HGE_PHASE_N2V_WALK = 23,
  HGE_PHASE_N2V_WINDOW = 24,
  HGE_PHASE_N2V_SHUFFLE = 25,
  HGE_PHASE_N2V_NEG = 26,
  HGE_PHASE_N2V_INIT = 27,
  // node2vec on a clique expansion (csrc/hge_n2v_clique.cu): walk w (item = w) reads its words in
  // proposal order, per proposal two words (high, low) per 64-bit rejection round for the position
  // r in [0, S(v)), one below(|e| - 1) for the member, then one acceptance word when a' < m
  HGE_PHASE_N2V_CLIQUE_WALK = 28,
};

#ifdef __CUDACC__
#define HGE_PHILOX_FN __host__ __device__ __forceinline__
#else
#define HGE_PHILOX_FN inline
#endif

struct HgeWords4 {
  uint32_t v[4];
};

HGE_PHILOX_FN HgeWords4 hge_philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                          uint32_t k0, uint32_t k1) {
  for (int round = 0; round < 10; ++round) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    c0 = n0;
    c1 = (uint32_t)p1;
    c2 = n2;
    c3 = (uint32_t)p0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  HgeWords4 r;
  r.v[0] = c0;
  r.v[1] = c1;
  r.v[2] = c2;
  r.v[3] = c3;
  return r;
}

// The word stream of one item.
struct HgeStreamRng {
  uint32_t k0, k1, item_lo, item_hi, phase, block;
  HgeWords4 buf;
  int used;

  HGE_PHILOX_FN HgeStreamRng(uint64_t seed, uint32_t phase_, uint64_t item)
      : k0((uint32_t)seed), k1((uint32_t)(seed >> 32)), item_lo((uint32_t)item),
        item_hi((uint32_t)(item >> 32)), phase(phase_), block(0), used(4) {}

  HGE_PHILOX_FN uint32_t next() {
    if (used == 4) {
      buf = hge_philox4x32_10(block++, item_lo, item_hi, phase, k0, k1);
      used = 0;
    }
    return buf.v[used++];
  }

  // uniform on [0, s), s >= 1 (Lemire)
  HGE_PHILOX_FN uint32_t below(uint32_t s) {
    uint64_t m = (uint64_t)next() * s;
    if ((uint32_t)m < s) {
      const uint32_t t = (0u - s) % s;
      while ((uint32_t)m < t) m = (uint64_t)next() * s;
    }
    return (uint32_t)(m >> 32);
  }
};

