"""node2vec on a hypergraph's node-edge bipartite graph on the GPU: the node2vec baseline embedder the
reference compares HOBE against (embedding.py:110-261 of the reference).

``Node2VecDevice`` walks the bipartite graph of V = N + E vertices (node r is vertex r, edge c is
vertex N + c) with node2vec's second-order rule, cuts word2vec's shrunk windows into (center,
context) pairs, and trains a skip-gram model with negative sampling in deterministic mini-batches
(DESIGN section 9.12).  ``Node2VecCliqueDevice`` runs the same pipeline on the weighted clique
expansion of the nodes or of the edges, walking it straight from the incidence (csrc/
hge_n2v_clique.cu, DESIGN section 9.13).  Walks, pairs, negatives and training run in
libhge_b200.so (csrc/hge_n2v.cu); this module sizes the buffers, builds the noise table and drives
the epochs.  Every draw comes from seeded Philox streams (phases 23-28), so numpy's global RNG and
Python's ``random`` are neither read nor advanced.
"""
import math

import numpy as np
import scipy.sparse as sps

from . import _native
from .algebraic_distance import make_incidence

MAX_DIM = 256
# Pairs per mini-batch; DESIGN section 9.12 records the float64 runs it was chosen from.
DEFAULT_BATCH_PAIRS = 256
# Node2VecCliqueDevice's sides, in the order of the library's side argument
SIDES = ("node", "edge")
# the clique walker's largest max / min of its scaled weights (q, p q, p); hge_n2v_clique_walks
# refuses the same
MAX_WEIGHT_RATIO = 65536.0


def check_arguments(dimension, walk_length, num_walks, p, q, window, negative, epochs, batch_pairs, side=None):
  """The refusals of Node2VecDevice and, with `side`, of Node2VecCliqueDevice, made before anything
  is computed."""
  assert 1 <= int(dimension) <= MAX_DIM, "dimension = %r not in [1, %d]" % (dimension, MAX_DIM)
  assert int(walk_length) >= 1, "walk_length = %r must be >= 1" % (walk_length,)
  assert int(num_walks) >= 1, "num_walks = %r must be >= 1" % (num_walks,)
  for name, v in (("p", p), ("q", q)):
    assert math.isfinite(float(v)) and float(v) > 0, "%s = %r must be positive and finite" % (name, v)
  assert int(window) >= 1, "window = %r must be >= 1" % (window,)
  assert int(negative) >= 0, "negative = %r must be >= 0" % (negative,)
  assert int(epochs) >= 1, "epochs = %r must be >= 1" % (epochs,)
  assert int(batch_pairs) >= 1, "batch_pairs = %r must be >= 1" % (batch_pairs,)
  if side is not None:
    assert side in SIDES, "side = %r must be 'node' or 'edge'" % (side,)
    a = (float(q), float(p) * float(q), float(p))
    ratio = max(a) / min(a) if min(a) > 0 else math.inf
    assert ratio <= MAX_WEIGHT_RATIO, ("p = %r, q = %r: max / min of (q, p q, p) = %g is above %g, the bound on the "
                                       "clique walker's expected proposals per step" % (p, q, ratio, MAX_WEIGHT_RATIO))


def noise_table(counts):
  """Cumulative int64 noise table [V + 1] of the unigram counts raised to 0.75 in float64:
  q_v = floor((c_v^0.75 / max_u c_u^0.75) 2^32), cum = [0, q_0, q_0 + q_1, ...]."""
  w = np.power(np.asarray(counts, dtype=np.float64), 0.75)
  q = np.floor((w / w.max()) * 2.0**32).astype(np.int64)
  return np.concatenate([[0], np.cumsum(q)]).astype(np.int64)


def _require_memory(torch, dev, needed, what):
  free, _ = torch.cuda.mem_get_info(dev)
  if needed > free:
    raise MemoryError("node2vec: %s needs %d bytes of device memory, %d are free" % (what, needed, free))


def Node2VecDevice(incidence, dimension, walk_length=80, num_walks=10, p=1.0, q=1.0, window=10, negative=5,
                   epochs=5, alpha=0.025, min_alpha=1e-4, batch_pairs=DEFAULT_BATCH_PAIRS, seed=0,
                   plan_bytes=0, timings=None):
  """node2vec embeddings of the N + E vertices of the N x E incidence pattern `incidence` (scipy
  sparse; every stored entry counts as 1).  Returns (X [V, dimension] float32, info): row r is node
  r, row N + c is edge c (the skip-gram input table).  info holds "losses" (per epoch), "num_pairs",
  "num_walks", "walk_length", "mean_walk_length" (valid vertices per walk) and "batch_pairs".
  plan_bytes bounds the training plan of one chunk of batches (0: the library's default); results
  do not depend on it.  `timings` (a dict) receives milliseconds of the walks, pairs and training
  (CUDA events).  The defaults are the published node2vec / word2vec ones."""
  check_arguments(dimension, walk_length, num_walks, p, q, window, negative, epochs, batch_pairs)
  A = _pattern(incidence)
  N, E = A.shape
  V = N + E
  assert 1 <= V < 2**31, "%d vertices" % V

  def walk(ctx, inc, walks, counts):
    _native.n2v_walks(ctx, inc, num_walks, walk_length, p, q, seed, walks, counts)

  return _node2vec(A, V, 0, walk, dimension, walk_length, num_walks, window, negative, epochs, alpha, min_alpha,
                   batch_pairs, seed, plan_bytes, timings)


def Node2VecCliqueDevice(incidence, dimension, side="node", walk_length=80, num_walks=10, p=1.0, q=1.0, window=10,
                         negative=5, epochs=5, alpha=0.025, min_alpha=1e-4, batch_pairs=DEFAULT_BATCH_PAIRS, seed=0,
                         plan_bytes=0, timings=None):
  """node2vec embeddings of the vertices of one weighted clique expansion of the N x E incidence
  pattern `incidence` (scipy sparse; every stored entry counts as 1), DESIGN section 9.13.
  side="node": the N nodes, w(u, x) = number of edges holding both; side="edge": the E edges,
  w(c, y) = number of shared members.  The walks are drawn from the incidence, so the expansion is
  never built; pairs, negatives and training are those of Node2VecDevice, with the same keywords,
  defaults, `info` and `timings`.  Returns (X [V, dimension] float32, info), row v = vertex v of
  the side.  A vertex with no neighbour in the expansion (only in single-member edges, or in none)
  has a walk of one vertex."""
  check_arguments(dimension, walk_length, num_walks, p, q, window, negative, epochs, batch_pairs, side=side)
  A = _pattern(incidence)
  V = A.shape[0] if side == "node" else A.shape[1]
  assert 1 <= V < 2**31, "%d vertices" % V
  s = SIDES.index(side)

  def walk(ctx, inc, walks, counts):
    _native.n2v_clique_walks(ctx, inc, s, num_walks, walk_length, p, q, seed, walks, counts)

  # the walker's row prefix: one int64 per incidence
  return _node2vec(A, V, 8 * A.nnz, walk, dimension, walk_length, num_walks, window, negative, epochs, alpha,
                   min_alpha, batch_pairs, seed, plan_bytes, timings)


def clique_edge_seed(seed):
  """The seed of the edge side of EmbedNode2VecCliqueDevice, so that the node and edge tables are
  not drawn from identical streams."""
  return (int(seed) & 0xFFFFFFFFFFFFFFFF) ^ 0x9E3779B97F4A7C15


def _pattern(incidence):
  A = sps.csr_matrix(incidence, dtype=np.float32)
  A.sum_duplicates()
  A.sort_indices()
  return A


def _node2vec(A, V, walk_extra_bytes, walk, dimension, walk_length, num_walks, window, negative, epochs, alpha,
              min_alpha, batch_pairs, seed, plan_bytes, timings):
  """The pipeline of both walkers over V vertices: walk(ctx, inc, walks, counts) fills the walks,
  then pairs, noise table, initial table and epochs.  walk_extra_bytes is the device memory the
  walker needs beyond its output."""
  import torch
  ctx = _native.default_context()
  dev = torch.device("cuda", ctx.device)
  ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)] if timings is not None else None
  inc = make_incidence(A, ctx=ctx)
  try:
    W = int(num_walks) * V
    _require_memory(torch, dev, W * int(walk_length) * 4 + V * 8 + walk_extra_bytes, "the walks")
    walks = torch.empty((W, int(walk_length)), dtype=torch.int32, device=dev)
    counts = torch.empty(V, dtype=torch.int64, device=dev)
    if ev:
      ev[0].record()
    walk(ctx, inc, walks, counts)
  finally:
    inc.close()
  if ev:
    ev[1].record()
  P = _native.n2v_pairs(ctx, walks, window, seed)
  S = int(negative) + 1
  table_bytes = 2 * V * int(dimension) * 4
  _require_memory(torch, dev, P * 8 + table_bytes + 8 * (V + 1) + 4 * P, "%d pairs" % P)
  pairs = torch.empty((P, 2), dtype=torch.int32, device=dev)
  _native.n2v_pairs(ctx, walks, window, seed, pairs)
  if ev:
    ev[2].record()
  counts_host = counts.cpu().numpy()
  mean_len = float((walks >= 0).sum().item()) / W
  del walks
  cum = torch.from_numpy(noise_table(counts_host)).to(dev)
  tin = torch.empty((V, int(dimension)), dtype=torch.float32, device=dev)
  tout = torch.empty_like(tin)
  _native.n2v_init(ctx, seed, tin, tout)
  losses = []
  for e in range(int(epochs)):
    losses.append(_native.n2v_train_epoch(ctx, tin, tout, pairs, cum, negative, seed, e, epochs, batch_pairs,
                                          alpha, min_alpha, plan_bytes))
  if ev:
    ev[3].record()
    ev[3].synchronize()
    timings.update(walks_ms=ev[0].elapsed_time(ev[1]), pairs_ms=ev[1].elapsed_time(ev[2]),
                   train_ms=ev[2].elapsed_time(ev[3]))
  info = {"losses": np.asarray(losses), "num_pairs": P, "num_walks": W, "walk_length": int(walk_length),
          "mean_walk_length": mean_len, "batch_pairs": int(batch_pairs), "slots": S}
  return tin.cpu().numpy(), info
