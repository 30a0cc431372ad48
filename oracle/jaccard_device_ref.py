"""Numpy restatement of the index and neighbour columns of WeightedJaccardSamplesDevice: the blocks
of oracle/device_sampler_ref.hobe_pairs (same factors, phases and Philox streams) with per-row counts
int(weight * num_samples).  Its probabilities are restated by the fp32 numpy restatement of
SparseWeightedJaccard / CentroidFromRows (tests/test_jaccard_restatement.py).

Test infrastructure only."""
import numpy as np
import scipy.sparse as sps

from oracle.device_sampler_ref import PHASE, _block, _concat, _node_edge, _pairs


def per_row(weights, count, base):
  if weights is None:
    return np.full(count, int(base), dtype=np.int64)
  return np.asarray([int(w * base) for w in weights], dtype=np.int64)


def jaccard_pairs(A, k, num_samples, seed=0, node_weights=None, edge_weights=None):
  """Index and neighbour columns of WeightedJaccardSamplesDevice; with unit weights those of
  hobe_pairs."""
  A = sps.csr_matrix(A)
  N, E = A.shape
  node_s, edge_s = per_row(node_weights, N, num_samples), per_row(edge_weights, E, num_samples)
  blocks = []
  for side, s, phase, l, r in ((0, node_s, "NN", "left_node", "right_node"),
                               (1, edge_s, "EE", "left_edge", "right_edge")):
    a, b = _pairs(A, side, 2, s, seed, PHASE[phase], False)
    blocks.append(_block(len(a), k, **{l: a, r: b}))
  blocks.append(_node_edge(A, k, node_s, edge_s, 3, seed, ("NE", "EN", "NEIGHBORS"), False, False))
  return _concat(blocks)
