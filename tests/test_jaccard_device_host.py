"""The numpy restatement of WeightedJaccardSamplesDevice's index and neighbour columns
(oracle/jaccard_device_ref.py): with unit weights it is the HOBE restatement, with row weights row r
draws int(w_r * num_samples) samples.  The GPU tests pin the sampler to it bit for bit."""
import numpy as np
import scipy.sparse as sps

from oracle import device_sampler_ref as dref
from oracle import jaccard_device_ref as jref


def _graph():
  from hypergraphembedding_b200 import synthetic
  return synthetic.zipf_hypergraph(300, 150, seed=3)


def test_unit_weights_give_the_hobe_pairs():
  A = _graph()
  want = dref.hobe_pairs(A, 3, 6, seed=21)
  for weights in ((None, None), (np.ones(A.shape[0]), np.ones(A.shape[1]))):
    got = jref.jaccard_pairs(A, 3, 6, seed=21, node_weights=weights[0], edge_weights=weights[1])
    assert set(got) == set(want)
    for name in want:
      assert np.array_equal(got[name], want[name], equal_nan=got[name].dtype.kind == "f"), name


def test_row_weights_set_the_per_row_counts():
  A = sps.csr_matrix(_graph())
  N, E = A.shape
  rng = np.random.default_rng(5)
  nw, ew = rng.random(N) * 2, rng.random(E) * 2
  nw[:7] = 0
  got = jref.jaccard_pairs(A, 2, 10, seed=4, node_weights=nw, edge_weights=ew)
  want_n = np.asarray([int(w * 10) for w in nw])
  want_e = np.asarray([int(w * 10) for w in ew])
  cptr_nn, _, _ = dref.candidate_rows(A, 0, 2)
  cptr_ee, _, _ = dref.candidate_rows(A, 1, 2)
  cptr_ne, _, _ = dref.candidate_rows(A, 0, 3)
  cptr_en, _, _ = dref.candidate_rows(A, 1, 3)
  nn = (got["left_node"] >= 0) & (got["right_node"] >= 0)
  ee = (got["left_edge"] >= 0) & (got["right_edge"] >= 0)
  ne = (got["left_node"] >= 0) & (got["right_edge"] >= 0)
  assert np.array_equal(np.bincount(got["left_node"][nn], minlength=N), np.minimum(want_n, np.diff(cptr_nn)))
  assert np.array_equal(np.bincount(got["left_edge"][ee], minlength=E), np.minimum(want_e, np.diff(cptr_ee)))
  # node-edge block: node rows, then edge rows
  m = int(np.minimum(want_n, np.diff(cptr_ne)).sum())
  nodes, edges = got["left_node"][ne], got["right_edge"][ne]
  assert np.array_equal(np.bincount(nodes[:m], minlength=N), np.minimum(want_n, np.diff(cptr_ne)))
  assert np.array_equal(np.bincount(edges[m:], minlength=E), np.minimum(want_e, np.diff(cptr_en)))
  assert got["neigh_node"][ne].shape == (len(nodes), 2) and np.all(got["neigh_node"][~ne] == -1)
