"""node2vec on a weighted clique expansion, restated in tests/n2v_clique_ref.py, on the CPU: the
restated walks follow node2vec's second-order rule and its first step on the expansion built
with scipy (chi-square), vertices without expansion neighbours give one-vertex walks, the float64
pipeline over the restated walks separates the communities of a planted partition (the bar the
GPU test holds the device to), and Node2VecCliqueDevice refuses bad arguments before anything is
computed."""
import numpy as np
import pytest
import scipy.sparse as sps
from scipy import stats

import n2v_clique_ref as cref
from oracle import node2vec_ref as ref

PQ = [(1.0, 1.0), (0.25, 4.0), (4.0, 0.25)]

# Planted-partition quality settings, shared with the GPU test.  The float64 pipeline reaches AUC
# 0.9377 (nodes) and 0.9936 (edges) here (DESIGN section 9.13); each bar is that value - 0.02.
QUALITY = dict(dim=32, walk_length=20, num_walks=5, p=1.0, q=1.0, window=5, negative=5, epochs=5, batch_pairs=256,
               seed=0)
AUC_BAR = {0: 0.917, 1: 0.973}


def community_labels(side):
  """communities of the vertices of ref.planted_partition() (8 of 40 nodes, 8 of 20 edges)"""
  return np.arange(320 if side == 0 else 160) // (40 if side == 0 else 20)


def _graph():
  A = sps.random(16, 10, density=0.3, random_state=4, format="csr")
  A.data[:] = 1
  return A


def _groups(a, b):
  out = {}
  for i, key in enumerate(zip(a.tolist(), b.tolist())):
    out.setdefault(key, []).append(i)
  return {k: np.asarray(v) for k, v in out.items()}


def _chi_square(groups, nxt, weights_of):
  """pooled chi-square statistic and degrees of freedom of the next-vertex counts of every group
  against weights_of(key) -> (candidates, weights)"""
  chi, dof = 0.0, 0
  for key, idx in groups.items():
    cand, wt = weights_of(key)
    got = np.array([np.sum(nxt[idx] == x) for x in cand])
    assert got.sum() == len(idx), "a step left the expansion's neighbours"
    if len(cand) < 2:
      continue
    expected = len(idx) * wt / wt.sum()
    chi += float(np.sum((got - expected) ** 2 / expected))
    dof += len(cand) - 1
  return chi, dof


@pytest.mark.parametrize("side", [0, 1])
@pytest.mark.parametrize("pq", PQ)
def test_walks_follow_the_second_order_rule(side, pq):
  """Step 2 of every walk, grouped by (t, v): counts of the next vertex x against alpha(t, x)
  w(v, x), alpha = 1/p (x = t), 1 (x shares an edge with t), 1/q otherwise, with w and the
  adjacency taken from the materialized expansion."""
  p, q = pq
  A = _graph()
  Wx = cref.expansion(A, side).toarray()
  walks, _ = cref.clique_walks(A, side, 1500, 3, p, q, seed=9)
  w = walks[walks[:, 2] >= 0].astype(np.int64)

  def weights_of(key):
    t, v = key
    cand = np.nonzero(Wx[v])[0]
    alpha = np.where(cand == t, 1 / p, np.where(Wx[t, cand] > 0, 1.0, 1 / q))
    return cand, alpha * Wx[v, cand]

  chi, dof = _chi_square(_groups(w[:, 0], w[:, 1]), w[:, 2], weights_of)
  assert dof > 50
  assert stats.chi2.sf(chi, dof) >= 1e-3, (chi, dof)


@pytest.mark.parametrize("side", [0, 1])
def test_first_step_is_the_weighted_first_order_step(side):
  """Step 1, grouped by the start v: counts against w(v, x) / S(v)."""
  A = _graph()
  Wx = cref.expansion(A, side).toarray()
  walks, _ = cref.clique_walks(A, side, 3000, 2, 0.25, 4.0, seed=3)
  w = walks[walks[:, 1] >= 0].astype(np.int64)

  def weights_of(key):
    cand = np.nonzero(Wx[key[0]])[0]
    return cand, Wx[key[0], cand].astype(np.float64)

  chi, dof = _chi_square(_groups(w[:, 0], np.zeros(len(w), np.int64)), w[:, 1], weights_of)
  assert dof > 50 if side == 0 else dof > 20
  assert stats.chi2.sf(chi, dof) >= 1e-3, (chi, dof)


def shape_graph():
  """random incidence with an isolated node (0), an empty edge (0), and node 1 alone in edge 1"""
  A = sps.random(60, 25, density=0.12, random_state=0, format="lil")
  A[0, :] = 0
  A[:, 0] = 0
  A[1, :] = 0
  A[:, 1] = 0
  A[1, 1] = 1
  A = sps.csr_matrix(A)
  A.data[:] = 1
  A.eliminate_zeros()
  return A


@pytest.mark.parametrize("side", [0, 1])
def test_walk_shape(side):
  A = shape_graph()
  S = np.asarray(cref.expansion(A, side).sum(axis=1)).ravel()
  isolated = np.nonzero(S == 0)[0]
  assert {0, 1} <= set(isolated.tolist())
  walks, counts = cref.clique_walks(A, side, 2, 10, 4.0, 0.25, seed=1)
  start = walks[:, 0].astype(np.int64)
  lone = np.isin(start, isolated)
  assert np.all(walks[lone, 1:] == -1)
  assert np.all(walks[~lone] >= 0)
  assert counts.sum() == np.sum(walks >= 0)


def test_quality_bar_of_the_float64_pipeline():
  A = ref.planted_partition()
  for side in (0, 1):
    X, losses = cref.embed64(A, side, **QUALITY)
    assert np.all(np.diff(losses) < 0)
    assert cref.community_auc(X, community_labels(side)) >= AUC_BAR[side]


@pytest.mark.parametrize("kw, match", [
    (dict(side="nodes"), "side"), (dict(side=0), "side"), (dict(p=0.0), "p ="), (dict(q=float("nan")), "q ="),
    (dict(p=1e-3, q=1e3), "max / min"), (dict(p=1e-200, q=1e-200), "max / min"), (dict(dimension=0), "dimension"),
    (dict(walk_length=0), "walk_length"), (dict(num_walks=0), "num_walks"), (dict(batch_pairs=0), "batch_pairs"),
])
def test_refusals_before_anything_is_computed(kw, match):
  from hypergraphembedding_b200 import Node2VecCliqueDevice
  args = dict(dimension=8)
  args.update(kw)
  dimension = args.pop("dimension")
  with pytest.raises(AssertionError, match=match):
    Node2VecCliqueDevice(_graph(), dimension, **args)


def test_edge_seed_matches_library():
  from hypergraphembedding_b200.node2vec import clique_edge_seed
  for seed in (0, 4, -1, 2**64 - 1, 0x9E3779B97F4A7C15):
    assert clique_edge_seed(seed) == cref.edge_seed(seed)
  assert clique_edge_seed(0) != 0
