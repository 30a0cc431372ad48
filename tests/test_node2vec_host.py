"""The node2vec restatement (oracle/node2vec_ref.py) on the CPU: its walks follow node2vec's general
second-order transition probabilities (distances from networkx on the bipartite graph) within a
chi-square bound; its fp32 trainer stays within 1e-5 of the float64 form; the float64 form's loss
falls every epoch on the youtube fixture at the default training settings; and Node2VecDevice
refuses bad arguments before anything is computed."""
import numpy as np
import pytest
import scipy.sparse as sps
from scipy import stats

from conftest import load_golden
from oracle import node2vec_ref as ref


def _graph():
  A = sps.random(14, 6, density=0.35, random_state=4, format="csr")
  A.data[:] = 1
  return A


@pytest.mark.parametrize("pq", [(1.0, 1.0), (0.25, 4.0), (4.0, 0.25)])
def test_walks_follow_the_second_order_rule(pq):
  """Step 2 of every walk, grouped by (t, v): counts of the next vertex x against weights 1/p
  (dist(t, x) = 0), 1 (dist 1) and 1/q (dist 2) normalised over v's neighbours; the pooled
  chi-square statistic must not be improbable (p-value >= 1e-3)."""
  import networkx as nx
  p, q = pq
  A = _graph()
  N, E = A.shape
  G = nx.Graph()
  G.add_nodes_from(range(N + E))
  coo = A.tocoo()
  G.add_edges_from(zip(coo.row.tolist(), (coo.col + N).tolist()))
  dist = dict(nx.all_pairs_shortest_path_length(G, cutoff=2))
  walks, _ = ref.walks(A, 3000, 3, p, q, seed=9)
  w = walks[walks[:, 2] >= 0].astype(np.int64)
  chi, dof = 0.0, 0
  for (t, v), idx in _groups(w[:, 0], w[:, 1]).items():
    nbrs = sorted(G.neighbors(v))
    if len(nbrs) < 2:
      assert np.all(w[idx, 2] == t)
      continue
    wt = np.array([1 / p if dist[t].get(x) == 0 else 1.0 if dist[t].get(x) == 1 else 1 / q for x in nbrs])
    expected = len(idx) * wt / wt.sum()
    got = np.array([np.sum(w[idx, 2] == x) for x in nbrs])
    assert got.sum() == len(idx)
    chi += float(np.sum((got - expected) ** 2 / expected))
    dof += len(nbrs) - 1
  assert dof > 50
  assert stats.chi2.sf(chi, dof) >= 1e-3, (chi, dof)


def _groups(a, b):
  out = {}
  for i, key in enumerate(zip(a.tolist(), b.tolist())):
    out.setdefault(key, []).append(i)
  return {k: np.asarray(v) for k, v in out.items()}


def test_fp32_trainer_within_bar_of_float64():
  A = _graph()
  walks, counts = ref.walks(A, 4, 20, 0.5, 2.0, 1)
  pairs = ref.pairs(walks, 5, 1)
  cum = ref.noise_table(counts)
  t32, o32 = ref.init_tables(2, sum(A.shape), 24)
  t64, o64 = t32.astype(np.float64), o32.astype(np.float64)
  for e in range(3):
    l32 = ref.train32(t32, o32, pairs, cum, 5, 2, e, 3, 64)
    l64 = ref.train64(t64, o64, pairs, cum, 5, 2, e, 3, 64)
    assert abs(l32 - l64) <= 1e-5 * abs(l64)
  assert np.max(np.abs(t32 - t64)) <= 1e-5 and np.max(np.abs(o32 - o64)) <= 1e-5


def test_float64_loss_falls_on_youtube_at_the_defaults():
  """Defaults of Node2VecDevice (window 10, 5 negatives, 5 epochs, alpha 0.025 -> 1e-4, the default
  batch_pairs); one walk of 20 vertices per vertex keeps the CPU run short."""
  from hypergraphembedding_b200.node2vec import DEFAULT_BATCH_PAIRS
  g = load_golden("algdist_youtube")
  nid, eid = np.unique(g["pairs"][:, 0]), np.unique(g["pairs"][:, 1])
  A = sps.csr_matrix((np.ones(len(g["pairs"])), (np.searchsorted(nid, g["pairs"][:, 0]),
                                                 np.searchsorted(eid, g["pairs"][:, 1]))), shape=(len(nid), len(eid)))
  walks, counts = ref.walks(A, 1, 20, 1.0, 1.0, 0)
  pairs = ref.pairs(walks, 10, 0)
  cum = ref.noise_table(counts)
  tin, tout = (t.astype(np.float64) for t in ref.init_tables(0, sum(A.shape), 32))
  losses = [ref.train64(tin, tout, pairs, cum, 5, 0, e, 5, DEFAULT_BATCH_PAIRS) for e in range(5)]
  assert np.all(np.isfinite(tin)) and np.all(np.isfinite(tout))
  assert np.all(np.diff(losses) < 0), losses


def test_noise_table_matches_library():
  from hypergraphembedding_b200.node2vec import noise_table
  counts = np.array([10, 0, 3, 1, 250, 7], np.int64)
  assert np.array_equal(noise_table(counts), ref.noise_table(counts))
  cum = noise_table(counts)
  assert cum[0] == 0 and cum[2] == cum[1] and cum[5] - cum[4] == 2**32


@pytest.mark.parametrize("kw, match", [
    (dict(p=0.0), "p ="), (dict(q=-1.0), "q ="), (dict(p=float("nan")), "p ="), (dict(q=float("inf")), "q ="),
    (dict(dimension=0), "dimension"), (dict(dimension=257), "dimension"), (dict(walk_length=0), "walk_length"),
    (dict(window=0), "window"), (dict(negative=-1), "negative"), (dict(epochs=0), "epochs"),
])
def test_refusals_before_anything_is_computed(kw, match):
  from hypergraphembedding_b200 import Node2VecDevice
  args = dict(dimension=8)
  args.update(kw)
  dimension = args.pop("dimension")
  with pytest.raises(AssertionError, match=match):
    Node2VecDevice(_graph(), dimension, **args)
