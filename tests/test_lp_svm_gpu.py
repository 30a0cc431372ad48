"""hge_lp_svm_predict and the device personalized classifiers: negatives bit-equal to their numpy
restatement (oracle/lp_svm_ref.py) on both sides; the exported model (coef, rho) against
scikit-learn fitted on the exported training sets, through its KKT gap and through decision values
recomputed from it on the host (ref.decision), with the keep mask's sign checked where
scikit-learn's value is clear of zero; every owner size class and the degenerate owners in one
call, bit-identical output for every workspace budget and run, the refusals, the untouched global
RNGs, the proto-level wrappers against the host predictors, and a 100 000-node run.  The device's
own coef, rho, iterations and decision values are pinned bit for bit to the restatement in
tests/test_lp_svm_exact_gpu.py."""
import functools
import random

import numpy as np
import pytest
import scipy.sparse as sps

from conftest import csr_from_pairs, hypergraph_from_pairs, load_golden
from oracle import lp_svm_ref as ref

pytestmark = pytest.mark.gpu


def _vectors(rows, d=16, seed=3):
  rng = np.random.RandomState(seed)
  return (rng.randn(rows, d) * 0.5 * np.sqrt(32.0 / d)).astype(np.float32)


def _youtube_plus():
  """The youtube fixture (50 edges, one of 2 217 members) plus edge 50 of 1 100 members (3 300
  points), edge 51 of 1 member, edge 52 without members and edge 53 holding every node."""
  pairs = load_golden("boolean_youtube_s10")["pairs"].astype(np.int64)
  N = int(pairs[:, 0].max()) + 1
  extra = [(n, 50) for n in range(1100)] + [(7, 51)] + [(n, 53) for n in range(N)]
  return csr_from_pairs(np.concatenate([pairs, np.asarray(extra)]), shape=(N, 54))


def _links(A, per_edge, count, seed):
  rng = np.random.RandomState(seed)
  N, E = A.shape
  return np.stack([rng.randint(0, N, count), rng.randint(0, E, count)], axis=1)


def _run(A, X, links, per_edge, **kw):
  from hypergraphembedding_b200 import evaluation_util as ev
  return ev.PersonalizedClassifierPredictionDevice(A, X, links, per_edge, return_model=True, **kw)


def _members(A, per_edge):
  M = sps.csr_matrix(A.T if per_edge else A)
  M.sort_indices()
  return M.indptr.astype(np.int64), M.indices.astype(np.int64)


def _check_model(A, X, links, per_edge, seed, keep, model, sklearn_owners=()):
  """negatives bit-equal to the restatement; sklearn and KKT on the owners `sklearn_owners`"""
  from sklearn.svm import SVC
  mptr, midx = _members(A, per_edge)
  items = X.shape[0]
  owner_col, item_col = (1, 0) if per_edge else (0, 1)
  named = np.unique(links[:, owner_col])
  assert model.owner_ids.tolist() == named.tolist()
  phase = ref.PHASE_LP_EDGE_OWNERS if per_edge else ref.PHASE_LP_NODE_OWNERS
  sets = ref.training_sets(mptr, midx, items, named, seed, phase)
  for u, o in enumerate(named.tolist()):
    pts = model.point_ids[model.offset[u]:model.offset[u + 1]]
    mem, neg = sets[o]
    assert pts.tolist() == mem.tolist() + neg.tolist(), o
    m = mptr[o + 1] - mptr[o]
    if len(pts) == 0:
      assert model.rho[u] == (np.inf if m == 0 else -np.inf)
      sel = links[:, owner_col] == o
      assert np.all(keep[sel] == (m > 0))
  for o in sklearn_owners:
    u = int(np.searchsorted(named, o))
    pts = model.point_ids[model.offset[u]:model.offset[u + 1]]
    coef = model.coef[model.offset[u]:model.offset[u + 1]]
    m = int(mptr[o + 1] - mptr[o])
    y = np.r_[np.ones(m), -np.ones(len(pts) - m)]
    Xo = X[pts]
    assert ref.kkt_gap(Xo, y, coef) <= 1e-3 + 1e-3
    sel = np.nonzero(links[:, owner_col] == o)[0]
    Z = X[links[sel, item_col]]
    want = SVC(C=1, gamma=0.1).fit(Xo, (y > 0).astype(int)).decision_function(Z)
    got = ref.decision(Xo, coef, model.rho[u], Z)
    assert np.abs(got - want).max() <= 5e-3, o
    sure = np.abs(want) > 5e-3
    assert np.array_equal(keep[sel][sure], want[sure] > 0), o


def test_edge_owners_of_every_size_class():
  A = _youtube_plus()
  X = _vectors(A.shape[0])
  sizes = np.diff(A.T.tocsr().indptr)
  big = int(np.argmax(sizes[:50]))
  assert sizes[big] == 2217
  small = [e for e in range(50) if 2 <= sizes[e] <= 10][:3]
  rng = np.random.RandomState(1)
  owners = [big, 50, 51, 52, 53] + small
  links = np.concatenate([np.stack([rng.randint(0, A.shape[0], 40), np.full(40, o)], axis=1) for o in owners] +
                         [_links(A, True, 300, 2)])
  keep, model = _run(A, X, links, True, seed=9)
  n = np.diff(model.offset)
  u = {o: int(np.searchsorted(model.owner_ids, o)) for o in owners}
  N = A.shape[0]
  assert n[u[51]] == 3 and n[u[50]] == 3300 and n[u[big]] == 2217 + min(N - 2217, 2 * 2217)
  assert n[u[52]] == 0 and n[u[53]] == 0
  assert any(0 < n[u[o]] <= 32 for o in small)
  _check_model(A, X, links, True, 9, keep, model, sklearn_owners=[big, 50, 51] + small)


@pytest.mark.parametrize("golden", ["boolean_rand25", "boolean_youtube_s10"])
def test_node_owners_equal_the_restatement(golden):
  A = csr_from_pairs(load_golden(golden)["pairs"])
  Xe = _vectors(A.shape[1], seed=4)
  links = _links(A, False, 2000, 5)
  keep, model = _run(A, Xe, links, False, seed=11)
  named = model.owner_ids
  _check_model(A, Xe, links, False, 11, keep, model, sklearn_owners=named[:: max(1, len(named) // 20)])


def test_budget_runs_and_link_order_change_no_bit():
  A = _youtube_plus()
  X = _vectors(A.shape[0])
  links = _links(A, True, 3000, 6)
  base, model = _run(A, X, links, True, seed=2)
  for mb in (1, 4, 0):
    keep, other = _run(A, X, links, True, seed=2, workspace_mb=mb)
    assert np.array_equal(keep, base)
    for f in ("rho", "iterations", "offset", "point_ids", "coef"):
      assert np.array_equal(getattr(other, f), getattr(model, f)), (mb, f)
  perm = np.random.RandomState(0).permutation(len(links))
  keep, other = _run(A, X, links[perm], True, seed=2)
  assert np.array_equal(keep, base[perm]) and np.array_equal(other.coef, model.coef)


def test_refusals_and_global_rngs():
  from hypergraphembedding_b200 import evaluation_util as ev
  A = csr_from_pairs(load_golden("boolean_rand25")["pairs"])
  X = _vectors(A.shape[0])
  random.seed(3)
  np.random.seed(3)
  py, npy = random.getstate(), np.random.get_state()
  ev.PersonalizedClassifierPredictionDevice(A, X, _links(A, True, 100, 1), True, seed=1)
  ev.PersonalizedClassifierPredictionDevice(A, _vectors(A.shape[1]), _links(A, False, 100, 1), False, seed=1)
  assert random.getstate() == py
  after = np.random.get_state()
  assert np.array_equal(after[1], npy[1]) and after[2] == npy[2]
  for bad in ([[A.shape[0], 0]], [[0, A.shape[1]]], [[-1, 0]]):
    with pytest.raises(AssertionError, match="outside"):
      ev.PersonalizedClassifierPredictionDevice(A, X, np.asarray(bad), True, seed=1)


def _communities(strays=False):
  """4 communities of 6 nodes, an edge per community (with `strays`, about 5 % more links at random)"""
  rng = np.random.RandomState(11)
  return hypergraph_from_pairs([(n, e) for n in range(24) for e in range(4)
                                if n // 6 == e or (strays and rng.rand() < 0.05)])


def test_wrappers_keep_what_the_host_predictors_keep():
  from hypergraphembedding_b200 import HypergraphEmbedding, evaluation_util as ev
  hg = _communities()
  emb = HypergraphEmbedding()
  emb.dim = 4
  for n in hg.node:
    emb.node[n].values.extend(np.eye(4)[n // 6].tolist())
  for e in hg.edge:
    emb.edge[e].values.extend(np.eye(4)[e].tolist())
  links = [(n, e) for n in range(24) for e in range(4)] + [(99, 0), (0, 99)]
  random.seed(0)
  for host, dev in ((ev.PersonalizedEdgeClassifierPrediction, ev.PersonalizedEdgeClassifierPredictionDevice),
                    (ev.PersonalizedNodeClassifierPrediction, ev.PersonalizedNodeClassifierPredictionDevice)):
    want = host(hg, emb, links)
    got = dev(hg, emb, links, seed=4)
    assert sorted(got) == sorted(want)
    asked = [l for l in links if l in set(got)]
    assert got == asked   # the asked order


def test_registered_wrappers_give_metrics():
  from hypergraphembedding_b200 import HypergraphEmbedding, evaluation_util as ev
  hg = _communities(strays=True)
  rng = np.random.RandomState(2)

  def embed(h):
    emb = HypergraphEmbedding()
    emb.dim = 2
    for n in h.node:
      emb.node[n].values.extend([float(n // 6), rng.rand() * 0.1])
    for e in h.edge:
      emb.edge[e].values.extend([float(e), 0.05])
    return emb

  random.seed(2)
  data = ev.PrepLinkPredictionExperiment(hg, 0.2, embed)
  for name, fn in (("LP_EDGE_DEVICE", ev.PersonalizedEdgeClassifierPredictionDevice),
                   ("LP_NODE_DEVICE", ev.PersonalizedNodeClassifierPredictionDevice)):
    ev.RegisterExperiment(name, functools.partial(fn, seed=7))
    try:
      m = ev.RunLinkPredictionExperiment(data, name)
    finally:
      del ev.EXPERIMENT_OPTIONS[name]
    assert m.experiment_name == name and len(m.records) == 2 * len(data.good_links)
    assert m.num_true_pos + m.num_false_neg == len(data.good_links)
    assert m.num_true_neg + m.num_false_pos == len(data.bad_links)


def test_a_member_without_a_vector_is_a_key_error():
  from hypergraphembedding_b200 import HypergraphEmbedding, evaluation_util as ev
  hg = _communities()
  emb = HypergraphEmbedding()
  emb.dim = 1
  for n in hg.node:
    if n != 0:
      emb.node[n].values.append(1.0)
  for e in hg.edge:
    emb.edge[e].values.append(0.0)
  with pytest.raises(KeyError):
    ev.PersonalizedEdgeClassifierPredictionDevice(hg, emb, [(1, 0)], seed=1)


def test_100k_nodes_both_sides():
  from hypergraphembedding_b200 import synthetic
  A = synthetic.zipf_hypergraph(100000, 50000, seed=2024)
  for per_edge in (True, False):
    X = _vectors(A.shape[0] if per_edge else A.shape[1], d=32, seed=5)
    links = _links(A, per_edge, 20000, 8)
    keep, model = _run(A, X, links, per_edge, seed=3)
    mptr, _ = _members(A, per_edge)
    owner_col = 1 if per_edge else 0
    named = np.unique(links[:, owner_col])
    m = (mptr[named + 1] - mptr[named])
    items = X.shape[0]
    want = np.where((m == 0) | (m == items), 0, m + np.minimum(items - m, 2 * m))
    assert np.array_equal(np.diff(model.offset), want)
    assert model.capped == 0 and np.all(model.iterations[want > 0] > 0)
    assert keep.dtype == bool and len(keep) == len(links)
    # negatives of a sample of owners against the restatement
    sample = named[:: max(1, len(named) // 200)]
    sub = links[np.isin(links[:, owner_col], sample)]
    k2, m2 = _run(A, X, sub, per_edge, seed=3)
    _check_model(A, X, sub, per_edge, 3, k2, m2)
