"""hge_lp_node_edge_train / _predict and NodeEdgeClassifierDevice on the GPU: the training set, every
epoch order and the initial weights bit-equal to their restatement (oracle/lp_node_edge_ref.py); the
trained weights and losses against the float64 trainer over the range of d, hidden, batch sizes and
epochs; bit-equal weights, losses and probabilities from run to run and batch to batch; the
proto-level predictor against NodeEdgeEmbeddingPrediction with the fitted classifier; the registry
and the global RNGs left alone; the refusals; the planted-community accuracy; a 100 000-node run."""
import functools
import random

import numpy as np
import pytest
import scipy.sparse as sps

from conftest import csr_from_pairs, hypergraph_from_pairs
from oracle import lp_node_edge_ref as ref
from test_lp_node_edge_host import PLANTED_ACCURACY, PLANTED_KW, PLANTED_SEED, planted_accuracy

pytestmark = pytest.mark.gpu

TOL = 2e-4   # trained weights and epoch losses against the float64 trainer (DESIGN 9.3 / 9.9)


def _graph(seed=0, N=40, E=20, p=0.25):
  rng = np.random.RandomState(seed)
  A = sps.csr_matrix((rng.rand(N, E) < p).astype(np.int8))
  A.sort_indices()
  return A


def _vectors(A, d, seed=1):
  rng = np.random.RandomState(seed)
  return ((rng.randn(A.shape[0], d) * 0.5).astype(np.float32), (rng.randn(A.shape[1], d) * 0.5).astype(np.float32))


def _ev():
  from hypergraphembedding_b200 import evaluation_util as ev
  return ev


def _samples(A, seed, epochs):
  from hypergraphembedding_b200 import _native
  from hypergraphembedding_b200.hg2v_sample import _Graph
  ctx = _native.default_context()
  inc = _Graph.from_csr(A).incidence(ctx)
  try:
    sn, se, orders = _native.lp_node_edge_samples(ctx, inc, seed, epochs)
  finally:
    inc.close()
  return sn.cpu().numpy(), se.cpu().numpy(), orders.cpu().numpy()


@pytest.mark.parametrize("shape,p,seed", [((40, 20), 0.25, 0), ((9, 7), 0.5, 3), ((300, 120), 0.02, 11)])
def test_training_set_and_orders_bit_exact(shape, p, seed):
  A = _graph(seed, *shape, p=p)
  sn, se, orders = _samples(A, seed, 3)
  nodes, edges, _ = ref.training_set(A.indptr, A.indices, A.shape[1], seed)
  assert np.array_equal(sn, nodes) and np.array_equal(se, edges)
  for e in range(3):
    assert np.array_equal(orders[e], ref.shuffle_order(seed, e, len(nodes)))


@pytest.mark.parametrize("d,hidden", [(1, 1), (3, 8), (32, 64), (33, 7), (256, 256)])
def test_initial_weights_bit_exact(d, hidden):
  A = _graph()
  xn, xe = _vectors(A, d)
  model = _ev().NodeEdgeClassifierDevice.fit(A, xn, xe, seed=4, hidden=hidden, epochs=0)
  for mine, theirs in zip(model.weights(), ref.init_weights(4, d, hidden)):
    assert mine.dtype == np.float32 and np.array_equal(mine, theirs)


CASES = [(1, 8, 7, 3), (3, 1, 1, 3), (32, 64, 256, 3), (33, 256, 7, 1), (200, 8, 1000, 3), (256, 256, 256, 3),
         (256, 64, 1, 1), (32, 64, 1000, 1)]


@pytest.mark.parametrize("d,hidden,batch,epochs", CASES)
def test_training_matches_float64(d, hidden, batch, epochs):
  A = _graph()
  xn, xe = _vectors(A, d)
  seed = 7
  nodes, edges, labels = ref.training_set(A.indptr, A.indices, A.shape[1], seed)
  assert len(nodes) % batch or batch == 1
  model = _ev().NodeEdgeClassifierDevice.fit(A, xn, xe, seed=seed, hidden=hidden, epochs=epochs, batch_size=batch)
  orders = [ref.shuffle_order(seed, e, len(nodes)) for e in range(epochs)]
  weights, losses = ref.train(xn, xe, nodes, edges, labels, ref.init_weights(seed, d, hidden), orders, batch)
  for mine, theirs in zip(model.weights(), weights):
    assert np.abs(mine - theirs).max() < TOL
  assert np.abs(model.losses - losses).max() < TOL


def test_reproducible_and_batch_independent():
  A = _graph(5)
  xn, xe = _vectors(A, 32)
  ev = _ev()
  m1 = ev.NodeEdgeClassifierDevice.fit(A, xn, xe, seed=3, hidden=64, epochs=2, batch_size=32)
  m2 = ev.NodeEdgeClassifierDevice.fit(A, xn, xe, seed=3, hidden=64, epochs=2, batch_size=32)
  for a, b in zip(m1.weights(), m2.weights()):
    assert np.array_equal(a, b)
  assert np.array_equal(m1.losses, m2.losses)
  rng = np.random.RandomState(0)
  L = 100000
  nodes, edges = rng.randint(0, A.shape[0], L), rng.randint(0, A.shape[1], L)
  together = m1.predict_links(nodes, edges)
  for i in (0, 1, 777, L - 1):
    assert together[i] == m1.predict_links(nodes[i:i + 1], edges[i:i + 1])[0]
  perm = rng.permutation(L)
  assert np.array_equal(m1.predict_links(nodes[perm], edges[perm]), together[perm])
  # predict() on concatenated rows runs the same kernel: the same bits
  x = np.concatenate([xn[nodes[:1000]], xe[edges[:1000]]], axis=1)
  assert np.array_equal(m1.predict(x), together[:1000])
  p64 = ref.predict(m1.weights(), xn, xe, nodes[:1000], edges[:1000])
  assert np.abs(together[:1000] - p64).max() < 1e-5


def _proto_case():
  from hypergraphembedding_b200 import HypergraphEmbedding
  rng = np.random.RandomState(8)
  pairs = [(3 * n + 1, 5 * e + 2) for n in range(30) for e in range(12) if rng.rand() < 0.2]
  hg = hypergraph_from_pairs(pairs)
  emb = HypergraphEmbedding()
  emb.dim = 6
  for n in hg.node:
    emb.node[n].values.extend(rng.randn(6).tolist())
  for e in hg.edge:
    emb.edge[e].values.extend(rng.randn(6).tolist())
  nodes, edges = sorted(hg.node), sorted(hg.edge)
  links = [(nodes[rng.randint(len(nodes))], edges[rng.randint(len(edges))]) for _ in range(300)]
  links += [(1000, edges[0]), (nodes[0], 1000), (2000, 3000)]   # absent node / edge
  return hg, emb, links


def _fit_from_proto(hg, emb, seed, **kw):
  nodes, edges = sorted(hg.node), sorted(hg.edge)
  nr, er = {n: i for i, n in enumerate(nodes)}, {e: i for i, e in enumerate(edges)}
  A = csr_from_pairs([(nr[n], er[e]) for n in hg.node for e in hg.node[n].edges], shape=(len(nodes), len(edges)))
  xn = np.asarray([emb.node[n].values for n in nodes], np.float32)
  xe = np.asarray([emb.edge[e].values for e in edges], np.float32)
  return _ev().NodeEdgeClassifierDevice.fit(A, xn, xe, seed=seed, **kw)


def test_proto_predictor_equals_host_hook_with_fitted_classifier():
  ev = _ev()
  hg, emb, links = _proto_case()
  got = ev.NodeEdgeEmbeddingPredictionDevice(hg, emb, links, seed=2, hidden=16, epochs=3, batch_size=32)
  want = ev.NodeEdgeEmbeddingPrediction(hg, emb, links,
                                        classifier=_fit_from_proto(hg, emb, 2, hidden=16, epochs=3, batch_size=32))
  assert got == want
  assert 0 < len(got) < len(links) - 3
  asked = [l for l in links if l in set(got)]
  assert got == asked


def test_registered_experiment_runs(monkeypatch):
  ev = _ev()
  before = dict(ev.EXPERIMENT_OPTIONS)
  hg, emb, links = _proto_case()
  monkeypatch.setattr(ev, "EXPERIMENT_OPTIONS", dict(ev.EXPERIMENT_OPTIONS))
  ev.RegisterExperiment("LP_NODE_EDGE_CLASSIFIER", functools.partial(ev.NodeEdgeEmbeddingPredictionDevice, seed=1))
  good = [(n, e) for n in sorted(hg.node)[:10] for e in hg.node[n].edges]
  member = {(n, e) for n in hg.node for e in hg.node[n].edges}
  bad = [l for l in links[:-3] if l not in member][:len(good)]
  lp = ev.LinkPredictionData(hypergraph=hg, embedding=emb, good_links=good, bad_links=bad, removal_prob=0.1)
  m = ev.RunLinkPredictionExperiment(lp, "LP_NODE_EDGE_CLASSIFIER")
  assert m.experiment_name == "LP_NODE_EDGE_CLASSIFIER" and len(m.records) == len(good) + len(bad)
  monkeypatch.undo()
  assert ev.EXPERIMENT_OPTIONS == before
  assert ev.EXPERIMENT_OPTIONS["LP_NODE_EDGE_CLASSIFIER"] is ev.NodeEdgeEmbeddingPrediction
  with pytest.raises(NotImplementedError):
    ev.NodeEdgeEmbeddingPrediction(hg, emb, links)


def test_global_rngs_untouched():
  ev = _ev()
  random.seed(123)
  np.random.seed(456)
  py, npy = random.getstate(), np.random.get_state()
  hg, emb, links = _proto_case()
  ev.NodeEdgeEmbeddingPredictionDevice(hg, emb, links, seed=0, epochs=1)
  assert random.getstate() == py
  after = np.random.get_state()
  assert after[0] == npy[0] and np.array_equal(after[1], npy[1]) and after[2:] == npy[2:]


def test_refusals():
  ev = _ev()
  A = _graph()
  xn, xe = _vectors(A, 4)
  m = ev.NodeEdgeClassifierDevice.fit(A, xn, xe, hidden=4, epochs=1)
  with pytest.raises(AssertionError):
    m.predict_links([A.shape[0]], [0])
  with pytest.raises(AssertionError):
    m.predict_links([0], [-1])
  big_n, big_e = _vectors(A, 257)
  with pytest.raises(AssertionError):
    ev.NodeEdgeClassifierDevice.fit(A, big_n, big_e, epochs=1)
  for hidden in (0, 257):
    with pytest.raises(AssertionError):
      ev.NodeEdgeClassifierDevice.fit(A, xn, xe, hidden=hidden, epochs=1)
  empty = sps.csr_matrix((5, 4), dtype=np.int8)
  with pytest.raises(AssertionError):
    ev.NodeEdgeClassifierDevice.fit(empty, *_vectors(empty, 4), epochs=1)
  full = sps.csr_matrix(np.ones((5, 4), dtype=np.int8))
  with pytest.raises(AssertionError):
    ev.NodeEdgeClassifierDevice.fit(full, *_vectors(full, 4), epochs=1)


def test_planted_communities_accuracy_on_device():
  A, xn, xe, pos, neg = ref.planted_communities()
  m = _ev().NodeEdgeClassifierDevice.fit(A, xn, xe, seed=PLANTED_SEED, **PLANTED_KW)
  acc = planted_accuracy(m.weights(), xn, xe, pos, neg)
  p = np.concatenate([m.predict_links(pos[:, 0], pos[:, 1]), m.predict_links(neg[:, 0], neg[:, 1])])
  dev_acc = (np.sum(p[:len(pos)] > 0.5) + np.sum(p[len(pos):] <= 0.5)) / len(p)
  assert acc >= PLANTED_ACCURACY and dev_acc >= PLANTED_ACCURACY


def test_zipf_100k_end_to_end():
  from hypergraphembedding_b200 import synthetic
  A = sps.csr_matrix(synthetic.zipf_hypergraph(100000, 50000, seed=2024))
  A.sort_indices()
  xn, xe = _vectors(A, 32)
  sn, se, orders = _samples(A, 9, 1)
  nodes, edges, _ = ref.training_set(A.indptr, A.indices, A.shape[1], 9)
  assert np.array_equal(sn, nodes) and np.array_equal(se, edges)
  assert np.array_equal(orders[0], ref.shuffle_order(9, 0, len(nodes)))
  m = _ev().NodeEdgeClassifierDevice.fit(A, xn, xe, seed=9, epochs=2)
  assert np.all(np.isfinite(m.losses)) and m.losses[1] < m.losses[0] < np.log(2) + 0.1
  p = m.predict_links(nodes[::97], edges[::97])
  assert np.all((p >= 0) & (p <= 1))
