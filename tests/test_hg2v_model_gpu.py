"""hypergraph2vec training (hg2v_model.py:51-203, embedding.py:269-305) on the GPU against the
numpy restatement of the Keras semantics (oracle/hg2v_model_ref.py; Keras itself is absent, so
this part of the path is not pinned against it -- see the oracle's header).

Tolerance: the kernels accumulate fp32 and sum duplicated rows' gradients with atomics, the
restatement is float64; after hundreds of Adagrad steps the tables agree to 2e-4 absolute on
values of magnitude 0.05-1 (stated per test)."""
import numpy as np
import pytest

from conftest import hypergraph_from_pairs, load_golden
from oracle import hg2v_model_ref as ref

pytestmark = pytest.mark.gpu


def _random_problem(seed, nodes=300, edges=120, k=3, m=5000):
  rng = np.random.default_rng(seed)
  kind = rng.integers(0, 3, m)
  z = np.zeros(m, np.int32)
  ln = np.where(kind != 1, rng.integers(1, nodes + 1, m), z).astype(np.int32)
  rn = np.where(kind == 0, rng.integers(1, nodes + 1, m), z).astype(np.int32)
  le = np.where(kind == 1, rng.integers(1, edges + 1, m), z).astype(np.int32)
  re = np.where(kind != 0, rng.integers(1, edges + 1, m), z).astype(np.int32)
  nbr_n = [np.where(kind == 2, rng.integers(1, nodes + 1, m), z).astype(np.int32) for _ in range(k)]
  nbr_e = [np.where(kind == 2, rng.integers(1, edges + 1, m), z).astype(np.int32) for _ in range(k)]
  prob = rng.random(m).astype(np.float32)
  targets = [np.where(kind == 0, prob, 0).astype(np.float32), np.where(kind == 1, prob, 0).astype(np.float32),
             np.where(kind == 2, prob, 0).astype(np.float32)]
  return [ln, le, rn, re] + nbr_n + nbr_e, targets


class _Graph(object):
  """Just enough of a Hypergraph for the model constructors: the id ranges."""

  def __init__(self, nodes, edges):
    self.node, self.edge = range(nodes), range(edges)


@pytest.mark.parametrize("activation,loss,dim,k,batch", [
    ("relu", "mean_squared_error", 16, 3, 256),
    ("sigmoid", "kullback_leibler_divergence", 32, 2, 256),
    ("relu", "mean_squared_error", 5, 0, 100),
    ("sigmoid", "kullback_leibler_divergence", 70, 5, 333),
    ("relu", "mean_squared_error", 200, 1, 1000),
])
def test_epochs_match_the_float64_restatement(activation, loss, dim, k, batch):
  from hypergraphembedding_b200.hg2v_model import Hg2vModel
  feats, targets = _random_problem(dim + k, k=k)
  np.random.seed(4)
  model = Hg2vModel(_Graph(300, 120), dim, k, activation, loss)
  n0, e0 = model.weights()
  assert n0.shape == (301, dim) and e0.shape == (121, dim) and np.abs(n0).max() <= 0.05
  # larger initial values than keras' 0.05 make every term of the gradient matter
  rng = np.random.default_rng(1)
  model.close()
  n0 = rng.uniform(-0.7, 0.7, n0.shape).astype(np.float32)
  e0 = rng.uniform(-0.7, 0.7, e0.shape).astype(np.float32)
  model = _model_with_tables(n0, e0, k, activation, loss)
  model.set_samples(feats, targets)
  m = len(feats[0])
  orders = [np.random.default_rng(10 + e).permutation(m) for e in range(3)]
  got_losses = [model.fit_epoch(o, batch) for o in orders]
  got_n, got_e = model.weights()
  want_n, want_e, want_losses = ref.fit(n0, e0, feats, targets, k, activation,
                                        "kld" if loss.startswith("kull") else "mse", batch, 3,
                                        order=orders, min_delta=-1e9)
  assert np.allclose(got_losses, want_losses, rtol=2e-5, atol=1e-6), (got_losses, want_losses)
  assert np.abs(got_n - want_n).max() < 2e-4 and np.abs(got_e - want_e).max() < 2e-4
  assert np.abs(got_n - n0).max() > 0.01            # and it did train
  model.close()


@pytest.mark.parametrize("activation,loss,dim,k,batch", [
    ("relu", "mean_squared_error", 32, 3, 1024),
    ("sigmoid", "kullback_leibler_divergence", 16, 5, 4096),
    ("relu", "mean_squared_error", 70, 2, 5000),
])
def test_large_batches_on_several_clusters_match_the_restatement(activation, loss, dim, k, batch):
  """Batches of more than 256 samples run on one cluster per 256 samples with a global barrier
  between the phases: same result (up to the order of the gradient atomics) as the float64
  restatement and as the same epochs forced onto one cluster."""
  from hypergraphembedding_b200 import _native
  feats, targets = _random_problem(50 + dim, nodes=3000, edges=1200, k=k, m=20000)
  rng = np.random.default_rng(2)
  n0 = rng.uniform(-0.7, 0.7, (3001, dim)).astype(np.float32)
  e0 = rng.uniform(-0.7, 0.7, (1201, dim)).astype(np.float32)
  m = len(feats[0])
  orders = [np.random.default_rng(20 + e).permutation(m) for e in range(3)]
  want_n, want_e, want_losses = ref.fit(n0, e0, feats, targets, k, activation,
                                        "kld" if loss.startswith("kull") else "mse", batch, 3,
                                        order=orders, min_delta=-1e9)
  ctx = _native.default_context()
  results = []
  try:
    for cap in (0, 1):
      ctx.set_trainer_clusters(cap)
      model = _model_with_tables(n0, e0, k, activation, loss)
      model.set_samples(feats, targets)
      losses = [model.fit_epoch(o, batch) for o in orders]
      clusters = model.last_clusters
      results.append((model.weights(), losses, clusters))
      model.close()
      assert np.allclose(losses, want_losses, rtol=2e-5, atol=1e-6), (cap, losses, want_losses)
      got_n, got_e = results[-1][0]
      assert np.abs(got_n - want_n).max() < 2e-4 and np.abs(got_e - want_e).max() < 2e-4, cap
  finally:
    ctx.reset_tuning()
  assert results[0][2] > 1 and results[1][2] == 1, (results[0][2], results[1][2])


def _model_with_tables(n0, e0, k, activation, loss):
  import ctypes
  from hypergraphembedding_b200 import _native
  from hypergraphembedding_b200.hg2v_model import ACTIVATIONS, LOSSES, Hg2vModel
  model = Hg2vModel.__new__(Hg2vModel)
  model.ctx = _native.default_context()
  model.dimension, model.num_neighbors = n0.shape[1], k
  model.node_rows, model.edge_rows = n0.shape[0], e0.shape[0]
  handle = _native.c_vp()
  _native.check(model.ctx.lib.hge_hg2v_create(model.ctx.handle, n0.shape[0], e0.shape[0], n0.shape[1], k,
                                              ACTIVATIONS[activation], LOSSES[loss], _native.ptr(n0),
                                              _native.ptr(e0), _native.MEM_HOST, ctypes.byref(handle)))
  model.handle = handle
  return model


def test_fit_shuffles_with_the_global_rng_and_stops_early():
  from hypergraphembedding_b200.hg2v_model import EarlyStopping, UnweightedFloatModel
  feats, targets = _random_problem(3, k=2, m=3000)
  np.random.seed(5)
  model = UnweightedFloatModel(_Graph(300, 120), 8, 2)
  n0, e0 = model.weights()
  state = np.random.get_state()
  history = model.fit(feats, targets, batch_size=256, epochs=10,
                      callbacks=[EarlyStopping(monitor="loss", min_delta=2.5e-3)], verbose=0)
  got_n, got_e = model.weights()
  np.random.set_state(state)
  want_n, want_e, want_losses = ref.fit(n0, e0, feats, targets, 2, "relu", "mse", 256, 10,
                                        min_delta=2.5e-3)
  assert 1 < len(history.history["loss"]) == len(want_losses) < 10   # EarlyStopping fired
  assert np.allclose(history.history["loss"], want_losses, rtol=1e-4, atol=1e-6)
  assert np.abs(got_n - want_n).max() < 2e-4 and np.abs(got_e - want_e).max() < 2e-4


def test_bad_indices_are_refused():
  import ctypes
  from hypergraphembedding_b200.hg2v_model import UnweightedFloatModel
  feats, targets = _random_problem(0, k=1, m=50)
  model = UnweightedFloatModel(_Graph(300, 120), 4, 1)
  feats[0][7] = 302                                  # rows are 0 .. 300
  good, good_targets = _random_problem(1, k=1, m=40)
  model.set_samples(good, good_targets)
  with pytest.raises(AssertionError):
    model.set_samples(feats, targets)
  with pytest.raises(AssertionError):
    model.set_samples(feats[:-1], targets)
  # a refused call leaves the samples of the last accepted one
  assert model.num_samples == 40
  got, got_targets = model.samples()
  assert all(np.array_equal(a, b) for a, b in zip(got + got_targets, good + good_targets))
  model.close()
  # and on a fresh model, none: there is nothing to read back and nothing to train on
  from hypergraphembedding_b200 import _native
  fresh = UnweightedFloatModel(_Graph(300, 120), 4, 1)
  try:
    with pytest.raises(AssertionError):
      fresh.set_samples(feats, targets)
    lib = fresh.ctx.lib
    _native.check(lib.hge_hg2v_get_samples(fresh.handle, None, None, _native.MEM_HOST), "hge_hg2v_get_samples")
    order = np.arange(50, dtype=np.int32)
    loss = ctypes.c_double()
    with pytest.raises(AssertionError, match="no samples"):
      _native.check(lib.hge_hg2v_fit_epoch(fresh.handle, _native.ptr(order), 8, _native.MEM_HOST,
                                           ctypes.byref(loss)))
  finally:
    fresh.close()


@pytest.mark.parametrize("method", ["HG2V_ALG_DIST", "HG2V_BOOLEAN", "HG2V_NEIGH_JAC"])
def test_embed_end_to_end_on_the_fixture(method):
  """The runner.py --embedding-method HG2V_* path (embedding.py:308-414) on the reference's own
  fixture: ids kept, dimension and method_name as the reference sets them, finite vectors, and
  the trained model reproduces its training targets better than the initial tables did."""
  import hypergraphembedding_b200 as H
  g = load_golden("algdist_youtube")
  node_ids, edge_ids = g["node_ids"], g["edge_ids"]
  hg = hypergraph_from_pairs(np.stack([node_ids[np.searchsorted(node_ids, g["pairs"][:, 0])],
                                       edge_ids[np.searchsorted(edge_ids, g["pairs"][:, 1])]], axis=1))
  np.random.seed(0)
  emb = H.EMBEDDING_OPTIONS[method](hg, 8, num_samples=20, epochs=3, disable_pbar=True)
  assert emb.method_name == method and emb.dim == 8
  assert sorted(emb.node) == sorted(hg.node) and sorted(emb.edge) == sorted(hg.edge)
  xn = np.asarray([emb.node[i].values for i in sorted(emb.node)])
  assert xn.shape == (len(hg.node), 8) and np.isfinite(xn).all() and np.abs(xn).max() > 0.05


def test_training_lowers_the_loss_on_real_samples():
  import hypergraphembedding_b200 as H
  g = load_golden("hobe_youtube_s2")
  hg = hypergraph_from_pairs(g["pairs"])
  emb = H.HypergraphEmbedding()
  for i, v in enumerate(g["xn"]):
    emb.node[i].values.extend(v.tolist())
  for i, v in enumerate(g["xe"]):
    emb.edge[i].values.extend(v.tolist())
  np.random.seed(int(g["seed"]))
  samples = H.AlgebraicDistanceSamples(hg, emb, int(g["k"]), 20)
  feats, targets = H.SamplesToModelInput(samples, int(g["k"]), weighted=False)
  model = H.UnweightedFloatModel(hg, 16, int(g["k"]))
  history = model.fit(feats, targets, batch_size=256, epochs=6, verbose=0)
  losses = history.history["loss"]
  assert losses[-1] < 0.7 * losses[0], losses
