"""The seeded sample -> train pipeline on the device: DeviceSampleColumns (keep_on_device=True) equal
to the host result, the sample buffer packed on the device equal to SamplesToModelInput, the
epoch order and the initial tables equal to their numpy restatements (oracle/seeded_training_ref.py)
bit for bit, training equal to the host path and to the float64 restatement
(oracle/hg2v_model_ref.py, same bars as tests/test_hg2v_model_gpu.py), the Embed*Device entry
points, and the refusals."""
import ctypes
import logging
import re

import numpy as np
import pytest

from conftest import hypergraph_from_pairs, load_golden
from oracle import seeded_training_ref as dref
from oracle import hg2v_model_ref as mref
from test_device_sampler_gpu import _graphs, _vectors

pytestmark = pytest.mark.gpu

GRAPHS = ["youtube", "rand25", "gadgets", "zipf2000"]


def _same_columns(a, b):
  from hypergraphembedding_b200 import SampleColumns
  for f in SampleColumns.FIELDS:
    x, y = np.asarray(getattr(a, f)), np.asarray(getattr(b, f))
    assert x.dtype == y.dtype and x.shape == y.shape, f
    assert np.array_equal(x, y, equal_nan=x.dtype.kind == "f"), f


def _same_model_input(got, want):
  for g, w in zip(got[0] + got[1], want[0] + want[1]):
    w = np.asarray(w)
    assert g.dtype == w.dtype and g.shape == w.shape
    assert np.array_equal(g, w)
  assert len(got[0]) == len(want[0]) and len(got[1]) == len(want[1])


@pytest.mark.parametrize("name", GRAPHS)
@pytest.mark.parametrize("neg", [0, 2])
def test_boolean_on_device_equals_the_host_result(name, neg):
  from hypergraphembedding_b200 import BooleanSamplesDevice, DeviceSampleColumns
  A = _graphs()[name]
  want = BooleanSamplesDevice(A, 3, 7, neg_samples=neg, seed=1234)
  for chunk in (0, 97):
    got = BooleanSamplesDevice(A, 3, 7, neg_samples=neg, seed=1234, chunk_rows=chunk, keep_on_device=True)
    assert isinstance(got, DeviceSampleColumns) and got.num_neighbors == 3
    assert len(got) == len(want) == sum(got.counts)
    assert all(t is None or t.is_cuda for b in got.blocks for t in list(b.cols.values()) + [b.prob])
    _same_columns(got.to_host(), want)


def test_boolean_on_device_with_row_weights_and_chunks():
  from hypergraphembedding_b200 import BooleanSamplesDevice
  A = _graphs()["zipf2000"]
  rng = np.random.default_rng(0)
  nw, ew = rng.random(A.shape[0]) * 2, rng.random(A.shape[1]) * 2
  want = BooleanSamplesDevice(A, 2, 5, neg_samples=3, node_weights=nw, edge_weights=ew, seed=9)
  for chunk in (0, 1, 64, 1000):
    got = BooleanSamplesDevice(A, 2, 5, neg_samples=3, node_weights=nw, edge_weights=ew, seed=9,
                               chunk_rows=chunk, keep_on_device=True)
    _same_columns(got.to_host(), want)
  with pytest.raises(AssertionError):
    BooleanSamplesDevice(A, 2, 5, stream=True, keep_on_device=True)


@pytest.mark.parametrize("name", GRAPHS)
def test_hobe_on_device_equals_the_host_result(name):
  from hypergraphembedding_b200 import AlgebraicDistanceSamplesDevice
  A = _graphs()[name]
  xn, xe = _vectors(A)
  want = AlgebraicDistanceSamplesDevice(A, xn, xe, 4, 9, seed=77)
  for chunk in (0, 101):
    timings = {}
    got = AlgebraicDistanceSamplesDevice(A, xn, xe, 4, 9, seed=77, chunk_rows=chunk, timings=timings,
                                         keep_on_device=True)
    assert set(timings) == {"pairs", "neighbours", "probabilities"}
    _same_columns(got.to_host(), want)
  with pytest.raises(AssertionError):
    AlgebraicDistanceSamplesDevice(A, xn, xe, 4, 9, stream=True, keep_on_device=True)


@pytest.mark.parametrize("name", GRAPHS)
@pytest.mark.parametrize("kind", ["fobe", "fobe_neg", "hobe"])
def test_packing_on_device_equals_samples_to_model_input(name, kind):
  import hypergraphembedding_b200 as H
  from hypergraphembedding_b200.hg2v_model import Hg2vModel
  A = _graphs()[name]
  k = 3
  if kind == "hobe":
    xn, xe = _vectors(A)
    sample = lambda **kw: H.AlgebraicDistanceSamplesDevice(A, xn, xe, k, 6, seed=5, **kw)
  else:
    sample = lambda **kw: H.BooleanSamplesDevice(A, k, 6, neg_samples=2 if kind == "fobe_neg" else 0,
                                                 seed=5, **kw)
  host = sample()
  dev = sample(keep_on_device=True)
  model = Hg2vModel.seeded(A.shape[0], A.shape[1], 8, k, "relu", "mean_squared_error", 3)
  try:
    history = model.fit_device(dev, batch_size=256, epochs=0, seed=1)
    assert history.history["loss"] == [] and dev.blocks == []
    assert model.num_samples == len(host)
    _same_model_input(model.samples(), H.SamplesToModelInput(host, k, weighted=False))
  finally:
    model.close()


@pytest.mark.parametrize("n", [1, 2, 1000, (1 << 20) + 3])
def test_shuffle_order_equals_the_restatement(n):
  from hypergraphembedding_b200 import _native
  ctx = _native.default_context()
  for seed, epoch in ((0, 0), (17, 1), (2**63 + 5, 6)):
    got = _native.shuffle_order(ctx, seed, epoch, n).cpu().numpy()
    assert np.array_equal(got, dref.shuffle_order(seed, epoch, n)), (n, seed, epoch)
  host = np.empty(n, np.int32)
  _native.check(ctx.lib.hge_shuffle_order(ctx.handle, 4, 2, n, _native.ptr(host), _native.MEM_HOST))
  assert np.array_equal(host, dref.shuffle_order(4, 2, n))


@pytest.mark.parametrize("dim", [1, 5, 32, 70])
def test_seeded_tables_equal_the_restatement(dim):
  from hypergraphembedding_b200.hg2v_model import Hg2vModel
  state = np.random.get_state()
  model = Hg2vModel.seeded(300, 120, dim, 2, "sigmoid", "kullback_leibler_divergence", 2024 + dim)
  try:
    n0, e0 = model.weights()
  finally:
    model.close()
  after = np.random.get_state()
  assert after[2] == state[2] and np.array_equal(after[1], state[1])
  assert n0.shape == (301, dim) and e0.shape == (121, dim)
  assert np.array_equal(n0, dref.init_table(2024 + dim, dref.PHASE["INIT_NODES"], 301, dim))
  assert np.array_equal(e0, dref.init_table(2024 + dim, dref.PHASE["INIT_EDGES"], 121, dim))


def _model_with_tables(n0, e0, k, activation, loss):
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


@pytest.mark.parametrize("kind,activation,loss,dim,batch", [
    ("fobe", "sigmoid", "kullback_leibler_divergence", 16, 256),
    ("hobe", "relu", "mean_squared_error", 32, 1024),
])
def test_fit_device_equals_the_host_path_and_the_restatement(kind, activation, loss, dim, batch):
  import hypergraphembedding_b200 as H
  from hypergraphembedding_b200.hg2v_model import Hg2vModel
  A = _graphs()["zipf2000"]
  k, seed = 3, 31
  if kind == "hobe":
    xn, xe = _vectors(A)
    sample = lambda **kw: H.AlgebraicDistanceSamplesDevice(A, xn, xe, k, 6, seed=2, **kw)
  else:
    sample = lambda **kw: H.BooleanSamplesDevice(A, k, 6, neg_samples=1, seed=2, **kw)
  feats, targets = H.SamplesToModelInput(sample(), k, weighted=False)
  m = len(feats[0])
  orders = [dref.shuffle_order(seed, e, m) for e in range(3)]
  model = Hg2vModel.seeded(A.shape[0], A.shape[1], dim, k, activation, loss, 8)
  n0, e0 = model.weights()
  try:
    history = model.fit_device(sample(keep_on_device=True), batch_size=batch, epochs=3, seed=seed, verbose=0)
    got_n, got_e = model.weights()
  finally:
    model.close()
  got_losses = history.history["loss"]
  # the existing host path on the same tables and orders
  host = _model_with_tables(n0, e0, k, activation, loss)
  try:
    host.set_samples(feats, targets)
    host_losses = [host.fit_epoch(o, batch) for o in orders]
    host_n, host_e = host.weights()
  finally:
    host.close()
  want_n, want_e, want_losses = mref.fit(n0, e0, feats, targets, k, activation,
                                         "kld" if loss.startswith("kull") else "mse", batch, 3,
                                         order=orders, min_delta=-1e9)
  for losses, n_, e_ in ((host_losses, host_n, host_e), (want_losses, want_n, want_e)):
    assert np.allclose(got_losses, losses, rtol=2e-5, atol=1e-6), (got_losses, losses)
    assert np.abs(got_n - n_).max() < 2e-4 and np.abs(got_e - e_).max() < 2e-4
  assert np.abs(got_n - n0).max() > 1e-3                # and it did train


def test_fit_device_stops_early_at_the_restatements_epoch():
  import hypergraphembedding_b200 as H
  from hypergraphembedding_b200.hg2v_model import EarlyStopping, Hg2vModel
  A = _graphs()["rand25"]
  k, seed, epochs, batch = 2, 3, 10, 128
  feats, targets = H.SamplesToModelInput(H.BooleanSamplesDevice(A, k, 8, seed=4), k, weighted=False)
  m = len(feats[0])
  orders = [dref.shuffle_order(seed, e, m) for e in range(epochs)]
  model = Hg2vModel.seeded(A.shape[0], A.shape[1], 8, k, "sigmoid", "kullback_leibler_divergence", 6)
  n0, e0 = model.weights()
  _, _, free = mref.fit(n0, e0, feats, targets, k, "sigmoid", "kld", batch, epochs, order=orders,
                        min_delta=-1e9)
  # a min_delta half way between the two successive improvements that differ most: the
  # restatement stops part way, with a margin far above the fp32 differences of the losses
  gains = -np.diff(free)
  j = 1 + int(np.argmax(gains[1:6] - gains[2:7]))
  assert gains[j] - gains[j + 1] > 1e-5, gains
  min_delta = (gains[j] + gains[j + 1]) / 2
  _, _, want = mref.fit(n0, e0, feats, targets, k, "sigmoid", "kld", batch, epochs, order=orders,
                        min_delta=min_delta)
  assert 1 < len(want) < epochs, (gains, want)
  try:
    history = model.fit_device(H.BooleanSamplesDevice(A, k, 8, seed=4, keep_on_device=True), batch_size=batch,
                               epochs=epochs, seed=seed, verbose=0,
                               callbacks=[EarlyStopping(monitor="loss", min_delta=min_delta)])
  finally:
    model.close()
  assert len(history.history["loss"]) == len(want)
  assert np.allclose(history.history["loss"], want, rtol=2e-5, atol=1e-6)


@pytest.mark.parametrize("method", ["EmbedHg2vBooleanDevice", "EmbedHg2vAlgDistDevice"])
def test_embed_device_end_to_end_on_the_fixture(method, caplog):
  import hypergraphembedding_b200 as H
  g = load_golden("algdist_youtube")
  node_ids, edge_ids = g["node_ids"], g["edge_ids"]
  hg = hypergraph_from_pairs(np.stack([node_ids[np.searchsorted(node_ids, g["pairs"][:, 0])],
                                       edge_ids[np.searchsorted(edge_ids, g["pairs"][:, 1])]], axis=1))
  np.random.seed(0)
  state = np.random.get_state()
  with caplog.at_level(logging.INFO):
    emb = getattr(H, method)(hg, 8, num_samples=20, epochs=3, seed=5)
  after = np.random.get_state()
  assert after[2] == state[2] and np.array_equal(after[1], state[1])
  assert emb.method_name == {"EmbedHg2vBooleanDevice": "HG2V_BOOLEAN",
                             "EmbedHg2vAlgDistDevice": "HG2V_ALG_DIST"}[method]
  assert emb.dim == 8
  assert sorted(emb.node) == sorted(hg.node) and sorted(emb.edge) == sorted(hg.edge)
  xn = np.asarray([emb.node[i].values for i in sorted(emb.node)])
  assert xn.shape == (len(hg.node), 8) and np.isfinite(xn).all()
  losses = [float(x) for x in re.findall(r"Epoch \d+/\d+ - loss: ([0-9.eE+-]+)", caplog.text)]
  assert len(losses) >= 2 and losses[-1] < losses[0], losses
  assert getattr(H, method) not in H.EMBEDDING_OPTIONS.values()


def _append(model, count, ln=None, le=None, rn=None, re_=None, nn=None, ne=None, prob=None, slot=-1):
  from hypergraphembedding_b200 import _native
  P = _native.ptr
  _native.check(model.ctx.lib.hge_hg2v_append_samples(model.handle, P(ln), P(le), P(rn), P(re_), P(nn), P(ne),
                                                      P(prob), slot, 1.0, count), "hge_hg2v_append_samples")


def test_refusals_leave_the_gpu_usable():
  import torch
  import hypergraphembedding_b200 as H
  from hypergraphembedding_b200 import _native
  from hypergraphembedding_b200.hg2v_model import Hg2vModel
  from hypergraphembedding_b200.hg2v_sample import _DeviceBlock
  dev = torch.device("cuda", _native.default_context().device)
  model = Hg2vModel.seeded(10, 4, 8, 2, "relu", "mean_squared_error", 1)
  try:
    lib = model.ctx.lib
    # an index past its table, in the last record of a neighbour column
    ln = torch.arange(6, dtype=torch.int32, device=dev)
    nbr = torch.zeros((6, 2), dtype=torch.int32, device=dev)
    nbr_e = nbr.clone()
    nbr_e[5, 1] = 4                                  # edge rows are 0 .. 4, index 4 + 1 is out
    bad = H.DeviceSampleColumns(2, [_DeviceBlock(6, "ne_prob", left_node=ln, right_edge=ln % 4, neigh_node=nbr,
                                                 neigh_edge=nbr_e)])
    with pytest.raises(AssertionError, match="column 7, record 5"):
      model.fit_device(bad, epochs=1, seed=0)
    # negative ids other than the padding -1 are refused too
    with pytest.raises(AssertionError, match="outside its table"):
      model.set_device_samples(H.DeviceSampleColumns(2, [_DeviceBlock(6, left_node=ln - 2)]))
    # past the reservation
    _native.check(lib.hge_hg2v_reserve_samples(model.handle, 10))
    _append(model, 6, ln=ln)
    with pytest.raises(AssertionError, match="do not fit"):
      _append(model, 6, ln=ln)
    # a half-filled buffer is not trained on
    order = torch.arange(10, dtype=torch.int32, device=dev)
    loss = ctypes.c_double()
    with pytest.raises(AssertionError, match="6 of the 10 reserved"):
      _native.check(lib.hge_hg2v_fit_epoch(model.handle, _native.ptr(order), 4, _native.MEM_DEVICE,
                                           ctypes.byref(loss)))
    with pytest.raises(AssertionError):
      _native.check(lib.hge_hg2v_reserve_samples(model.handle, 1 << 31))
    # a neighbour count that is not the model's
    A = _graphs()["gadgets"]
    with pytest.raises(AssertionError, match="neighbours"):
      model.fit_device(H.BooleanSamplesDevice(A, 3, 2, keep_on_device=True), epochs=1, seed=0)
    # and the device still works: filling the rest lets the epoch run
    _native.check(lib.hge_hg2v_reserve_samples(model.handle, 10))
    _append(model, 6, ln=ln)
    _append(model, 4, ln=ln[:4], rn=ln[:4], prob=torch.full((4,), 0.5, device=dev), slot=0)
    _native.check(lib.hge_hg2v_fit_epoch(model.handle, _native.ptr(order), 4, _native.MEM_DEVICE,
                                         ctypes.byref(loss)))
    torch.cuda.synchronize()
    model.num_samples = 10                           # reserved through the C ABI above
    feats, targets = model.samples()
    assert np.array_equal(feats[0], np.r_[np.arange(1, 7), np.arange(1, 5)])
    assert np.array_equal(feats[2], np.r_[np.zeros(6), np.arange(1, 5)])
    assert np.array_equal(targets[0], np.r_[np.zeros(6), np.full(4, 0.5)]) and not targets[1].any()
    assert np.isfinite(loss.value)
  finally:
    model.close()


def test_fit_device_at_100k_nodes():
  import hypergraphembedding_b200 as H
  from hypergraphembedding_b200 import synthetic
  from hypergraphembedding_b200.hg2v_model import Hg2vModel
  A = synthetic.zipf_hypergraph(100000, 50000, seed=2024)
  k = 5
  samples = H.BooleanSamplesDevice(A, k, 10, neg_samples=1, seed=3, keep_on_device=True)
  records = len(samples)
  model = Hg2vModel.seeded(A.shape[0], A.shape[1], 32, k, "sigmoid", "kullback_leibler_divergence", 3)
  try:
    history = model.fit_device(samples, batch_size=4096, epochs=3, seed=3, verbose=0)
    assert model.num_samples == records > 1000000
    feats, targets = model.samples()
  finally:
    model.close()
  assert all(len(f) == records for f in feats + targets)
  for c, f in enumerate(feats):
    node = c in (0, 2) or 4 <= c < 4 + k
    assert f.min() >= 0 and f.max() <= (A.shape[0] if node else A.shape[1]), c
  losses = history.history["loss"]
  assert len(losses) == 3 and losses[2] < losses[0], losses
