"""Drop-in for the reference's ``hypergraph_embedding/hg2v_model.py``: ``BooleanModel``:51,
``UnweightedFloatModel``:129 and ``KerasModelToEmbedding``:31, without Keras.

The reference builds a Keras graph and calls ``model.fit`` (embedding.py:289-299).  Here a model
is two fp32 embedding tables on the device and ``fit`` runs the same mini-batch Adagrad loop in
libhge_b200.so (csrc/hge_hg2v_train.cu: one thread-block cluster walks all batches of an epoch in
one launch).  The objects answer the calls the reference makes on a Keras model: ``fit(x, y,
batch_size, epochs, callbacks, verbose)`` returning a history, and
``get_layer(name).get_weights()[0]``.

What is and is not the same as Keras 2.x / TensorFlow 1.x (absent here, so this part of the path
is not pinned against it -- oracle/hg2v_model_ref.py restates the semantics and the kernels are
tested against that):
  same       model arithmetic, losses (kullback_leibler_divergence with its 1e-7 clipping /
             mean_squared_error, summed over the three outputs), Adagrad defaults (lr 0.01,
             epsilon 1e-7, accumulators from 0), batching, the per-epoch
             ``np.random.shuffle`` of the sample order from the global numpy RNG, the epoch
             ``loss`` and EarlyStopping(monitor="loss") on it, the trained padding row 0;
             what the GLOBAL numpy stream is advanced by: Keras' backend seeds each
             RandomUniform initializer with one ``np.random.randint(10e6)`` (one draw per Embedding
             layer, node layer first), then one shuffle per epoch;
  different  the initial VALUES: Keras feeds that seed to TensorFlow's generator, here it seeds a
             private ``np.random.RandomState`` per table (same distribution U(-0.05, 0.05));
             sums of duplicated rows' gradients inside a batch are fp32 atomics (order varies).
"""
import ctypes
import logging

import numpy as np

from . import _native
from .hypergraph_pb2 import HypergraphEmbedding
from .hypergraph_util import embedding_to_wire

log = logging.getLogger()

ACTIVATIONS = {"sigmoid": 0, "relu": 1}
LOSSES = {"kullback_leibler_divergence": 0, "mean_squared_error": 1}


class EarlyStopping(object):
  """keras.callbacks.EarlyStopping for a loss-like quantity (mode "min")."""

  def __init__(self, monitor="loss", min_delta=0, patience=0):
    assert monitor == "loss", "only the training loss is available to monitor"
    self.monitor, self.min_delta, self.patience = monitor, abs(min_delta), patience
    self.best, self.wait, self.stopped_epoch = np.inf, 0, None

  def on_train_begin(self):
    self.best, self.wait, self.stopped_epoch = np.inf, 0, None

  def on_epoch_end(self, epoch, loss):
    """True when training should stop."""
    if loss + self.min_delta < self.best:
      self.best, self.wait = loss, 0
      return False
    self.wait += 1
    if self.wait >= self.patience:
      self.stopped_epoch = epoch
      return True
    return False


class History(object):
  def __init__(self):
    self.history = {"loss": []}
    self.epoch = []


class _EmbeddingLayer(object):
  def __init__(self, model, which, name):
    self._model, self._which, self.name = model, which, name

  def get_weights(self):
    return [self._model.weights()[self._which]]


class Hg2vModel(object):
  """The hypergraph2vec model family of hg2v_model.py as two device-resident tables."""

  def __init__(self, hypergraph, dimension, num_neighbors, activation, loss, ctx=None):
    log.info("Constructing model")
    max_node_idx = max([i for i in hypergraph.node])
    max_edge_idx = max([i for i in hypergraph.edge])
    self.dimension, self.num_neighbors = int(dimension), int(num_neighbors)
    self.activation, self.loss = activation, loss
    self.ctx = ctx or _native.default_context()
    # Embedding(input_dim=max + 2): index 0 pads absent inputs (hg2v_model.py:75-84);
    # keras 'uniform' initializer = RandomUniform(-0.05, 0.05)
    # the global stream moves by one randint per layer, as under Keras (K.random_uniform with
    # seed=None draws np.random.randint(10e6)); the tables come from private generators
    node_seed = np.random.randint(10e6)
    edge_seed = np.random.randint(10e6)
    node0 = np.random.RandomState(node_seed).uniform(
        -0.05, 0.05, (max_node_idx + 2, self.dimension)).astype(np.float32)
    edge0 = np.random.RandomState(edge_seed).uniform(
        -0.05, 0.05, (max_edge_idx + 2, self.dimension)).astype(np.float32)
    self.node_rows, self.edge_rows = node0.shape[0], edge0.shape[0]
    lib = self.ctx.lib
    handle = _native.c_vp()
    _native.check(lib.hge_hg2v_create(self.ctx.handle, self.node_rows, self.edge_rows, self.dimension,
                                      self.num_neighbors, ACTIVATIONS[activation], LOSSES[loss],
                                      _native.ptr(node0), _native.ptr(edge0), _native.MEM_HOST,
                                      ctypes.byref(handle)), "hge_hg2v_create")
    self.handle = handle
    self._layers = {"node_embedding": _EmbeddingLayer(self, 0, "node_embedding"),
                    "edge_embedding": _EmbeddingLayer(self, 1, "edge_embedding")}
    self.stop_training = False

  @classmethod
  def seeded(cls, num_nodes, num_edges, dimension, num_neighbors, activation, loss, seed, ctx=None):
    """The model for `num_nodes` / `num_edges` compressed ids (num + 1 table rows, as
    Embedding(input_dim = max id + 2) gives), its tables drawn on the device from U(-0.05, 0.05)
    by seeded Philox streams (hge_hg2v_create_seeded).  numpy's global RNG is neither read nor
    advanced."""
    self = cls.__new__(cls)
    self.dimension, self.num_neighbors = int(dimension), int(num_neighbors)
    self.activation, self.loss = activation, loss
    self.ctx = ctx or _native.default_context()
    self.node_rows, self.edge_rows = int(num_nodes) + 1, int(num_edges) + 1
    handle = _native.c_vp()
    _native.check(self.ctx.lib.hge_hg2v_create_seeded(self.ctx.handle, self.node_rows, self.edge_rows,
                                                      self.dimension, self.num_neighbors,
                                                      ACTIVATIONS[activation], LOSSES[loss],
                                                      int(seed) & 0xFFFFFFFFFFFFFFFF, ctypes.byref(handle)),
                  "hge_hg2v_create_seeded")
    self.handle = handle
    self._layers = {"node_embedding": _EmbeddingLayer(self, 0, "node_embedding"),
                    "edge_embedding": _EmbeddingLayer(self, 1, "edge_embedding")}
    self.stop_training = False
    return self

  def get_layer(self, name):
    return self._layers[name]

  def weights(self):
    node = np.empty((self.node_rows, self.dimension), np.float32)
    edge = np.empty((self.edge_rows, self.dimension), np.float32)
    _native.check(self.ctx.lib.hge_hg2v_get_weights(self.handle, _native.ptr(node), _native.ptr(edge),
                                                    _native.MEM_HOST), "hge_hg2v_get_weights")
    return node, edge

  def set_samples(self, x, y):
    cols = 4 + 2 * self.num_neighbors
    assert len(x) == cols, "expected %d input columns (SamplesToModelInput, weighted=False), got %d" % (
        cols, len(x))
    assert len(y) == 3
    feats = np.ascontiguousarray(np.stack([np.asarray(c).reshape(-1) for c in x]), dtype=np.int32)
    targets = np.ascontiguousarray(np.stack([np.asarray(c).reshape(-1) for c in y]), dtype=np.float32)
    assert feats.shape[1] == targets.shape[1]
    _native.check(self.ctx.lib.hge_hg2v_set_samples(self.handle, _native.ptr(feats), _native.ptr(targets),
                                                    feats.shape[1], _native.MEM_HOST),
                  "hge_hg2v_set_samples")
    self.num_samples = feats.shape[1]

  def fit_epoch(self, order, batch_size):
    order = np.ascontiguousarray(order, dtype=np.int32)
    assert order.shape == (self.num_samples,)
    loss = ctypes.c_double(0.0)
    _native.check(self.ctx.lib.hge_hg2v_fit_epoch(self.handle, _native.ptr(order), int(batch_size),
                                                  _native.MEM_HOST, ctypes.byref(loss)),
                  "hge_hg2v_fit_epoch")
    return loss.value

  def set_device_samples(self, samples):
    """Packs a DeviceSampleColumns into the model's sample buffer on the device, as
    SamplesToModelInput(samples.to_host(), k, weighted=False) would, then releases the blocks and
    the memory torch cached for them.  Every index is range-checked on the device."""
    import torch
    assert samples.num_neighbors == self.num_neighbors, \
        "samples have %d neighbours, the model %d" % (samples.num_neighbors, self.num_neighbors)
    lib = self.ctx.lib
    self.num_samples = len(samples)
    _native.check(lib.hge_hg2v_reserve_samples(self.handle, self.num_samples), "hge_hg2v_reserve_samples")
    for b in samples.blocks:
      c = b.cols
      _native.check(lib.hge_hg2v_append_samples(
          self.handle, _native.ptr(c["left_node"]), _native.ptr(c["left_edge"]), _native.ptr(c["right_node"]),
          _native.ptr(c["right_edge"]), _native.ptr(c["neigh_node"]), _native.ptr(c["neigh_edge"]),
          _native.ptr(b.prob), b.prob_slot, b.prob_value, b.count),
                    "hge_hg2v_append_samples")
    samples.release()
    torch.cuda.empty_cache()

  def samples(self):
    """The packed sample buffer as SamplesToModelInput's (features, targets) lists."""
    cols = 4 + 2 * self.num_neighbors
    feats = np.empty((cols, self.num_samples), np.int32)
    targets = np.empty((3, self.num_samples), np.float32)
    _native.check(self.ctx.lib.hge_hg2v_get_samples(self.handle, _native.ptr(feats), _native.ptr(targets),
                                                    _native.MEM_HOST), "hge_hg2v_get_samples")
    return list(feats), list(targets)

  def fit_device(self, samples, batch_size=32, epochs=1, seed=0, callbacks=None, verbose=1):
    """fit() on a DeviceSampleColumns without a host round trip: the blocks are packed into the
    model's buffer on the device and then released (the caller's `samples` is empty afterwards),
    and epoch e trains in the order hge_shuffle_order(seed, e) draws on the device.  Callbacks and
    the returned history are those of fit(); numpy's global RNG is neither read nor advanced."""
    import torch
    self.set_device_samples(samples)
    order = torch.empty(max(self.num_samples, 1), dtype=torch.int32,
                        device=torch.device("cuda", self.ctx.device))[:self.num_samples]
    history = History()
    stoppers = [c for c in (callbacks or []) if isinstance(c, EarlyStopping)]
    for c in stoppers:
      c.on_train_begin()
    for epoch in range(int(epochs)):
      _native.shuffle_order(self.ctx, seed, epoch, self.num_samples, out=order)
      loss = ctypes.c_double(0.0)
      _native.check(self.ctx.lib.hge_hg2v_fit_epoch(self.handle, _native.ptr(order), int(batch_size),
                                                    _native.MEM_DEVICE, ctypes.byref(loss)),
                    "hge_hg2v_fit_epoch")
      history.epoch.append(epoch)
      history.history["loss"].append(loss.value)
      if verbose:
        log.info("Epoch %d/%d - loss: %.6f", epoch + 1, epochs, loss.value)
      if any([c.on_epoch_end(epoch, loss.value) for c in stoppers]):
        break
    return history

  @property
  def last_clusters(self):
    """Thread-block clusters the last epoch ran on (one per 256 samples of a batch)."""
    return int(self.ctx.lib.hge_hg2v_last_clusters(self.handle))

  def fit(self, x, y, batch_size=32, epochs=1, callbacks=None, verbose=1, shuffle=True):
    """keras Model.fit for this model family: per epoch the sample order is shuffled with the
    global numpy RNG (as keras.engine.training_arrays does), batches are consecutive slices of
    it, and callbacks see the epoch's sample-weighted mean loss."""
    self.set_samples(x, y)
    history = History()
    stoppers = [c for c in (callbacks or []) if isinstance(c, EarlyStopping)]
    for c in stoppers:
      c.on_train_begin()
    for epoch in range(int(epochs)):
      index = np.arange(self.num_samples)
      if shuffle:
        np.random.shuffle(index)
      loss = self.fit_epoch(index, batch_size)
      history.epoch.append(epoch)
      history.history["loss"].append(loss)
      if verbose:
        log.info("Epoch %d/%d - loss: %.6f", epoch + 1, epochs, loss)
      if any([c.on_epoch_end(epoch, loss) for c in stoppers]):
        break
    return history

  def close(self):
    if getattr(self, "handle", None):
      self.ctx.lib.hge_hg2v_destroy(self.handle)
      self.handle = None

  def __del__(self):
    try:
      self.close()
    except Exception:
      pass


def BooleanModel(hypergraph, dimension, num_neighbors):
  """hg2v_model.py:51-126: sigmoid outputs, KL-divergence loss (trains on BooleanSamples)."""
  return Hg2vModel(hypergraph, dimension, num_neighbors, "sigmoid", "kullback_leibler_divergence")


def UnweightedFloatModel(hypergraph, dimension, num_neighbors):
  """hg2v_model.py:129-203: relu outputs, squared-error loss (trains on the weighted samplers)."""
  return Hg2vModel(hypergraph, dimension, num_neighbors, "relu", "mean_squared_error")


def KerasModelToEmbedding(hypergraph, model, node_map, edge_map, node_layer_name="node_embedding",
                          edge_layer_name="edge_embedding"):
  """hg2v_model.py:31-48: row idx + 1 of each table becomes the vector of node_map[idx] /
  edge_map[idx] (row 0 is the padding row)."""
  node_weights = model.get_layer(node_layer_name).get_weights()[0]
  edge_weights = model.get_layer(edge_layer_name).get_weights()[0]
  node_idx = np.asarray(sorted(hypergraph.node), dtype=np.int64)
  edge_idx = np.asarray(sorted(hypergraph.edge), dtype=np.int64)
  node_ids = np.asarray([node_map[int(i)] for i in node_idx], dtype=np.int64)
  edge_ids = np.asarray([edge_map[int(i)] for i in edge_idx], dtype=np.int64)
  no, eo = np.argsort(node_ids), np.argsort(edge_ids)
  embedding = HypergraphEmbedding()
  embedding.ParseFromString(embedding_to_wire(node_ids[no], node_weights[node_idx[no] + 1],
                                              edge_ids[eo], edge_weights[edge_idx[eo] + 1],
                                              len(node_weights[0]), None))
  return embedding
