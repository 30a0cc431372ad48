"""Link-prediction evaluation hooks -- the piece that closes the loop from an embedding to the
``ExperimentalResult`` files the reference's ``utilities/`` consume (SURVEY.md section 8f rank 4).

Mirrors the hook surface of the reference's ``evaluation_util.py``:

  ``LinkPredictionData``                    :33-35   (same field tuple, by contract)
  ``AddPredictionRecords``                  :38-53
  ``RunLinkPredictionExperiment``           :56-71
  ``LinkPredictionDataToResultProto``       :74-81
  ``RemoveRandomConnections``               :84-124  (same consumption of Python's ``random``)
  ``SampleMissingConnections``              :127-157 (same consumption of Python's ``random``)
  ``CalculateCommunityPredictionMetrics``   :160-204
  ``EXPERIMENT_OPTIONS``                    :586-590

The predictors themselves (one SVC per edge / node, a Keras classifier) are downstream of the
embeddings and out of scope (SURVEY.md section 2 row 11); ``EXPERIMENT_OPTIONS`` is a registry a
caller fills with ``RegisterExperiment`` -- ``RunLinkPredictionExperiment`` looks the predictor up
in it exactly as the reference does.  The per-edge / per-node SVC predictors are provided on top
of scikit-learn (imported on first use) because they need nothing else; the Keras one raises.
Their GPU forms (``Personalized*ClassifierPredictionDevice``, csrc/hge_lp_svm.cu) train the same
classifiers with seeded negatives and are not registered.  ``NodeEdgeEmbeddingPredictionDevice``
(csrc/hge_lp_node_edge.cu) trains a seeded GPU classifier for the node-edge experiment, a documented
model of the Keras kind rather than the reference's; it is not registered either.
"""
import logging
import random
from collections import namedtuple

import numpy as np

from . import _native
from .hypergraph_pb2 import EvaluationMetrics, ExperimentalResult, Hypergraph

log = logging.getLogger()

LinkPredictionData = namedtuple("LinkPredictionData",
                                ("hypergraph", "embedding", "good_links", "bad_links", "removal_prob"))


def _pairs(links):
  return [(int(n), int(e)) for n, e in links]


def AddPredictionRecords(eval_metric, good_links, bad_links, predictions):
  """Appends one record per evaluated link: the good links (label true) in their order, then the
  bad ones; ``prediction`` says whether the predictor kept the link."""
  log.info("Adding link data...")
  kept = set(_pairs(predictions))
  for label, links in ((True, good_links), (False, bad_links)):
    for node, edge in links:
      eval_metric.records.add(node_idx=node, edge_idx=edge, label=label,
                              prediction=(node, edge) in kept)
  return eval_metric


def CalculateCommunityPredictionMetrics(predicted_connections, good_links, bad_links):
  """Precision / recall / F1 / accuracy and the confusion counts of a set of predicted links
  against disjoint positive and negative sets.  Precision, recall and F1 stay unset (proto2
  presence) where the reference leaves them unset: no predictions, no positives, both zero."""
  predicted, pos, neg = set(predicted_connections), set(good_links), set(bad_links)
  assert pos.isdisjoint(neg)
  assert predicted <= (pos | neg)
  assert pos or neg
  hits = len(predicted & pos)
  m = EvaluationMetrics()
  if predicted:
    m.precision = hits / len(predicted)
  if pos:
    m.recall = hits / len(pos)
  if m.precision + m.recall:
    m.f1 = 2 * m.precision * m.recall / (m.precision + m.recall)
  m.num_true_pos = hits
  m.num_false_pos = len(predicted) - hits
  m.num_false_neg = len(pos) - hits
  m.num_true_neg = len(neg - predicted)
  m.accuracy = (m.num_true_pos + m.num_true_neg) / (len(pos) + len(neg))
  return m


def RemoveRandomConnections(original_hypergraph, probability):
  """Copy of the hypergraph with each node-edge connection dropped with `probability`, never a
  node's or an edge's last one; returns (copy, removed (node, edge) pairs in removal order).
  Draws from Python's global ``random`` exactly as the reference: one shuffle of the
  connection list in proto iteration order, then one ``random()`` per connection whose node and
  edge both still have another connection."""
  assert 0 <= probability <= 1
  out = Hypergraph()
  out.CopyFrom(original_hypergraph)
  links = [(n, e) for n, node in original_hypergraph.node.items() for e in node.edges]
  random.shuffle(links)
  node_left = {n: len(node.edges) for n, node in out.node.items()}
  edge_left = {e: len(edge.nodes) for e, edge in out.edge.items()}
  removed = []
  for n, e in links:
    if node_left[n] == 1 or edge_left[e] == 1:
      continue
    if random.random() < probability and probability > 0:
      out.node[n].edges.remove(e)
      out.edge[e].nodes.remove(n)
      node_left[n] -= 1
      edge_left[e] -= 1
      removed.append((n, e))
  return out, removed


def SampleMissingConnections(hypergraph, num_samples):
  """`num_samples` distinct (node, edge) pairs with the node not in the edge -- the negatives of
  the link-prediction task.  Rejection sampling with the reference's draws (``random.choice`` of
  a node, then of an edge, at most 10 x num_samples attempts) and its result order (a set's)."""
  nodes, edges = list(hypergraph.node), list(hypergraph.edge)
  assert num_samples < len(nodes) * len(edges)
  assert nodes and edges
  member = {n: set(node.edges) for n, node in hypergraph.node.items()}
  found = set()
  tries = 10 * num_samples
  while len(found) < num_samples and tries:
    tries -= 1
    n = random.choice(nodes)
    e = random.choice(edges)
    if e not in member[n]:
      found.add((n, e))
  if len(found) < num_samples:
    log.critical("SampleMissingConnections failed to find %i samples", num_samples)
  return list(found)


def RunLinkPredictionExperiment(link_prediction_data, experiment_name):
  """Runs the predictor registered under `experiment_name` on bad + good links and returns the
  ``EvaluationMetrics`` proto (metrics, experiment name, one record per link)."""
  assert experiment_name in EXPERIMENT_OPTIONS
  hypergraph, embedding, good_links, bad_links, _ = link_prediction_data
  log.info("Predicting links on subset graph")
  predicted = EXPERIMENT_OPTIONS[experiment_name](hypergraph, embedding, bad_links + good_links)
  log.info("Evaluating link prediction performance")
  metrics = CalculateCommunityPredictionMetrics(predicted, good_links, bad_links)
  metrics.experiment_name = experiment_name
  log.info("Result:\n%s", metrics)
  AddPredictionRecords(metrics, good_links, bad_links, predicted)
  return metrics


def LinkPredictionDataToResultProto(lp_data):
  """``ExperimentalResult`` holding the (reduced) hypergraph, its embedding and the removal
  probability; the caller appends the metrics of each experiment it runs."""
  log.info("Storing data into Experimental Result proto")
  res = ExperimentalResult()
  res.removal_probability = lp_data.removal_prob
  res.hypergraph.CopyFrom(lp_data.hypergraph)
  res.embedding.CopyFrom(lp_data.embedding)
  return res


def PrepLinkPredictionExperiment(hypergraph, removal_prob, embedding_function):
  """The caller side of the hook (runner.py:366-375 flow, experiment_util): hide connections
  with `removal_prob`, sample as many negatives, embed the reduced hypergraph with
  `embedding_function(hypergraph) -> HypergraphEmbedding`."""
  reduced, good_links = RemoveRandomConnections(hypergraph, removal_prob)
  bad_links = SampleMissingConnections(hypergraph, len(good_links))
  return LinkPredictionData(hypergraph=reduced, embedding=embedding_function(reduced),
                            good_links=good_links, bad_links=bad_links, removal_prob=removal_prob)


# ---- predictors -------------------------------------------------------------------------------


def _personalized_classifier_prediction(hypergraph, embedding, links, per_edge):
  """One RBF SVC (C = 1, gamma = 0.1) per edge over node vectors (or per node over edge vectors),
  trained on the members against twice as many sampled non-members
  (evaluation_util.py:317-350, :389-447); the degenerate classifiers accept everything (no
  non-member) or nothing (no member)."""
  from sklearn.svm import SVC
  from sklearn.utils import shuffle
  assert embedding.dim > 0
  vectors = embedding.node if per_edge else embedding.edge
  owners = hypergraph.edge if per_edge else hypergraph.node
  asked = [(n, e) if per_edge else (e, n) for n, e in links if n in embedding.node and e in embedding.edge]
  models = {}
  for owner in set(o for _, o in asked):
    members = set(owners[owner].nodes if per_edge else owners[owner].edges) if owner in owners else set()
    if not members:
      models[owner] = 0
      continue
    others = vectors.keys() - members
    if not others:
      models[owner] = 1
      continue
    others = random.sample(sorted(others), min(len(others), 2 * len(members)))
    x = [list(vectors[i].values) for i in members] + [list(vectors[i].values) for i in others]
    y = [1] * len(members) + [0] * len(others)
    x, y = shuffle(x, y)
    models[owner] = SVC(C=1, gamma=0.1).fit(x, y)
  kept = []
  for item, owner in asked:
    model = models[owner]
    verdict = model if isinstance(model, int) else model.predict([list(vectors[item].values)])[0]
    if verdict > 0:
      kept.append((item, owner) if per_edge else (owner, item))
  return kept


def PersonalizedEdgeClassifierPrediction(hypergraph, embedding, links, run_in_parallel=False):
  return _personalized_classifier_prediction(hypergraph, embedding, links, per_edge=True)


def PersonalizedNodeClassifierPrediction(hypergraph, embedding, links, run_in_parallel=False):
  return _personalized_classifier_prediction(hypergraph, embedding, links, per_edge=False)


def PersonalizedClassifierPredictionDevice(incidence, item_vectors, links, per_edge, seed=0, C=1.0, gamma=0.1,
                                          tol=1e-3, workspace_mb=0, return_model=False):
  """The personalized classifiers on the GPU (csrc/hge_lp_svm.cu) over dense row ids.  `incidence`
  is an N x E incidence CSR (or an hg2v_sample._Graph), `item_vectors` fp32 [N, d] node vectors
  (`per_edge`: one classifier per edge over its nodes) or [E, d] edge vectors (one per node over its
  edges), `links` an [L, 2] array of (node, edge) rows.  Each owner named by a link trains an RBF
  SVC (C, gamma, tol as libsvm) on its members against min(non-members, 2 x members) non-members
  drawn from the owner's own Philox stream of `seed`; the draw and the result depend only on
  (seed, side, owner, graph), never on the links' order or `workspace_mb` (megabytes of solver
  workspace per batch of large owners, 0 = 2048).  Returns the boolean keep mask of the links (a
  numpy array), and with ``return_model`` also the _native.LpSvmModel.  Python's ``random`` and
  numpy's global RNG are neither read nor advanced; owners that hit libsvm's iteration cap are
  logged as a warning, as libsvm warns."""
  import torch
  from .hg2v_sample import _Graph
  g = incidence if isinstance(incidence, _Graph) else _Graph.from_csr(incidence)
  links = np.asarray(links, dtype=np.int64).reshape(-1, 2)
  items, owners = (links[:, 0], links[:, 1]) if per_edge else (links[:, 1], links[:, 0])
  ctx = _native.default_context()
  dev = torch.device("cuda", ctx.device)
  if torch.is_tensor(item_vectors):
    vectors = item_vectors.to(dev, torch.float32).contiguous()
  else:
    vectors = torch.as_tensor(np.ascontiguousarray(item_vectors, dtype=np.float32)).to(dev)
  assert vectors.dim() == 2 and vectors.shape[0] == (g.num_nodes if per_edge else g.num_edges)
  as_i32 = lambda a: torch.as_tensor(np.asarray(a).astype(np.int32)).to(dev)
  inc = g.incidence(ctx)
  try:
    out = _native.lp_svm_predict(ctx, inc, 1 if per_edge else 0, vectors, as_i32(items), as_i32(owners), seed,
                                 C, gamma, tol, workspace_mb, return_model)
  finally:
    inc.close()
  if out[2]:
    log.warning("%d personalized classifiers reached the maximum number of iterations", out[2])
  keep = out[0].cpu().numpy()
  return (keep, out[3]) if return_model else keep


def _embedding_tables(embedding):
  """((sorted node ids, fp32 rows in that order), (sorted edge ids, rows)) of an embedding proto."""
  from .hypergraph_util import embedding_from_wire
  ids_n, ptr_n, val_n, ids_e, ptr_e, val_e, _ = embedding_from_wire(embedding)
  table = []
  for ids, ptr, val in ((ids_n, ptr_n, val_n), (ids_e, ptr_e, val_e)):
    order = np.argsort(ids, kind="stable")
    width = int(ptr[1] - ptr[0]) if len(ids) else 0
    assert width > 0 and np.all(np.diff(ptr) == width), "embedding rows must all have the same length"
    table.append((ids[order].astype(np.int64), val.reshape(-1, width)[order]))
  return table


def _personalized_classifier_prediction_device(hypergraph, embedding, links, per_edge, seed, **kw):
  """The host form's semantics on PersonalizedClassifierPredictionDevice: the asked links are those
  whose node and edge both have vectors, item rows are the embedding's sorted ids, an owner absent
  from the hypergraph has no members, a member without a vector is a KeyError; the kept links come
  back in the asked order."""
  (node_ids, xn), (edge_ids, xe) = _embedding_tables(embedding)
  pairs = np.asarray(_pairs(links), dtype=np.int64).reshape(-1, 2)
  asked = pairs[np.isin(pairs[:, 0], node_ids) & np.isin(pairs[:, 1], edge_ids)]
  rows = np.stack([np.searchsorted(node_ids, asked[:, 0]), np.searchsorted(edge_ids, asked[:, 1])], axis=1)
  owner_ids, member_ids, owner_map = (edge_ids, node_ids, hypergraph.edge) if per_edge else (
      node_ids, edge_ids, hypergraph.node)
  member_rows = {int(i): r for r, i in enumerate(member_ids.tolist())}
  inc = []   # (node row, edge row) of every named owner's members
  for r in np.unique(rows[:, 1 if per_edge else 0]).tolist():
    owner = int(owner_ids[r])
    if owner not in owner_map:
      continue
    members = set(owner_map[owner].nodes if per_edge else owner_map[owner].edges)
    for m in members:
      inc.append((member_rows[m], r) if per_edge else (r, member_rows[m]))   # KeyError: no vector
  import scipy.sparse as sps
  inc = np.asarray(inc, dtype=np.int64).reshape(-1, 2)
  A = sps.csr_matrix((np.ones(len(inc), dtype=np.int8), (inc[:, 0], inc[:, 1])),
                     shape=(len(node_ids), len(edge_ids)))
  A.sum_duplicates()
  A.sort_indices()
  keep = PersonalizedClassifierPredictionDevice(A, xn if per_edge else xe, rows, per_edge, seed=seed, **kw)
  return [(int(n), int(e)) for n, e in asked[keep]]


def PersonalizedEdgeClassifierPredictionDevice(hypergraph, embedding, links, seed=0, **kw):
  """LP_EDGE_CLASSIFIERS with the classifiers trained on the GPU from `seed` (not registered in
  EXPERIMENT_OPTIONS: add it with RegisterExperiment(name, functools.partial(fn, seed=s))).  `kw`:
  C, gamma, tol, workspace_mb of PersonalizedClassifierPredictionDevice."""
  return _personalized_classifier_prediction_device(hypergraph, embedding, links, True, seed, **kw)


def PersonalizedNodeClassifierPredictionDevice(hypergraph, embedding, links, seed=0, **kw):
  """LP_NODE_CLASSIFIERS with the classifiers trained on the GPU from `seed` (see
  PersonalizedEdgeClassifierPredictionDevice)."""
  return _personalized_classifier_prediction_device(hypergraph, embedding, links, False, seed, **kw)


def NodeEdgeEmbeddingPrediction(hypergraph, embedding, potential_links, classifier=None,
                                disable_pbar=False):
  """Keeps the links a binary classifier over [node vector, edge vector] scores above 0.5
  (evaluation_util.py:508-548).  The reference trains a Keras model when `classifier` is None;
  Keras is not part of this build, so a classifier with ``predict`` must be passed."""
  if classifier is None:
    raise NotImplementedError("NodeEdgeEmbeddingPrediction needs a classifier: the Keras model of "
                              "evaluation_util.py:466-505 is out of scope of this build")
  links = [(n, e) for n, e in potential_links if n in hypergraph.node and e in hypergraph.edge]
  if not links:
    return []
  for n, e in links:
    assert n in embedding.node and e in embedding.edge
  x = np.array([np.concatenate((embedding.node[n].values, embedding.edge[e].values)) for n, e in links])
  return [link for link, p in zip(links, classifier.predict(x)) if p > 0.5]


def _device_f32(x, dev):
  import torch
  if torch.is_tensor(x):
    return x.to(dev, torch.float32).contiguous()
  return torch.as_tensor(np.ascontiguousarray(x, dtype=np.float32)).to(dev)


class NodeEdgeClassifierDevice(object):
  """The node-edge link classifier on the GPU (csrc/hge_lp_node_edge.cu): p = sigmoid(w2 . relu(W1^T
  [xn[n], xe[e]] + b1) + b2), trained on the incidences (label 1) against as many non-incidences drawn
  uniformly from `seed` (label 0), with Glorot-uniform kernels, zero biases, Adagrad and binary
  cross-entropy.  This is a documented model of the usual Keras kind, not the reference's Keras
  model, whose architecture is not recorded; oracle/lp_node_edge_ref.py restates it.  Weights and
  losses are bit-identical from run to run; Python's ``random`` and numpy's global RNG are neither
  read nor advanced.  Use ``fit``; the object satisfies the ``classifier=`` protocol of
  NodeEdgeEmbeddingPrediction (``predict`` of [L, 2d] rows [node vector, edge vector])."""

  def __init__(self, ctx, xn, xe, weights, losses):
    self._ctx, self._xn, self._xe, self._weights, self.losses = ctx, xn, xe, weights, losses

  @classmethod
  def fit(cls, incidence, xn, xe, seed=0, hidden=64, epochs=10, batch_size=256, lr=0.01, timings=None):
    """Trains on an N x E incidence CSR (or an hg2v_sample._Graph) with node vectors `xn` [N, d] and
    edge vectors `xe` [E, d] (numpy or torch, fp32); 1 <= d, hidden <= 256.  ``losses``: the mean
    sample loss of each epoch.  `timings` (a dict) receives the set-up and per-epoch seconds."""
    import torch
    from .hg2v_sample import _Graph
    g = incidence if isinstance(incidence, _Graph) else _Graph.from_csr(incidence)
    ctx = _native.default_context()
    dev = torch.device("cuda", ctx.device)
    xn, xe = _device_f32(xn, dev), _device_f32(xe, dev)
    assert xn.dim() == 2 and xn.shape[0] == g.num_nodes and xe.dim() == 2 and xe.shape[0] == g.num_edges
    inc = g.incidence(ctx)
    try:
      weights, losses = _native.lp_node_edge_train(ctx, inc, xn, xe, seed, hidden, epochs, batch_size, lr,
                                                   timings=timings)
    finally:
      inc.close()
    return cls(ctx, xn, xe, weights, losses)

  def weights(self):
    """(W1 [2d, hidden], b1 [hidden], w2 [hidden], b2 [1]) as numpy arrays."""
    return tuple(w.cpu().numpy() for w in self._weights)

  def _predict(self, xn, xe, nodes, edges):
    import torch
    dev = self._xn.device
    as_i32 = lambda a: torch.as_tensor(np.asarray(a, dtype=np.int64).astype(np.int32)).to(dev)
    prob, _ = _native.lp_node_edge_predict(self._ctx, xn, xe, self._weights, as_i32(nodes), as_i32(edges))
    return prob.cpu().numpy()

  def predict_links(self, nodes, edges):
    """p of the links (nodes[l], edges[l]) over the training vectors (fp32 numpy array)."""
    return self._predict(self._xn, self._xe, nodes, edges)

  def predict(self, x):
    """p of each row [node vector, edge vector] of the [L, 2d] matrix `x`, by the same kernel."""
    x = _device_f32(x, self._xn.device)
    d = int(self._xn.shape[1])
    assert x.dim() == 2 and x.shape[1] == 2 * d, "rows must be [node vector, edge vector]"
    rows = np.arange(int(x.shape[0]))
    return self._predict(x[:, :d].contiguous(), x[:, d:].contiguous(), rows, rows)


def NodeEdgeEmbeddingPredictionDevice(hypergraph, embedding, links, seed=0, **kw):
  """LP_NODE_EDGE_CLASSIFIER with NodeEdgeClassifierDevice trained from `seed` (not registered in
  EXPERIMENT_OPTIONS: add it with RegisterExperiment(name, functools.partial(fn, seed=s))).  Rows are
  the embedding's sorted ids, the positives the hypergraph's connections (one without a vector is a
  KeyError); the links are filtered as NodeEdgeEmbeddingPrediction filters them and the kept ones come
  back in the asked order.  `kw`: hidden, epochs, batch_size, lr of NodeEdgeClassifierDevice.fit."""
  import scipy.sparse as sps
  (node_ids, xn), (edge_ids, xe) = _embedding_tables(embedding)
  links = [(n, e) for n, e in _pairs(links) if n in hypergraph.node and e in hypergraph.edge]
  if not links:
    return []
  for n, e in links:
    assert n in embedding.node and e in embedding.edge
  node_rows = {int(i): r for r, i in enumerate(node_ids.tolist())}
  edge_rows = {int(i): r for r, i in enumerate(edge_ids.tolist())}
  inc = [(node_rows[n], edge_rows[e]) for n, node in hypergraph.node.items() for e in node.edges]
  inc = np.asarray(inc, dtype=np.int64).reshape(-1, 2)
  A = sps.csr_matrix((np.ones(len(inc), dtype=np.int8), (inc[:, 0], inc[:, 1])),
                     shape=(len(node_ids), len(edge_ids)))
  A.sum_duplicates()
  A.sort_indices()
  model = NodeEdgeClassifierDevice.fit(A, xn, xe, seed=seed, **kw)
  rows = np.asarray([(node_rows[n], edge_rows[e]) for n, e in links], dtype=np.int64)
  p = model.predict_links(rows[:, 0], rows[:, 1])
  return [link for link, q in zip(links, p) if q > 0.5]


# Each entry is a function taking (hypergraph, embedding, links) -> predicted links
EXPERIMENT_OPTIONS = {
    "LP_EDGE_CLASSIFIERS": PersonalizedEdgeClassifierPrediction,
    "LP_NODE_CLASSIFIERS": PersonalizedNodeClassifierPrediction,
    "LP_NODE_EDGE_CLASSIFIER": NodeEdgeEmbeddingPrediction,
}


def RegisterExperiment(name, predictor):
  """Adds a predictor ``(hypergraph, embedding, links) -> links`` to ``EXPERIMENT_OPTIONS``."""
  EXPERIMENT_OPTIONS[name] = predictor
  return predictor
