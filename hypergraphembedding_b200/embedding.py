"""Drop-in for the hypergraph2vec part of the reference's ``hypergraph_embedding/embedding.py``:
``_hypergraph2vec_skeleton``:269, ``EmbedHg2vBoolean``:308 (FOBE), ``EmbedHg2vAdjJaccard``:330,
``EmbedHg2vNeighborhoodWeightedJaccard``:358, ``EmbedHg2vAlgDist``:387 (HOBE) and the matching
entries of ``EMBEDDING_OPTIONS``:417 -- what ``runner.py --embedding-method HG2V_*`` calls.

Same arguments, defaults, consumption of the global numpy RNG (the sampler's draws, then one
seed draw per embedding table as Keras' initializers make, then one shuffle per epoch) and result (a ``HypergraphEmbedding`` keyed by the original
ids with the reference's ``method_name``).  Sampling and training run in libhge_b200.so.
"""
import logging

import numpy as np

from . import _native
from .algebraic_distance import EmbedAlgebraicDistance
from .hg2v_model import (BooleanModel, EarlyStopping, Hg2vModel, KerasModelToEmbedding,
                         UnweightedFloatModel)
from .hg2v_sample import (AlgebraicDistanceSamples, AlgebraicDistanceSamplesDevice, BooleanSamples,
                          BooleanSamplesDevice, PlotDistributions, SamplesToModelInput,
                          WeightedJaccardSamples, WeightedJaccardSamplesDevice, _Graph)
from .hg2v_weighting import UniformWeight, WeightByNeighborhood
from .hypergraph_pb2 import HypergraphEmbedding
from .hypergraph_util import (CompressRange, ToCsrMatrix, ToEdgeCsrMatrix, compressed_incidence,
                              embedding_to_wire)
from .nmf import NonNegativeFactorizationDevice
from .node2vec import DEFAULT_BATCH_PAIRS, Node2VecCliqueDevice, Node2VecDevice, clique_edge_seed
from .svd import TruncatedSVDDevice

log = logging.getLogger()


def _hypergraph2vec_skeleton(hypergraph, dimension, num_neighbors, sampler_fn, model_fn,
                             fit_batch_size, fit_epochs, debug_summary_path, disable_pbar):
  """embedding.py:269-305."""
  log.info("Compressing index space")
  # we want to do this in order to reduce the embedding problem size
  compressed_hg, inv_node_map, inv_edge_map = CompressRange(hypergraph)

  log.info("Sampling")
  samples = sampler_fn(compressed_hg)

  if debug_summary_path is not None:
    PlotDistributions(debug_summary_path, samples)

  log.info("Converting samples to model input")
  input_features, output_probs = SamplesToModelInput(samples, num_neighbors=num_neighbors,
                                                     weighted=False)

  log.info("Getting model")
  model = model_fn(compressed_hg)
  stopper = EarlyStopping(monitor="loss", min_delta=1e-3)
  try:
    model.fit(input_features, output_probs, batch_size=fit_batch_size, epochs=fit_epochs,
              callbacks=[stopper], verbose=0 if disable_pbar else 1)
    log.info("Recording embeddings.")
    return KerasModelToEmbedding(compressed_hg, model, inv_node_map, inv_edge_map)
  finally:
    model.close()


def EmbedHg2vBoolean(hypergraph, dimension, num_neighbors=5, num_samples=200, batch_size=256,
                     epochs=10, neg_samples=0, debug_summary_path=None, disable_pbar=False):
  """embedding.py:308-327 (FOBE)."""
  sampler_fn = lambda hg: BooleanSamples(hg, num_neighbors=num_neighbors, num_samples=num_samples,
                                         neg_samples=neg_samples, disable_pbar=disable_pbar)
  model_fn = lambda hg: BooleanModel(hg, dimension=dimension, num_neighbors=num_neighbors)
  embedding = _hypergraph2vec_skeleton(hypergraph, dimension, num_neighbors, sampler_fn, model_fn,
                                       batch_size, epochs, debug_summary_path, disable_pbar)
  embedding.method_name = "HG2V_BOOLEAN"
  return embedding


def EmbedHg2vAdjJaccard(hypergraph, dimension, num_neighbors=5, num_samples=200, batch_size=256,
                        epochs=10, debug_summary_path=None, disable_pbar=False):
  """embedding.py:330-355."""

  def sampler_fn(hypergraph):
    node2weight, edge2weight = UniformWeight(hypergraph)
    return WeightedJaccardSamples(hypergraph, node2weight, edge2weight, num_neighbors=num_neighbors,
                                  num_samples=num_samples, disable_pbar=disable_pbar)

  model_fn = lambda hg: UnweightedFloatModel(hg, dimension=dimension, num_neighbors=num_neighbors)
  embedding = _hypergraph2vec_skeleton(hypergraph, dimension, num_neighbors, sampler_fn, model_fn,
                                       batch_size, epochs, debug_summary_path, disable_pbar)
  embedding.method_name = "HG2V_ADJ_JAC"
  return embedding


def EmbedHg2vNeighborhoodWeightedJaccard(hypergraph, dimension, alpha=0, num_neighbors=5,
                                         num_samples=200, batch_size=256, epochs=10,
                                         debug_summary_path=None, disable_pbar=False):
  """embedding.py:358-384."""

  def sampler_fn(hypergraph):
    node2feature, edge2feature = WeightByNeighborhood(hypergraph, alpha)
    return WeightedJaccardSamples(hypergraph, node2feature, edge2feature,
                                  num_neighbors=num_neighbors, num_samples=num_samples,
                                  disable_pbar=disable_pbar)

  model_fn = lambda hg: UnweightedFloatModel(hg, dimension=dimension, num_neighbors=num_neighbors)
  embedding = _hypergraph2vec_skeleton(hypergraph, dimension, num_neighbors, sampler_fn, model_fn,
                                       batch_size, epochs, debug_summary_path, disable_pbar)
  embedding.method_name = "HG2V_NEIGH_JAC"
  return embedding


def EmbedHg2vAlgDist(hypergraph, dimension, alpha=0, num_neighbors=5, num_samples=200,
                     batch_size=256, epochs=10, debug_summary_path=None, disable_pbar=False):
  """embedding.py:387-414 (HOBE): algebraic-distance embedding (dimension 10, 20 sweeps), samples
  weighted by it, UnweightedFloatModel trained on them."""
  del alpha   # accepted and unused, as in the reference

  def sampler_fn(hypergraph):
    log.info("Embedding weighted by algebraic distance.")
    alg_emb = EmbedAlgebraicDistance(hypergraph, dimension=10, iterations=20,
                                     disable_pbar=disable_pbar)
    return AlgebraicDistanceSamples(hypergraph, alg_emb, num_neighbors=num_neighbors,
                                    num_samples=num_samples, disable_pbar=disable_pbar)

  model_fn = lambda hg: UnweightedFloatModel(hg, dimension=dimension, num_neighbors=num_neighbors)
  embedding = _hypergraph2vec_skeleton(hypergraph, dimension, num_neighbors, sampler_fn, model_fn,
                                       batch_size, epochs, debug_summary_path, disable_pbar)
  embedding.method_name = "HG2V_ALG_DIST"
  return embedding


def _hypergraph2vec_device(hypergraph, dimension, num_neighbors, sampler_fn, activation, loss,
                           batch_size, epochs, seed):
  """_hypergraph2vec_skeleton with the samples kept on the device: CompressRange, sampler_fn(the
  compressed graph's _Graph) -> DeviceSampleColumns, Hg2vModel.seeded, fit_device,
  KerasModelToEmbedding.  Sampling, tables and epoch orders all derive from `seed`."""
  compressed_hg, inv_node_map, inv_edge_map = CompressRange(hypergraph)
  g = _Graph.from_csr(ToCsrMatrix(compressed_hg), ToEdgeCsrMatrix(compressed_hg))
  log.info("Sampling on the device")
  samples = sampler_fn(g, compressed_hg)
  model = Hg2vModel.seeded(g.num_nodes, g.num_edges, dimension, num_neighbors, activation, loss, seed)
  stopper = EarlyStopping(monitor="loss", min_delta=1e-3)
  try:
    model.fit_device(samples, batch_size=batch_size, epochs=epochs, seed=seed, callbacks=[stopper])
    log.info("Recording embeddings.")
    return KerasModelToEmbedding(compressed_hg, model, inv_node_map, inv_edge_map)
  finally:
    model.close()


def EmbedHg2vBooleanDevice(hypergraph, dimension, num_neighbors=5, num_samples=200, batch_size=256,
                           epochs=10, neg_samples=0, seed=0, chunk_rows=0):
  """EmbedHg2vBoolean (FOBE) as a seeded pipeline whose samples never leave the GPU:
  BooleanSamplesDevice (per-row counts from the node / edge weights, as BooleanSamples), a
  BooleanModel with seeded tables, and per-epoch orders from hge_shuffle_order.  The result
  depends on `seed`, not on numpy's global RNG, which is neither read nor advanced."""

  def sampler_fn(g, hg):
    nw = [hg.node[i].weight for i in range(g.num_nodes)]
    ew = [hg.edge[i].weight for i in range(g.num_edges)]
    return BooleanSamplesDevice(g, num_neighbors, num_samples, neg_samples=neg_samples, node_weights=nw,
                                edge_weights=ew, seed=seed, chunk_rows=chunk_rows, keep_on_device=True)

  embedding = _hypergraph2vec_device(hypergraph, dimension, num_neighbors, sampler_fn, "sigmoid",
                                     "kullback_leibler_divergence", batch_size, epochs, seed)
  embedding.method_name = "HG2V_BOOLEAN"
  return embedding


def EmbedHg2vAlgDistDevice(hypergraph, dimension, num_neighbors=5, num_samples=200, batch_size=256,
                           epochs=10, seed=0, chunk_rows=0):
  """EmbedHg2vAlgDist (HOBE) as a seeded pipeline whose samples never leave the GPU: the
  algebraic-distance relaxation (dimension 10, 20 sweeps, initial vectors from a private
  RandomState seeded by `seed`), AlgebraicDistanceSamplesDevice, an UnweightedFloatModel with
  seeded tables, per-epoch orders from hge_shuffle_order.  numpy's global RNG is neither read
  nor advanced."""

  def sampler_fn(g, hg):
    del hg
    log.info("Embedding weighted by algebraic distance.")
    rng = np.random.RandomState(seed & 0xFFFFFFFF)
    xn = rng.random_sample((g.num_nodes, 10)).astype(np.float32)
    xe = rng.random_sample((g.num_edges, 10)).astype(np.float32)
    _native.algdist_run_csr(_native.default_context(), g.num_nodes, g.num_edges, g.a.ptr, g.a.idx, xn, xe,
                            20, e2n_ptr=g.b.ptr, e2n_idx=g.b.idx)
    return AlgebraicDistanceSamplesDevice(g, xn, xe, num_neighbors, num_samples, seed=seed,
                                          chunk_rows=chunk_rows, keep_on_device=True)

  embedding = _hypergraph2vec_device(hypergraph, dimension, num_neighbors, sampler_fn, "relu",
                                     "mean_squared_error", batch_size, epochs, seed)
  embedding.method_name = "HG2V_ALG_DIST"
  return embedding


def _jaccard_device(hypergraph, dimension, features_fn, num_neighbors, num_samples, batch_size, epochs,
                    seed, chunk_rows):
  """The Jaccard methods as a seeded pipeline whose samples never leave the GPU: features_fn(the
  compressed hypergraph) on the host, WeightedJaccardSamplesDevice (per-row counts from the node /
  edge weights, as WeightedJaccardSamples), an UnweightedFloatModel with seeded tables, per-epoch
  orders from hge_shuffle_order."""

  def sampler_fn(g, hg):
    node2features, edge2features = features_fn(hg)
    nw = [hg.node[i].weight for i in range(g.num_nodes)]
    ew = [hg.edge[i].weight for i in range(g.num_edges)]
    return WeightedJaccardSamplesDevice(g, node2features, edge2features, num_neighbors, num_samples,
                                        node_weights=nw, edge_weights=ew, seed=seed, chunk_rows=chunk_rows,
                                        keep_on_device=True)

  return _hypergraph2vec_device(hypergraph, dimension, num_neighbors, sampler_fn, "relu",
                                "mean_squared_error", batch_size, epochs, seed)


def EmbedHg2vAdjJaccardDevice(hypergraph, dimension, num_neighbors=5, num_samples=200, batch_size=256,
                              epochs=10, seed=0, chunk_rows=0):
  """EmbedHg2vAdjJaccard (uniform features) as a seeded pipeline whose samples never leave the GPU
  (see _jaccard_device).  The result depends on `seed`, not on numpy's global RNG, which is
  neither read nor advanced."""
  embedding = _jaccard_device(hypergraph, dimension, UniformWeight, num_neighbors, num_samples, batch_size,
                              epochs, seed, chunk_rows)
  embedding.method_name = "HG2V_ADJ_JAC"
  return embedding


def EmbedHg2vNeighborhoodWeightedJaccardDevice(hypergraph, dimension, alpha=0, num_neighbors=5,
                                               num_samples=200, batch_size=256, epochs=10, seed=0,
                                               chunk_rows=0):
  """EmbedHg2vNeighborhoodWeightedJaccard (WeightByNeighborhood(alpha) features) as a seeded
  pipeline whose samples never leave the GPU (see _jaccard_device).  numpy's global RNG is neither
  read nor advanced."""
  embedding = _jaccard_device(hypergraph, dimension, lambda hg: WeightByNeighborhood(hg, alpha),
                              num_neighbors, num_samples, batch_size, epochs, seed, chunk_rows)
  embedding.method_name = "HG2V_NEIGH_JAC"
  return embedding


def EmbedNMFDevice(hypergraph, dimension, max_iter=200, tol=1e-4, seed=0):
  """The NMF baseline (embedding.py:110-261 of the reference) on the GPU: the compressed incidence
  A ~ W H by NonNegativeFactorizationDevice with the seeded start of `seed`; node vectors are the
  rows of W, edge vectors the columns of H, keyed by the original ids, method_name "NMF".  Not the
  reference's NMF, whose start (init="nndsvda") draws numpy's global RNG: this one neither reads
  nor advances it, so it is not in EMBEDDING_OPTIONS."""
  node_ids, edge_ids, A = compressed_incidence(hypergraph)
  W, H, _ = NonNegativeFactorizationDevice(A, dimension, seed=seed, max_iter=max_iter, tol=tol)
  embedding = HypergraphEmbedding()
  embedding.ParseFromString(embedding_to_wire(node_ids, W, edge_ids, np.ascontiguousarray(H.T), dimension,
                                              "NMF"))
  return embedding


def EmbedSVDDevice(hypergraph, dimension, n_iter=5, oversamples=10, seed=0):
  """The SVD baseline (embedding.py:110-261 of the reference) on the GPU: the compressed incidence
  A ~ U diag(s) V^T by TruncatedSVDDevice (randomized subspace iteration from the seeded start of
  `seed`); node vectors are the rows of U, edge vectors the rows of V, keyed by the original ids,
  method_name "SVD".  Triplets beyond the incidence's numerical rank give zero columns.  numpy's
  global RNG is neither read nor advanced, so this is not the reference's call and not in
  EMBEDDING_OPTIONS."""
  node_ids, edge_ids, A = compressed_incidence(hypergraph)
  U, _, Vt, _ = TruncatedSVDDevice(A, dimension, n_iter=n_iter, oversamples=oversamples, seed=seed)
  embedding = HypergraphEmbedding()
  embedding.ParseFromString(embedding_to_wire(node_ids, U, edge_ids, np.ascontiguousarray(Vt.T), dimension,
                                              "SVD"))
  return embedding


def EmbedNode2VecDevice(hypergraph, dimension, walk_length=80, num_walks=10, p=1.0, q=1.0, window=10, negative=5,
                        epochs=5, alpha=0.025, min_alpha=1e-4, batch_pairs=DEFAULT_BATCH_PAIRS, seed=0):
  """The node2vec baseline (embedding.py:110-261 of the reference) on the GPU: Node2VecDevice on the
  node-edge bipartite graph of the compressed incidence; node vectors are the input-table rows of
  the nodes, edge vectors those of the edges, keyed by the original ids, method_name "N2V".  numpy's
  global RNG and Python's ``random`` are neither read nor advanced, so this is not the reference's
  call and not in EMBEDDING_OPTIONS."""
  node_ids, edge_ids, A = compressed_incidence(hypergraph)
  X, _ = Node2VecDevice(A, dimension, walk_length=walk_length, num_walks=num_walks, p=p, q=q, window=window,
                        negative=negative, epochs=epochs, alpha=alpha, min_alpha=min_alpha, batch_pairs=batch_pairs,
                        seed=seed)
  N = len(node_ids)
  embedding = HypergraphEmbedding()
  embedding.ParseFromString(embedding_to_wire(node_ids, np.ascontiguousarray(X[:N]), edge_ids,
                                              np.ascontiguousarray(X[N:]), dimension, "N2V"))
  return embedding


def EmbedNode2VecCliqueDevice(hypergraph, dimension, walk_length=80, num_walks=10, p=1.0, q=1.0, window=10,
                              negative=5, epochs=5, alpha=0.025, min_alpha=1e-4, batch_pairs=DEFAULT_BATCH_PAIRS,
                              seed=0):
  """node2vec on the weighted clique expansions of the compressed incidence on the GPU
  (Node2VecCliqueDevice): node vectors from the node-side expansion with `seed`, edge vectors from
  the edge-side expansion with clique_edge_seed(seed), keyed by the original ids, method_name
  "N2V_CLIQUE".  The two tables are trained apart, so node and edge vectors do not share a space.
  numpy's global RNG and Python's ``random`` are neither read nor advanced; not in
  EMBEDDING_OPTIONS."""
  node_ids, edge_ids, A = compressed_incidence(hypergraph)
  kw = dict(walk_length=walk_length, num_walks=num_walks, p=p, q=q, window=window, negative=negative, epochs=epochs,
            alpha=alpha, min_alpha=min_alpha, batch_pairs=batch_pairs)
  Xn, _ = Node2VecCliqueDevice(A, dimension, side="node", seed=seed, **kw)
  Xe, _ = Node2VecCliqueDevice(A, dimension, side="edge", seed=clique_edge_seed(seed), **kw)
  embedding = HypergraphEmbedding()
  embedding.ParseFromString(embedding_to_wire(node_ids, Xn, edge_ids, Xe, dimension, "N2V_CLIQUE"))
  return embedding


# the part of embedding.py:417-436 that is on this path
EMBEDDING_OPTIONS = {
    "ALG_DIST": EmbedAlgebraicDistance,
    "HG2V_BOOLEAN": EmbedHg2vBoolean,
    "HG2V_ADJ_JAC": EmbedHg2vAdjJaccard,
    "HG2V_NEIGH_JAC": EmbedHg2vNeighborhoodWeightedJaccard,
    "HG2V_ALG_DIST": EmbedHg2vAlgDist,
}
