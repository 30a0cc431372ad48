"""Drop-in for the sampling half of the reference's ``hypergraph_embedding/hg2v_sample.py``:
``SimilarityRecord``:29, ``_sample_adj_matrix``:53, ``_sample_neighbors``:49, ``BooleanSamples``:125
(FOBE), ``AlgebraicDistanceSamples``:632 (HOBE) with ``SameTypeDistanceSample``:546 /
``DiffTypeDistanceSample``:588, and ``SamplesToModelInput``:751.

Same names, arguments, RNG consumption (the process-global legacy numpy stream is advanced
exactly as the reference advances it) and record contents.  Where the work happens:
  * candidate rows (scipy CSR-product order) and every draw: csrc/hge_sampler.cpp (host; the
    MT19937 stream is sequential with data-dependent rejection);
  * incidence weights and the max-min probabilities of all sampled pairs: csrc/hge_weighting.cu.

The samplers return a ``SampleColumns``: a sequence of ``SimilarityRecord`` backed by columnar
arrays (a 755k-record result on the youtube fixture is 7 arrays, not 755k tuples); iterating or
indexing it yields ordinary records, ``list(result)`` materialises them.
"""
import collections.abc
import logging
from collections import namedtuple

import numpy as np
import scipy.sparse as sps

from . import _native
from .hypergraph_util import ToCsrMatrix, ToEdgeCsrMatrix

log = logging.getLogger()

SimilarityRecord = namedtuple(
    "SimilarityRecord",
    (
        "left_node_idx",
        "left_edge_idx",
        "right_node_idx",
        "right_edge_idx",
        "left_weight",  # Only used in weighted cases
        "right_weight",  # Only used in weighted cases
        "neighbor_node_indices",
        "neighbor_node_weights",  # Only used in weighted cases
        "neighbor_edge_indices",
        "neighbor_edge_weights",  # Only used in weighted cases
        "node_node_prob",
        "edge_edge_prob",
        "node_edge_prob"))
# Set all field defaults to none
SimilarityRecord.__new__.__defaults__ = (None,) * len(SimilarityRecord._fields)

NONE_IDX = -1


class SampleColumns(collections.abc.Sequence):
  """Columnar list of SimilarityRecord.  -1 marks a ``None`` index, NaN a ``None``
  probability, ``has_neighbors`` False a record without neighbour arrays."""

  FIELDS = ("left_node", "left_edge", "right_node", "right_edge", "neigh_node", "neigh_edge",
            "nn_prob", "ee_prob", "ne_prob", "has_neighbors", "left_weight", "right_weight")

  def __init__(self, num_neighbors, **cols):
    self.num_neighbors = int(num_neighbors)
    for name in self.FIELDS:
      setattr(self, name, cols[name])

  @classmethod
  def build(cls, num_neighbors, count, left_node=None, left_edge=None, right_node=None,
            right_edge=None, neigh_node=None, neigh_edge=None, nn_prob=None, ee_prob=None,
            ne_prob=None, left_weight=None, right_weight=None):
    # absent columns are constant read-only views (no memory): a chunk of a streamed 1e9-record
    # result only pays for the columns it has; concatenate() materialises them
    def idx(a):
      return (np.broadcast_to(np.int32(NONE_IDX), (count,)) if a is None
              else np.asarray(a, dtype=np.int32))

    def prob(a):
      return (np.broadcast_to(np.float32(np.nan), (count,)) if a is None
              else np.asarray(a, dtype=np.float32))

    k = int(num_neighbors)
    has = neigh_node is not None
    none = np.broadcast_to(np.int32(NONE_IDX), (count, k))
    return cls(k, left_node=idx(left_node), left_edge=idx(left_edge), right_node=idx(right_node),
               right_edge=idx(right_edge),
               neigh_node=np.asarray(neigh_node, np.int32).reshape(count, k) if has else none,
               neigh_edge=np.asarray(neigh_edge, np.int32).reshape(count, k) if has else none,
               nn_prob=prob(nn_prob), ee_prob=prob(ee_prob), ne_prob=prob(ne_prob),
               has_neighbors=np.broadcast_to(np.bool_(has), (count,)),
               left_weight=prob(left_weight), right_weight=prob(right_weight))

  @classmethod
  def concatenate(cls, parts):
    parts = list(parts)
    k = parts[0].num_neighbors
    return cls(k, **{name: np.concatenate([getattr(p, name) for p in parts])
                     for name in cls.FIELDS})

  def arrays(self):
    return {name: getattr(self, name) for name in self.FIELDS}

  def __len__(self):
    return len(self.left_node)

  def _record(self, i):
    def idx(v):
      return None if v == NONE_IDX else v

    def prob(v):
      return None if np.isnan(v) else v

    has = bool(self.has_neighbors[i])
    return SimilarityRecord(
        left_node_idx=idx(self.left_node[i]), left_edge_idx=idx(self.left_edge[i]),
        right_node_idx=idx(self.right_node[i]), right_edge_idx=idx(self.right_edge[i]),
        left_weight=prob(self.left_weight[i]), right_weight=prob(self.right_weight[i]),
        neighbor_node_indices=self.neigh_node[i] if has else None,
        neighbor_edge_indices=self.neigh_edge[i] if has else None,
        node_node_prob=prob(self.nn_prob[i]), edge_edge_prob=prob(self.ee_prob[i]),
        node_edge_prob=prob(self.ne_prob[i]))

  def __getitem__(self, i):
    if isinstance(i, slice):
      return [self._record(j) for j in range(*i.indices(len(self)))]
    if i < 0:
      i += len(self)
    if not 0 <= i < len(self):
      raise IndexError(i)
    return self._record(i)

  def __iter__(self):
    for i in range(len(self)):
      yield self._record(i)


# -----------------------------------------------------------------------------------------
# sampling primitives
# -----------------------------------------------------------------------------------------


def _sample_neighbors(idx, idx2neighbors, num_neighbors):
  """hg2v_sample.py:49-51: np.random.choice(neighbours of idx, k, replace=True)."""
  m = _native.CsrArrays(idx2neighbors)
  state = _native.LegacyRngState()
  out = np.empty(num_neighbors, dtype=np.uint32)
  deg = int(m.ptr[idx + 1] - m.ptr[idx])
  if deg == 0 and num_neighbors > 0:
    raise ValueError("'a' cannot be empty unless no samples are taken")
  if num_neighbors:
    _native.check(_native.load_library().hge_mt19937_interval(
        _native.ptr(state.buf), max(deg - 1, 0), num_neighbors, _native.ptr(out)))
  state.commit()
  return m.idx[m.ptr[idx] + out.astype(np.int64)]


def _sample_adj_matrix(matrix, interesting_rows, samples_per_row, disable_pbar=False,
                       replace=False, negative=False):
  """hg2v_sample.py:53-86 on an explicit scipy matrix: list of (row, col) samples.  The row's
  candidates are its stored columns in stored order (which is what ``matrix[row].nonzero()``
  returns, sorted or not)."""
  del disable_pbar
  rows = list(interesting_rows)
  if type(samples_per_row) == int:
    samples_per_row = [samples_per_row for _ in rows]
  assert len(samples_per_row) == len(rows)
  assert len(samples_per_row) > 0
  state = _native.LegacyRngState()
  r, c = _native.sample_adj_rows((_native.CsrArrays(matrix),), rows, samples_per_row, state,
                                 replace=replace, negative=negative)
  state.commit()
  return list(zip(r.tolist(), c.tolist()))


def _alpha_scale(val, alpha=0):
  """hg2v_sample.py:89-94."""
  assert alpha >= 0
  assert alpha <= 1
  assert val <= 1
  assert val >= 0
  return alpha + (1 - alpha) * (val)


class _Graph(object):
  """Host CSR arrays of a hypergraph the way the samplers see it: A from ``node.edges``
  (ToCsrMatrix), B from ``edge.nodes`` (ToEdgeCsrMatrix), their transposes for the products
  ``A * A.T`` / ``B * B.T``, and the proto-map iteration orders."""

  def __init__(self, hypergraph):
    A = ToCsrMatrix(hypergraph)
    B = ToEdgeCsrMatrix(hypergraph)
    self._set(A, B, list(hypergraph.node), list(hypergraph.edge))

  @classmethod
  def from_csr(cls, A, B=None, node_rows=None, edge_rows=None):
    """The same view of a hypergraph given as a canonical N x E incidence CSR (and optionally
    the E x N CSR of ``edge.nodes``; default: the transpose).  Row orders default to ascending
    ids, which is the proto-map order for dense ids."""
    g = cls.__new__(cls)
    A = sps.csr_matrix(A)
    if B is None:
      B = A.T.tocsr()
      B.sort_indices()
    g._set(A, sps.csr_matrix(B),
           np.arange(A.shape[0], dtype=np.int32) if node_rows is None else node_rows,
           np.arange(A.shape[1], dtype=np.int32) if edge_rows is None else edge_rows)
    return g

  def _set(self, A, B, node_rows, edge_rows):
    n = max(A.shape[0], B.shape[1])
    e = max(A.shape[1], B.shape[0])
    A = sps.csr_matrix((A.data, A.indices, _pad(A.indptr, n)), shape=(n, e))
    B = sps.csr_matrix((B.data, B.indices, _pad(B.indptr, e)), shape=(e, n))
    self.A, self.B = A, B
    self.a, self.b = _native.CsrArrays(A), _native.CsrArrays(B)
    consistent = A.nnz == B.nnz and _is_transpose(self.a, self.b)
    if consistent:
      self.at, self.bt = self.b, self.a
    else:
      At = A.T.tocsr()
      At.sort_indices()
      Bt = B.T.tocsr()
      Bt.sort_indices()
      self.at, self.bt = _native.CsrArrays(At), _native.CsrArrays(Bt)
    self.node_rows = node_rows
    self.edge_rows = edge_rows
    self.num_nodes, self.num_edges = n, e

  def incidence(self, ctx):
    return _native.Incidence(ctx, self.num_nodes, self.num_edges, self.a.ptr, self.a.idx,
                             self.b.ptr, self.b.idx)


def _is_transpose(a, b):
  """True when the canonical CSR `b` is the transpose of the canonical CSR `a`."""
  At = sps.csr_matrix((np.ones(len(a.idx), dtype=np.int8), a.idx, a.ptr), shape=a.shape).T.tocsr()
  At.sort_indices()
  return bool(np.array_equal(At.indptr, b.ptr) and np.array_equal(At.indices, b.idx))


def _pad(indptr, rows):
  indptr = np.asarray(indptr)
  if len(indptr) - 1 >= rows:
    return indptr
  return np.concatenate([indptr, np.full(rows - (len(indptr) - 1), indptr[-1], indptr.dtype)])


def embedding_to_arrays(embedding, num_nodes, num_edges):
  """Dense fp32 [num_nodes, R] / [num_edges, R] from a HypergraphEmbedding proto (rows of ids
  without a vector stay zero), read from the serialized message (csrc/hge_proto.cpp)."""
  from .hypergraph_util import embedding_from_wire
  ids_n, ptr_n, val_n, ids_e, ptr_e, val_e, _ = embedding_from_wire(embedding)
  assert len(ids_n) > 0 and ptr_n[-1] > 0, "embedding has no node vectors"

  def dense(ids, ptr, vals, rows, dim):
    out = np.zeros((rows, dim), dtype=np.float32)
    lens = np.diff(ptr)
    keep = (ids >= 0) & (ids < rows)
    assert np.all(lens[keep] == dim), "embedding vectors have different lengths"
    if np.all(lens == dim):
      out[ids[keep]] = vals.reshape(-1, dim)[keep]
    else:
      for i in np.nonzero(keep)[0]:
        out[ids[i]] = vals[ptr[i]:ptr[i + 1]]
    return out

  dim = int(np.diff(ptr_n).max())
  return dense(ids_n, ptr_n, val_n, num_nodes, dim), dense(ids_e, ptr_e, val_e, num_edges, dim)


################################################################################
# BooleanSamples                                                               #
################################################################################


def _row_chunks(rows, samples, chunk_rows):
  rows = np.asarray(rows, dtype=np.int32)
  samples = np.asarray(samples, dtype=np.int32)
  assert len(samples) == len(rows)
  assert len(samples) > 0          # hg2v_sample.py:67
  step = len(rows) if not chunk_rows else int(chunk_rows)
  for lo in range(0, len(rows), step):
    yield rows[lo:lo + step], samples[lo:lo + step]


def _boolean_sample_chunks(g, k, node_samples, edge_samples, neg_node_samples, neg_edge_samples,
                           state, chunk_rows=0):
  """BooleanSamples as a stream of SampleColumns chunks in the reference's record order.  The
  RNG stream is consumed row after row exactly as one call over all rows would consume it, so
  the concatenation of the chunks does not depend on `chunk_rows` (0 = one chunk per phase)."""
  ones = lambda m: np.broadcast_to(np.float32(1.0), (m,))

  def same_type(mats, rows, samples, left, right, prob, negative=False):
    for r_rows, r_samples in _row_chunks(rows, samples, chunk_rows):
      r, c = _native.sample_adj_rows(mats, r_rows, r_samples, state, negative=negative)
      cols = {left: r, right: c}
      if prob and not negative:
        cols[prob] = ones(len(r))
      yield SampleColumns.build(k, len(r), **cols)

  def node_edge(node_s, edge_s, negative=False):
    # all (node, edge) pairs are drawn first (node rows, then edge rows), then the neighbour
    # arrays of every pair in that order (hg2v_sample.py:170-195)
    pairs_n, pairs_e = [], []
    for r_rows, r_samples in _row_chunks(g.node_rows, node_s, chunk_rows):
      n1, e1 = _native.sample_adj_rows((g.a,), r_rows, r_samples, state, negative=negative)
      pairs_n.append(n1)
      pairs_e.append(e1)
    for r_rows, r_samples in _row_chunks(g.edge_rows, edge_s, chunk_rows):
      e2, n2 = _native.sample_adj_rows((g.b,), r_rows, r_samples, state, negative=negative)
      pairs_n.append(n2)
      pairs_e.append(e2)
    nodes, edges = np.concatenate(pairs_n), np.concatenate(pairs_e)
    step = len(nodes) if not chunk_rows else max(1, int(chunk_rows) * 8)
    for lo in range(0, max(len(nodes), 1), max(step, 1)):
      sn, se = nodes[lo:lo + step], edges[lo:lo + step]
      nbr_e, nbr_n = _native.sample_neighbors(g.a, g.b, sn, se, k, state)
      cols = dict(left_node=sn, right_edge=se, neigh_node=nbr_n, neigh_edge=nbr_e)
      if not negative:
        cols["ne_prob"] = ones(len(sn))
      yield SampleColumns.build(k, len(sn), **cols)

  log.info("Sampling node-node probabilities")
  for part in same_type((g.a, g.at), g.node_rows, node_samples, "left_node", "right_node", "nn_prob"):
    yield part
  log.info("Sampling edge-edge probabilities")
  for part in same_type((g.b, g.bt), g.edge_rows, edge_samples, "left_edge", "right_edge", "ee_prob"):
    yield part
  log.info("Getting node-edge / edge-node relationships")
  for part in node_edge(node_samples, edge_samples):
    yield part

  if neg_node_samples is not None:
    log.info("Node-Node Negatives")
    for part in same_type((g.a, g.at), g.node_rows, neg_node_samples, "left_node", "right_node",
                          None, negative=True):
      yield part
    for label in ("Edge-Edge Negatives", "Node-Edge Negatives"):   # sic: both are edge-edge
      log.info(label)
      for part in same_type((g.b, g.bt), g.edge_rows, neg_edge_samples, "left_edge", "right_edge",
                            None, negative=True):
        yield part
    log.info("Getting node-edge / edge-node negatives")
    for part in node_edge(neg_node_samples, neg_edge_samples, negative=True):
      yield part


def BooleanSamples(hypergraph, num_neighbors, num_samples, neg_samples=0, disable_pbar=False):
  """hg2v_sample.py:125-242 (FOBE): up to num_samples node-node, edge-edge and node-edge /
  edge-node first-order samples per row with probability 1, optionally neg_samples uniform
  negatives per row (including the reference's duplicated edge-edge negative block, :215-221)."""
  del disable_pbar
  node_samples = [int(node.weight * num_samples) for _, node in hypergraph.node.items()]
  edge_samples = [int(edge.weight * num_samples) for _, edge in hypergraph.edge.items()]
  neg_node_samples = [int(node.weight * neg_samples) for _, node in hypergraph.node.items()]
  neg_edge_samples = [int(edge.weight * neg_samples) for _, edge in hypergraph.edge.items()]
  g = _Graph(hypergraph)
  state = _native.LegacyRngState()
  parts = list(_boolean_sample_chunks(g, num_neighbors, node_samples, edge_samples,
                                      neg_node_samples if neg_samples > 0 else None,
                                      neg_edge_samples if neg_samples > 0 else None, state))
  state.commit()
  return SampleColumns.concatenate(parts)


def BooleanSamplesCsr(incidence, num_neighbors, num_samples, neg_samples=0, node_weights=None,
                      edge_weights=None, chunk_rows=0, stream=False):
  """BooleanSamples on a canonical N x E incidence CSR instead of a proto (the 10M-node case of
  BASELINE.json configs[3]: building the proto alone would take minutes of Python).  Same
  records, same RNG consumption as BooleanSamples on the equivalent proto with dense ids.
  With ``stream=True`` returns an iterator of SampleColumns chunks of about `chunk_rows` rows
  (record order preserved) that commits the RNG state when exhausted; otherwise one
  SampleColumns."""
  g = incidence if isinstance(incidence, _Graph) else _Graph.from_csr(incidence)

  def per_row(weights, count, base):
    if weights is None:
      return np.full(count, int(base), dtype=np.int32)
    return np.asarray([int(w * base) for w in weights], dtype=np.int32)

  node_samples = per_row(node_weights, len(g.node_rows), num_samples)
  edge_samples = per_row(edge_weights, len(g.edge_rows), num_samples)
  neg_node = per_row(node_weights, len(g.node_rows), neg_samples) if neg_samples > 0 else None
  neg_edge = per_row(edge_weights, len(g.edge_rows), neg_samples) if neg_samples > 0 else None
  state = _native.LegacyRngState()

  def chunks():
    for part in _boolean_sample_chunks(g, num_neighbors, node_samples, edge_samples, neg_node,
                                       neg_edge, state, chunk_rows=chunk_rows):
      yield part
    state.commit()

  if stream:
    return chunks()
  return SampleColumns.concatenate(list(chunks()))


################################################################################
# Device sampling from seeded Philox streams                                   #
################################################################################


class _DeviceSampler(object):
  """Pair and neighbour draws of csrc/hge_device_sampler.cu over a device incidence, in row chunks
  of `chunk_rows` (0 = one call per block).  Every row and every record owns its Philox stream
  (csrc/hge_philox.cuh), so the chunking does not change the result.  `spent` receives the seconds
  of the pair ("pairs") and neighbour ("neighbours") calls; both end in a device synchronise."""

  def __init__(self, g, ctx, inc, k, seed, chunk_rows, workspace_mb=0):
    assert np.array_equal(g.node_rows, np.arange(g.num_nodes)) and \
        np.array_equal(g.edge_rows, np.arange(g.num_edges)), \
        "the device sampler emits rows in ascending id order"
    self.ctx, self.inc, self.k, self.seed = ctx, inc, int(k), int(seed)
    self.chunk_rows, self.workspace_mb = int(chunk_rows), int(workspace_mb)
    self.spent = {"pairs": 0.0, "neighbours": 0.0}

  def _timed(self, kind, fn, *args, **kw):
    import time
    t = time.perf_counter()
    out = fn(*args, **kw)
    self.spent[kind] += time.perf_counter() - t
    return out

  def pairs(self, side, factors, samples, phase, negative=False):
    """(row, col) CUDA tensors, chunk by chunk, rows ascending."""
    samples = np.asarray(samples, dtype=np.int32)
    step = len(samples) if not self.chunk_rows else self.chunk_rows
    for lo in range(0, len(samples), max(step, 1)):
      yield self._timed("pairs", _native.sample_pairs_device, self.ctx, self.inc, side, factors, lo,
                        samples[lo:lo + step], self.seed, phase, negative=negative,
                        workspace_mb=self.workspace_mb)

  def node_edge(self, node_s, edge_s, factors, phases, negative=False):
    """(nodes, edges, neighbour nodes, neighbour edges) CUDA tensors of the node-edge block: node
    rows, then edge rows; the neighbour streams are numbered by record inside the block."""
    ne, en, nbr = phases
    first = 0
    for side, samples, phase in ((0, node_s, ne), (1, edge_s, en)):
      for r, c in self.pairs(side, factors, samples, phase, negative):
        nodes, edges = (r, c) if side == 0 else (c, r)
        nbr_e, nbr_n = self._timed("neighbours", _native.sample_neighbors_device, self.ctx, self.inc,
                                   nodes, edges, self.k, self.seed, nbr, first)
        first += int(nodes.shape[0])
        yield nodes, edges, nbr_n, nbr_e


def _host(t):
  return t.cpu().numpy()


def _per_row(weights, count, base):
  if weights is None:
    return np.full(count, int(base), dtype=np.int32)
  return np.asarray([int(w * base) for w in weights], dtype=np.int32)


class _DeviceBlock(object):
  """One block of device sampler output: int32 CUDA tensors of the index columns it has ([m, k]
  for the neighbour arrays), the one probability column it fills, `prob_field`, as an fp32
  CUDA tensor `prob` or the constant `prob_value`, and optionally the fp32 CUDA tensors
  `left_weight` / `right_weight` (the Jaccard factors of node-edge records)."""

  INDEX = ("left_node", "left_edge", "right_node", "right_edge", "neigh_node", "neigh_edge")
  PROB_SLOT = {"nn_prob": 0, "ee_prob": 1, "ne_prob": 2}

  def __init__(self, count, prob_field=None, prob=None, prob_value=1.0, left_weight=None,
               right_weight=None, **cols):
    assert set(cols) <= set(self.INDEX)
    self.count = int(count)
    self.cols = {name: cols.get(name) for name in self.INDEX}
    self.prob_field, self.prob, self.prob_value = prob_field, prob, float(prob_value)
    self.left_weight, self.right_weight = left_weight, right_weight

  @property
  def prob_slot(self):
    """Target slot of the probability column (hge_hg2v_append_samples), -1 for none."""
    return self.PROB_SLOT.get(self.prob_field, -1)

  def compact(self):
    """Copies every column that is a view of a larger buffer (the sampler's output buffers are
    sized for sum(k_r) records) into one of its own, so a kept block holds only its records."""
    def own(t):
      return t if t is None or t.untyped_storage().nbytes() == t.nbytes else t.clone()
    self.cols = {name: own(t) for name, t in self.cols.items()}
    self.prob = own(self.prob)
    self.left_weight, self.right_weight = own(self.left_weight), own(self.right_weight)
    return self

  def to_host(self, k):
    cols = {name: _host(t) for name, t in self.cols.items() if t is not None}
    if self.prob_field is not None:
      cols[self.prob_field] = (_host(self.prob) if self.prob is not None else
                               np.broadcast_to(np.float32(self.prob_value), (self.count,)))
    for name in ("left_weight", "right_weight"):
      if getattr(self, name) is not None:
        cols[name] = _host(getattr(self, name))
    return SampleColumns.build(k, self.count, **cols)


class DeviceSampleColumns(object):
  """Output of BooleanSamplesDevice / AlgebraicDistanceSamplesDevice /
  WeightedJaccardSamplesDevice with ``keep_on_device=True``:
  the sampler's blocks in record order, each a set of CUDA tensors (``blocks[i].cols``,
  ``.prob``) with its record count.  ``to_host()`` is the SampleColumns the default call returns;
  ``Hg2vModel.fit_device`` packs the blocks into the model's sample buffer on the device."""

  def __init__(self, num_neighbors, blocks):
    self.num_neighbors = int(num_neighbors)
    self.blocks = list(blocks)

  @property
  def counts(self):
    return [b.count for b in self.blocks]

  def __len__(self):
    return sum(self.counts)

  def to_host(self):
    assert self.blocks, "the device blocks were released"
    return SampleColumns.concatenate([b.to_host(self.num_neighbors) for b in self.blocks])

  def release(self):
    """Drops the device tensors (the caller frees the cached memory, e.g. torch.cuda.empty_cache)."""
    self.blocks = []


def _device_result(blocks, k, stream, keep_on_device):
  """The three forms of a device sampler's result from its generator of _DeviceBlock."""
  if keep_on_device:
    assert not stream, "keep_on_device=True holds every block on the device; it does not stream"
    return DeviceSampleColumns(k, (b.compact() for b in blocks))
  chunks = (b.to_host(k) for b in blocks)
  if stream:
    return chunks
  return SampleColumns.concatenate(list(chunks))


def BooleanSamplesDevice(incidence, num_neighbors, num_samples, neg_samples=0, node_weights=None,
                         edge_weights=None, seed=0, chunk_rows=0, stream=False, keep_on_device=False):
  """BooleanSamplesCsr drawn on the GPU from seeded Philox streams instead of numpy's global
  MT19937 (which is neither read nor advanced).  Same distribution of every record as the
  reference's FOBE sampler, same blocks in the same order (node-node, edge-edge, node-edge rows,
  edge-node rows; with negatives their negative blocks, the edge-edge one twice as in the
  reference), same columns; not the reference's stream.  The result depends only on the graph,
  the counts and `seed`, not on `chunk_rows`.  With ``stream=True`` returns an iterator of
  SampleColumns chunks of about `chunk_rows` rows; with ``keep_on_device=True`` a
  DeviceSampleColumns whose blocks stay on the GPU; otherwise one SampleColumns."""
  assert num_neighbors >= 0
  assert num_samples >= 0
  assert neg_samples >= 0
  g = incidence if isinstance(incidence, _Graph) else _Graph.from_csr(incidence)
  node_s = _per_row(node_weights, g.num_nodes, num_samples)
  edge_s = _per_row(edge_weights, g.num_edges, num_samples)
  assert node_s.min(initial=0) >= 0 and edge_s.min(initial=0) >= 0
  k = num_neighbors

  def blocks():
    ctx = _native.default_context()
    inc = g.incidence(ctx)
    s = _DeviceSampler(g, ctx, inc, k, seed, chunk_rows)
    try:
      for side, samples, phase, left, right, prob in (
          (0, node_s, _native.PHASE_NN, "left_node", "right_node", "nn_prob"),
          (1, edge_s, _native.PHASE_EE, "left_edge", "right_edge", "ee_prob")):
        for r, c in s.pairs(side, 2, samples, phase):
          yield _DeviceBlock(r.shape[0], prob, **{left: r, right: c})
      phases = (_native.PHASE_NE, _native.PHASE_EN, _native.PHASE_NEIGHBORS)
      for nodes, edges, nbr_n, nbr_e in s.node_edge(node_s, edge_s, 1, phases):
        yield _DeviceBlock(nodes.shape[0], "ne_prob", left_node=nodes, right_edge=edges, neigh_node=nbr_n,
                           neigh_edge=nbr_e)
      if neg_samples > 0:
        neg_n = _per_row(node_weights, g.num_nodes, neg_samples)
        neg_e = _per_row(edge_weights, g.num_edges, neg_samples)
        for side, samples, phase, left, right in (
            (0, neg_n, _native.PHASE_NEG_NN, "left_node", "right_node"),
            (1, neg_e, _native.PHASE_NEG_EE, "left_edge", "right_edge"),
            (1, neg_e, _native.PHASE_NEG_EE_AGAIN, "left_edge", "right_edge")):   # sic, :215-221
          for r, c in s.pairs(side, 2, samples, phase, negative=True):
            yield _DeviceBlock(r.shape[0], **{left: r, right: c})
        phases = (_native.PHASE_NEG_NE, _native.PHASE_NEG_EN, _native.PHASE_NEG_NEIGHBORS)
        for nodes, edges, nbr_n, nbr_e in s.node_edge(neg_n, neg_e, 1, phases, negative=True):
          yield _DeviceBlock(nodes.shape[0], left_node=nodes, right_edge=edges, neigh_node=nbr_n,
                             neigh_edge=nbr_e)
    finally:
      inc.close()

  return _device_result(blocks(), k, stream, keep_on_device)


################################################################################
# WeightedJaccard Samples - helper and sampler                                 #
################################################################################


def SparseWeightedJaccard(row_i, row_j):
  """hg2v_sample.py:250-275: sum of minima over sum of maxima of two sparse 1 x F rows (0 when
  the denominator is 0)."""
  assert row_i.shape[0] == 1
  assert row_j.shape[0] == 1
  assert row_i.shape[1] == row_j.shape[1]
  feat = _native.FeatureCsr(sps.vstack([sps.csr_matrix(row_i), sps.csr_matrix(row_j)]))
  return _native.jaccard_rows(_native.default_context(), feat, [0], [1])[0]


def CentroidFromRows(idx, idx2targets=None, targets2features=None):
  """hg2v_sample.py:284-299: mean of the feature rows of idx's targets as (vals, (rows, cols)).
  Host bookkeeping kept for API compatibility; the sampler itself never materialises centroids
  (csrc/hge_jaccard.cu evaluates them on the fly)."""
  assert idx2targets is not None and targets2features is not None
  rows = sps.csr_matrix(idx2targets)[idx].nonzero()[1]
  centroid = sps.csr_matrix(targets2features)[rows].sum(axis=0) / len(rows)
  cols = centroid.nonzero()[1]
  return ([centroid[0, c] for c in cols], ([idx] * len(cols), list(cols)))


def GetAllCentroids(important_indices, idx2targets, targets2features, disable_pbar):
  """hg2v_sample.py:302-320."""
  del disable_pbar
  rows, cols, vals = [], [], []
  for idx in important_indices:
    v, (r, c) = CentroidFromRows(idx, idx2targets, targets2features)
    vals.extend(v)
    rows.extend(r)
    cols.extend(c)
  return sps.csr_matrix((vals, (rows, cols)),
                        shape=(idx2targets.shape[0], targets2features.shape[1]))


def SameTypeJaccardSample(indices, idx2features=None, is_edge=None):
  """hg2v_sample.py:323-340 with explicit arguments."""
  assert idx2features is not None
  idx, neighbor_idx = indices
  m = sps.csr_matrix(idx2features)
  prob = SparseWeightedJaccard(m[idx], m[neighbor_idx])
  if is_edge:
    return SimilarityRecord(left_edge_idx=idx, right_edge_idx=neighbor_idx,
                            edge_edge_prob=_alpha_scale(prob))
  return SimilarityRecord(left_node_idx=idx, right_node_idx=neighbor_idx,
                          node_node_prob=_alpha_scale(prob))


def DiffTypeJaccardSample(indices, node2edge=None, edge2node=None, num_neighbors=None,
                          node2features=None, edge2features=None, node2edge_centroid=None,
                          edge2node_centroid=None):
  """hg2v_sample.py:343-392 with explicit arguments: neighbour arrays from the global RNG (edges
  of the node first), the two Jaccard factors as left / right weight, their product as the
  probability.  The centroid matrices are accepted for compatibility and not needed: the
  kernel evaluates the centroids on the fly."""
  del node2edge_centroid, edge2node_centroid
  assert None not in (node2edge, edge2node, num_neighbors, node2features, edge2features)
  node_idx, edge_idx = indices
  assert node2edge.shape[0] == node2features.shape[0]
  assert node2edge.shape[1] == edge2node.shape[0]
  assert edge2node.shape[0] == edge2features.shape[0]
  neighbor_edge_indices = _sample_neighbors(node_idx, node2edge, num_neighbors)
  neighbor_node_indices = _sample_neighbors(edge_idx, edge2node, num_neighbors)
  ctx = _native.default_context()
  nf, ef = _native.FeatureCsr(node2features), _native.FeatureCsr(edge2features)
  prob_by_node = _native.jaccard_centroid(ctx, nf, _native.CsrArrays(edge2node), nf, [node_idx],
                                          [edge_idx])[0]
  prob_by_edge = _native.jaccard_centroid(ctx, ef, _native.CsrArrays(node2edge), ef, [edge_idx],
                                          [node_idx])[0]
  return SimilarityRecord(left_node_idx=node_idx, right_edge_idx=edge_idx, left_weight=prob_by_node,
                          right_weight=prob_by_edge, neighbor_node_indices=neighbor_node_indices,
                          neighbor_edge_indices=neighbor_edge_indices,
                          node_edge_prob=_alpha_scale(prob_by_node * prob_by_edge))


def WeightedJaccardSamples(hypergraph, node2features, edge2features, num_neighbors, num_samples,
                           run_in_parallel=True, disable_pbar=False):
  """hg2v_sample.py:398-510: node-node / edge-edge samples weighted by the sparse weighted
  Jaccard of their feature rows, node-edge samples by the product of J(node features, centroid
  of the edge's members' features) and J(edge features, centroid of the node's edges'
  features), both factors recorded as left / right weight.

  Pair sets come from the global RNG exactly as the reference draws them; the neighbour arrays
  are drawn the way the reference's single worker (``run_in_parallel=False``) draws them, from
  a copy of the RNG state the parent had when the pair sampling ended."""
  del run_in_parallel, disable_pbar
  log.info("Performing input checks")
  assert num_neighbors >= 0
  assert num_samples >= 0
  node_samples = [int(node.weight * num_samples) for _, node in hypergraph.node.items()]
  edge_samples = [int(edge.weight * num_samples) for _, edge in hypergraph.edge.items()]

  g = _Graph(hypergraph)
  k = num_neighbors
  log.info("Checking that feature matrices agree with the sparse matrices")
  assert g.num_nodes == node2features.shape[0]     # hg2v_sample.py:430
  assert g.num_edges == edge2features.shape[0]     # hg2v_sample.py:458
  nf = _native.FeatureCsr(node2features)
  ef = _native.FeatureCsr(edge2features)
  ctx = _native.default_context()
  state = _native.LegacyRngState()
  parts = []

  log.info("Getting node-node samples")
  r, c = _native.sample_adj_rows((g.a, g.at), g.node_rows, node_samples, state)
  log.info("Sampling node-node probabilities")
  parts.append(SampleColumns.build(k, len(r), left_node=r, right_node=c,
                                   nn_prob=_native.jaccard_rows(ctx, nf, r, c)))
  log.info("Getting edge-edge samples")
  r, c = _native.sample_adj_rows((g.b, g.bt), g.edge_rows, edge_samples, state)
  log.info("Sampling edge-edge probabilities")
  parts.append(SampleColumns.build(k, len(r), left_edge=r, right_edge=c,
                                   ee_prob=_native.jaccard_rows(ctx, ef, r, c)))
  log.info("Getting node-edge samples")
  n1, e1 = _native.sample_adj_rows((g.a, g.at, g.a), g.node_rows, node_samples, state)
  log.info("Getting edge-node samples")
  e2, n2 = _native.sample_adj_rows((g.b, g.bt, g.b), g.edge_rows, edge_samples, state)
  state.commit()   # the parent's stream ends here (the worker draws from a copy)
  nodes, edges = np.concatenate([n1, n2]), np.concatenate([e1, e2])
  nbr_e, nbr_n = _native.sample_neighbors(g.a, g.b, nodes, edges, k, state.copy())
  log.info("Getting node-edge relationships")
  # centroid of an edge = mean of its member nodes' feature rows, and vice versa
  prob_by_node = _native.jaccard_centroid(ctx, nf, g.b, nf, nodes, edges)
  prob_by_edge = _native.jaccard_centroid(ctx, ef, g.a, ef, edges, nodes)
  parts.append(SampleColumns.build(k, len(nodes), left_node=nodes, right_edge=edges,
                                   neigh_node=nbr_n, neigh_edge=nbr_e,
                                   left_weight=prob_by_node, right_weight=prob_by_edge,
                                   ne_prob=prob_by_node * prob_by_edge))
  return SampleColumns.concatenate(parts)


def WeightedJaccardSamplesDevice(incidence, node2features, edge2features, num_neighbors, num_samples,
                                 node_weights=None, edge_weights=None, seed=0, chunk_rows=0, stream=False,
                                 timings=None, keep_on_device=False, workspace_mb=0):
  """WeightedJaccardSamples on an N x E incidence CSR (or a _Graph) with the pairs and neighbour
  arrays drawn on the GPU from seeded Philox streams, as AlgebraicDistanceSamplesDevice draws them
  (numpy's global MT19937 is neither read nor advanced), and every probability computed on the
  device from the drawn pairs.  Row r emits int(weight_r * num_samples) samples (weights default
  to 1).  Same blocks and columns as the reference's Jaccard sampler: node-node (nn_prob),
  edge-edge (ee_prob), then node-edge rows and edge-node rows with left_weight = J(node features,
  centroid of the edge's nodes' features), right_weight = J(edge features, centroid of the node's
  edges' features) and ne_prob their fp32 product; not the reference's stream.  The feature
  matrices (any scipy sparse matrices) are uploaded once per call.  The result depends on the
  graph, the features, the counts and `seed`, not on `chunk_rows` or `workspace_mb` (megabytes of
  one expansion batch of the candidate and centroid rows, 0 = 2048).  With ``stream=True`` returns
  an iterator of SampleColumns chunks of about `chunk_rows` rows, with ``keep_on_device=True`` a
  DeviceSampleColumns (see BooleanSamplesDevice).  `timings` (a dict) receives the seconds spent
  drawing pairs ("pairs") and neighbour arrays ("neighbours") and uploading the features and
  computing the probabilities ("probabilities"); it is filled when the result is complete."""
  import time
  import torch
  assert num_neighbors >= 0
  assert num_samples >= 0
  g = incidence if isinstance(incidence, _Graph) else _Graph.from_csr(incidence)
  assert g.num_nodes == node2features.shape[0]     # hg2v_sample.py:430
  assert g.num_edges == edge2features.shape[0]     # hg2v_sample.py:458
  nf, ef = _native.FeatureCsr(node2features), _native.FeatureCsr(edge2features)
  node_s = _per_row(node_weights, g.num_nodes, num_samples)
  edge_s = _per_row(edge_weights, g.num_edges, num_samples)
  assert node_s.min(initial=0) >= 0 and edge_s.min(initial=0) >= 0
  k = num_neighbors

  def blocks():
    ctx = _native.default_context()
    spent = {"probabilities": 0.0}

    def prob(fn, *args, **kw):
      t = time.perf_counter()
      out = fn(*args, **kw)
      ctx.sync()
      spent["probabilities"] += time.perf_counter() - t
      return out

    dev = torch.device("cuda", ctx.device)
    nfd, efd = prob(nf.to_device, dev), prob(ef.to_device, dev)
    inc = g.incidence(ctx)
    s = _DeviceSampler(g, ctx, inc, k, seed, chunk_rows, workspace_mb)
    try:
      for side, samples, phase, left, right, field, feat in (
          (0, node_s, _native.PHASE_NN, "left_node", "right_node", "nn_prob", nfd),
          (1, edge_s, _native.PHASE_EE, "left_edge", "right_edge", "ee_prob", efd)):
        for r, c in s.pairs(side, 2, samples, phase):
          p = prob(_native.jaccard_rows, ctx, feat, r, c)
          yield _DeviceBlock(p.shape[0], field, p, **{left: r, right: c})
      phases = (_native.PHASE_NE, _native.PHASE_EN, _native.PHASE_NEIGHBORS)
      for nodes, edges, nbr_n, nbr_e in s.node_edge(node_s, edge_s, 3, phases):
        # centroid of an edge = mean of its member nodes' feature rows, and vice versa
        by_node = prob(_native.jaccard_centroid_grouped, ctx, inc, 1, nfd, nfd, nodes, edges, workspace_mb)
        by_edge = prob(_native.jaccard_centroid_grouped, ctx, inc, 0, efd, efd, edges, nodes, workspace_mb)
        yield _DeviceBlock(nodes.shape[0], "ne_prob", by_node * by_edge, left_weight=by_node,
                           right_weight=by_edge, left_node=nodes, right_edge=edges, neigh_node=nbr_n,
                           neigh_edge=nbr_e)
    finally:
      inc.close()
    if timings is not None:
      timings.update(s.spent)
      timings.update(spent)

  return _device_result(blocks(), k, stream, keep_on_device)


################################################################################
# AlgebraicDistanceSamples - With helpers                                      #
################################################################################


class _HobeWeights(object):
  """Incidence weights W(n, e) = (sqrt(R) - ||xn[n] - xe[e]||) / sqrt(R) in both storage
  orders, resident on the device; every w(.,.) the reference evaluates is one of them
  (SURVEY.md section 0.2)."""

  def __init__(self, graph, xn, xe, ctx=None):
    import torch
    self.ctx = ctx or _native.default_context()
    self.graph = graph
    self.inc = graph.incidence(self.ctx)
    dev = torch.device("cuda", self.ctx.device)
    xn_d = torch.from_numpy(np.ascontiguousarray(xn, dtype=np.float32)).to(dev)
    xe_d = torch.from_numpy(np.ascontiguousarray(xe, dtype=np.float32)).to(dev)
    self.w_n2e = _native.incidence_l2(self.ctx, self.inc, xn_d, xe_d, order=0, as_weight=True)
    self.w_e2n = _native.incidence_l2(self.ctx, self.inc, xn_d, xe_d, order=1, as_weight=True)
    self.dev = dev

  def _dev(self, a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(self.dev)

  def same_type(self, side, pi, pj):
    w = self.w_n2e if side == 0 else self.w_e2n
    return _native.same_type_prob(self.ctx, self.inc, side, w, self._dev(pi),
                                  self._dev(pj)).cpu().numpy()

  def diff_type(self, pn, pe):
    return _native.diff_type_prob(self.ctx, self.inc, self.w_e2n, self._dev(pn),
                                  self._dev(pe)).cpu().numpy()

  def close(self):
    self.inc.close()


def _same_type_dist_calc(indices, idx2target, source_half_emb, target_half_emb):
  """hg2v_sample.py:527-543 for one pair (compat entry point; the samplers batch this)."""
  m = sps.csr_matrix(idx2target)
  n_src, n_tgt = m.shape
  xs = np.zeros((n_src, len(source_half_emb[indices[0]].values)), np.float32)
  xt = np.zeros((n_tgt, xs.shape[1]), np.float32)
  for i in (indices[0], indices[1]):
    xs[i] = source_half_emb[i].values
  for k in set(m[indices[0]].indices) | set(m[indices[1]].indices):
    xt[k] = target_half_emb[int(k)].values
  ctx = _native.default_context()
  ptr_, idx_ = _native.CsrArrays(m).ptr, _native.CsrArrays(m).idx
  mt = m.T.tocsr()
  mt.sort_indices()
  inc = _native.Incidence(ctx, n_src, n_tgt, ptr_, idx_, np.asarray(mt.indptr, np.int64),
                          np.asarray(mt.indices, np.int32))
  try:
    w = _native.incidence_l2(ctx, inc, xs, xt, order=0, as_weight=True)
    prob = _native.same_type_prob(ctx, inc, 0, w, [indices[0]], [indices[1]])[0]
  finally:
    inc.close()
  has_shared = len(set(m[indices[0]].indices) & set(m[indices[1]].indices)) > 0
  return prob if has_shared else 0


def AlgebraicDistanceSamples(hypergraph, algebraic_embedding, num_neighbors, num_samples,
                             run_in_parallel=True, disable_pbar=False):
  """hg2v_sample.py:632-717 (HOBE): node-node, edge-edge and node-edge samples whose
  probability is the max-min algebraic-distance weight over shared neighbours.

  Pair sets are drawn from the global RNG exactly as the reference's parent process draws
  them.  The neighbour arrays of node-edge records are drawn by the reference inside forked
  workers that inherit a copy of the parent's RNG; this implementation reproduces the
  ``run_in_parallel=False`` behaviour (one worker, records in order) for either flag value,
  and like the reference leaves the global RNG where the pair sampling left it."""
  del run_in_parallel, disable_pbar
  log.info("Performing input checks")
  assert num_neighbors >= 0
  assert num_samples >= 0

  g = _Graph(hypergraph)
  xn, xe = embedding_to_arrays(algebraic_embedding, g.num_nodes, g.num_edges)
  return _hobe_samples(g, xn, xe, num_neighbors, num_samples)


def AlgebraicDistanceSamplesCsr(incidence, xn, xe, num_neighbors, num_samples, timings=None):
  """AlgebraicDistanceSamples on an N x E incidence given as a scipy CSR matrix and dense fp32
  vector blocks [N, R], [E, R] -- the form a caller at scale holds (building the proto alone
  takes longer than the sampling; cf. BooleanSamplesCsr).  Same records, same consumption of the
  global numpy RNG.  `timings` (a dict) receives the seconds spent replaying the RNG stream on
  the host ("draw") and computing probabilities on the device ("probabilities")."""
  assert num_neighbors >= 0
  assert num_samples >= 0
  g = incidence if isinstance(incidence, _Graph) else _Graph.from_csr(incidence)
  xn = np.ascontiguousarray(xn, dtype=np.float32)
  xe = np.ascontiguousarray(xe, dtype=np.float32)
  assert xn.shape[0] == g.num_nodes and xe.shape[0] == g.num_edges and xn.shape[1] == xe.shape[1]
  return _hobe_samples(g, xn, xe, num_neighbors, num_samples, timings)


def _hobe_samples(g, xn, xe, k, num_samples, timings=None):
  import time
  spent = {"draw": 0.0, "probabilities": 0.0, "weights": 0.0}

  def timed(kind, fn, *args):
    t = time.perf_counter()
    out = fn(*args)
    spent[kind] += time.perf_counter() - t
    return out

  weights = timed("weights", _HobeWeights, g, xn, xe)
  try:
    state = _native.LegacyRngState()
    parts = []
    log.info("Getting node-node samples")
    per_node = [num_samples] * len(g.node_rows)
    per_edge = [num_samples] * len(g.edge_rows)
    r, c = timed("draw", _native.sample_adj_rows, (g.a, g.at), g.node_rows, per_node, state)
    log.info("Sampling node-node probabilities")
    parts.append(SampleColumns.build(k, len(r), left_node=r, right_node=c,
                                     nn_prob=timed("probabilities", weights.same_type, 0, r, c)))
    log.info("Getting edge-edge samples")
    r, c = timed("draw", _native.sample_adj_rows, (g.b, g.bt), g.edge_rows, per_edge, state)
    log.info("Sampling edge-edge probabilities")
    parts.append(SampleColumns.build(k, len(r), left_edge=r, right_edge=c,
                                     ee_prob=timed("probabilities", weights.same_type, 1, r, c)))
    log.info("Getting node-edge samples")
    n1, e1 = timed("draw", _native.sample_adj_rows, (g.a, g.at, g.a), g.node_rows, per_node, state)
    log.info("Getting edge-node samples")
    e2, n2 = timed("draw", _native.sample_adj_rows, (g.b, g.bt, g.b), g.edge_rows, per_edge, state)
    state.commit()   # the parent's stream ends here (workers draw from a copy)
    nodes, edges = np.concatenate([n1, n2]), np.concatenate([e1, e2])
    nbr_e, nbr_n = timed("draw", _native.sample_neighbors, g.a, g.b, nodes, edges, k, state.copy())
    parts.append(SampleColumns.build(k, len(nodes), left_node=nodes, right_edge=edges,
                                     neigh_node=nbr_n, neigh_edge=nbr_e,
                                     ne_prob=timed("probabilities", weights.diff_type, nodes, edges)))
  finally:
    weights.close()
  if timings is not None:
    timings.update(spent)
  return SampleColumns.concatenate(parts)


def AlgebraicDistanceSamplesDevice(incidence, xn, xe, num_neighbors, num_samples, seed=0,
                                   chunk_rows=0, stream=False, timings=None, keep_on_device=False):
  """AlgebraicDistanceSamplesCsr with the pairs and neighbour arrays drawn on the GPU from seeded
  Philox streams (see BooleanSamplesDevice) instead of numpy's global MT19937, which is neither
  read nor advanced.  The pairs stay on the device and go straight into the probability kernels.
  Same blocks, columns and probabilities as the reference's HOBE sampler; not its stream.  With
  ``stream=True`` returns an iterator of SampleColumns chunks of about `chunk_rows` rows, with
  ``keep_on_device=True`` a DeviceSampleColumns (see BooleanSamplesDevice).
  `timings` (a dict) receives the seconds spent drawing pairs ("pairs") and neighbour arrays
  ("neighbours") and computing the incidence weights and probabilities ("probabilities"); it is
  filled when the result is complete."""
  import time
  assert num_neighbors >= 0
  assert num_samples >= 0
  g = incidence if isinstance(incidence, _Graph) else _Graph.from_csr(incidence)
  xn = np.ascontiguousarray(xn, dtype=np.float32)
  xe = np.ascontiguousarray(xe, dtype=np.float32)
  assert xn.shape[0] == g.num_nodes and xe.shape[0] == g.num_edges and xn.shape[1] == xe.shape[1]
  k = num_neighbors
  per_node = _per_row(None, g.num_nodes, num_samples)
  per_edge = _per_row(None, g.num_edges, num_samples)

  def blocks():
    spent = {"probabilities": 0.0}
    t = time.perf_counter()
    weights = _HobeWeights(g, xn, xe)
    spent["probabilities"] += time.perf_counter() - t
    ctx, inc = weights.ctx, weights.inc

    def prob(fn, *args):
      t = time.perf_counter()
      out = fn(*args)
      ctx.sync()
      spent["probabilities"] += time.perf_counter() - t
      return out

    s = _DeviceSampler(g, ctx, inc, k, seed, chunk_rows)
    try:
      for side, samples, phase, left, right, field, w in (
          (0, per_node, _native.PHASE_NN, "left_node", "right_node", "nn_prob", weights.w_n2e),
          (1, per_edge, _native.PHASE_EE, "left_edge", "right_edge", "ee_prob", weights.w_e2n)):
        for r, c in s.pairs(side, 2, samples, phase):
          p = prob(_native.same_type_prob, ctx, inc, side, w, r, c)
          yield _DeviceBlock(p.shape[0], field, p, **{left: r, right: c})
      phases = (_native.PHASE_NE, _native.PHASE_EN, _native.PHASE_NEIGHBORS)
      for nodes, edges, nbr_n, nbr_e in s.node_edge(per_node, per_edge, 3, phases):
        p = prob(_native.diff_type_prob, ctx, inc, weights.w_e2n, nodes, edges)
        yield _DeviceBlock(p.shape[0], "ne_prob", p, left_node=nodes, right_edge=edges, neigh_node=nbr_n,
                           neigh_edge=nbr_e)
    finally:
      weights.close()
    if timings is not None:
      timings.update(s.spent)
      timings.update(spent)

  return _device_result(blocks(), k, stream, keep_on_device)


def SameTypeDistanceSample(indices, idx2target=None, source_half_emb=None, target_half_emb=None,
                           is_edge=None):
  """hg2v_sample.py:546-576 with explicit arguments (the reference's worker-global fallback
  does not exist here: there are no worker processes)."""
  assert idx2target is not None and source_half_emb is not None and target_half_emb is not None
  prob = _same_type_dist_calc(indices, idx2target, source_half_emb, target_half_emb)
  if is_edge:
    return SimilarityRecord(left_edge_idx=indices[0], right_edge_idx=indices[1],
                            edge_edge_prob=_alpha_scale(prob))
  return SimilarityRecord(left_node_idx=indices[0], right_node_idx=indices[1],
                          node_node_prob=_alpha_scale(prob))


def DiffTypeDistanceSample(indices, node2edge=None, edge2node=None, num_neighbors=None,
                           algebraic_embedding=None):
  """hg2v_sample.py:588-629 with explicit arguments: neighbour arrays from the global RNG and
  the max over the node's edges of the edge-edge probability."""
  assert None not in (node2edge, edge2node, num_neighbors, algebraic_embedding)
  node_idx, edge_idx = indices
  neighbor_edge_indices = _sample_neighbors(node_idx, node2edge, num_neighbors)
  neighbor_node_indices = _sample_neighbors(edge_idx, edge2node, num_neighbors)
  a, b = _native.CsrArrays(node2edge), _native.CsrArrays(edge2node)
  xn, xe = embedding_to_arrays(algebraic_embedding, a.shape[0], b.shape[0])
  ctx = _native.default_context()
  inc = _native.Incidence(ctx, a.shape[0], b.shape[0], a.ptr, a.idx, b.ptr, b.idx)
  try:
    w_e2n = _native.incidence_l2(ctx, inc, xn, xe, order=1, as_weight=True)
    prob = _native.diff_type_prob(ctx, inc, w_e2n, [node_idx], [edge_idx])[0]
  finally:
    inc.close()
  return SimilarityRecord(left_node_idx=node_idx, right_edge_idx=edge_idx,
                          neighbor_node_indices=neighbor_node_indices,
                          neighbor_edge_indices=neighbor_edge_indices,
                          node_edge_prob=_alpha_scale(prob))


################################################################################
# Samples to Model Input w/ Helper functions                                   #
################################################################################


def _columns_to_model_input(cols, num_neighbors, weighted):
  m = len(cols)
  zeros_i = np.zeros(m, dtype=np.int32)
  zeros_f = np.zeros(m, dtype=np.float32)

  def inc(a):
    return (a + 1).astype(np.int32)      # -1 (None) becomes the padding index 0

  def neigh(a):
    out = []
    for i in range(num_neighbors):
      out.append(inc(a[:, i]) if i < a.shape[1] else zeros_i.copy())
    return out

  features = [inc(cols.left_node), inc(cols.left_edge), inc(cols.right_node), inc(cols.right_edge)]
  if weighted:
    features += [np.nan_to_num(cols.left_weight, nan=0.0), np.nan_to_num(cols.right_weight, nan=0.0)]
  features += neigh(cols.neigh_node)
  if weighted:
    features += [zeros_f.copy() for _ in range(num_neighbors)]
  features += neigh(cols.neigh_edge)
  if weighted:
    features += [zeros_f.copy() for _ in range(num_neighbors)]
  targets = [np.nan_to_num(cols.nn_prob, nan=0.0), np.nan_to_num(cols.ee_prob, nan=0.0),
             np.nan_to_num(cols.ne_prob, nan=0.0)]
  return (features, targets)


def SamplesToModelInput(similarity_records, num_neighbors, weighted=True):
  """hg2v_sample.py:751-797: (input arrays, output arrays).  Indices are shifted by +1 because
  0 is the padding row of the embedding tables; None becomes 0; neighbour lists are padded
  to num_neighbors.  A ``SampleColumns`` is packed column-wise into numpy arrays; any other
  iterable of records goes through the reference's record loop and yields Python lists."""
  if isinstance(similarity_records, SampleColumns):
    return _columns_to_model_input(similarity_records, num_neighbors, weighted)

  records = list(similarity_records)

  def scalar(field, shift):
    # None -> 0; indices are shifted past the padding row
    return [0 if getattr(r, field) is None else getattr(r, field) + shift for r in records]

  def padded(field, shift):
    cols = []
    for i in range(num_neighbors):
      col = []
      for r in records:
        arr = getattr(r, field)
        col.append(0 if arr is None or i >= len(arr) else arr[i] + shift)
      cols.append(col)
    return cols

  features = [scalar("left_node_idx", 1), scalar("left_edge_idx", 1), scalar("right_node_idx", 1),
              scalar("right_edge_idx", 1)]
  if weighted:
    features += [scalar("left_weight", 0), scalar("right_weight", 0)]
  features += padded("neighbor_node_indices", 1)
  if weighted:
    features += padded("neighbor_node_weights", 0)
  features += padded("neighbor_edge_indices", 1)
  if weighted:
    features += padded("neighbor_edge_weights", 0)
  targets = [scalar("node_node_prob", 0), scalar("edge_edge_prob", 0), scalar("node_edge_prob", 0)]
  return (features, targets)


################################################################################
# Debug summary                                                                #
################################################################################


def PlotDistributions(debug_summary_path, sim_records):
  """hg2v_sample.py:805-853: histograms of the per-entity weights and of the three probability
  kinds, written to `debug_summary_path`.  matplotlib is an optional dependency; without it this
  raises (the reference would have failed at import), it never skips the file silently."""
  try:
    import matplotlib
    matplotlib.use("Agg")
    import matplotlib.pyplot as plt
  except ImportError as exc:
    raise ImportError("debug_summary_path needs matplotlib for PlotDistributions "
                      "(hg2v_sample.py:805-853): %s" % exc)
  log.info("Writing Debug Summary to %s", debug_summary_path)
  node2features, edge2features = {}, {}
  for r in sim_records:
    if r.left_weight is not None:
      if r.left_node_idx is not None and r.left_node_idx not in node2features:
        node2features[r.left_node_idx] = r.left_weight
      if r.left_edge_idx is not None and r.left_edge_idx not in edge2features:
        edge2features[r.left_edge_idx] = r.left_weight
    if r.right_weight is not None:
      if r.right_node_idx is not None and r.right_node_idx not in node2features:
        node2features[r.right_node_idx] = r.right_weight
      if r.right_edge_idx is not None and r.right_edge_idx not in edge2features:
        edge2features[r.right_edge_idx] = r.right_weight
  nn_probs = [r.node_node_prob for r in sim_records if r.node_node_prob is not None]
  ee_probs = [r.edge_edge_prob for r in sim_records if r.edge_edge_prob is not None]
  ne_probs = [r.node_edge_prob for r in sim_records if r.node_edge_prob is not None]
  fig, (node_spans, edge_spans, nn_ax, ee_ax, ne_ax) = plt.subplots(5, 1, figsize=(8.5, 11))
  if node2features:
    node_spans.set_title("Node Weights")
    node_spans.hist(list(node2features.values()))
    node_spans.set_yscale("log")
  if edge2features:
    edge_spans.set_title("Edge Weights")
    edge_spans.hist(list(edge2features.values()))
    edge_spans.set_yscale("log")
  for ax, title, probs in ((nn_ax, "Node-Node Probability Distribution", nn_probs),
                           (ee_ax, "Edge-Edge Probability Distribution", ee_probs),
                           (ne_ax, "Node-Edge Probability Distribution", ne_probs)):
    ax.set_title(title)
    ax.hist(probs)
    ax.set_yscale("log")
  fig.tight_layout()
  fig.savefig(debug_summary_path)
  plt.close(fig)
