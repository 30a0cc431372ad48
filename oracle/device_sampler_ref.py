"""Numpy restatement of the device sampler (csrc/hge_device_sampler.cu, csrc/hge_philox.cuh):
Philox4x32-10 word streams keyed by the seed with counter {block, item lo, item hi, phase},
Lemire's bounded draws with rejection, Floyd's selection over the sorted distinct candidates of a
product row, one stream per row (pairs) or per record of a block (neighbour arrays), and the
blocks of BooleanSamplesDevice / AlgebraicDistanceSamplesDevice in their order.

Test infrastructure only.  Everything is vectorised over rows / records: step s of every row's
sequential loop runs at once for all rows that still have a step s.
"""
import numpy as np
import scipy.sparse as sps

MASK = np.uint64(0xFFFFFFFF)
_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)

PHASE = dict(NN=1, EE=2, NE=3, EN=4, NEIGHBORS=5, NEG_NN=6, NEG_EE=7, NEG_EE_AGAIN=8, NEG_NE=9,
             NEG_EN=10, NEG_NEIGHBORS=11)


def philox4x32_10(ctr, key):
  """ctr: 4 arrays (or ints) of uint32 values, key: 2; returns the 4 output words as uint64 arrays."""
  c = [np.asarray(x, dtype=np.uint64) for x in ctr]
  k0, k1 = (np.asarray(x, dtype=np.uint64) for x in key)
  for _ in range(10):
    p0 = _M0 * c[0]
    p1 = _M1 * c[2]
    c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & MASK, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & MASK]
    k0 = (k0 + _W0) & MASK
    k1 = (k1 + _W1) & MASK
  return c


class Streams(object):
  """The word streams of many items of one (seed, phase), each with its own read position."""

  def __init__(self, seed, phase, items):
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    self.key = (np.uint64(seed & 0xFFFFFFFF), np.uint64(seed >> 32))
    self.phase = np.uint64(phase)
    self.items = np.asarray(items, dtype=np.uint64)
    self.word = np.zeros(len(self.items), dtype=np.int64)

  def next(self, sel):
    """Next word of the items `sel` (an index array)."""
    w = self.word[sel]
    it = self.items[sel]
    out = philox4x32_10((w // 4, it & MASK, it >> np.uint64(32), self.phase), self.key)
    self.word[sel] += 1
    return np.choose(w % 4, out).astype(np.uint64)

  def below(self, sel, s):
    """Uniform on [0, s) for the items `sel` (Lemire: m = x * s, redraw while low32(m) <
    (2^32 - s) mod s)."""
    sel = np.asarray(sel, dtype=np.int64)
    s = np.broadcast_to(np.asarray(s, dtype=np.uint64), sel.shape).copy()
    t = (np.uint64(1 << 32) - s) % s
    m = self.next(sel) * s
    redo = np.nonzero((m & MASK) < t)[0]
    while len(redo):
      m[redo] = self.next(sel[redo]) * s[redo]
      redo = redo[(m[redo] & MASK) < t[redo]]
    return (m >> np.uint64(32)).astype(np.int64)


def transpose(A):
  B = sps.csr_matrix(A).T.tocsr()
  B.sort_indices()
  return B


def candidate_rows(A, side, factors):
  """(indptr, indices) of the sorted distinct candidates of every row of M1, M1 * M2 or
  (M1 * M2) * M3, with M1 = M3 = A, M2 = A^T for side 0 and the other way round for side 1."""
  A = sps.csr_matrix(A, dtype=np.int64)
  B = transpose(A)
  m1, m2 = (A, B) if side == 0 else (B, A)
  p = m1
  if factors >= 2:
    p = (m1 @ m2).astype(bool).astype(np.int64)
  if factors == 3:
    p = p @ m1
  p = sps.csr_matrix(p)
  p.sum_duplicates()
  p.sort_indices()
  return np.asarray(p.indptr, dtype=np.int64), np.asarray(p.indices, dtype=np.int64), p.shape[1]


def select(cptr, ccol, k, seed, phase, row0=0):
  """Positives of rows row0, row0 + 1, ...: min(k_r, n_r) of the row's candidates by Floyd's
  algorithm (a row with k_r >= n_r takes all and draws nothing), ascending."""
  rows = row0 + np.arange(len(cptr) - 1, dtype=np.int64)
  n = np.diff(cptr)
  kk = np.minimum(np.maximum(np.asarray(k, dtype=np.int64), 0), n)
  flags = np.repeat(kk == n, n)
  part = np.nonzero((kk > 0) & (kk < n))[0]
  st = Streams(seed, phase, rows[part])
  steps = kk[part]
  start = n[part] - steps
  base = cptr[part]
  for s in range(int(steps.max(initial=0))):
    act = np.nonzero(s < steps)[0]
    j = start[act] + s
    t = st.below(act, j + 1)
    hit = flags[base[act] + t]
    flags[base[act] + np.where(hit, j, t)] = True
  return np.repeat(rows, n)[flags], np.asarray(ccol)[flags]


def negatives(k, out_cols, seed, phase, row0=0):
  """k_r draws with replacement, uniform on [0, out_cols), of rows row0, row0 + 1, ..."""
  k = np.maximum(np.asarray(k, dtype=np.int64), 0)
  rows = row0 + np.arange(len(k), dtype=np.int64)
  st = Streams(seed, phase, rows)
  kmax = int(k.max(initial=0))
  out = np.zeros((len(k), kmax), dtype=np.int64)
  for j in range(kmax):
    act = np.nonzero(j < k)[0]
    out[act, j] = st.below(act, out_cols)
  keep = np.arange(kmax)[None, :] < k[:, None]
  return np.repeat(rows, k), out[keep]


def neighbors(A, nodes, edges, k, seed, phase, first=0):
  """([m, k] draws from the nodes' edges, [m, k] draws from the edges' nodes), record i owning
  stream first + i."""
  A = sps.csr_matrix(A)
  B = transpose(A)
  nodes = np.asarray(nodes, dtype=np.int64)
  edges = np.asarray(edges, dtype=np.int64)
  m = len(nodes)
  nbr_e = np.zeros((m, k), dtype=np.int64)
  nbr_n = np.zeros((m, k), dtype=np.int64)
  if m == 0 or k == 0:
    return nbr_e, nbr_n
  ns, nd = A.indptr[nodes], np.diff(A.indptr)[nodes]
  es, ed = B.indptr[edges], np.diff(B.indptr)[edges]
  if np.any(nd == 0) or np.any(ed == 0):
    raise ValueError("'a' cannot be empty unless no samples are taken")
  st = Streams(seed, phase, first + np.arange(m))
  every = np.arange(m)
  for j in range(k):
    nbr_e[:, j] = A.indices[ns + st.below(every, nd)]
  for j in range(k):
    nbr_n[:, j] = B.indices[es + st.below(every, ed)]
  return nbr_e, nbr_n


def _block(count, k, **cols):
  out = {name: np.full(count, -1, dtype=np.int64)
         for name in ("left_node", "left_edge", "right_node", "right_edge")}
  for name in ("nn_prob", "ee_prob", "ne_prob"):
    out[name] = np.full(count, np.nan, dtype=np.float32)
  out["neigh_node"] = np.full((count, k), -1, dtype=np.int64)
  out["neigh_edge"] = np.full((count, k), -1, dtype=np.int64)
  out["has_neighbors"] = np.full(count, "neigh_node" in cols)
  out.update(cols)
  return out


def _concat(blocks):
  return {name: np.concatenate([b[name] for b in blocks]) for name in blocks[0]}


def _pairs(A, side, factors, k, seed, phase, negative):
  cptr, ccol, out_cols = candidate_rows(A, side, factors)
  if negative:
    return negatives(k, out_cols, seed, phase)
  return select(cptr, ccol, k, seed, phase)


def _node_edge(A, k, node_s, edge_s, factors, seed, phases, negative, ones):
  ne, en, nbr = phases
  n1, e1 = _pairs(A, 0, factors, node_s, seed, PHASE[ne], negative)
  e2, n2 = _pairs(A, 1, factors, edge_s, seed, PHASE[en], negative)
  nodes, edges = np.concatenate([n1, n2]), np.concatenate([e1, e2])
  nbr_e, nbr_n = neighbors(A, nodes, edges, k, seed, PHASE[nbr])
  cols = dict(left_node=nodes, right_edge=edges, neigh_node=nbr_n, neigh_edge=nbr_e)
  if ones:
    cols["ne_prob"] = np.ones(len(nodes), dtype=np.float32)
  return _block(len(nodes), k, **cols)


def boolean_samples(A, k, num_samples, neg_samples=0, seed=0, node_weights=None, edge_weights=None):
  """Columns of BooleanSamplesDevice (SampleColumns.FIELDS without the weights)."""
  A = sps.csr_matrix(A)
  N, E = A.shape

  def per_row(w, count, base):
    if w is None:
      return np.full(count, int(base), dtype=np.int64)
    return np.asarray([int(x * base) for x in w], dtype=np.int64)

  node_s, edge_s = per_row(node_weights, N, num_samples), per_row(edge_weights, E, num_samples)
  blocks = []
  for side, s, phase, l, r, p in ((0, node_s, "NN", "left_node", "right_node", "nn_prob"),
                                  (1, edge_s, "EE", "left_edge", "right_edge", "ee_prob")):
    a, b = _pairs(A, side, 2, s, seed, PHASE[phase], False)
    blocks.append(_block(len(a), k, **{l: a, r: b, p: np.ones(len(a), dtype=np.float32)}))
  blocks.append(_node_edge(A, k, node_s, edge_s, 1, seed, ("NE", "EN", "NEIGHBORS"), False, True))
  if neg_samples > 0:
    neg_n, neg_e = per_row(node_weights, N, neg_samples), per_row(edge_weights, E, neg_samples)
    for side, s, phase, l, r in ((0, neg_n, "NEG_NN", "left_node", "right_node"),
                                 (1, neg_e, "NEG_EE", "left_edge", "right_edge"),
                                 (1, neg_e, "NEG_EE_AGAIN", "left_edge", "right_edge")):
      a, b = _pairs(A, side, 2, s, seed, PHASE[phase], True)
      blocks.append(_block(len(a), k, **{l: a, r: b}))
    blocks.append(_node_edge(A, k, neg_n, neg_e, 1, seed, ("NEG_NE", "NEG_EN", "NEG_NEIGHBORS"),
                             True, False))
  return _concat(blocks)


def hobe_pairs(A, k, num_samples, seed=0):
  """Index and neighbour columns of AlgebraicDistanceSamplesDevice (its probabilities come from
  the existing HOBE kernels)."""
  A = sps.csr_matrix(A)
  N, E = A.shape
  node_s, edge_s = np.full(N, num_samples), np.full(E, num_samples)
  blocks = []
  for side, s, phase, l, r in ((0, node_s, "NN", "left_node", "right_node"),
                               (1, edge_s, "EE", "left_edge", "right_edge")):
    a, b = _pairs(A, side, 2, s, seed, PHASE[phase], False)
    blocks.append(_block(len(a), k, **{l: a, r: b}))
  blocks.append(_node_edge(A, k, node_s, edge_s, 3, seed, ("NE", "EN", "NEIGHBORS"), False, False))
  return _concat(blocks)
