"""Numpy restatement of the node-edge link-prediction classifier (csrc/hge_lp_node_edge.cu): the
training set (positives in CSR order, negatives by 64-bit masked rejection from the Philox streams of
phase HGE_PHASE_LP_NODE_EDGE_NEG), the initial weights (phase HGE_PHASE_LP_NODE_EDGE_INIT) and the
epoch orders (phase HGE_PHASE_LP_NODE_EDGE_SHUFFLE), all bit for bit, and a float64 trainer and
predictor of the same model:

  x = [xn[n], xe[e]],  h = relu(x W1 + b1),  p = sigmoid(h . w2 + b2),
  loss = max(z, 0) - z y + log1p(exp(-|z|)) of the logit z, batch mean, Adagrad on every parameter.

Test infrastructure only.
"""
import numpy as np

from oracle.device_sampler_ref import MASK, Streams, philox4x32_10
from oracle.seeded_training_ref import _key

PHASE = dict(NEG=17, SHUFFLE=18, INIT=19)


def rejection_mask(S):
  """smallest 2^k - 1 >= S - 1"""
  mask = 0
  while mask < S - 1:
    mask = (mask << 1) | 1
  return mask


def draw_ranks(seed, count, S):
  """r_i uniform on [0, S) for items 0 .. count - 1: r = ((w0 << 32) | w1) & mask, redrawn while
  r >= S, words from item i's NEG stream"""
  mask = np.uint64(rejection_mask(int(S)))
  st = Streams(seed, PHASE["NEG"], np.arange(int(count)))
  r = np.zeros(int(count), dtype=np.uint64)
  todo = np.arange(int(count))
  while len(todo):
    w0 = st.next(todo)
    w1 = st.next(todo)
    r[todo] = ((w0 << np.uint64(32)) | w1) & mask
    todo = todo[r[todo] >= np.uint64(S)]
  return r.astype(np.int64)


def rank_to_pair(indptr, indices, num_edges, r):
  """(node, edge) of non-incidence ranks r: node n with C[n] <= r < C[n + 1] (C the exclusive sum
  of E - deg), edge the (r - C[n])-th edge id not in n's row"""
  indptr = np.asarray(indptr, dtype=np.int64)
  indices = np.asarray(indices, dtype=np.int64)
  N, E = len(indptr) - 1, int(num_edges)
  deg = np.diff(indptr)
  C = np.concatenate([[0], np.cumsum(E - deg)])
  r = np.asarray(r, dtype=np.int64)
  n = np.searchsorted(C, r, side="right") - 1
  q = r - C[n]
  # within a row mem[c] - c is non-decreasing: key row-major, so one global search finds the first
  # c of row n with mem[c] - c > q
  row = np.repeat(np.arange(N, dtype=np.int64), deg)
  key = row * (E + 1) + (indices - (np.arange(len(indices)) - indptr[row]))
  c = np.searchsorted(key, n * (E + 1) + q, side="right") - indptr[n]
  return n, q + c


def training_set(indptr, indices, num_edges, seed):
  """(nodes, edges, labels) of the 2 nnz samples"""
  indptr = np.asarray(indptr, dtype=np.int64)
  nnz = int(indptr[-1])
  N = len(indptr) - 1
  S = N * int(num_edges) - nnz
  assert nnz > 0 and S > 0
  pos_n = np.repeat(np.arange(N, dtype=np.int64), np.diff(indptr))
  neg_n, neg_e = rank_to_pair(indptr, indices, num_edges, draw_ranks(seed, nnz, S))
  nodes = np.concatenate([pos_n, neg_n])
  edges = np.concatenate([np.asarray(indices, dtype=np.int64), neg_e])
  return nodes, edges, np.r_[np.ones(nnz), np.zeros(nnz)]


def shuffle_order(seed, epoch, n):
  """hge_shuffle_order with the SHUFFLE phase of this classifier"""
  items = np.arange(int(n), dtype=np.uint64)
  w = philox4x32_10((np.uint64(epoch // 2), items & MASK, items >> np.uint64(32), np.uint64(PHASE["SHUFFLE"])),
                    _key(seed))
  j = 2 * (int(epoch) % 2)
  keys = (w[j] << np.uint64(32)) | w[j + 1]
  return np.argsort(keys, kind="stable").astype(np.int64)


def init_weights(seed, d, hidden):
  """(W1 [2d, hidden], b1, w2 [hidden], b2) fp32: glorot_uniform kernels from the INIT streams (row i
  of W1 = item i, w2 = item 2d, word j = column j), zero biases"""
  rows = np.arange(2 * int(d) + 1, dtype=np.uint64)
  cols = []
  for b in range((int(hidden) + 3) // 4):
    cols += philox4x32_10((np.uint64(b), rows & MASK, rows >> np.uint64(32), np.uint64(PHASE["INIT"])), _key(seed))
  w = np.stack(cols[:int(hidden)], axis=1)
  u = (w >> np.uint64(8)).astype(np.float32) * np.float32(2.0**-24)
  L = np.full((len(rows), 1), np.float32(np.sqrt(6.0 / (2 * d + hidden))), dtype=np.float32)
  L[-1] = np.float32(np.sqrt(6.0 / (hidden + 1)))
  vals = -L + (np.float32(2) * L) * u
  return vals[:-1], np.zeros(int(hidden), np.float32), vals[-1], np.zeros(1, np.float32)


def forward(W1, b1, w2, b2, x):
  z1 = x @ W1 + b1
  h = np.maximum(z1, 0.0)
  return z1, h, h @ w2 + b2[0]


def sample_loss(z, y):
  return np.maximum(z, 0.0) - z * y + np.log1p(np.exp(-np.abs(z)))


def train(xn, xe, nodes, edges, labels, weights, orders, batch, lr=0.01, eps=1e-7):
  """float64 trainer: weights (W1, b1, w2, b2) from `weights`, epoch e visits the samples in
  orders[e] in batches of `batch`.  Returns ((W1, b1, w2, b2), per-epoch mean sample losses)."""
  W1, b1, w2, b2 = (np.asarray(w, dtype=np.float64).copy() for w in weights)
  params = [W1, b1, w2, b2]
  acc = [np.zeros_like(p) for p in params]
  xn, xe = np.asarray(xn, dtype=np.float64), np.asarray(xe, dtype=np.float64)
  losses = []
  for order in orders:
    total = 0.0
    for first in range(0, len(order), batch):
      s = np.asarray(order[first:first + batch])
      x = np.concatenate([xn[nodes[s]], xe[edges[s]]], axis=1)
      y = labels[s]
      z1, h, z = forward(W1, b1, w2, b2, x)
      total += sample_loss(z, y).sum()
      p = 1.0 / (1.0 + np.exp(-z))
      dz = (p - y) / len(s)
      dh = np.outer(dz, w2) * (z1 > 0)
      grads = [x.T @ dh, dh.sum(axis=0), h.T @ dz, np.array([dz.sum()])]
      for prm, a, g in zip(params, acc, grads):
        a += g * g
        prm -= lr * g / (np.sqrt(a) + eps)
    losses.append(total / len(order))
  return (W1, b1, w2, b2), np.asarray(losses)


def predict(weights, xn, xe, nodes, edges):
  """float64 p of the links (nodes[l], edges[l])"""
  W1, b1, w2, b2 = (np.asarray(w, dtype=np.float64) for w in weights)
  x = np.concatenate([np.asarray(xn, np.float64)[nodes], np.asarray(xe, np.float64)[edges]], axis=1)
  return 1.0 / (1.0 + np.exp(-forward(W1, b1, w2, b2, x)[2]))


def planted_communities(communities=6, nodes_per=12, edges_per=6, p_in=0.7, d=8, noise=0.25, seed=0):
  """A graph whose incidences all lie inside communities, vectors near one-hot(community) (d >=
  communities), 15 % of the incidences held out: (A train CSR, xn, xe, held-out positives,
  held-out negatives (cross-community pairs, as many))."""
  import scipy.sparse as sps
  rng = np.random.RandomState(seed)
  N, E = communities * nodes_per, communities * edges_per
  cn, ce = np.arange(N) // nodes_per, np.arange(E) // edges_per
  inc = [(n, e) for n in range(N) for e in range(E) if cn[n] == ce[e] and rng.rand() < p_in]
  inc = np.asarray(inc, dtype=np.int64)
  held = rng.rand(len(inc)) < 0.15
  A = sps.csr_matrix((np.ones(int((~held).sum()), np.int8), (inc[~held, 0], inc[~held, 1])), shape=(N, E))
  A.sort_indices()
  pos = inc[held]
  neg = []
  while len(neg) < len(pos):
    n, e = rng.randint(N), rng.randint(E)
    if cn[n] != ce[e]:
      neg.append((n, e))
  xn = (np.eye(d)[cn] + noise * rng.randn(N, d)).astype(np.float32)
  xe = (np.eye(d)[ce] + noise * rng.randn(E, d)).astype(np.float32)
  return A, xn, xe, pos, np.asarray(neg, dtype=np.int64)
