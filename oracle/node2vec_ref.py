"""Numpy restatement of node2vec on the node-edge bipartite graph (csrc/hge_n2v.cu, DESIGN section
9.12): the walks, windows, pairs, noise table, negatives, epoch orders and initial table bit for bit;
the mini-batch skip-gram trainer in fp32 in the device's operation order (the tables bit for bit up
to the `exp` / `log` hooks, which stand for __expf / __logf); and the same trainer in float64.

Vertices: compressed node r is vertex r, compressed edge c is vertex N + c.

Test infrastructure only.
"""
import numpy as np
import scipy.sparse as sps

from oracle.device_sampler_ref import MASK, Streams, philox4x32_10
from oracle.hg2v_train_ref import warp_sum
from oracle.seeded_training_ref import _key
from oracle.sweep_ref import fma32

PHASE = dict(WALK=23, WINDOW=24, SHUFFLE=25, NEG=26, INIT=27)
F32 = np.float32
_XOR = [np.arange(32) ^ off for off in (16, 8, 4, 2, 1)]


def exp32(x):
  return np.exp(np.asarray(x, F32)).astype(F32)


def log32(x):
  return np.log(np.asarray(x, F32)).astype(F32)


def bipartite(A):
  """(vptr [V + 1], vidx): the sorted neighbour rows of the V = N + E vertices of incidence A."""
  A = sps.csr_matrix(A, dtype=np.float32)
  A.sum_duplicates()
  A.sort_indices()
  N, E = A.shape
  B = A.T.tocsr()
  B.sort_indices()
  vptr = np.concatenate([A.indptr, A.indptr[-1] + B.indptr[1:]]).astype(np.int64)
  vidx = np.concatenate([A.indices.astype(np.int64) + N, B.indices.astype(np.int64)])
  return vptr, vidx


def walks(A, num_walks, walk_length, p, q, seed):
  """(walks [num_walks V, L] int32, counts [V] int64) of hge_n2v_walks."""
  vptr, vidx = bipartite(A)
  V = len(vptr) - 1
  deg = np.diff(vptr)
  W, L = int(num_walks) * V, int(walk_length)
  row_of = np.repeat(np.arange(V, dtype=np.int64), deg)
  comp = row_of * (V + 1) + vidx                     # sorted: row-major, ascending inside a row
  out = np.full((W, L), -1, dtype=np.int64)
  cur = np.arange(W, dtype=np.int64) % V
  prev = np.full(W, -1, dtype=np.int64)
  out[:, 0] = cur
  st = Streams(seed, PHASE["WALK"], np.arange(W))
  live = np.nonzero(deg[cur] > 0)[0]
  for i in range(1, L):
    v, t, d = cur[live], prev[live], deg[cur[live]]
    x = np.empty(len(live), dtype=np.int64)
    first = t < 0
    if first.any():
      sel = live[first]
      x[first] = vidx[vptr[v[first]] + st.below(sel, d[first])]
    one = ~first & (d == 1)
    x[one] = t[one]
    many = np.nonzero(~first & (d >= 2))[0]
    if len(many):
      u = st.next(live[many]).astype(np.float64) * 2.0**-32
      c = q + (d[many] - 1).astype(np.float64) * p
      ret = u * c < q
      x[many[ret]] = t[many[ret]]
      go = many[~ret]
      if len(go):
        j = st.below(live[go], d[go] - 1)
        pos = np.searchsorted(comp, v[go] * (V + 1) + t[go], side="left") - vptr[v[go]]
        x[go] = vidx[vptr[v[go]] + np.where(j < pos, j, j + 1)]
    out[live, i] = x
    prev[live] = v
    cur[live] = x
  counts = np.bincount(out[out >= 0], minlength=V).astype(np.int64)
  return out.astype(np.int32), counts


def pairs(walks_, window, seed):
  """int32 pairs [P, 2] of hge_n2v_pairs: token g = w L + i draws b = 1 + below(window) (item g of
  WINDOW) and pairs with tokens j != i, |i - j| <= b, of its walk; (g, j) ascending."""
  w = np.asarray(walks_)
  W, L = w.shape
  length = np.full(W, L)
  if L > 1:
    length[w[:, 1] < 0] = 1
  g = np.nonzero(w.reshape(-1) >= 0)[0]
  b = 1 + Streams(seed, PHASE["WINDOW"], g).below(np.arange(len(g)), int(window))
  i = g % L
  n = length[g // L]
  lo, hi = np.maximum(0, i - b), np.minimum(n - 1, i + b)
  off = np.arange(-int(window), int(window) + 1)
  j = i[:, None] + off[None, :]
  keep = (j >= lo[:, None]) & (j <= hi[:, None]) & (off[None, :] != 0)
  flat = w.reshape(-1)
  center = np.broadcast_to(flat[g][:, None], j.shape)[keep]
  context = flat[(g - i)[:, None] + j.clip(0, L - 1)][keep]
  return np.stack([center, context], axis=1).astype(np.int32)


def noise_table(counts):
  """Cumulative int64 noise table [V + 1]: q_v = floor((c_v^0.75 / max c^0.75) 2^32) in f64."""
  w = np.power(np.asarray(counts, dtype=np.float64), 0.75)
  q = np.floor((w / w.max()) * 2.0**32).astype(np.int64)
  return np.concatenate([[0], np.cumsum(q)]).astype(np.int64)


def negatives(cum, num_pairs, negative, seed, epoch, ids=None):
  """int32 [len(ids), negative]: pair i's negatives in `epoch` (item epoch P + i of NEG; per sample
  r = ((w0 << 32) | w1) & mask redrawn while r >= total, then v with cum[v] <= r < cum[v + 1])."""
  cum = np.asarray(cum, dtype=np.int64)
  total = int(cum[-1])
  mask = 0
  while mask < total - 1:
    mask = (mask << 1) | 1
  ids = np.arange(int(num_pairs)) if ids is None else np.asarray(ids, dtype=np.int64)
  st = Streams(seed, PHASE["NEG"], int(epoch) * int(num_pairs) + ids)
  out = np.zeros((len(ids), int(negative)), dtype=np.int64)
  for k in range(int(negative)):
    r = np.zeros(len(ids), dtype=np.uint64)
    todo = np.arange(len(ids))
    while len(todo):
      w0 = st.next(todo)
      w1 = st.next(todo)
      r[todo] = ((w0 << np.uint64(32)) | w1) & np.uint64(mask)
      todo = todo[r[todo] >= np.uint64(total)]
    out[:, k] = np.searchsorted(cum, r.astype(np.int64), side="right") - 1
  return out.astype(np.int32)


def shuffle_order(seed, epoch, n):
  """hge_shuffle_order in phase N2V_SHUFFLE"""
  items = np.arange(int(n), dtype=np.uint64)
  w = philox4x32_10((np.uint64(epoch // 2), items & MASK, items >> np.uint64(32), np.uint64(PHASE["SHUFFLE"])),
                    _key(seed))
  j = 2 * (int(epoch) % 2)
  keys = (w[j] << np.uint64(32)) | w[j + 1]
  return np.argsort(keys, kind="stable").astype(np.int64)


def init_tables(seed, V, dim):
  """hge_n2v_init: (in, out) fp32 [V, dim]; in = -0.5/dim + (1/dim) ((w >> 8) 2^-24), out = 0."""
  r = np.arange(int(V), dtype=np.uint64)
  cols = []
  for b in range((int(dim) + 3) // 4):
    cols += philox4x32_10((np.uint64(b), r & MASK, r >> np.uint64(32), np.uint64(PHASE["INIT"])), _key(seed))
  w = np.stack(cols[:int(dim)], axis=1)
  u = (w >> np.uint64(8)).astype(F32) * F32(2.0**-24)
  off, scale = F32(-0.5) / F32(dim), F32(1) / F32(dim)
  return (off + scale * u).astype(F32), np.zeros((int(V), int(dim)), F32)


def lanes_per_dim(dim):
  dpl = (int(dim) + 31) // 32
  return 1 if dpl <= 1 else 2 if dpl <= 2 else 4 if dpl <= 4 else 8


def epoch_plan(pairs_, cum, negative, seed, epoch):
  """(centers [P], targets [P, 1 + negative]) in the epoch's order; target -1 = a skipped negative."""
  P = len(pairs_)
  order = shuffle_order(seed, epoch, P)
  pr = np.asarray(pairs_, dtype=np.int64)[order]
  neg = negatives(cum, P, negative, seed, epoch, ids=order).astype(np.int64)
  neg[neg == pr[:, 1:2]] = -1
  return pr[:, 0], np.concatenate([pr[:, 1:2], neg], axis=1)


def learning_rate(alpha, min_alpha, t, T):
  return alpha - (alpha - min_alpha) * (t / T)


def _segment_ranks(keys):
  """stable order of keys, and for it each entry's segment id and rank inside its segment"""
  o = np.argsort(keys, kind="stable")
  k = keys[o]
  head = np.ones(len(k), bool)
  head[1:] = k[1:] != k[:-1]
  seg = np.cumsum(head) - 1
  start = np.nonzero(head)[0]
  rank = np.arange(len(k)) - start[seg]
  return o, seg, rank, k[head]


def _ordered_sums(rows, g, vecs, dim):
  """per distinct row (ascending): fp32 fma chain from +0 of g_i vecs_i in the given entry order"""
  o, seg, rank, uniq = _segment_ranks(rows)
  acc = np.zeros((len(uniq), dim), F32)
  g, vecs = g[o], vecs[o]
  for r in range(int(rank.max()) + 1 if len(rank) else 0):
    s = rank == r
    acc[seg[s]] = fma32(g[s][:, None], vecs[s], acc[seg[s]])
  return uniq, acc


def _batch_loss(l):
  """lane l sums l[lane::32] in f64 in order, then the xor butterfly"""
  lanes = np.zeros(32)
  for i, v in enumerate(l):
    lanes[i % 32] = lanes[i % 32] + v
  for x in _XOR:
    lanes = lanes + lanes[x]
  return lanes[0]


def train32(tin, tout, pairs_, cum, negative, seed, epoch, epochs, batch_pairs, alpha=0.025, min_alpha=1e-4,
            exp=exp32, log=log32):
  """One epoch of hge_n2v_train_epoch in place on fp32 tin / tout; returns the epoch loss."""
  P, dim = len(pairs_), tin.shape[1]
  if P == 0:
    return 0.0
  B = min(int(batch_pairs), P)
  nb_total = (P + B - 1) // B
  T = float(epochs) * float(nb_total)
  dpl = lanes_per_dim(dim)
  cen, tgt = epoch_plan(pairs_, cum, negative, seed, epoch)
  S = tgt.shape[1]
  total = 0.0
  for b in range(nb_total):
    c, x = cen[b * B:(b + 1) * B], tgt[b * B:(b + 1) * B]
    nb = len(c)
    lr = F32(learning_rate(alpha, min_alpha, float(epoch * nb_total + b), T))
    a = np.zeros((nb, dpl * 32), F32)
    a[:, :dim] = tin[c]
    a = a.reshape(nb, dpl, 32)
    G = np.zeros((nb, S), F32)
    loss = np.zeros(nb)
    for s in range(S):
      ok = x[:, s] >= 0
      bv = np.zeros((nb, dpl * 32), F32)
      bv[ok, :dim] = tout[x[ok, s]]
      bv = bv.reshape(nb, dpl, 32)
      z = np.zeros((nb, 32), F32)
      for j in range(dpl):
        z = fma32(a[:, j], bv[:, j], z)
      z = warp_sum(z)
      sg = F32(1) / (F32(1) + exp(-z))
      sy = sg if s == 0 else F32(1) / (F32(1) + exp(z))
      label = F32(1) if s == 0 else F32(0)
      G[ok, s] = (lr * (label - sg))[ok]
      loss[ok] = loss[ok] + (-log(sy)).astype(np.float64)[ok]
    total = total + _batch_loss(loss)
    p_idx, s_idx = np.nonzero(x >= 0)                  # (pair, slot) ascending
    g = G[p_idx, s_idx]
    rin, din = _ordered_sums(c[p_idx], g, tout[x[p_idx, s_idx]], dim)
    rout, dout = _ordered_sums(x[p_idx, s_idx], g, tin[c[p_idx]], dim)
    tin[rin] = tin[rin] + din
    tout[rout] = tout[rout] + dout
  return total


def train64(tin, tout, pairs_, cum, negative, seed, epoch, epochs, batch_pairs, alpha=0.025, min_alpha=1e-4):
  """The same epoch in float64 (tin / tout float64, in place); returns the epoch loss."""
  P = len(pairs_)
  if P == 0:
    return 0.0
  B = min(int(batch_pairs), P)
  nb_total = (P + B - 1) // B
  T = float(epochs) * float(nb_total)
  cen, tgt = epoch_plan(pairs_, cum, negative, seed, epoch)
  total = 0.0
  for b in range(nb_total):
    c, x = cen[b * B:(b + 1) * B], tgt[b * B:(b + 1) * B]
    lr = learning_rate(alpha, min_alpha, float(epoch * nb_total + b), T)
    p_idx, s_idx = np.nonzero(x >= 0)
    rows_in, rows_out = c[p_idx], x[p_idx, s_idx]
    z = np.einsum("ij,ij->i", tin[rows_in], tout[rows_out])
    label = (s_idx == 0).astype(np.float64)
    sg = 1.0 / (1.0 + np.exp(-z))
    total += float(np.sum(np.logaddexp(0.0, -np.where(s_idx == 0, z, -z))))
    g = lr * (label - sg)
    din = np.zeros_like(tin)
    dout = np.zeros_like(tout)
    np.add.at(din, rows_in, g[:, None] * tout[rows_out])
    np.add.at(dout, rows_out, g[:, None] * tin[rows_in])
    tin += din
    tout += dout
  return total


def planted_partition(communities=8, nodes_per=40, edges_per=20, edge_size=8, p_in=0.9, seed=0):
  """Seeded planted-partition hypergraph: community k owns nodes_per nodes and edges_per edges; each
  edge takes edge_size distinct members, each from its own community with probability p_in, else
  uniformly from all nodes.  Returns the N x E 0/1 CSR incidence."""
  rng = np.random.RandomState(seed)
  N, E = communities * nodes_per, communities * edges_per
  rows, cols = [], []
  for e in range(E):
    k = e // edges_per
    members = set()
    while len(members) < edge_size:
      members.add(k * nodes_per + rng.randint(nodes_per) if rng.rand() < p_in else rng.randint(N))
    rows += sorted(members)
    cols += [e] * edge_size
  return sps.csr_matrix((np.ones(len(rows), np.float32), (rows, cols)), shape=(N, E))


def held_out_auc(A, seed, fraction=0.1, negatives_per=1):
  """(training incidence, scorer): removes `fraction` of A's incidences (seeded); scorer(X) is the ROC
  AUC of node . edge scores of the held-out incidences against as many sampled non-incidences."""
  A = sps.csr_matrix(A)
  N, E = A.shape
  rng = np.random.RandomState(seed)
  coo = A.tocoo()
  held = rng.rand(coo.nnz) < fraction
  train = sps.csr_matrix((coo.data[~held], (coo.row[~held], coo.col[~held])), shape=(N, E))
  pos = np.stack([coo.row[held], coo.col[held]], 1)
  dense = A.toarray() > 0
  neg = []
  while len(neg) < negatives_per * len(pos):
    n, e = rng.randint(N), rng.randint(E)
    if not dense[n, e]:
      neg.append((n, e))
  neg = np.asarray(neg)

  def score(X):
    s = lambda pr: np.einsum("ij,ij->i", X[pr[:, 0]].astype(np.float64), X[N + pr[:, 1]].astype(np.float64))
    sp, sn = s(pos), s(neg)
    return float(np.mean(sp[:, None] > sn[None, :]) + 0.5 * np.mean(sp[:, None] == sn[None, :]))

  return train, score
