"""Numpy restatement of node2vec's walks on a weighted clique expansion (csrc/hge_n2v_clique.cu,
DESIGN section 9.13), bit for bit, reusing the Philox streams of oracle/device_sampler_ref.py; the
pairs, noise table, negatives and trainers are those of oracle/node2vec_ref.py.  Also the weighted
expansion itself, built with scipy for the host tests (it is never built by the library), and the
same- against cross-community pair AUC the quality tests use.

Side 0: vertices are the nodes; side 1: the edges.  Test infrastructure only.
"""
import numpy as np
import scipy.sparse as sps
from scipy import stats as sps_stats

from oracle import node2vec_ref as ref
from oracle.device_sampler_ref import Streams

PHASE_CLIQUE_WALK = 28


def edge_seed(seed):
  """clique_edge_seed of hypergraphembedding_b200.node2vec"""
  return (int(seed) & 0xFFFFFFFFFFFFFFFF) ^ 0x9E3779B97F4A7C15


def _pattern(A):
  A = sps.csr_matrix(A, dtype=np.float32)
  A.sum_duplicates()
  A.sort_indices()
  A.data[:] = 1
  return A


def side_rows(A, side):
  """(ptr, idx, optr, oidx): every vertex's sorted incident edges idx[ptr[v]:ptr[v + 1]] and every
  edge's sorted members oidx[optr[e]:optr[e + 1]], for side 0 (nodes) or 1 (edges)."""
  A = _pattern(A)
  B = A.T.tocsr()
  B.sort_indices()
  X, Y = (A, B) if side == 0 else (B, A)
  as64 = lambda a: np.asarray(a, dtype=np.int64)
  return as64(X.indptr), as64(X.indices), as64(Y.indptr), as64(Y.indices)


def expansion(A, side):
  """The weighted clique expansion [V, V] (int64 CSR): A A^T (side 0) or A^T A (side 1) without its
  diagonal."""
  A = sps.csr_matrix(_pattern(A), dtype=np.int64)
  M = (A @ A.T if side == 0 else A.T @ A).tolil()
  M.setdiag(0)
  M = M.tocsr()
  M.eliminate_zeros()
  M.sort_indices()
  return M


def _shares_edge(ptr, idx, vkey, M, a, b):
  """bool [n]: whether a[i] and b[i] have an incident edge in common (rows of the shorter
  searched in the longer)"""
  da, db = np.diff(ptr)[a], np.diff(ptr)[b]
  short, long_ = np.where(da <= db, a, b), np.where(da <= db, b, a)
  n_short = np.diff(ptr)[short]
  rep = np.repeat(np.arange(len(a)), n_short)
  off = np.arange(len(rep)) - np.repeat(np.cumsum(n_short) - n_short, n_short)
  keys = long_[rep] * (M + 1) + idx[ptr[short][rep] + off]
  pos = np.searchsorted(vkey, keys)
  hit = (pos < len(vkey)) & (vkey[np.minimum(pos, len(vkey) - 1)] == keys)
  return np.bincount(rep, weights=hit, minlength=len(a)) > 0


def clique_walks(A, side, num_walks, walk_length, p, q, seed, stats=None):
  """(walks [num_walks V, L] int32, counts [V] int64) of hge_n2v_clique_walks.  With a dict
  `stats`, adds "proposals" and "steps" (accepted steps after the first vertex)."""
  ptr, idx, optr, oidx = side_rows(A, side)
  V, M = len(ptr) - 1, len(optr) - 1
  deg, esize = np.diff(ptr), np.diff(optr)
  cum = np.cumsum(esize[idx] - 1)                                  # inclusive, row after row
  base = np.zeros(V, np.int64)
  base[ptr[:-1] > 0] = cum[ptr[:-1][ptr[:-1] > 0] - 1]
  S = np.zeros(V, np.int64)
  S[deg > 0] = cum[ptr[1:][deg > 0] - 1] - base[deg > 0]
  vkey = np.repeat(np.arange(V, dtype=np.int64), deg) * (M + 1) + idx     # sorted
  mkey = np.repeat(np.arange(M, dtype=np.int64), esize) * (V + 1) + oidx  # sorted
  p, q = float(p), float(q)
  pq = p * q
  m = max(q, pq, p)
  W, L = int(num_walks) * V, int(walk_length)
  out = np.full((W, L), -1, dtype=np.int64)
  cur = np.arange(W, dtype=np.int64) % V
  prev = np.full(W, -1, dtype=np.int64)
  out[:, 0] = cur
  st = Streams(seed, PHASE_CLIQUE_WALK, np.arange(W))
  live = np.nonzero(S[cur] > 0)[0]
  proposals = 0
  for i in range(1, L):
    pend = live
    while len(pend):
      proposals += len(pend)
      v, t = cur[pend], prev[pend]
      s = S[v].astype(np.uint64)
      mask = np.zeros(len(pend), np.uint64)
      grow = mask < s - np.uint64(1)
      while grow.any():
        mask[grow] = (mask[grow] << np.uint64(1)) | np.uint64(1)
        grow = mask < s - np.uint64(1)
      r = np.zeros(len(pend), np.uint64)
      todo = np.arange(len(pend))
      while len(todo):
        w0 = st.next(pend[todo])
        w1 = st.next(pend[todo])
        r[todo] = ((w0 << np.uint64(32)) | w1) & mask[todo]
        todo = todo[r[todo] >= s[todo]]
      k = np.searchsorted(cum, base[v] + r.astype(np.int64), side="right")
      e = idx[k]
      j = st.below(pend, esize[e] - 1)
      pos = np.searchsorted(mkey, e * (V + 1) + v) - optr[e]
      x = oidx[optr[e] + np.where(j < pos, j, j + 1)]
      first = t < 0
      a = np.full(len(pend), p)
      a[x == t] = q
      if pq != p:
        cand = np.nonzero(~first & (x != t))[0]
        if len(cand):
          tk = e[cand] * (V + 1) + t[cand]
          pt = np.searchsorted(mkey, tk)
          adj = (pt < len(mkey)) & (mkey[np.minimum(pt, len(mkey) - 1)] == tk)
          rest = np.nonzero(~adj)[0]
          if len(rest):
            adj[rest] = _shares_edge(ptr, idx, vkey, M, t[cand[rest]], x[cand[rest]])
          a[cand[adj]] = pq
      accept = first | ~(a < m)
      draw = np.nonzero(~accept)[0]
      if len(draw):
        u = st.next(pend[draw]).astype(np.float64) * 2.0**-32
        accept[draw] = u * m < a[draw]
      done = pend[accept]
      out[done, i] = x[accept]
      prev[done] = cur[done]
      cur[done] = x[accept]
      pend = pend[~accept]
  if stats is not None:
    stats["proposals"] = stats.get("proposals", 0) + proposals
    stats["steps"] = stats.get("steps", 0) + len(live) * (L - 1)
  counts = np.bincount(out[out >= 0], minlength=V).astype(np.int64)
  return out.astype(np.int32), counts


def embed64(A, side, dim, walk_length, num_walks, p, q, window, negative, epochs, batch_pairs, seed):
  """float64 tables of the whole pipeline (clique_walks, pairs, noise, initial table, train64):
  (in [V, dim], losses)"""
  walks, counts = clique_walks(A, side, num_walks, walk_length, p, q, seed)
  pairs = ref.pairs(walks, window, seed)
  cum = ref.noise_table(counts)
  tin, tout = (t.astype(np.float64) for t in ref.init_tables(seed, len(counts), dim))
  losses = [ref.train64(tin, tout, pairs, cum, negative, seed, e, epochs, batch_pairs) for e in range(epochs)]
  return tin, losses


def community_auc(X, labels):
  """ROC AUC of the dot products of all same-community vertex pairs against all cross-community
  ones (ties count one half)."""
  X = np.asarray(X, dtype=np.float64)
  i, j = np.triu_indices(len(X), k=1)
  score = np.einsum("ij,ij->i", X[i], X[j])
  same = np.asarray(labels)[i] == np.asarray(labels)[j]
  rank = sps_stats.rankdata(score)
  n1, n0 = int(same.sum()), int((~same).sum())
  return float((rank[same].sum() - n1 * (n1 + 1) / 2.0) / (n1 * n0))
