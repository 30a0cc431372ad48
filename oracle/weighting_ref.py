"""Numpy restatements of the results of the distance, span and HOBE-probability kernels of
csrc/hge_weighting.cu (k_incidence_l2, k_pair_l2, k_row_span, k_same_type_prob,
k_diff_type_prob).

- Spans and probabilities are selections: a max / min over values the kernel computes with single
  IEEE operations (build.NVCC_FLAGS has no fast-math flag), so `row_span_f32`, `same_type_prob`
  and `diff_type_prob` equal the kernels bit for bit on any fp32 input (up to the sign of a zero).
- Distances are sums whose order is the kernel's own (lanes, slabs, FMA); `incidence_l2_f64` and
  `pair_l2_f64` give the float64 value they approximate.

Rows are int64 CSR pointers `ptr` with sorted int32 column ids `idx`, weights `w` in storage
order.  Test infrastructure only."""
import numpy as np

_CHUNK = 1 << 24      # elements of one [incidences, R] difference block


def _rows_of(ptr):
  ptr = np.asarray(ptr, dtype=np.int64)
  return np.repeat(np.arange(len(ptr) - 1, dtype=np.int64), np.diff(ptr))


def row_span_f32(ptr, idx, x_self, x_other):
  """k_row_span: per row r, hi - lo in fp32 with lo = min(0, x_other[c][k] - x_self[r][k]) and
  hi = max(0, ...) over the row's columns c and the components k < R (each difference one fp32
  subtraction).  An empty row gives 0."""
  x_self = np.asarray(x_self, dtype=np.float32)
  x_other = np.asarray(x_other, dtype=np.float32)
  idx = np.asarray(idx, dtype=np.int64)
  rows = _rows_of(ptr)
  lo = np.zeros(len(ptr) - 1, dtype=np.float32)
  hi = np.zeros(len(ptr) - 1, dtype=np.float32)
  step = max(1, _CHUNK // max(1, x_self.shape[1]))
  for s in range(0, len(idx), step):
    r, c = rows[s:s + step], idx[s:s + step]
    d = x_other[c] - x_self[r]
    np.minimum.at(lo, r, d.min(axis=1))
    np.maximum.at(hi, r, d.max(axis=1))
  return hi - lo


def same_type_prob(ptr, idx, w, pi, pj):
  """k_same_type_prob: per pair (i, j), max(0, max over columns k shared by rows i and j of
  min(w(i, k), w(j, k))) in fp32.  Vectorised: every column of the shorter row is looked up in
  the longer row by searchsorted on row * cols + col keys."""
  ptr = np.asarray(ptr, dtype=np.int64)
  idx = np.asarray(idx, dtype=np.int64)
  w = np.asarray(w, dtype=np.float32)
  pi = np.asarray(pi, dtype=np.int64)
  pj = np.asarray(pj, dtype=np.int64)
  out = np.zeros(len(pi), dtype=np.float32)
  if len(pi) == 0 or len(idx) == 0:
    return out
  cols = int(idx.max()) + 1
  keys = _rows_of(ptr) * cols + idx              # ascending: rows in order, sorted columns
  deg = np.diff(ptr)
  short = np.where(deg[pi] <= deg[pj], pi, pj)
  long_ = np.where(deg[pi] <= deg[pj], pj, pi)
  n = deg[short]
  step = 1 << 22
  first = 0
  while first < len(pi):                          # pairs in batches of about `step` lookups
    csum = np.cumsum(n[first:])
    last = first + max(1, int(np.searchsorted(csum, step, side="right")))
    p = np.repeat(np.arange(first, last), n[first:last])
    t = np.arange(len(p)) - np.repeat(np.cumsum(n[first:last]) - n[first:last], n[first:last])
    a = ptr[short[p]] + t                         # incidence of the shorter row
    key = long_[p] * cols + idx[a]
    b = np.minimum(np.searchsorted(keys, key), len(keys) - 1)
    hit = keys[b] == key
    np.maximum.at(out, p[hit], np.minimum(w[a[hit]], w[b[hit]]))
    first = last
  return out


def diff_type_prob(n2e_ptr, n2e_idx, e2n_ptr, e2n_idx, w_e2n, pn, pe):
  """k_diff_type_prob: per pair (node n, edge e), max(0, max over the node's edges e' of the
  edge-edge same_type_prob(e, e')) on the edge -> node rows."""
  n2e_ptr = np.asarray(n2e_ptr, dtype=np.int64)
  n2e_idx = np.asarray(n2e_idx, dtype=np.int64)
  pn = np.asarray(pn, dtype=np.int64)
  pe = np.asarray(pe, dtype=np.int64)
  deg = np.diff(n2e_ptr)[pn]
  p = np.repeat(np.arange(len(pn)), deg)
  t = np.arange(len(p)) - np.repeat(np.cumsum(deg) - deg, deg)
  other = n2e_idx[n2e_ptr[pn[p]] + t]
  out = np.zeros(len(pn), dtype=np.float32)
  np.maximum.at(out, p, same_type_prob(e2n_ptr, e2n_idx, w_e2n, pe[p], other))
  return out


def pair_sq_f64(xa, xb, ia, ib):
  """||xa[ia[p]] - xb[ib[p]]||_2^2 in float64.  Exact when every component is a multiple of 2^-4
  in [0, 1): each square is then a multiple of 2^-8 below 1 and, for R <= 1024, every partial sum
  has at most 18 significant bits, so fp32 holds it exactly in any order of summation."""
  xa = np.asarray(xa, dtype=np.float64)
  xb = np.asarray(xb, dtype=np.float64)
  ia = np.asarray(ia, dtype=np.int64)
  ib = np.asarray(ib, dtype=np.int64)
  out = np.empty(len(ia), dtype=np.float64)
  step = max(1, _CHUNK // max(1, xa.shape[1]))
  for s in range(0, len(ia), step):
    d = xa[ia[s:s + step]] - xb[ib[s:s + step]]
    out[s:s + step] = np.einsum("ij,ij->i", d, d)
  return out


def pair_l2_f64(xa, xb, ia, ib):
  """||xa[ia[p]] - xb[ib[p]]||_2 in float64 (k_pair_l2)."""
  return np.sqrt(pair_sq_f64(xa, xb, ia, ib))


def incidence_l2_f64(ptr, idx, x_self, x_other):
  """||x_self[r] - x_other[c]||_2 in float64 for every stored incidence (r, c), in storage order
  (k_incidence_l2)."""
  return pair_l2_f64(x_self, x_other, _rows_of(ptr), idx)


def hobe_weight_f64(d, R):
  """The HOBE incidence weight (sqrt(R) - d) / sqrt(R) in float64."""
  m = np.sqrt(np.float64(R))
  return (m - np.asarray(d, dtype=np.float64)) / m
