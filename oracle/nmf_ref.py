"""Numpy restatements of the non-negative factorization of csrc/hge_nmf.cu (scikit-learn's
coordinate-descent NMF: _fit_coordinate_descent, _update_cdnmf_fast; Frobenius loss, no
regularization, no shuffling) of the 0/1 incidence A [N, E] ~ W [N, k] H [k, E].

- `fit32`: the fp32 operation order of the device, bit for bit (tests/test_nmf_gpu.py compares the
  kernels with it):
    the seeded start (`start`): scale * ((w >> 8) 2^-24), Philox of oracle/device_sampler_ref.py;
    the products P = A Ht, A^T W: each row adds its neighbours' rows in ascending order, one fp32
    add each, from +0;
    the Gram matrices: one fma chain per entry over each chunk of 4096 consecutive rows, from +0,
    then the chunk partials added in ascending chunk order;
    the coordinate descent: per row and coordinate t, grad = fma chain over r = 0..k-1 of
    G[t,r] * Y[i,r] from -P[i,t]; an IEEE division, a subtraction and max(., 0) for the update;
    the violation: per row an f64 sum over t in order, a halving tree over the 64 rows of a block,
    the block sums in ascending order per half, then (W half) + (H half); the stop rule.
  Read from `cuobjdump -sass` of the sm_100a build: k_nmf_cd computes its chain as written with
  FFMA (explicit __fmaf_rn), the division is the IEEE div.rn.f32 subroutine, k_nmf_gram is FFMA
  (explicit __fmaf_rn), k_nmf_spmm is FADD only.  No other contraction exists to emulate.
- `fit64`: the same algorithm in float64 in scikit-learn's own order (np.dot Gram, scipy products,
  t-major / row-minor violation sum), which tests/test_nmf_host.py pins to scikit-learn.

Test infrastructure only."""
import numpy as np
import scipy.sparse as sps

from oracle.device_sampler_ref import philox4x32_10
from oracle.sweep_ref import fma32

F32 = np.float32
PHASE_W = 20
PHASE_H = 21
GRAM_CHUNK = 4096
CD_ROWS = 64


# ---- seeded start ------------------------------------------------------------------------------

def table(rows, k, seed, phase, scale):
  """[rows, k] float32: element (r, c) = scale * (fp32(w >> 8) * 2^-24), w = word c of row r's
  stream (counter {c // 4, r lo, r hi, phase}, word c % 4), each operation rounded on its own."""
  seed = int(seed) & 0xFFFFFFFFFFFFFFFF
  key = (np.uint64(seed & 0xFFFFFFFF), np.uint64(seed >> 32))
  r = np.arange(rows, dtype=np.uint64)
  out = np.empty((rows, k), dtype=F32)
  for b in range((k + 3) // 4):
    words = philox4x32_10((np.uint64(b), r & np.uint64(0xFFFFFFFF), r >> np.uint64(32), np.uint64(phase)), key)
    for j in range(4):
      c = 4 * b + j
      if c < k:
        u = (words[j] >> np.uint64(8)).astype(F32) * F32(2.0 ** -24)
        out[:, c] = F32(scale) * u
  return out


def start(num_nodes, num_edges, k, seed, scale):
  """(W [N, k], Ht [E, k]) of hge_nmf_init."""
  return table(num_nodes, k, seed, PHASE_W, scale), table(num_edges, k, seed, PHASE_H, scale)


# ---- fp32 device order ---------------------------------------------------------------------------

def spmm32(ptr, idx, Y):
  """P[i] = (((0 + Y[n_0]) + Y[n_1]) + ...) over row i's neighbours in stored (ascending) order."""
  ptr = np.asarray(ptr, np.int64)
  idx = np.asarray(idx, np.int64)
  rows = len(ptr) - 1
  P = np.zeros((rows, Y.shape[1]), dtype=F32)
  deg = np.diff(ptr)
  order = np.argsort(-deg, kind="stable")
  sdeg = deg[order]
  for s in range(int(deg.max()) if rows else 0):
    live = order[:np.searchsorted(-sdeg, -s, side="left")]   # rows with deg > s
    P[live] += Y[idx[ptr[live] + s]]
  return P


def gram32(Y):
  """G = Y^T Y: per chunk of GRAM_CHUNK rows an fma chain from +0 in row order, then the chunk
  partials summed in ascending order."""
  rows, k = Y.shape
  chunks = max(1, -(-rows // GRAM_CHUNK))
  part = np.zeros((chunks, k, k), dtype=F32)
  for j in range(min(rows, GRAM_CHUNK)):
    sel = np.arange(j, rows, GRAM_CHUNK)
    y = Y[sel]
    part[:len(sel)] = fma32(y[:, :, None], y[:, None, :], part[:len(sel)])
  G = part[0].copy()
  for c in range(1, chunks):
    G = G + part[c]
  return G


def _block_sum(v):
  """Per-row f64 sums -> fixed halving tree per block of CD_ROWS rows -> ascending sum of blocks."""
  if len(v) == 0:
    return 0.0
  blocks = -(-len(v) // CD_ROWS)
  s = np.zeros(blocks * CD_ROWS, dtype=np.float64)
  s[:len(v)] = v
  s = s.reshape(blocks, CD_ROWS)
  h = CD_ROWS // 2
  while h >= 1:
    s[:, :h] = s[:, :h] + s[:, h:2 * h]
    h //= 2
  return float(np.add.accumulate(np.concatenate([[0.0], s[:, 0]]))[-1])


def cd32(Y, G, P):
  """One coordinate-descent pass over every row of Y (in place); returns the half's violation."""
  rows, k = Y.shape
  viol = np.zeros(rows, dtype=np.float64)
  for t in range(k):
    grad = -P[:, t]
    for r in range(k):
      grad = fma32(G[t, r], Y[:, r], grad)
    yt = Y[:, t].copy()
    pg = np.where(yt == 0, np.minimum(F32(0), grad), grad)
    viol = viol + np.abs(pg.astype(np.float64))
    hess = G[t, t]
    if hess != 0:
      x = yt - grad / hess
      Y[:, t] = np.where(x > 0, x, F32(0))
  return _block_sum(viol)


def fit32(n2e_ptr, n2e_idx, e2n_ptr, e2n_idx, W0, Ht0, max_iter=200, tol=1e-4):
  """(W [N, k], Ht [E, k], n_iter, violations [n_iter]) of hge_nmf_fit, bit for bit."""
  W = np.array(W0, dtype=F32)
  Ht = np.array(Ht0, dtype=F32)
  viols = []
  viol0 = 0.0
  it = 0
  while it < max_iter:
    it += 1
    vw = cd32(W, gram32(Ht), spmm32(n2e_ptr, n2e_idx, Ht))
    vh = cd32(Ht, gram32(W), spmm32(e2n_ptr, e2n_idx, W))
    v = vw + vh
    viols.append(v)
    if it == 1:
      viol0 = v
    if viol0 == 0 or v / viol0 <= tol:
      break
  return W, Ht, it, np.asarray(viols)


# ---- float64, scikit-learn's order -------------------------------------------------------------------

def _cd64(X, W, Ht):
  HHt = np.dot(Ht.T, Ht)
  XHt = X @ Ht
  violation = 0.0
  for t in range(W.shape[1]):
    grad = -XHt[:, t]
    for r in range(W.shape[1]):
      grad = grad + HHt[t, r] * W[:, r]
    pg = np.where(W[:, t] == 0, np.minimum(0.0, grad), grad)
    violation = float(np.add.accumulate(np.concatenate([[violation], np.abs(pg)]))[-1])
    hess = HHt[t, t]
    if hess != 0:
      W[:, t] = np.maximum(W[:, t] - grad / hess, 0.0)
  return violation


def fit64(A, W0, H0, max_iter=200, tol=1e-4):
  """(W [N, k], H [k, E], n_iter, violations) of scikit-learn's coordinate descent in float64 from
  the start (W0, H0)."""
  X = sps.csr_matrix(A, dtype=np.float64)
  W = np.array(W0, dtype=np.float64, order="C")
  Ht = np.ascontiguousarray(np.asarray(H0, dtype=np.float64).T)
  viols = []
  viol0 = 0.0
  it = 0
  for it in range(1, max_iter + 1):
    v = _cd64(X, W, Ht)
    v += _cd64(X.T, Ht, W)
    viols.append(v)
    if it == 1:
      viol0 = v
    if viol0 == 0 or v / viol0 <= tol:
      break
  return W, np.ascontiguousarray(Ht.T), it, np.asarray(viols)
