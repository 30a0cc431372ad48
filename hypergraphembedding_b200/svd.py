"""Truncated SVD of a hypergraph's node-edge incidence on the GPU: the SVD baseline embedder the
reference compares HOBE against (embedding.py:110-261 of the reference).

``TruncatedSVDDevice`` runs randomized subspace iteration with Rayleigh-Ritz (Halko, Martinsson and
Tropp 2011) on the 0/1 incidence A [N, E] (DESIGN section 9.11).  The products, Gram matrices and
row-times-matrix steps run in libhge_b200.so (csrc/hge_svd.cu); this module drives the loop and
does the l x l steps in float64 with numpy's ``eigh``.  The start block is seeded (Philox phase 22),
so numpy's global RNG is neither read nor advanced.
"""
import time

import numpy as np
import scipy.sparse as sps

from . import _native
from .algebraic_distance import make_incidence

MAX_K = 256
RANK_CUT = 1e-6   # 1 / sigma is 0 where sigma <= RANK_CUT * sigma_1 (numerical rank)


def block_width(k, oversamples, num_nodes, num_edges):
  """l = min(k + oversamples, min(N, E), 256): the width of the iterated block."""
  return min(int(k) + int(oversamples), int(num_nodes), int(num_edges), MAX_K)


def check_arguments(num_nodes, num_edges, k, n_iter, oversamples, tol):
  """The refusals of TruncatedSVDDevice, made before anything is computed."""
  assert 1 <= k <= min(num_nodes, num_edges) and k <= MAX_K, \
      "k = %r not in [1, min(N, E) = %d] or above %d" % (k, min(num_nodes, num_edges), MAX_K)
  assert n_iter >= 1, "n_iter = %r must be >= 1" % (n_iter,)
  assert oversamples >= 0, "oversamples = %r must be >= 0" % (oversamples,)
  assert tol >= 0, "tol = %r must be non-negative (and not NaN)" % (tol,)


def ritz_step(G):
  """The host step of one half, in float64: eigh(G) = (lambda, U~) with sigma = sqrt(lambda)
  descending; M = U~ diag(1 / sigma) rounded to float32, 1 / sigma = 0 where sigma <= RANK_CUT *
  sigma_1.  Returns (sigma [l], U~ [l, l], M [l, l] float32, kept [l] bool)."""
  lam, vec = np.linalg.eigh(G)
  lam, vec = lam[::-1], vec[:, ::-1]
  sigma = np.sqrt(np.maximum(lam, 0.0))
  kept = sigma > RANK_CUT * sigma[0]
  inv = np.zeros_like(sigma)
  inv[kept] = 1.0 / sigma[kept]
  return sigma, vec, np.ascontiguousarray((vec * inv).astype(np.float32)), kept


def truncated_svd(ctx, inc, k, n_iter=5, oversamples=10, tol=0.0, seed=0, device=True, timings=None):
  """The loop of TruncatedSVDDevice on an incidence made by make_incidence.  device: the working
  arrays are CUDA tensors (True) or numpy arrays staged by the library on every call (False); the
  results are the same bits.  Returns (U [N, k], s [k] float64, V [E, k], info) with U and V as
  [rows, k] views of the padded working arrays.  `timings` (a list) receives one dict per
  iteration: wall, product, Gram and row-product milliseconds, and the host's eigh milliseconds."""
  N, E = inc.num_nodes, inc.num_edges
  check_arguments(N, E, k, n_iter, oversamples, tol)
  l = block_width(k, oversamples, N, E)
  ld = _native.svd_ld(l)
  if device:
    import torch
    dev = torch.device("cuda", ctx.device)

    def new(rows):
      return torch.zeros((rows, ld), dtype=torch.float32, device=dev)
  else:
    def new(rows):
      return np.zeros((rows, ld), dtype=np.float32)
  omega, Z, Y, Q = new(E), new(E), new(N), new(N)
  _native.svd_start(ctx, E, l, seed, omega)
  phase = np.zeros(2) if timings is not None else None
  ritz = []
  prev = None
  it = 0
  while it < n_iter:
    it += 1
    t = _Timer(timings is not None and device)
    G = _native.svd_half(ctx, inc, 0, l, omega, Y, phase)
    t.device_phase(phase)
    _, _, M, _ = t.host(ritz_step, G)
    t.row(lambda: _native.svd_rowmat(ctx, l, Y, M, Q))
    G = _native.svd_half(ctx, inc, 1, l, Q, Z, phase)
    t.device_phase(phase)
    sigma, vec, M, kept = t.host(ritz_step, G)
    t.row(lambda: _native.svd_rowmat(ctx, l, Z, M, omega))
    if timings is not None:
      timings.append(t.result())
    ritz.append(sigma.copy())
    if tol > 0 and prev is not None and np.max(np.abs(sigma[:k] - prev)) <= tol * sigma[0]:
      break
    prev = sigma[:k]
  # U = Q U~ (first k columns, zero beyond the numerical rank) into Y; V = the first k columns of omega
  _native.svd_rowmat(ctx, l, Q, vec[:, :k] * kept[:k], Y)
  s = np.where(kept[:k], sigma[:k], 0.0)
  _native.svd_flip(ctx, l, k, Y, omega)
  resid = _native.svd_residuals(ctx, inc, l, k, Y, omega, s)
  info = {"n_iter": it, "ritz_values": np.asarray(ritz), "residuals": resid, "block_width": l}
  return Y[:, :k], s, omega[:, :k], info


class _Timer(object):
  """Per-iteration timing of truncated_svd (device working arrays only; a no-op otherwise)."""

  def __init__(self, on):
    self.on = on
    self.t0 = time.perf_counter()
    self.ms = {"spmm": 0.0, "gram": 0.0, "rowmat": 0.0, "eigh_host": 0.0}

  def device_phase(self, phase):
    if self.on:
      self.ms["spmm"] += float(phase[0])
      self.ms["gram"] += float(phase[1])

  def host(self, fn, *args):
    t0 = time.perf_counter()
    out = fn(*args)
    self.ms["eigh_host"] += (time.perf_counter() - t0) * 1e3
    return out

  def row(self, fn):
    if not self.on:
      fn()
      return
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    self.ms["rowmat"] += a.elapsed_time(b)

  def result(self):
    out = dict(self.ms)
    out["wall"] = (time.perf_counter() - self.t0) * 1e3
    return out


def TruncatedSVDDevice(incidence, k, n_iter=5, oversamples=10, tol=0.0, seed=0):
  """A ~ U diag(s) V^T for the N x E incidence pattern `incidence` (scipy sparse; every stored
  entry counts as 1), 1 <= k <= min(N, E), k <= 256.  Returns (U [N, k] float32, s [k] float64,
  Vt [k, E] float32, info) as numpy arrays, in the shapes of scikit-learn's ``randomized_svd``;
  info holds "n_iter" (iterations run), "ritz_values" ([n_iter, l], each iteration's, l the block
  width), "block_width" and "residuals" ([k], ||A v_i - s_i u_i|| / s_0).  s is descending; each
  pair (u_i, v_i) is signed so that the entry of u_i of largest magnitude is positive
  (scikit-learn's svd_flip).  Triplets beyond the numerical rank (sigma <= 1e-6 sigma_1) come back
  as s_i = 0 with zero vectors.  numpy's global RNG is neither read nor advanced."""
  A = sps.csr_matrix(incidence)
  N, E = A.shape
  check_arguments(N, E, k, n_iter, oversamples, tol)
  ctx = _native.default_context()
  inc = make_incidence(A, ctx=ctx)
  try:
    U, s, V, info = truncated_svd(ctx, inc, k, n_iter, oversamples, tol, seed, device=True)
    U, V = U.cpu().numpy(), V.cpu().numpy()
  finally:
    inc.close()
  return np.ascontiguousarray(U), s, np.ascontiguousarray(V.T), info
