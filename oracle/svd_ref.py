"""Numpy restatements of the truncated SVD of csrc/hge_svd.cu and hypergraphembedding_b200/svd.py:
randomized subspace iteration with Rayleigh-Ritz on the node-edge incidence A [N, E].

- `fit32`: the device's operation order, bit for bit (tests/test_svd_gpu.py compares the library
  with it), with its own copy of the host driver:
    the start (`start`): -1 + 2 ((w >> 8) 2^-24), Philox phase 22, padded to ld = l rounded up to 4;
    the products: nmf_ref.spmm32 (each row adds its neighbours' rows in ascending order from +0);
    the Gram matrices (`gram64`): per chunk of 4096 rows a float64 sum in row order from +0 of the
    exact products Y[i,t] Y[i,r] (the device's f64 fma equals it, as the product of two floats is
    exact in f64), then the chunk partials in ascending chunk order;
    the row-times-matrix step (`rowmat32`): per entry an fp32 fma chain over r ascending from +0;
    the sign flip and the residuals (`flip`, `residuals`).
  Read from `cuobjdump -sass` of the sm_100a build: k_svd_rowmat is FFMA (explicit __fmaf_rn),
  k_svd_gram DFMA (explicit __fma_rn), the residual DMUL / DADD (explicit __dmul_rn, __dsub_rn,
  __dadd_rn) and the IEEE square root and division.
- `fit64`: the same algorithm in float64 on any real matrix (dense or scipy sparse), from a given
  start block; tests/test_svd_host.py holds it to numpy's dense SVD on matrices of known spectrum.

Test infrastructure only."""
import numpy as np
import scipy.sparse as sps

from oracle.nmf_ref import spmm32, table
from oracle.sweep_ref import fma32

F32 = np.float32
PHASE_SVD = 22
GRAM_CHUNK = 4096
RANK_CUT = 1e-6
MAX_L = 256


def ld_of(l):
  return (int(l) + 3) & ~3


def block_width(k, oversamples, N, E):
  return min(int(k) + int(oversamples), int(N), int(E), MAX_L)


def start(num_edges, l, seed):
  """Omega [E, ld] float32: element (r, c < l) = fp32(-1 + fp32(2 u)), u = (w >> 8) 2^-24, w = word c
  of row r's stream in phase 22; the padding columns are 0."""
  out = np.zeros((int(num_edges), ld_of(l)), dtype=F32)
  out[:, :l] = F32(-1) + table(num_edges, l, seed, PHASE_SVD, 2.0)
  return out


# ---- fp32 device order ---------------------------------------------------------------------------

def gram64(Y, l):
  """G = Y^T Y over the first l columns in float64: per chunk a sum in row order from +0, then the
  chunk partials in ascending order."""
  rows = Y.shape[0]
  Y = np.asarray(Y[:, :l], dtype=np.float64)
  chunks = max(1, -(-rows // GRAM_CHUNK))
  part = np.zeros((chunks, l, l), dtype=np.float64)
  for j in range(min(rows, GRAM_CHUNK)):
    sel = np.arange(j, rows, GRAM_CHUNK)
    y = Y[sel]
    part[:len(sel)] = part[:len(sel)] + y[:, :, None] * y[:, None, :]
  G = part[0].copy()
  for c in range(1, chunks):
    G = G + part[c]
  return G


def rowmat32(Y, M, l):
  """out [rows, ld] = Y[:, :l] M (M [l, cols] float32): per entry an fp32 fma chain over r = 0..l-1
  from +0; columns cols .. ld - 1 are 0."""
  rows = Y.shape[0]
  cols = M.shape[1]
  acc = np.zeros((rows, cols), dtype=F32)
  for r in range(l):
    acc = fma32(Y[:, r:r + 1], M[r:r + 1, :], acc)
  out = np.zeros((rows, ld_of(l)), dtype=F32)
  out[:, :cols] = acc
  return out


def flip(U, V, k):
  """In place on the first k columns: negate (u_i, v_i) where the entry of u_i of largest
  magnitude (lowest row on a tie) is negative."""
  idx = np.argmax(np.abs(U[:, :k]), axis=0)
  neg = U[idx, np.arange(k)] < 0
  U[:, :k] = np.where(neg, -U[:, :k], U[:, :k])
  V[:, :k] = np.where(neg, -V[:, :k], V[:, :k])


def residuals(n2e_ptr, n2e_idx, U, V, sigma, k):
  """||A v_i - sigma_i u_i|| / sigma_0: P = A V (spmm32), then d = P - sigma U and s = s + d d in
  float64 per chunk of 4096 rows in row order, the chunk sums in ascending order."""
  P = spmm32(n2e_ptr, n2e_idx, V).astype(np.float64)[:, :k]
  D = P - np.asarray(sigma, np.float64)[None, :] * U[:, :k].astype(np.float64)
  rows = D.shape[0]
  chunks = max(1, -(-rows // GRAM_CHUNK))
  part = np.zeros((chunks, k), dtype=np.float64)
  for j in range(min(rows, GRAM_CHUNK)):
    sel = np.arange(j, rows, GRAM_CHUNK)
    part[:len(sel)] = part[:len(sel)] + D[sel] * D[sel]
  s = part[0].copy()
  for c in range(1, chunks):
    s = s + part[c]
  norm = np.sqrt(s)
  return norm / sigma[0] if sigma[0] > 0 else norm


def ritz_step(G):
  """eigh in float64, sigma descending, M = U~ diag(1 / sigma) (0 beyond the numerical rank)."""
  lam, vec = np.linalg.eigh(G)
  lam, vec = lam[::-1], vec[:, ::-1]
  sigma = np.sqrt(np.maximum(lam, 0.0))
  kept = sigma > RANK_CUT * sigma[0]
  inv = np.zeros_like(sigma)
  inv[kept] = 1.0 / sigma[kept]
  return sigma, vec, vec * inv, kept


def fit32(n2e_ptr, n2e_idx, e2n_ptr, e2n_idx, num_nodes, num_edges, k, n_iter=5, oversamples=10, tol=0.0,
          seed=0):
  """(U [N, k] float32, s [k] float64, V [E, k] float32, info) of the library, bit for bit."""
  l = block_width(k, oversamples, num_nodes, num_edges)
  omega = start(num_edges, l, seed)
  ritz = []
  prev = None
  it = 0
  while it < n_iter:
    it += 1
    Y = spmm32(n2e_ptr, n2e_idx, omega)
    _, _, M, _ = ritz_step(gram64(Y, l))
    Q = rowmat32(Y, M.astype(F32), l)
    Z = spmm32(e2n_ptr, e2n_idx, Q)
    sigma, vec, M, kept = ritz_step(gram64(Z, l))
    omega = rowmat32(Z, M.astype(F32), l)
    ritz.append(sigma.copy())
    if tol > 0 and prev is not None and np.max(np.abs(sigma[:k] - prev)) <= tol * sigma[0]:
      break
    prev = sigma[:k]
  U = rowmat32(Q, (vec[:, :k] * kept[:k]).astype(F32), l)
  s = np.where(kept[:k], sigma[:k], 0.0)
  flip(U, omega, k)
  resid = residuals(n2e_ptr, n2e_idx, U, omega, s, k)
  return U[:, :k].copy(), s, omega[:, :k].copy(), {"n_iter": it, "ritz_values": np.asarray(ritz),
                                                     "residuals": resid}


# ---- float64 -----------------------------------------------------------------------------------------

def fit64(A, k, omega0, n_iter=5, tol=0.0):
  """The same algorithm in float64 on any real N x E matrix A (dense or scipy sparse) from the start
  block omega0 [E, l] (its first l columns are used, l = omega0's columns): (U [N, k], s [k],
  V [E, k], info) with info's residuals ||A v_i - s_i u_i|| / s_0."""
  A = sps.csr_matrix(A, dtype=np.float64) if sps.issparse(A) else np.asarray(A, dtype=np.float64)
  omega = np.array(omega0, dtype=np.float64)
  ritz = []
  prev = None
  it = 0
  while it < n_iter:
    it += 1
    Y = np.asarray(A @ omega)
    _, _, M, _ = ritz_step(Y.T @ Y)
    Q = Y @ M
    Z = np.asarray(A.T @ Q)
    sigma, vec, M, kept = ritz_step(Z.T @ Z)
    omega = Z @ M
    ritz.append(sigma.copy())
    if tol > 0 and prev is not None and np.max(np.abs(sigma[:k] - prev)) <= tol * sigma[0]:
      break
    prev = sigma[:k]
  U = Q @ (vec[:, :k] * kept[:k])
  V = omega[:, :k].copy()
  s = np.where(kept[:k], sigma[:k], 0.0)
  idx = np.argmax(np.abs(U), axis=0)
  sign = np.where(U[idx, np.arange(k)] < 0, -1.0, 1.0)
  U, V = U * sign, V * sign
  R = np.asarray(A @ V) - U * s
  resid = np.linalg.norm(R, axis=0) / (s[0] if s[0] > 0 else 1.0)
  return U, s, V, {"n_iter": it, "ritz_values": np.asarray(ritz), "residuals": resid}
