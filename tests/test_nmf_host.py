"""The restatements of the non-negative factorization (oracle/nmf_ref.py) on the CPU: the float64
form equals scikit-learn's coordinate descent from the same start, the fp32 form of the device's
operation order stays within the GPU test's bars of scikit-learn's float64 run, its products equal
scipy's float32 products, and the seeded start equals the Philox formula evaluated element by
element with Python integers."""
import warnings

import numpy as np
import pytest
import scipy.sparse as sps

from hypergraphembedding_b200 import synthetic
from oracle import nmf_ref as ref


def _incidence(N, E, nnz, seed=1234):
  A = synthetic.power_law_hypergraph(N, E, nnz, seed=seed).astype(np.float32)
  A.sort_indices()
  return sps.csr_matrix(A)


def _start(A, k, seed=3):
  N, E = A.shape
  scale = np.float32(2) * np.float32(np.sqrt(A.nnz / (N * E * k)))
  W, Ht = ref.start(N, E, k, seed, scale)
  return W, np.ascontiguousarray(Ht.T)


def _sklearn(A, W0, H0, k, max_iter, tol):
  from sklearn.decomposition import non_negative_factorization
  with warnings.catch_warnings():
    warnings.simplefilter("ignore")
    return non_negative_factorization(A.astype(np.float64), W=W0.astype(np.float64), H=H0.astype(np.float64),
                                      n_components=k, init="custom", solver="cd", max_iter=max_iter, tol=tol)


def _rel(a, b):
  return np.linalg.norm(np.asarray(a, np.float64) - b) / np.linalg.norm(b)


def _fit32(A, W0, H0, max_iter, tol):
  B = sps.csr_matrix(A.T)
  B.sort_indices()
  W, Ht, it, viols = ref.fit32(A.indptr, A.indices, B.indptr, B.indices, W0, H0.T, max_iter, tol)
  return W, Ht.T, it, viols


@pytest.mark.parametrize("k", [8, 32])
@pytest.mark.parametrize("max_iter,tol", [(1, 0.0), (5, 0.0), (20, 0.0), (200, 1e-4)])
def test_f64_restatement_equals_scikit_learn(k, max_iter, tol):
  A = _incidence(3000, 1800, 40000)
  W0, H0 = _start(A, k)
  W, H, it = _sklearn(A, W0, H0, k, max_iter, tol)
  W64, H64, it64, viols = ref.fit64(A, W0, H0, max_iter, tol)
  assert it64 == it and len(viols) == it
  assert _rel(W64, W) < 1e-10 and _rel(H64, H) < 1e-10
  if tol > 0:
    assert it < max_iter and viols[-1] / viols[0] <= tol < viols[-2] / viols[0]


@pytest.mark.parametrize("max_iter", [1, 5, 20])
def test_fp32_restatement_is_close_to_scikit_learn(max_iter):
  A = _incidence(2000, 1200, 25000, seed=7)
  k = 8
  W0, H0 = _start(A, k, seed=11)
  W, H, _ = _sklearn(A, W0, H0, k, max_iter, 0.0)
  W32, H32, it, _ = _fit32(A, W0, H0, max_iter, 0.0)
  assert it == max_iter
  assert _rel(W32, W) < 2e-3 and _rel(H32, H) < 2e-3


def test_fp32_restatement_default_stop_is_close_to_scikit_learn():
  A = _incidence(1200, 700, 12000, seed=5)
  k = 8
  W0, H0 = _start(A, k, seed=2)
  W, H, it = _sklearn(A, W0, H0, k, 200, 1e-4)
  W32, H32, it32, _ = _fit32(A, W0, H0, 200, 1e-4)
  assert abs(it32 - it) <= 1
  X = A.toarray().astype(np.float64)
  err = np.linalg.norm(X - W @ H)
  err32 = np.linalg.norm(X - W32.astype(np.float64) @ H32)
  assert abs(err32 - err) / err < 1e-4


def test_products_equal_scipy_float32():
  A = _incidence(3000, 1800, 40000)
  rng = np.random.default_rng(0)
  Ht = rng.random((A.shape[1], 20), dtype=np.float32)
  W = rng.random((A.shape[0], 20), dtype=np.float32)
  B = sps.csr_matrix(A.T)
  B.sort_indices()
  for got, want in ((ref.spmm32(A.indptr, A.indices, Ht), A @ Ht), (ref.spmm32(B.indptr, B.indices, W), A.T @ W)):
    assert want.dtype == np.float32
    assert np.array_equal(got.view(np.uint32), np.asarray(want).view(np.uint32))


def _philox_word(seed, phase, item, word):
  M = 0xFFFFFFFF
  c = [word // 4, item & M, item >> 32, phase]
  k0, k1 = seed & M, seed >> 32
  for _ in range(10):
    p0, p1 = 0xD2511F53 * c[0], 0xCD9E8D57 * c[2]
    c = [((p1 >> 32) ^ c[1] ^ k0) & M, p1 & M, ((p0 >> 32) ^ c[3] ^ k1) & M, p0 & M]
    k0, k1 = (k0 + 0x9E3779B9) & M, (k1 + 0xBB67AE85) & M
  return c[word % 4]


def test_seeded_start_equals_the_philox_formula():
  seed, k, scale = 0x123456789ABCDEF, 7, np.float32(0.0625)
  W, Ht = ref.start(5, 4, k, seed, scale)
  assert W.dtype == np.float32 and W.shape == (5, k) and Ht.shape == (4, k)
  for phase, table in ((20, W), (21, Ht)):
    for r in range(table.shape[0]):
      for c in range(k):
        u = (_philox_word(seed, phase, r, c) >> 8) / 2.0 ** 24     # exact in float64
        assert table[r, c] == np.float32(np.float64(scale) * u)   # one rounding, as scale * u in fp32
  assert (W >= 0).all() and (W < scale).all() and not np.array_equal(W[:4], Ht)


def test_stop_rule_and_zero_hessian_branch():
  A = _incidence(600, 400, 5000, seed=9)
  k = 4
  W0, H0 = _start(A, k)
  W0[:, 2] = 0     # component 2 of W is zero: G[2, 2] == 0 in the H half of iteration 1
  W, H, it = _sklearn(A, W0, H0, k, 3, 0.0)
  W64, H64, it64, _ = ref.fit64(A, W0, H0, 3, 0.0)
  assert it64 == it == 3
  assert _rel(W64, W) < 1e-10 and _rel(H64, H) < 1e-10
  W32, H32, _, _ = _fit32(A, W0, H0, 3, 0.0)
  assert _rel(W32, W) < 2e-3 and _rel(H32, H) < 2e-3
