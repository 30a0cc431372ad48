"""The restatements of the truncated SVD (oracle/svd_ref.py) on the CPU: the float64 form equals
numpy's dense SVD on matrices of known spectrum, the fp32 form's Gram and row-times-matrix steps
equal plain numpy formulas on dyadic inputs (where the order of the sums does not matter), the fp32
form stays close to the float64 form on an incidence, and TruncatedSVDDevice refuses bad
arguments before it needs a device."""
import numpy as np
import pytest
import scipy.sparse as sps

from hypergraphembedding_b200 import synthetic
from oracle import svd_ref as ref


def _orthonormal(rng, n, r):
  q, _ = np.linalg.qr(rng.standard_normal((n, r)))
  return q


@pytest.mark.parametrize("k", [8, 32])
def test_f64_form_equals_dense_svd_on_a_known_spectrum(k):
  rng = np.random.default_rng(k)
  N, E = 300, 200
  s_true = 3.0 * 0.95 ** np.arange(E)             # geometric gaps of 5.3 %
  U0, V0 = _orthonormal(rng, N, E), _orthonormal(rng, E, E)
  A = (U0 * s_true) @ V0.T
  l = ref.block_width(k, 10, N, E)
  omega = ref.start(E, l, seed=k)[:, :l].astype(np.float64)
  U, s, V, info = ref.fit64(A, k, omega, n_iter=100)
  Ud, sd, Vdt = np.linalg.svd(A, full_matrices=False)
  assert info["n_iter"] == 100 and info["ritz_values"].shape == (100, l)
  assert np.abs(s - sd[:k]).max() <= 1e-10 * sd[0]
  assert np.abs(np.sum(U * Ud[:, :k], axis=0)).min() >= 1 - 1e-8
  assert np.abs(np.sum(V * Vdt[:k].T, axis=0)).min() >= 1 - 1e-8
  assert info["residuals"].max() < 1e-8
  # the sign rule: the entry of largest magnitude of each u_i is positive
  assert (U[np.argmax(np.abs(U), axis=0), np.arange(k)] > 0).all()


def test_f64_form_zeroes_the_triplets_beyond_the_numerical_rank():
  rng = np.random.default_rng(3)
  N, E, r = 120, 90, 6
  A = (_orthonormal(rng, N, r) * (1.0 + np.arange(r)[::-1])) @ _orthonormal(rng, E, r).T
  k = 10
  l = ref.block_width(k, 10, N, E)
  U, s, V, _ = ref.fit64(A, k, ref.start(E, l, 1)[:, :l], n_iter=5)
  assert np.allclose(s[:r], np.arange(r, 0, -1), rtol=0, atol=1e-12)
  assert (s[r:] == 0).all() and (U[:, r:] == 0).all() and (V[:, r:] == 0).all()


def _dyadic(rng, shape, bits=6):
  return (rng.integers(-2 ** bits, 2 ** bits, shape) / 2.0 ** bits).astype(np.float32)


def test_gram_and_row_times_matrix_equal_numpy_on_dyadic_inputs():
  rng = np.random.default_rng(7)
  for rows, l, cols in ((1, 1, 1), (37, 5, 3), (5000, 19, 19), (9000, 42, 8), (300, 256, 256)):
    Y = np.zeros((rows, ref.ld_of(l)), dtype=np.float32)
    Y[:, :l] = _dyadic(rng, (rows, l))
    M = _dyadic(rng, (l, cols))
    G = ref.gram64(Y, l)
    assert G.dtype == np.float64 and np.array_equal(G, Y[:, :l].astype(np.float64).T @ Y[:, :l])
    out = ref.rowmat32(Y, M, l)
    assert out.shape == (rows, ref.ld_of(l)) and (out[:, cols:] == 0).all()
    assert np.array_equal(out[:, :cols], (Y[:, :l].astype(np.float64) @ M).astype(np.float32))


def test_start_is_uniform_on_minus_one_one_and_padded():
  seed, l = 0x123456789ABCDEF, 7
  omega = ref.start(500, l, seed)
  assert omega.shape == (500, 8) and omega.dtype == np.float32
  assert (omega[:, l:] == 0).all() and (omega[:, :l] >= -1).all() and (omega[:, :l] < 1).all()
  from oracle.nmf_ref import table
  u = table(500, l, seed, ref.PHASE_SVD, 1.0)          # (w >> 8) 2^-24 of phase 22
  assert np.array_equal(omega[:, :l], np.float32(-1) + np.float32(2) * u)
  assert abs(float(omega[:, :l].mean())) < 0.05


def test_flip_takes_the_lowest_row_on_a_tie():
  U = np.array([[0.5, -2.0, 1.0], [-0.5, 2.0, -3.0], [0.25, 0.0, 3.0]], dtype=np.float32)
  V = np.ones((2, 3), dtype=np.float32)
  ref.flip(U, V, 3)
  assert np.array_equal(U[:, 0], [0.5, -0.5, 0.25]) and np.array_equal(V[:, 0], [1, 1])
  assert np.array_equal(U[:, 1], [2.0, -2.0, -0.0]) and np.array_equal(V[:, 1], [-1, -1])
  assert np.array_equal(U[:, 2], [-1.0, 3.0, -3.0]) and np.array_equal(V[:, 2], [-1, -1])


@pytest.mark.parametrize("k", [4, 17])
def test_fp32_form_is_close_to_the_f64_form_on_an_incidence(k):
  A = synthetic.power_law_hypergraph(900, 600, 9000, seed=5).astype(np.float32)
  A = sps.csr_matrix(A)
  A.sort_indices()
  B = sps.csr_matrix(A.T)
  B.sort_indices()
  N, E = A.shape
  U, s, V, info = ref.fit32(A.indptr, A.indices, B.indptr, B.indices, N, E, k, n_iter=4, seed=2)
  l = ref.block_width(k, 10, N, E)
  U64, s64, V64, info64 = ref.fit64(A, k, ref.start(E, l, 2)[:, :l], n_iter=4)
  assert U.dtype == np.float32 and V.dtype == np.float32 and s.dtype == np.float64
  assert np.abs(s - s64).max() <= 1e-5 * s64[0]
  assert np.abs(info["residuals"] - info64["residuals"]).max() <= 1e-4
  assert np.abs(U.T.astype(np.float64) @ U - np.eye(k)).max() <= 1e-4
  assert np.abs(V.T.astype(np.float64) @ V - np.eye(k)).max() <= 1e-4


def test_refusals_need_no_device():
  from hypergraphembedding_b200 import TruncatedSVDDevice
  A = synthetic.power_law_hypergraph(60, 40, 400, seed=1)
  for kwargs in ({"k": 0}, {"k": 41}, {"k": 257}, {"k": 4, "n_iter": 0}, {"k": 4, "oversamples": -1},
                 {"k": 4, "tol": -1e-9}, {"k": 4, "tol": float("nan")}):
    with pytest.raises(AssertionError):
      TruncatedSVDDevice(A, **kwargs)
