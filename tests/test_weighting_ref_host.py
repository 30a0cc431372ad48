"""The numpy restatements of the span and HOBE-probability kernels (oracle/weighting_ref.py) against
the oracle port (oracle/port.py, itself pinned to the unmodified reference).  The GPU tests
(tests/test_weighting_kernels_gpu.py) pin the kernels to these restatements bit for bit."""
import numpy as np

from conftest import csr_from_pairs, load_golden
from oracle import port
from oracle import weighting_ref as wref


def _golden(name):
  g = load_golden("weights_" + name)
  A = csr_from_pairs(g["pairs"], shape=(len(g["xn"]), len(g["xe"])))
  return A, A.T.tocsr(), g["xn"], g["xe"]


def _port_weights(M, x_src, x_tgt):
  """port.incidence_weight of every stored incidence of M, in storage order (fp32)."""
  rows = np.repeat(np.arange(M.shape[0]), np.diff(M.indptr))
  return np.asarray([port.incidence_weight(x_src[r], x_tgt[c]) for r, c in zip(rows, M.indices)],
                    dtype=np.float32)


def test_spans_match_the_port_on_the_goldens():
  for name in ("rand25", "youtube"):
    A, B, xn, xe = _golden(name)
    for M, xs, xo in ((A, xn, xe), (B, xe, xn)):
      got = wref.row_span_f32(M.indptr, M.indices, xs, xo)
      want = port.compute_span_rows(M, xs, xo)
      assert got.dtype == np.float32
      assert np.all(np.abs(got - want) <= 1e-6 * np.abs(want)), name


def test_same_type_prob_matches_the_port():
  rng = np.random.default_rng(0)
  for name in ("rand25", "youtube"):
    A, B, xn, xe = _golden(name)
    for M, xs, xo in ((A, xn, xe), (B, xe, xn)):
      w = _port_weights(M, xs, xo)
      pi, pj = (M @ M.T).nonzero()       # every pair that shares a column, i == j included
      if name != "rand25":
        # 5 000 random pairs: half uniform (mostly nothing shared), half among those that share
        pick = rng.integers(0, len(pi), 2500)
        ri, rj = rng.integers(0, M.shape[0], (2, 2500))
        pi, pj = np.concatenate([ri, pi[pick]]), np.concatenate([rj, pj[pick]])
      got = wref.same_type_prob(M.indptr, M.indices, w, pi, pj)
      want = np.asarray([port.same_type_dist_calc(int(i), int(j), M, xs, xo) for i, j in zip(pi, pj)],
                        dtype=np.float32)
      assert np.array_equal(got, want), name
      assert (got > 0).sum() > len(got) // 10, name


def test_diff_type_prob_matches_the_port():
  rng = np.random.default_rng(1)
  for name, count in (("rand25", None), ("youtube", 2000)):
    A, B, xn, xe = _golden(name)
    w_e2n = _port_weights(B, xe, xn)
    if count is None:
      pn, pe = np.meshgrid(np.arange(A.shape[0]), np.arange(A.shape[1]), indexing="ij")
      pn, pe = pn.ravel(), pe.ravel()
    else:
      pn, pe = rng.integers(0, A.shape[0], count), rng.integers(0, A.shape[1], count)
    got = wref.diff_type_prob(A.indptr, A.indices, B.indptr, B.indices, w_e2n, pn, pe)
    want = np.asarray([port.diff_type_prob(int(n), int(e), A, B, xn, xe) for n, e in zip(pn, pe)],
                      dtype=np.float32)
    assert np.array_equal(got, want), name
    assert (got > 0).any()


def _csr(rows):
  """CSR of `rows` lists of sorted column ids, as (ptr, idx)."""
  ptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
  idx = np.asarray([c for r in rows for c in r], dtype=np.int32)
  return ptr, idx


def test_hand_built_probabilities():
  #         row 0      row 1   row 2  row 3      row 4
  ptr, idx = _csr([[0, 2, 5], [2, 5], [], [0, 1, 2], [1, 5]])
  w = np.asarray([0.5, 0.25, 0.75,     # row 0
                  0.25, 0.75,          # row 1: ties with row 0 on both shared columns
                  -0.5, -0.25, -1.0,   # row 3: all negative
                  -2.0, -3.0],         # row 4
                 dtype=np.float32)
  pi = [0, 2, 2, 0, 1, 0, 3, 3, 4, 0, 1]
  pj = [0, 2, 0, 1, 0, 3, 3, 4, 3, 4, 4]
  want = [0.75,    # i == j: the largest weight of the row
          0.0,     # i == j on an empty row
          0.0,     # against an empty row
          0.75,    # ties: min(0.25, 0.25), min(0.75, 0.75)
          0.75,    # the same pair swapped
          0.0,     # shared {0, 2}: min(0.5, -0.5), min(0.25, -1) < 0, so the floor of 0 wins
          0.0,     # i == j on an all-negative row: the floor of 0 wins
          0.0,     # shared {1}: min(-0.25, -2) < 0
          0.0,
          0.0,     # shared {5}: min(0.75, -3) < 0
          0.0]
  got = wref.same_type_prob(ptr, idx, w, pi, pj)
  assert np.array_equal(got, np.asarray(want, dtype=np.float32))


def test_hand_built_spans_and_diff_type():
  ptr, idx = _csr([[1, 2], [], [0]])
  xs = np.asarray([[0, 1], [5, 5], [1, -1]], dtype=np.float32)
  xo = np.asarray([[2, 2], [1, 3], [-1, 0]], dtype=np.float32)
  # row 0: diffs (1, 2), (-1, -1) -> hi 2, lo -1; row 1 empty; row 2: (1, 3) -> hi 3, lo 0
  assert np.array_equal(wref.row_span_f32(ptr, idx, xs, xo), np.asarray([3, 0, 3], np.float32))
  # node 0 in edges {0, 1}, node 1 in none; edges: 0 -> {0, 2}, 1 -> {0}, 2 -> {1}
  n2e_ptr, n2e_idx = _csr([[0, 1], [], []])
  e2n_ptr, e2n_idx = _csr([[0, 2], [0], [1]])
  w_e2n = np.asarray([0.5, 0.9, 0.25, 0.8], dtype=np.float32)
  got = wref.diff_type_prob(n2e_ptr, n2e_idx, e2n_ptr, e2n_idx, w_e2n, [0, 0, 0, 1], [0, 1, 2, 0])
  # (0, 0): max(pr(0, 0) = 0.9, pr(0, 1) = min(0.5, 0.25)); (0, 1): max(0.25, 0.25);
  # (0, 2): edge 2 shares nothing with edges 0 and 1; node 1 has no edge
  assert np.array_equal(got, np.asarray([0.9, 0.25, 0, 0], np.float32))


def test_float64_distances_and_weights():
  rng = np.random.default_rng(2)
  xa, xb = rng.random((7, 5)).astype(np.float32), rng.random((4, 5)).astype(np.float32)
  ia, ib = rng.integers(0, 7, 50), rng.integers(0, 4, 50)
  want = np.asarray([np.linalg.norm(xa[i].astype(np.float64) - xb[j]) for i, j in zip(ia, ib)])
  assert np.allclose(wref.pair_l2_f64(xa, xb, ia, ib), want, rtol=1e-15, atol=0)
  ptr, idx = _csr([[0, 3], [], [1]])
  d = wref.incidence_l2_f64(ptr, idx, xa[:3], xb)
  assert np.allclose(d, wref.pair_l2_f64(xa, xb, [0, 0, 2], [0, 3, 1]), rtol=1e-15, atol=0)
  assert np.allclose(wref.hobe_weight_f64(d, 5), (np.sqrt(5) - d) / np.sqrt(5), rtol=1e-15, atol=0)
