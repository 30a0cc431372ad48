"""The numpy restatement of the device sampler (oracle/device_sampler_ref.py): Philox known answers,
and the distribution of what it draws on many disjoint copies of small gadgets whose candidate
sets are known.  Every check is a chi-square test at p = 1e-6 on fixed seeds, so each outcome is
deterministic.  The GPU tests pin the kernels to this restatement bit for bit."""
import itertools

import numpy as np
import scipy.sparse as sps
from scipy import stats

from oracle import device_sampler_ref as ref

P_FAIL = 1e-6


def _chi2_ok(counts, expected=None):
  counts = np.asarray(counts, dtype=np.float64).ravel()
  if expected is None:
    expected = np.full(len(counts), counts.sum() / len(counts))
  stat = ((counts - expected)**2 / expected).sum()
  return stat < stats.chi2.ppf(1.0 - P_FAIL, len(counts) - 1), stat


def _copies(block, copies):
  """Block-diagonal incidence of `copies` disjoint copies of a small N x E pattern."""
  return sps.block_diag([sps.csr_matrix(np.asarray(block, dtype=bool))] * copies, format="csr")


def test_philox_known_answers():
  cases = [((0, 0, 0, 0), (0, 0), "6627e8d5 e169c58d bc57ac4c 9b00dbd8"),
           ((0xffffffff,) * 4, (0xffffffff,) * 2, "408f276d 41c83b0e a20bc7c6 6d5451fd"),
           ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
            "d16cfe09 94fdcceb 5001e420 24126ea1")]
  for ctr, key, want in cases:
    assert " ".join("%08x" % int(w) for w in ref.philox4x32_10(ctr, key)) == want


def test_word_stream_layout():
  """Word i of an item is word i % 4 of block i // 4 under counter {block, item lo, item hi, phase}
  and key {seed lo, seed hi}."""
  seed, phase, item = 0x0123456789ABCDEF, 7, (5 << 32) | 9
  st = ref.Streams(seed, phase, [item])
  words = [int(st.next(np.array([0]))[0]) for _ in range(8)]
  for b in range(2):
    block = ref.philox4x32_10((b, 9, 5, phase), (0x89ABCDEF, 0x01234567))
    assert words[4 * b:4 * b + 4] == [int(w) for w in block]


def test_bounded_draws_are_uniform_even_where_rejection_is_frequent():
  # s = 3 * 2^30: a quarter of all words is rejected; bins of equal width must stay equally likely
  s = 3 << 30
  st = ref.Streams(3, 1, np.arange(40000))
  draws = st.below(np.arange(40000), s)
  assert draws.min() >= 0 and draws.max() < s
  assert st.word.sum() > 40000          # some draws were redone
  ok, stat = _chi2_ok(np.bincount(draws // (1 << 28), minlength=12))
  assert ok, stat


def test_every_5_subset_of_a_7_candidate_row_is_equally_likely():
  # one edge of 7 nodes: every node row of A * A^T has the 7 nodes of the copy as candidates
  copies = 3000
  A = _copies(np.ones((7, 1)), copies)
  cptr, ccol, _ = ref.candidate_rows(A, 0, 2)
  assert np.all(np.diff(cptr) == 7)
  rows, cols = ref.select(cptr, ccol, np.full(A.shape[0], 5), seed=11, phase=ref.PHASE["NN"])
  assert np.all(np.bincount(rows, minlength=A.shape[0]) == 5)
  local = (cols - (rows // 7) * 7).reshape(-1, 5)
  assert np.all(np.diff(local, axis=1) > 0)             # distinct and ascending
  index = {c: i for i, c in enumerate(itertools.combinations(range(7), 5))}
  counts = np.bincount([index[tuple(r)] for r in local.tolist()], minlength=len(index))
  ok, stat = _chi2_ok(counts)
  assert ok, stat


def test_inclusion_probability_on_64_candidate_rows_is_k_over_n():
  copies, k = 400, 10
  A = _copies(np.ones((64, 1)), copies)
  cptr, ccol, _ = ref.candidate_rows(A, 0, 2)
  rows, cols = ref.select(cptr, ccol, np.full(A.shape[0], k), seed=12, phase=ref.PHASE["NN"])
  local = cols - (rows // 64) * 64
  counts = np.bincount(local, minlength=64)
  assert counts.sum() == A.shape[0] * k
  ok, stat = _chi2_ok(counts)
  assert ok, stat


def test_three_factor_gadget():
  # node 0 shares edge 0 with node 1, which is also in edges 1..6: both node rows of
  # (A * A^T) * A have the 7 edges of their copy as candidates
  block = np.zeros((2, 7), dtype=bool)
  block[0, 0] = True
  block[1, :] = True
  copies = 1500
  A = _copies(block, copies)
  cptr, ccol, out_cols = ref.candidate_rows(A, 0, 3)
  assert out_cols == 7 * copies and np.all(np.diff(cptr) == 7)
  rows, cols = ref.select(cptr, ccol, np.full(A.shape[0], 5), seed=13, phase=ref.PHASE["NE"])
  local = (cols - (rows // 2) * 7).reshape(-1, 5)
  index = {c: i for i, c in enumerate(itertools.combinations(range(7), 5))}
  counts = np.bincount([index[tuple(r)] for r in local.tolist()], minlength=len(index))
  ok, stat = _chi2_ok(counts)
  assert ok, stat
  # per-position inclusion 5 / 7
  ok, stat = _chi2_ok(np.bincount(local.ravel(), minlength=7))
  assert ok, stat


def test_neighbour_draws_are_uniform_and_independent():
  # node 0 in edges 0..4, edge 0 holds nodes 0..3
  A = np.zeros((4, 5), dtype=bool)
  A[0, :] = True
  A[1:, 0] = True
  A = sps.csr_matrix(A)
  m, k = 20000, 4
  nbr_e, nbr_n = ref.neighbors(A, np.zeros(m, np.int64), np.zeros(m, np.int64), k, seed=14,
                               phase=ref.PHASE["NEIGHBORS"], first=1000)
  for j in range(k):
    ok, stat = _chi2_ok(np.bincount(nbr_e[:, j], minlength=5))
    assert ok, (j, stat)
    ok, stat = _chi2_ok(np.bincount(nbr_n[:, j], minlength=4))
    assert ok, (j, stat)
  for j in range(k - 1):
    ok, stat = _chi2_ok(np.bincount(nbr_e[:, j] * 5 + nbr_e[:, j + 1], minlength=25))
    assert ok, (j, stat)
    ok, stat = _chi2_ok(np.bincount(nbr_n[:, j] * 4 + nbr_n[:, j + 1], minlength=16))
    assert ok, (j, stat)
  # the last edge draw and the first node draw come from the same stream, one word apart
  ok, stat = _chi2_ok(np.bincount(nbr_e[:, -1] * 4 + nbr_n[:, 0], minlength=20))
  assert ok, stat


def test_negatives_are_uniform_on_the_output_columns():
  rows, cols = ref.negatives(np.full(3000, 10), 37, seed=15, phase=ref.PHASE["NEG_NN"])
  assert len(rows) == 30000 and np.all(np.bincount(rows) == 10)
  ok, stat = _chi2_ok(np.bincount(cols, minlength=37))
  assert ok, stat


def test_block_layout_of_the_restated_samplers():
  A = _copies(np.ones((3, 2)), 4)
  out = ref.boolean_samples(A, 2, 2, neg_samples=1, seed=1)
  nn = ~np.isnan(out["nn_prob"])
  assert nn[:nn.sum()].all()                        # node-node block first
  # 12 nodes in 2 edges each, 8 edges of 3 nodes: 12 * 2 + 8 * 2 node-edge records with neighbour
  # arrays and probability 1, then 12 + 8 negative ones without a probability
  assert out["has_neighbors"].sum() == 40 + 20
  assert np.isnan(out["ne_prob"][out["has_neighbors"]]).sum() == 20
