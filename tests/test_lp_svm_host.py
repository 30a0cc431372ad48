"""The numpy restatement of the device link-prediction classifiers (oracle/lp_svm_ref.py): the
distribution of the negatives, the solver against scikit-learn's SVC, the predictor's summation
order against the plain product, and the branches the solver's trace counts."""
import functools
import itertools

import numpy as np
import pytest
import scipy.stats

from oracle import lp_svm_ref as ref


def _same_members(owners, members):
  mptr = np.arange(owners + 1, dtype=np.int64) * len(members)
  return mptr, np.tile(np.asarray(members, dtype=np.int64), owners)


def test_negatives_are_uniform_over_subsets():
  # N = 7 items, members {1, 4}: k = 4 of the 5 non-members, 5 subsets; N = 8, members {2, 5}:
  # k = 4 of 6, 15 subsets
  for items, members in ((7, (1, 4)), (8, (2, 5))):
    owners = 6000
    mptr, midx = _same_members(owners, members)
    sets = ref.training_sets(mptr, midx, items, np.arange(owners), seed=5, phase=ref.PHASE_LP_EDGE_OWNERS)
    others = [i for i in range(items) if i not in members]
    subsets = {s: 0 for s in itertools.combinations(others, 4)}
    for o in range(owners):
      m, neg = sets[o]
      assert m.tolist() == list(members)
      assert not set(neg.tolist()) & set(members)
      assert neg.tolist() == sorted(set(neg.tolist())) and len(neg) == 4
      subsets[tuple(neg.tolist())] += 1
    assert scipy.stats.chisquare(list(subsets.values())).pvalue > 1e-3


def test_every_non_member_is_taken_when_there_are_few():
  mptr, midx = np.array([0, 2, 2, 5]), np.array([0, 1, 0, 1, 2])
  sets = ref.training_sets(mptr, midx, 5, [0, 1, 2], seed=1, phase=ref.PHASE_LP_NODE_OWNERS)
  assert sets[0][1].tolist() == [2, 3, 4]            # k = min(3, 4) = 3: all of them
  assert len(sets[1][0]) == 0 and len(sets[1][1]) == 0   # no member: nothing
  assert sets[2][1].tolist() == [3, 4]               # k = 2 = every non-member


def test_the_stream_is_the_owners():
  mptr, midx = _same_members(40, (3, 9, 20))
  a = ref.training_sets(mptr, midx, 50, np.arange(40), seed=8, phase=ref.PHASE_LP_EDGE_OWNERS)
  b = ref.training_sets(mptr, midx, 50, [17, 3], seed=8, phase=ref.PHASE_LP_EDGE_OWNERS)
  c = ref.training_sets(mptr, midx, 50, [17], seed=8, phase=ref.PHASE_LP_NODE_OWNERS)
  assert a[17][1].tolist() == b[17][1].tolist() and a[3][1].tolist() == b[3][1].tolist()
  assert a[17][1].tolist() != a[3][1].tolist() and a[17][1].tolist() != c[17][1].tolist()


def test_nonmember_ids():
  rng = np.random.RandomState(0)
  for _ in range(20):
    n = rng.randint(1, 40)
    members = np.sort(rng.choice(n, rng.randint(0, n), replace=False))
    others = np.setdiff1d(np.arange(n), members)
    assert ref.nonmember_ids(members, np.arange(len(others))).tolist() == others.tolist()


def _problems():
  rng = np.random.RandomState(2024)
  sizes = [1, 500, 2] + rng.randint(1, 200, 57).tolist()
  for p, m in enumerate(sizes):
    d = (2, 32, 200)[p % 3]
    if d == 2:
      # hundreds of points crowd the plane and flatten the dual's optimum, so two solvers stopped
      # at the same tol differ by more than the bar; keep the planar problems small
      m = 1 + m % 60
    k = 2 * m
    sd = 0.5 * np.sqrt(32.0 / d)   # the same typical squared distance (16) at every d
    centre = rng.randn(d) * sd
    X = np.concatenate([rng.randn(m, d) * sd + centre, rng.randn(k, d) * sd]).astype(np.float32)
    Z = np.concatenate([rng.randn(50, d) * sd + centre, rng.randn(50, d) * sd]).astype(np.float32)
    yield X, np.r_[np.ones(m), -np.ones(k)], Z


@functools.lru_cache(maxsize=None)
def _solved():
  return [(X, y, Z) + ref.solve(X, y) for X, y, Z in _problems()]


def test_solver_matches_sklearn():
  from sklearn.svm import SVC
  count = 0
  for X, y, Z, A, rho, it in _solved():
    assert 0 < it < 10000000
    coef = y * A
    f = ref.decision(X, coef, rho, Z)
    want = SVC(C=1, gamma=0.1).fit(X, (y > 0).astype(int)).decision_function(Z)
    assert np.abs(f - want).max() <= 5e-3
    sure = np.abs(want) > 5e-3
    assert np.array_equal(f[sure] > 0, want[sure] > 0)
    assert ref.kkt_gap(X, y, coef) < 1e-3
    assert np.all((A >= 0) & (A <= 1)) and abs(np.dot(A, y)) < 1e-9
    count += 1
  assert count >= 60


@pytest.mark.parametrize("C,gamma", [(1.0, 0.1), (10.0, 0.5)])
def test_solver_parameters(C, gamma):
  from sklearn.svm import SVC
  rng = np.random.RandomState(7)
  X = rng.randn(60, 4).astype(np.float32)
  y = np.where(X[:, 0] + 0.3 * rng.randn(60) > 0, 1.0, -1.0)
  A, rho, _ = ref.solve(X, y, C=C, gamma=gamma)
  Z = rng.randn(40, 4).astype(np.float32)
  want = SVC(C=C, gamma=gamma).fit(X, (y > 0).astype(int)).decision_function(Z)
  assert np.abs(ref.decision(X, y * A, rho, Z, gamma) - want).max() <= 5e-3 * max(1.0, C)


def test_device_order_decision_is_the_decision():
  for X, y, Z, A, rho, _ in _solved():
    coef = y * A
    want = ref.decision(X, coef, rho, Z)
    got = ref.decision_device_order(X, coef, rho, Z)
    # relative to the sum of the terms' magnitudes, the scale of any summation order's rounding
    scale = np.abs(ref.kernel(Z, X, 0.1).astype(np.float64) * coef).sum(axis=1) + abs(rho)
    assert np.all(np.abs(got - want) <= 1e-12 * scale)
  Z = np.zeros((3, 4), np.float32)
  assert ref.decision_device_order(np.zeros((0, 4), np.float32), [], np.inf, Z).tolist() == [-np.inf] * 3
  assert ref.decision_device_order(np.zeros((0, 4), np.float32), [], -np.inf, Z).tolist() == [np.inf] * 3


def test_device_order_decision_sums_by_lane():
  # K = 1 everywhere, and 2^53 + 1 rounds back to 2^53 (ties to even) while 2^53 + 2 is exact, so
  # where the two 1s meet the big term decides the sum
  X = np.zeros((70, 1), np.float32)
  Z = np.zeros((1, 1), np.float32)
  for ones, want in (((1, 3), 2.0 ** 53 + 2),   # lanes 1 and 3 meet first (o = 2), then lane 0
                     ((1, 2), 2.0 ** 53),       # lane 2 meets lane 0 first
                     ((32, 64), 2.0 ** 53)):    # lane 0 adds its terms one at a time
    coef = np.zeros(70)
    coef[0] = 2.0 ** 53
    coef[list(ones)] = 1.0
    assert ref.decision_device_order(X, coef, 0.5, Z)[0] == want - 0.5, ones


def test_rho_sums_the_free_gradients_in_order():
  # calculate_rho adds y G of the free alphas one at a time: (1e16 + 1) - 1e16 = 0, where a
  # compensated sum would give 1
  yG = np.array([1e16, 1.0, -1e16, 3.0])
  assert ref._rho(np.ones(4), yG, np.full(4, 0.5), 1.0) == 3.0 / 4
  # no free alpha: (min of ub candidates + max of lb candidates) / 2
  y, A = np.array([1.0, 1.0, -1.0, -1.0]), np.array([0.0, 1.0, 0.0, 1.0])
  assert ref._rho(y, np.array([-3.0, -0.5, 0.25, 2.0]), A, 1.0) == (-3.0 + -0.25) / 2


def _trace_cases():
  rng = np.random.RandomState(6)
  palette = rng.randn(3, 3).astype(np.float32)
  yield palette[rng.randint(0, 3, 150)], 50, {}                             # shared vectors
  yield np.ones((60, 4), np.float32), 20, {}                                # identical points
  for _ in range(2):
    yield rng.randn(300, 8).astype(np.float32), 100, dict(C=50, tol=1e-6)   # random
  yield rng.randn(257, 3).astype(np.float32), 200, dict(C=0.05)            # random, members the majority


def test_trace_reaches_every_branch():
  trace = {}
  for X, m, kw in _trace_cases():
    y = np.r_[np.ones(m), -np.ones(len(X) - m)]
    plain = ref.solve(X, y, **kw)
    traced = ref.solve(X, y, trace=trace, **kw)
    assert np.array_equal(plain[0], traced[0]) and plain[1:] == traced[1:]
  assert {k for k in ref.TRACE_KEYS if trace.get(k, 0) > 0} == set(ref.TRACE_KEYS), trace
  assert set(trace) == set(ref.TRACE_KEYS)


def test_exp_hook():
  X = np.random.RandomState(0).randn(5, 3).astype(np.float32)
  seen = []

  def exp(a):
    seen.append(a.dtype)
    return np.ones_like(a)

  assert np.all(ref.kernel(X, X, 0.1, exp) == 1) and seen == [np.float32]
  assert np.array_equal(ref.kernel(X, X, 0.1), ref.exp32(ref.kernel(X, X, 0.1, lambda a: a)))
