"""The numpy restatement of the device link-prediction classifiers (oracle/lp_svm_ref.py): the
distribution of the negatives, and the solver against scikit-learn's SVC."""
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


def test_solver_matches_sklearn():
  from sklearn.svm import SVC
  count = 0
  for X, y, Z in _problems():
    A, rho, it = ref.solve(X, y)
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
