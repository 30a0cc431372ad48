"""The numpy restatements of the seeded epoch order and the seeded initial tables
(oracle/seeded_training_ref.py: shuffle_order, init_table) that hge_shuffle_order and
hge_hg2v_create_seeded are checked against bit for bit: layout on the Philox word streams and
distribution."""
import itertools

import numpy as np
import pytest
from scipy import stats

from oracle import device_sampler_ref as dsr
from oracle import seeded_training_ref as ref


@pytest.mark.parametrize("n", [1, 2, 7, 1000])
def test_shuffle_order_is_a_permutation(n):
  for seed, epoch in ((0, 0), (5, 1), (2**40 + 3, 7)):
    order = ref.shuffle_order(seed, epoch, n)
    assert order.dtype == np.int32 and order.shape == (n,)
    assert np.array_equal(np.sort(order), np.arange(n))


def test_shuffle_order_depends_on_epoch_and_seed():
  base = ref.shuffle_order(11, 0, 1000)
  assert np.array_equal(base, ref.shuffle_order(11, 0, 1000))
  others = [ref.shuffle_order(11, e, 1000) for e in (1, 2, 3)] + \
      [ref.shuffle_order(s, 0, 1000) for s in (12, 11 + 2**32)]
  for other in others:
    assert not np.array_equal(base, other)
  assert not np.array_equal(others[0], others[1])


def test_shuffle_keys_are_words_2e_and_2e_plus_1_of_the_item_stream():
  seed, n = 99, 6
  for epoch in (0, 1, 2, 5):
    st = dsr.Streams(seed, ref.PHASE["SHUFFLE"], np.arange(n))
    every = np.arange(n)
    words = [st.next(every) for _ in range(2 * epoch + 2)]
    keys = (words[2 * epoch] << np.uint64(32)) | words[2 * epoch + 1]
    assert np.array_equal(ref.shuffle_order(seed, epoch, n), np.argsort(keys, kind="stable"))


def test_shuffle_order_is_uniform_over_the_permutations_of_five():
  """Chi-square over 6 000 seeds: each of the 120 orders of 5 items is about equally likely."""
  index = {p: i for i, p in enumerate(itertools.permutations(range(5)))}
  counts = np.zeros(len(index), dtype=np.int64)
  for seed in range(6000):
    counts[index[tuple(ref.shuffle_order(seed, 3, 5).tolist())]] += 1
  assert counts.min() > 0
  assert stats.chisquare(counts).pvalue > 1e-3, counts


def test_init_table_word_layout():
  seed, rows, dim = 7, 5, 6
  t = ref.init_table(seed, ref.PHASE["INIT_NODES"], rows, dim)
  st = dsr.Streams(seed, ref.PHASE["INIT_NODES"], np.arange(rows))
  every = np.arange(rows)
  w = np.stack([st.next(every) for _ in range(dim)], axis=1)
  u = (w >> np.uint64(8)).astype(np.float32) * np.float32(2.0**-24)
  assert t.dtype == np.float32
  assert np.array_equal(t, np.float32(-0.05) + np.float32(0.1) * u)
  assert not np.array_equal(t, ref.init_table(seed, ref.PHASE["INIT_EDGES"], rows, dim))


def test_init_table_is_uniform_on_keras_range():
  t = ref.init_table(3, ref.PHASE["INIT_EDGES"], 20000, 9).astype(np.float64)
  assert t.min() >= -0.05 and t.max() <= 0.05
  var = 0.1**2 / 12
  # standard error of a column mean: sqrt(var / rows) = 2.0e-4; of a column variance: 0.63 %
  assert np.all(np.abs(t.mean(axis=0)) < 1e-3), t.mean(axis=0)
  assert np.all(np.abs(t.var(axis=0) / var - 1) < 0.04), t.var(axis=0) / var
  assert stats.kstest(t[:, 0], stats.uniform(loc=-0.05, scale=0.1).cdf).pvalue > 1e-3
