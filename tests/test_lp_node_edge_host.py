"""The restatement of the node-edge link classifier (oracle/lp_node_edge_ref.py) on the CPU: its
float64 trainer against torch autograd + torch.optim.Adagrad, the negatives (never incidences,
uniform over the complement), the rank -> pair map against enumeration, the 64-bit draw against
Python integers, and the held-out accuracy the model reaches on planted communities."""
import numpy as np
import pytest
import scipy.sparse as sps
from scipy import stats

from oracle import lp_node_edge_ref as ref
from oracle.device_sampler_ref import Streams

# Held-out accuracy of the restatement on ref.planted_communities() (graph seed 0, hidden 32, 30
# epochs, batch 16, lr 0.1, training seed 5): 0.941 (96 of 102 links) measured with the float64
# trainer; the bar leaves a margin of 0.09 (9 links) for the fp32 device run.
PLANTED_ACCURACY = 0.85
PLANTED_KW = dict(hidden=32, epochs=30, batch_size=16, lr=0.1)
PLANTED_SEED = 5


def _graph(seed=0, N=9, E=7, p=0.4, full_rows=(), empty_rows=()):
  rng = np.random.RandomState(seed)
  A = (rng.rand(N, E) < p).astype(np.int8)
  for n in full_rows:
    A[n] = 1
  for n in empty_rows:
    A[n] = 0
  A = sps.csr_matrix(A)
  A.sort_indices()
  return A


def test_trainer_matches_torch_autograd():
  import torch
  A = _graph(1)
  rng = np.random.RandomState(2)
  d, H, batch, lr, eps = 3, 5, 7, 0.01, 1e-7
  xn, xe = rng.randn(A.shape[0], d), rng.randn(A.shape[1], d)
  nodes, edges, labels = ref.training_set(A.indptr, A.indices, A.shape[1], 3)
  weights = ref.init_weights(3, d, H)
  orders = [ref.shuffle_order(3, e, len(nodes)) for e in range(2)]
  (W1, b1, w2, b2), losses = ref.train(xn, xe, nodes, edges, labels, weights, orders, batch, lr, eps)

  prm = [torch.tensor(np.asarray(w, np.float64), requires_grad=True) for w in weights]
  opt = torch.optim.Adagrad(prm, lr=lr, eps=eps, initial_accumulator_value=0)
  X = torch.tensor(np.concatenate([xn[nodes], xe[edges]], axis=1))
  Y = torch.tensor(labels)
  t_losses = []
  for order in orders:
    total = 0.0
    for first in range(0, len(order), batch):
      s = torch.as_tensor(order[first:first + batch])
      z = torch.relu(X[s] @ prm[0] + prm[1]) @ prm[2] + prm[3][0]
      loss = torch.nn.functional.binary_cross_entropy_with_logits(z, Y[s], reduction="sum")
      total += float(loss.detach())
      opt.zero_grad()
      (loss / len(s)).backward()
      opt.step()
    t_losses.append(total / len(order))
  for mine, theirs in zip((W1, b1, w2, b2), prm):
    assert np.abs(mine - theirs.detach().numpy()).max() < 1e-12
  assert np.abs(losses - np.asarray(t_losses)).max() < 1e-12


def test_negatives_are_uniform_non_incidences():
  A = _graph(3, N=20, E=15, p=0.3)
  N, E = A.shape
  S = N * E - A.nnz
  assert 150 < S < 400
  r = ref.draw_ranks(11, 40 * S, S)
  n, e = ref.rank_to_pair(A.indptr, A.indices, E, r)
  assert not np.any(np.asarray(A[n, e]).ravel())
  counts = np.bincount(n * E + e, minlength=N * E)
  present = np.asarray(A.todense()).ravel() > 0
  assert np.all(counts[present] == 0)
  _, pvalue = stats.chisquare(counts[~present])
  assert pvalue > 1e-3


def test_rank_to_pair_matches_enumeration():
  A = _graph(4, N=10, E=6, p=0.5, full_rows=(2, 7), empty_rows=(0, 5, 9))
  N, E = A.shape
  dense = np.asarray(A.todense()) > 0
  expect = [(n, e) for n in range(N) for e in range(E) if not dense[n, e]]
  n, e = ref.rank_to_pair(A.indptr, A.indices, E, np.arange(len(expect)))
  assert list(zip(n.tolist(), e.tolist())) == expect


@pytest.mark.parametrize("S", [2**32 - 5, 2**32 + 3, 2**40 - 1, 2**40 + 12345])
def test_draw_matches_python_integers(S):
  count = 64
  r = ref.draw_ranks(9, count, S)
  mask = (1 << (S - 1).bit_length()) - 1
  assert mask >= S - 1 and (mask >> 1) < S - 1
  st = Streams(9, ref.PHASE["NEG"], np.arange(count))
  for i in range(count):
    while True:
      w0 = int(st.next(np.array([i]))[0])
      w1 = int(st.next(np.array([i]))[0])
      v = ((w0 << 32) | w1) & mask
      if v < S:
        break
    assert int(r[i]) == v


def planted_accuracy(weights, xn, xe, pos, neg):
  p_pos = ref.predict(weights, xn, xe, pos[:, 0], pos[:, 1])
  p_neg = ref.predict(weights, xn, xe, neg[:, 0], neg[:, 1])
  return (np.sum(p_pos > 0.5) + np.sum(p_neg <= 0.5)) / (len(pos) + len(neg))


def test_planted_communities_accuracy():
  A, xn, xe, pos, neg = ref.planted_communities()
  d = xn.shape[1]
  nodes, edges, labels = ref.training_set(A.indptr, A.indices, A.shape[1], PLANTED_SEED)
  orders = [ref.shuffle_order(PLANTED_SEED, e, len(nodes)) for e in range(PLANTED_KW["epochs"])]
  weights, _ = ref.train(xn, xe, nodes, edges, labels, ref.init_weights(PLANTED_SEED, d, PLANTED_KW["hidden"]),
                         orders, PLANTED_KW["batch_size"], PLANTED_KW["lr"])
  assert planted_accuracy(weights, xn, xe, pos, neg) >= PLANTED_ACCURACY
