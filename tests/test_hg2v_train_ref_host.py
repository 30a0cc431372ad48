"""The fp32 restatement of k_hg2v_epoch (oracle/hg2v_train_ref.py) on the CPU: it trains as the
float64 Keras restatement (oracle/hg2v_model_ref.py) does, and hand-built batches fix its
bookkeeping -- FTZ of subnormal contributions to rows != 0, the row-0 split between one CTA's plain
sum and the FTZ atomic per CTA, the da == 0 skip, both KL clip branches and p == 1, relu at z = 0,
elements with g == 0 left alone, and k = 0.  tests/test_hg2v_train_exact_gpu.py compares the
kernel with this restatement bit for bit."""
import numpy as np
import pytest

from oracle import hg2v_model_ref
from oracle import hg2v_train_ref as ref
from oracle.sweep_ref import fma32

F32 = np.float32
T = np.finfo(F32).tiny


def _random_problem(seed, nodes, edges, k, m):
  rng = np.random.default_rng(seed)
  kind = rng.integers(0, 3, m)
  z = np.zeros(m, np.int64)
  ln = np.where(kind != 1, rng.integers(1, nodes + 1, m), z)
  rn = np.where(kind == 0, rng.integers(1, nodes + 1, m), z)
  le = np.where(kind == 1, rng.integers(1, edges + 1, m), z)
  re = np.where(kind != 0, rng.integers(1, edges + 1, m), z)
  nn = [np.where(kind == 2, rng.integers(1, nodes + 1, m), z) for _ in range(k)]
  ne = [np.where(kind == 2, rng.integers(1, edges + 1, m), z) for _ in range(k)]
  p = rng.random(m).astype(F32)
  t = [np.where(kind == i, p, 0).astype(F32) for i in range(3)]
  return np.array([ln, le, rn, re] + nn + ne), np.array(t)


@pytest.mark.parametrize("activation,loss,dim,k,batch", [
    ("relu", "mse", 16, 3, 256),
    ("sigmoid", "kld", 40, 9, 100),
    ("relu", "kld", 70, 2, 333),
    ("sigmoid", "mse", 5, 0, 64),
    ("relu", "mse", 130, 14, 500),
])
def test_three_epochs_agree_with_the_float64_restatement(activation, loss, dim, k, batch):
  """Realistic inputs (heavy duplication, row 0 in most samples), uniform +-0.7 tables.  Measured:
  tables within 2.6e-5 of the float64 fit (relu / MSE, dim 130, k 14; the rest within 1.3e-6) and
  epoch losses within 1e-6 relative; the bar is 5e-5 and 1e-5, well inside the GPU tests' 2e-4."""
  f, t = _random_problem(dim + k, 300, 120, k, 2000)
  rng = np.random.default_rng(1)
  n0 = rng.uniform(-0.7, 0.7, (301, dim)).astype(F32)
  e0 = rng.uniform(-0.7, 0.7, (121, dim)).astype(F32)
  orders = [np.random.default_rng(10 + e).permutation(f.shape[1]) for e in range(3)]
  trainer = ref.Trainer(n0, e0, k, activation, loss)
  losses = [trainer.epoch(f, t, o, batch) for o in orders]
  want_n, want_e, want_losses = hg2v_model_ref.fit(n0, e0, list(f), list(t), k, activation, loss, batch, 3,
                                                   order=orders, min_delta=-1e9)
  assert np.abs(trainer.N - want_n).max() < 5e-5 and np.abs(trainer.E - want_e).max() < 5e-5
  assert np.allclose(losses, want_losses, rtol=1e-5, atol=0)
  assert np.abs(trainer.N - n0).max() > 0.01


# ---- hand-built batches -------------------------------------------------------------------------

def _batch(N, E, feats, targets, k=0, activation="relu", loss="mse", clusters=1):
  """One batch of the restatement; returns the trainer after it."""
  tr = ref.Trainer(np.asarray(N, F32), np.asarray(E, F32), k, activation, loss)
  tr.batch(np.asarray(feats, np.int64).reshape(4 + 2 * k, -1), np.asarray(targets, F32).reshape(3, -1), clusters)
  return tr


def _adagrad(p, g):
  """one fresh Adagrad step in fp32 as compiled: acc = fma(g, g, 0)"""
  g = F32(g)
  acc = fma32(g, g, F32(0))
  return F32(p) - (ref.LR * g) / (np.sqrt(acc) + ref.EPS)


def _subnormal_pair(row, bs=2, pos=(0, 1)):
  """sigmoid / MSE, dim 1, k 0: sample A at batch position pos[0] (le 3, re 1) gives edge row 3
  d_ee * E[1], sample B at pos[1] (le 2, re 3) gives it d_ee * E[2] (row 0 instead of 3 when asked);
  E[3] = 0, so z = 0, p = 1/2, y = 0 and d_ee = ((2 * 1/2) * (1 / bs)) * 1/4 in both."""
  feats = np.zeros((4, bs), np.int64)
  feats[:, :] = [[4], [5], [4], [5]]         # fillers: ln = rn = 4, le = re = 5
  feats[:, pos[0]] = [4, 3, 4, 1]
  feats[:, pos[1]] = [4, 2, 4, 3]
  if row == 0:
    feats[:, pos[0]] = [4, 0, 4, 1]
    feats[:, pos[1]] = [4, 2, 4, 0]
  targets = np.zeros((3, bs), F32)
  return feats, targets


def test_a_subnormal_contribution_to_a_row_other_than_0_is_flushed():
  d = F32(0.5) * F32(0.25)                    # d_ee = ((2 * 0.5) * (1 / 2)) * 0.25
  E = np.zeros((6, 1), F32)
  E[1], E[2] = F32(0.5 * T) / d, F32(1.5 * T) / d    # contributions 0.5 T (subnormal) and 1.5 T
  E[5] = 0.5
  N = np.full((5, 1), 0.5, F32)
  feats, targets = _subnormal_pair(3)
  tr = _batch(N, E, feats, targets, activation="sigmoid")
  assert tr.E[3, 0] == _adagrad(0, F32(1.5 * T))
  assert tr.E[3, 0] != _adagrad(0, F32(2.0 * T))     # what an unflushed sum would give


@pytest.mark.parametrize("positions,clusters,same_cta", [
    ((0, 1), 1, True), ((0, 32), 1, False), ((0, 256), 1, True), ((0, 256), 2, False)])
def test_row_0_sums_plainly_inside_a_cta_and_flushes_per_cta(positions, clusters, same_cta):
  """Two subnormal contributions (0.5 T and 0.75 T) to row 0: one CTA adds them in shared memory
  without flushing and passes on the normal 1.25 T; two CTAs each flush theirs.  Position p runs
  on warp p mod (clusters * 256), CTA warp // 32."""
  bs = positions[1] + 1
  d = (F32(1) * (F32(1) / F32(bs))) * F32(0.25)
  E = np.zeros((6, 1), F32)
  E[1], E[2] = F32(0.5 * T) / d, F32(0.75 * T) / d
  a, b = d * E[1, 0], d * E[2, 0]
  assert 0 < a < T and 0 < b < T and a + b >= T
  E[5] = 0.5
  N = np.full((5, 1), 0.5, F32)
  feats, targets = _subnormal_pair(0, bs, positions)
  tr = _batch(N, E, feats, targets, activation="sigmoid", clusters=clusters)
  if same_cta:
    assert tr.E[0, 0] == _adagrad(0, a + b) and tr.E[0, 0] != 0
  else:
    assert tr.E[0, 0].view(np.uint32) == 0 and tr.gE[0, 0] == 0      # untouched: nothing reached g


def test_a_neighbour_with_da_0_is_skipped():
  """relu, k 1: the neighbour's pre-activation is negative, so da = 0: its row is left alone (table,
  accumulator and gradient) and ln's gradient is the direct term only."""
  N = np.array([[0.0, 0.0], [0.5, 0.25], [1.0, -0.5], [-1.0, -1.0]], F32)
  E = np.array([[0.0, 0.0], [0.5, 0.5], [0.25, 0.5], [1.0, 1.0]], F32)
  feats = [1, 1, 2, 2, 3, 3]                 # ln le rn re nn ne
  targets = [0.0, 0.0, 0.5]
  tr = _batch(N, E, feats, targets, k=1)
  assert np.array_equal(tr.N[3], N[3]) and not tr.accN[3].any() and not tr.gN[3].any()
  z = F32(0.5) * F32(1.0) + F32(0.25) * F32(-0.5)       # exact: 0.375
  d_nn = (F32(2) * z) * F32(1)
  assert np.array_equal(tr.N[1], [_adagrad(N[1, c], d_nn * N[2, c]) for c in range(2)])


@pytest.mark.parametrize("z,updated", [(2.0 ** -24, False), (0.5, True), (1.0, True), (2.0, False)])
def test_kl_clips_below_1e_7_and_above_1_and_keeps_1(z, updated):
  """relu / KL, dim 1: p = z.  The gradient -yc / pc flows for 1e-7 <= p <= 1 (p == 1 included, the
  boundary a `p < 1` would lose) and is zero outside, where the rows are left alone."""
  N = np.array([[0.0], [1.0], [z]], F32)
  E = np.array([[0.0], [0.5], [0.5]], F32)
  tr = _batch(N, E, [1, 1, 2, 2], [0.5, 0.0, 0.0], activation="relu", loss="kld")
  if updated:
    g = -F32(0.5) / F32(z)
    assert tr.N[1, 0] == _adagrad(1.0, g * F32(z)) and tr.N[2, 0] == _adagrad(z, g * F32(1))
  else:
    assert tr.N[1, 0] == 1.0 and tr.N[2, 0] == F32(z) and not tr.accN.any()


def test_relu_gradient_is_zero_at_z_0():
  """dyadic rows with an exactly zero dot product: relu'(0) = 0, so MSE's non-zero gradient stops"""
  N = np.array([[0.0, 0.0], [1.0, 1.0], [1.0, -1.0]], F32)
  E = np.array([[0.0, 0.0], [0.5, 0.5], [0.5, 0.5]], F32)
  tr = _batch(N, E, [1, 1, 2, 2], [0.5, 0.0, 0.0])
  assert np.array_equal(tr.N, N) and not tr.accN.any()


def test_elements_with_a_zero_gradient_are_left_alone():
  """ln's gradient is d_nn * Rn: the column where Rn is 0 keeps its value and its accumulator"""
  N = np.array([[0.0, 0.0, 0.0], [0.5, 0.5, 0.5], [1.0, 0.0, -1.0]], F32)
  N[1, 1] = -0.0
  E = np.array([[0.0, 0.0, 0.0], [0.5, 0.5, 0.5], [0.5, 0.5, 0.5]], F32)
  tr = _batch(N, E, [1, 1, 2, 2], [0.0, 0.0, 0.0])
  assert np.array_equal(tr.N, N)           # z = 0.5 + (-0) * 0 + 0.5 * -1 = 0: relu' = 0 ...
  N[2, 2] = -0.5                           # ... so make z > 0
  tr = _batch(N, E, [1, 1, 2, 2], [0.0, 0.0, 0.0])
  z = F32(0.5) * F32(1.0) + F32(0.5) * F32(-0.5)
  d = F32(2) * z
  assert tr.N[1, 0] == _adagrad(0.5, d * F32(1.0)) and tr.N[1, 2] == _adagrad(0.5, d * F32(-0.5))
  assert tr.N[1, 1].view(np.uint32) == np.float32(-0.0).view(np.uint32) and tr.accN[1, 1] == 0


def test_k_0_has_p_ne_0_and_its_loss_counts_y_squared():
  N = np.array([[0.0], [0.5], [0.5]], F32)
  E = np.array([[0.0], [0.5], [0.5]], F32)
  tr = ref.Trainer(N, E, 0, "relu", "mse")
  loss = tr.batch(np.array([[1], [1], [2], [2]]), np.array([[0.25], [0.25], [0.75]], F32))
  # z = 0.25 = y on both direct terms: no gradient; p_ne = fma(0, 0, -0.75)
  assert loss == float(F32(0.75) * F32(0.75))
  assert np.array_equal(tr.N, N) and np.array_equal(tr.E, E)


def test_heavy_duplication_is_summed_in_a_fixed_order():
  """More than two contributions per row: the restatement still sums all of them (its own order)."""
  g = np.zeros((3, 1), F32)
  ref._scatter_ftz(g, np.array([1, 2, 1, 1]), np.array([[1.0], [2.0], [3.0], [F32(0.25 * T)]], F32))
  assert g[1, 0] == 4.0 and g[2, 0] == 2.0
