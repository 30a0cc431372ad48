"""The non-negative factorization on the GPU (csrc/hge_nmf.cu): bit for bit equal to the fp32
restatement of its operation order (oracle/nmf_ref.py) at every k class of the product kernel, for
1 to 200 iterations, host and device factors, a row of more than 100 000 incidences, empty rows and
k > min(N, E); close to scikit-learn's float64 run from the same start; reproducible under other
launch settings; its refusals; and EmbedNMFDevice end to end."""
import numpy as np
import pytest
import scipy.sparse as sps

from conftest import hypergraph_from_pairs, load_golden
from hypergraphembedding_b200 import synthetic
from oracle import nmf_ref as ref

pytestmark = pytest.mark.gpu

# k classes of k_nmf_spmm: lanes per row 1 | 2 | 4 | 8 | 16 | 32 | 32 x 2 slabs, split at these k
BOUNDARIES = [4, 5, 8, 9, 16, 17, 32, 33, 64, 65, 128, 129, 256]
KS = sorted(set([1, 2, 31, 32, 33, 64, 65, 128, 200, 256] + BOUNDARIES))


def _csr(A):
  A = sps.csr_matrix(A, dtype=np.float32)
  A.sum_duplicates()
  A.sort_indices()
  return A


def _graph(N, E, nnz, seed):
  return _csr(synthetic.power_law_hypergraph(N, E, nnz, seed=seed))


def _start(A, k, seed=3):
  from hypergraphembedding_b200.nmf import start_scale
  N, E = A.shape
  return ref.start(N, E, k, seed, start_scale(N, E, A.nnz, k))


def _device(A, W0, Ht0, max_iter, tol, on_device=False, ctx=None):
  from hypergraphembedding_b200 import _native
  from hypergraphembedding_b200.algebraic_distance import make_incidence
  ctx = ctx or _native.default_context()
  inc = make_incidence(A, ctx=ctx)
  try:
    if on_device:
      import torch
      W = torch.from_numpy(W0.copy()).cuda()
      Ht = torch.from_numpy(Ht0.copy()).cuda()
      it, viols = _native.nmf_fit(ctx, inc, W, Ht, max_iter, tol)
      return W.cpu().numpy(), Ht.cpu().numpy(), it, viols
    W, Ht = W0.copy(), Ht0.copy()
    it, viols = _native.nmf_fit(ctx, inc, W, Ht, max_iter, tol)
    return W, Ht, it, viols
  finally:
    inc.close()


def _oracle(A, W0, Ht0, max_iter, tol):
  B = _csr(A.T)
  return ref.fit32(A.indptr, A.indices, B.indptr, B.indices, W0, Ht0, max_iter, tol)


def _same(got, want):
  W, Ht, it, viols = got
  rW, rHt, rit, rviols = want
  assert it == rit
  assert np.array_equal(viols, rviols), (viols, rviols)
  assert np.array_equal(W.view(np.uint32), rW.view(np.uint32))
  assert np.array_equal(Ht.view(np.uint32), rHt.view(np.uint32))


@pytest.mark.parametrize("k", KS)
def test_bit_exact_at_every_k(k):
  A = _graph(150, 90, 1200, seed=k)
  W0, Ht0 = _start(A, k, seed=k)
  iters = 2 if k <= 65 else 1
  _same(_device(A, W0, Ht0, iters, 0.0), _oracle(A, W0, Ht0, iters, 0.0))


@pytest.mark.parametrize("max_iter,tol", [(1, 0.0), (3, 0.0), (20, 0.0), (200, 1e-4)])
@pytest.mark.parametrize("k", [5, 33])
def test_bit_exact_over_iterations_with_host_and_device_factors(max_iter, tol, k):
  A = _graph(700, 400, 6000, seed=21)
  W0, Ht0 = _start(A, k, seed=4)
  want = _oracle(A, W0, Ht0, max_iter, tol)
  if tol > 0:
    assert 3 < want[2] < max_iter     # the stop rule ends the fit (81 iterations at k 5, 138 at k 33)
  for on_device in (False, True):
    _same(_device(A, W0, Ht0, max_iter, tol, on_device), want)


def test_bit_exact_on_a_row_of_more_than_100000_incidences():
  rng = np.random.default_rng(5)
  N, E = 120000, 40
  rows = np.concatenate([np.arange(N), rng.integers(0, N, 30000)])
  cols = np.concatenate([np.zeros(N, np.int64), rng.integers(1, E, 30000)])
  A = _csr(sps.csr_matrix((np.ones(len(rows)), (rows, cols)), shape=(N, E)) > 0)
  assert np.diff(_csr(A.T).indptr).max() >= 100000
  W0, Ht0 = _start(A, 9, seed=6)
  _same(_device(A, W0, Ht0, 2, 0.0), _oracle(A, W0, Ht0, 2, 0.0))


def test_bit_exact_with_empty_rows_and_k_above_min_n_e():
  A = np.zeros((12, 7), dtype=np.float32)
  rng = np.random.default_rng(8)
  A[rng.random((12, 7)) < 0.4] = 1
  A[3] = 0          # a node without edges
  A[:, 5] = 0       # an edge without members
  A = _csr(A)
  for k in (10, 33):
    W0, Ht0 = _start(A, k, seed=k)
    _same(_device(A, W0, Ht0, 5, 0.0), _oracle(A, W0, Ht0, 5, 0.0))


def test_bit_exact_with_an_all_zero_component():
  A = _graph(300, 200, 3000, seed=2)
  W0, Ht0 = _start(A, 6, seed=1)
  W0[:, 2] = 0      # G[2, 2] == 0 in the H half of the first iteration
  Ht0[:, 4] = 0     # and G[4, 4] == 0 in its W half
  _same(_device(A, W0, Ht0, 3, 0.0), _oracle(A, W0, Ht0, 3, 0.0))


def _sklearn(A, W0, H0, k, max_iter, tol):
  import warnings
  from sklearn.decomposition import non_negative_factorization
  with warnings.catch_warnings():
    warnings.simplefilter("ignore")
    return non_negative_factorization(A.astype(np.float64), W=W0.astype(np.float64), H=H0.astype(np.float64),
                                      n_components=k, init="custom", solver="cd", max_iter=max_iter, tol=tol)


def _rel(a, b):
  return float(np.linalg.norm(np.asarray(a, np.float64) - b) / np.linalg.norm(b))


@pytest.mark.parametrize("k", [8, 32])
def test_close_to_scikit_learn_float64(k):
  from hypergraphembedding_b200 import NonNegativeFactorizationDevice
  A = _graph(3942, 8000, 114297, seed=1234)
  W0, Ht0 = _start(A, k, seed=9)
  H0 = np.ascontiguousarray(Ht0.T)
  for T in (1, 5, 20):
    W, H, _ = _sklearn(A, W0, H0, k, T, 0.0)
    Wd, Hd, it = NonNegativeFactorizationDevice(A, k, W=W0, H=H0, max_iter=T, tol=0.0)
    dw, dh = _rel(Wd, W), _rel(Hd, H)
    print("k %d after %d iterations: W %.2e, H %.2e relative" % (k, T, dw, dh))
    assert it == T and dw < 2e-3 and dh < 2e-3
  W, H, it = _sklearn(A, W0, H0, k, 200, 1e-4)
  Wd, Hd, itd = NonNegativeFactorizationDevice(A, k, W=W0, H=H0)
  X = A.toarray().astype(np.float64)
  err, errd = np.linalg.norm(X - W @ H), np.linalg.norm(X - Wd.astype(np.float64) @ Hd)
  print("k %d default stop: n_iter %d (scikit-learn %d), reconstruction error %.2e relative" %
        (k, itd, it, abs(errd - err) / err))
  assert abs(itd - it) <= 1 and abs(errd - err) / err < 1e-4


def test_reproducible_under_other_launch_settings():
  from hypergraphembedding_b200 import _native
  A = _graph(5000, 3000, 60000, seed=3)
  W0, Ht0 = _start(A, 24, seed=2)
  first = _device(A, W0, Ht0, 4, 0.0)
  _same(_device(A, W0, Ht0, 4, 0.0), first)
  _same(_device(A, W0, Ht0, 4, 0.0, on_device=True), first)
  ctx = _native.Context(0)
  try:
    for per_sm in (1, 32):
      ctx.set_tuning(blocks_per_sm=per_sm)
      _same(_device(A, W0, Ht0, 4, 0.0, ctx=ctx), first)
  finally:
    ctx.close()


def test_seeded_start_equals_the_restatement():
  import torch
  from hypergraphembedding_b200 import _native
  from hypergraphembedding_b200.nmf import seeded_start, start_scale
  for N, E, k, seed in ((37, 11, 1, 0), (300, 200, 33, 2 ** 40 + 7), (10, 1000, 256, 5)):
    scale = start_scale(N, E, 500, k)
    W, Ht = seeded_start(N, E, 500, k, seed)
    rW, rHt = ref.start(N, E, k, seed, scale)
    assert np.array_equal(W.view(np.uint32), rW.view(np.uint32))
    assert np.array_equal(Ht.view(np.uint32), rHt.view(np.uint32))
    Wd = torch.empty((N, k), dtype=torch.float32, device="cuda")
    Hd = torch.empty((E, k), dtype=torch.float32, device="cuda")
    _native.nmf_init(_native.default_context(), N, E, k, seed, scale, Wd, Hd)
    assert np.array_equal(Wd.cpu().numpy().view(np.uint32), rW.view(np.uint32))
    assert np.array_equal(Hd.cpu().numpy().view(np.uint32), rHt.view(np.uint32))


def test_refusals():
  from hypergraphembedding_b200 import _native
  from hypergraphembedding_b200.algebraic_distance import make_incidence
  A = _graph(60, 40, 400, seed=1)
  ctx = _native.default_context()
  inc = make_incidence(A, ctx=ctx)
  try:
    W0, Ht0 = _start(A, 4)

    def fit(W=W0, Ht=Ht0, max_iter=5, tol=1e-4):
      W, Ht = W.copy(), Ht.copy()
      before = (W.copy(), Ht.copy())
      with pytest.raises(AssertionError):
        _native.nmf_fit(ctx, inc, W, Ht, max_iter, tol)
      assert np.array_equal(W, before[0], equal_nan=True) and np.array_equal(Ht, before[1], equal_nan=True)

    for k in (0, 257):
      fit(np.ones((60, k), np.float32), np.ones((40, k), np.float32))
    fit(max_iter=0)
    fit(tol=-1e-9)
    fit(tol=float("nan"))
    for bad in (-1.0, float("nan"), float("inf")):
      W = W0.copy()
      W[7, 1] = bad
      fit(W=W)
      Ht = Ht0.copy()
      Ht[3, 2] = bad
      fit(Ht=Ht)
    fit(W=np.zeros_like(W0))
    fit(Ht=np.zeros_like(Ht0))
    fit(W=np.ones((61, 4), np.float32))
    fit(Ht=np.ones((39, 4), np.float32))
    with pytest.raises(AssertionError):
      _native.nmf_init(ctx, 60, 40, 0, 0, 1.0, np.zeros((60, 0), np.float32), np.zeros((40, 0), np.float32))
  finally:
    inc.close()
  from hypergraphembedding_b200 import NonNegativeFactorizationDevice
  with pytest.raises(AssertionError):
    NonNegativeFactorizationDevice(A, 4, W=W0)


def _youtube():
  g = load_golden("algdist_youtube")
  node_ids, edge_ids = g["node_ids"], g["edge_ids"]
  return hypergraph_from_pairs(np.stack([node_ids[np.searchsorted(node_ids, g["pairs"][:, 0])],
                                         edge_ids[np.searchsorted(edge_ids, g["pairs"][:, 1])]], axis=1))


@pytest.mark.parametrize("dim", [8, 16])
def test_embed_nmf_device_end_to_end(dim):
  import hypergraphembedding_b200 as H
  from hypergraphembedding_b200.hypergraph_util import compressed_incidence
  hg = _youtube()
  np.random.seed(0)
  state = np.random.get_state()
  emb = H.EmbedNMFDevice(hg, dim, seed=5)
  after = np.random.get_state()
  assert after[2] == state[2] and np.array_equal(after[1], state[1])
  assert emb.method_name == "NMF" and emb.dim == dim
  assert sorted(emb.node) == sorted(hg.node) and sorted(emb.edge) == sorted(hg.edge)
  node_ids, edge_ids, A = compressed_incidence(hg)
  xn = np.asarray([emb.node[int(i)].values for i in node_ids], dtype=np.float32)
  xe = np.asarray([emb.edge[int(i)].values for i in edge_ids], dtype=np.float32)
  assert np.isfinite(xn).all() and np.isfinite(xe).all() and (xn >= 0).all() and (xe >= 0).all()
  W, Hm, _ = H.NonNegativeFactorizationDevice(A, dim, seed=5)
  assert np.array_equal(xn.view(np.uint32), W.view(np.uint32))
  assert np.array_equal(xe.view(np.uint32), np.ascontiguousarray(Hm.T).view(np.uint32))
  assert H.EmbedNMFDevice not in H.EMBEDDING_OPTIONS.values()
