"""The truncated SVD on the GPU (csrc/hge_svd.cu driven by hypergraphembedding_b200/svd.py): bit for
bit equal to the fp32 restatement of its operation order (oracle/svd_ref.py) at every k class of
the product kernel, for 1 to 10 iterations and the tol stop, host and device working arrays, an edge
of 120 000 members, empty rows and a rank-deficient incidence; within the fp32 bars of the float64
form of the same algorithm and of numpy's dense SVD; reproducible under other launch settings; its
refusals; and EmbedSVDDevice end to end."""
import numpy as np
import pytest
import scipy.sparse as sps

from conftest import hypergraph_from_pairs, load_golden
from hypergraphembedding_b200 import synthetic
from oracle import svd_ref as ref

pytestmark = pytest.mark.gpu

# l = k + 10 crosses every class of k_nmf_spmm (ld / 4 of 1 | 2 | 4 | 8 | 16 | 32 | 64 float4 lanes)
KS = [1, 2, 4, 5, 8, 9, 16, 17, 31, 32, 33, 64, 65, 128, 129, 200, 246, 256]


def _csr(A):
  A = sps.csr_matrix(A, dtype=np.float32)
  A.sum_duplicates()
  A.sort_indices()
  return A


def _graph(N, E, nnz, seed):
  return _csr(synthetic.power_law_hypergraph(N, E, nnz, seed=seed))


def _device(A, k, n_iter=5, oversamples=10, tol=0.0, seed=0, device=True, ctx=None):
  from hypergraphembedding_b200 import _native
  from hypergraphembedding_b200.algebraic_distance import make_incidence
  from hypergraphembedding_b200.svd import truncated_svd
  ctx = ctx or _native.default_context()
  inc = make_incidence(A, ctx=ctx)
  try:
    U, s, V, info = truncated_svd(ctx, inc, k, n_iter, oversamples, tol, seed, device=device)
    if device:
      U, V = U.cpu().numpy(), V.cpu().numpy()
    return np.ascontiguousarray(U), s, np.ascontiguousarray(V), info
  finally:
    inc.close()


def _oracle(A, k, n_iter=5, oversamples=10, tol=0.0, seed=0):
  B = _csr(A.T)
  return ref.fit32(A.indptr, A.indices, B.indptr, B.indices, A.shape[0], A.shape[1], k, n_iter, oversamples, tol,
                   seed)


def _same(got, want):
  U, s, V, info = got
  rU, rs, rV, rinfo = want
  assert info["n_iter"] == rinfo["n_iter"]
  assert np.array_equal(info["ritz_values"].view(np.uint64), rinfo["ritz_values"].view(np.uint64))
  assert np.array_equal(s.view(np.uint64), rs.view(np.uint64))
  assert np.array_equal(U.view(np.uint32), rU.view(np.uint32))
  assert np.array_equal(V.view(np.uint32), rV.view(np.uint32))
  assert np.array_equal(info["residuals"].view(np.uint64), rinfo["residuals"].view(np.uint64))


@pytest.mark.parametrize("k", KS)
def test_bit_exact_at_every_k(k):
  A = _graph(420, 300, 4000, seed=k)
  n_iter = 2 if k <= 65 else 1
  _same(_device(A, k, n_iter, seed=k), _oracle(A, k, n_iter, seed=k))


@pytest.mark.parametrize("n_iter,tol", [(1, 0.0), (3, 0.0), (10, 0.0), (60, 1e-7)])
@pytest.mark.parametrize("k", [5, 33])
def test_bit_exact_over_iterations_with_host_and_device_arrays(n_iter, tol, k):
  A = _graph(700, 400, 6000, seed=21)
  want = _oracle(A, k, n_iter, tol=tol, seed=4)
  if tol > 0:
    assert 2 < want[3]["n_iter"] < n_iter     # the tol rule ends the loop
  for device in (False, True):
    _same(_device(A, k, n_iter, tol=tol, seed=4, device=device), want)


def test_bit_exact_on_an_edge_of_120000_members():
  rng = np.random.default_rng(5)
  N, E = 120000, 40
  rows = np.concatenate([np.arange(N), rng.integers(0, N, 30000)])
  cols = np.concatenate([np.zeros(N, np.int64), rng.integers(1, E, 30000)])
  A = _csr(sps.csr_matrix((np.ones(len(rows)), (rows, cols)), shape=(N, E)) > 0)
  assert np.diff(_csr(A.T).indptr).max() >= 120000
  _same(_device(A, 9, 2, seed=6), _oracle(A, 9, 2, seed=6))


def test_bit_exact_with_empty_rows():
  rng = np.random.default_rng(8)
  A = np.zeros((40, 30), dtype=np.float32)
  A[rng.random((40, 30)) < 0.3] = 1
  A[3] = 0          # a node without edges
  A[:, 5] = 0       # an edge without members
  A = _csr(A)
  for k in (4, 20, 30):
    _same(_device(A, k, 3, seed=k), _oracle(A, k, 3, seed=k))


def test_rank_deficient_incidence_gives_zero_triplets():
  rng = np.random.default_rng(9)
  B = (rng.random((6, 5)) < 0.5).astype(np.float32)
  B[0, :] = 1
  rank = np.linalg.matrix_rank(B)
  A = _csr(np.kron(B, np.ones((30, 20), dtype=np.float32)))    # 180 x 100, rank <= 5
  k = 12
  got = _device(A, k, 4, seed=3)
  _same(got, _oracle(A, k, 4, seed=3))
  U, s, V, _ = got
  assert (s[:rank] > 0).all() and (s[rank:] == 0).all()
  assert (U[:, rank:] == 0).all() and (V[:, rank:] == 0).all()
  np.testing.assert_allclose(s[:rank], np.linalg.svd(A.toarray().astype(np.float64), compute_uv=False)[:rank],
                             rtol=1e-5)


def _sin_max_angle(X, Y):
  qx, _ = np.linalg.qr(X)
  qy, _ = np.linalg.qr(Y)
  c = np.linalg.svd(qx.T @ qy, compute_uv=False)
  return float(np.sqrt(max(0.0, 1.0 - c.min() ** 2)))


@pytest.mark.parametrize("k", [8, 32])
@pytest.mark.parametrize("n_iter", [5, 50])
def test_close_to_the_float64_form_and_to_numpy(k, n_iter):
  A = _graph(4000, 8000, 120000, seed=1234)
  N, E = A.shape
  U, s, V, info = _device(A, k, n_iter, seed=1)
  l = info["block_width"]
  U64, s64, V64, info64 = ref.fit64(A, k, ref.start(E, l, 1)[:, :l], n_iter=n_iter)
  ritz = info64["ritz_values"][-1]
  gap = (ritz[k - 1] - ritz[k]) / ritz[k - 1]
  ds = float(np.abs(s - s64).max() / s64[0])
  sin_u, sin_v = _sin_max_angle(U.astype(np.float64), U64), _sin_max_angle(V.astype(np.float64), V64)
  ou = float(np.abs(U.T.astype(np.float64) @ U - np.eye(k)).max())
  ov = float(np.abs(V.T.astype(np.float64) @ V - np.eye(k)).max())
  dr = float(np.abs(info["residuals"] - info64["residuals"]).max())
  print("k %d, %d iterations: sigma %.2e sigma_1, gap %.2e, sin U %.2e, sin V %.2e, orthonormality %.2e / %.2e, "
        "residuals %.2e" % (k, n_iter, ds, gap, sin_u, sin_v, ou, ov, dr))
  assert ds <= 1e-5 and ou <= 1e-4 and ov <= 1e-4 and dr <= 1e-4
  assert gap > 1e-3, "pick a graph seed with a gap between Ritz values k and k + 1"
  assert sin_u <= 1e-3 and sin_v <= 1e-3
  # numpy's dense SVD, for the triplets the float64 form has converged
  Ud, sd, Vdt = np.linalg.svd(A.toarray().astype(np.float64), full_matrices=False)
  conv = np.flatnonzero(info64["residuals"] <= 1e-8)
  print("converged triplets: %d of %d" % (len(conv), k))
  assert np.abs(s[conv] - sd[conv]).max(initial=0.0) <= 1e-5 * sd[0]
  for i in conv:
    lo = sd[i - 1] if i > 0 else np.inf
    if (lo - sd[i]) / sd[i] > 1e-3 and (sd[i] - sd[i + 1]) / sd[i] > 1e-3:
      assert abs(float(U[:, i].astype(np.float64) @ Ud[:, i])) >= 1 - 1e-3
      assert abs(float(V[:, i].astype(np.float64) @ Vdt[i])) >= 1 - 1e-3


def test_reproducible_under_other_launch_settings():
  from hypergraphembedding_b200 import _native
  A = _graph(5000, 3000, 60000, seed=3)
  first = _device(A, 24, 4, seed=2)
  _same(_device(A, 24, 4, seed=2), first)
  _same(_device(A, 24, 4, seed=2, device=False), first)
  ctx = _native.Context(0)
  try:
    for per_sm in (1, 32):
      ctx.set_tuning(blocks_per_sm=per_sm)
      _same(_device(A, 24, 4, seed=2, ctx=ctx), first)
  finally:
    ctx.close()


def test_seeded_start_equals_the_restatement():
  import torch
  from hypergraphembedding_b200 import _native
  ctx = _native.default_context()
  for E, l, seed in ((37, 1, 0), (300, 33, 2 ** 40 + 7), (1000, 256, 5)):
    want = ref.start(E, l, seed)
    host = np.full((E, _native.svd_ld(l)), 7, dtype=np.float32)
    _native.svd_start(ctx, E, l, seed, host)
    assert np.array_equal(host.view(np.uint32), want.view(np.uint32))
    dev = torch.full((E, _native.svd_ld(l)), 7.0, device="cuda")
    _native.svd_start(ctx, E, l, seed, dev)
    assert np.array_equal(dev.cpu().numpy().view(np.uint32), want.view(np.uint32))


def test_refusals():
  from hypergraphembedding_b200 import TruncatedSVDDevice, _native
  from hypergraphembedding_b200.algebraic_distance import make_incidence
  A = _graph(60, 40, 400, seed=1)
  ctx = _native.default_context()
  inc = make_incidence(A, ctx=ctx)
  try:
    l, ld = 8, 8
    rng = np.random.default_rng(0)
    xe, xn = rng.random((40, ld), dtype=np.float32), rng.random((60, ld), dtype=np.float32)

    def refused(fn, *arrays):
      before = [a.copy() for a in arrays]
      with pytest.raises(AssertionError):
        fn()
      for a, b in zip(arrays, before):
        assert np.array_equal(a, b)

    y = np.full((60, ld), 3.0, np.float32)
    y4 = np.full((60, 4), 3.0, np.float32)
    refused(lambda: _native.svd_half(ctx, inc, 0, 0, np.zeros((40, 4), np.float32), y4), y4)
    refused(lambda: _native.svd_half(ctx, inc, 0, 257, np.zeros((40, 260), np.float32),
                                     np.zeros((60, 260), np.float32)))
    refused(lambda: _native.svd_half(ctx, inc, 2, l, xe, y), y)
    refused(lambda: _native.svd_half(ctx, inc, 0, l, xe[:39], y), y)           # edge rows
    refused(lambda: _native.svd_half(ctx, inc, 0, l, xe, np.ascontiguousarray(y[:59])))
    refused(lambda: _native.svd_half(ctx, inc, 1, l, xn[:59], np.zeros((40, ld), np.float32)))
    out = np.full((60, ld), 5.0, np.float32)
    refused(lambda: _native.svd_rowmat(ctx, l, xn, np.ones((l, l + 1), np.float32), out), out)
    refused(lambda: _native.svd_rowmat(ctx, l, xn, np.ones((l, 0), np.float32), out), out)
    u, v = xn.copy(), xe.copy()
    refused(lambda: _native.svd_flip(ctx, l, 0, u, v), u, v)
    refused(lambda: _native.svd_flip(ctx, l, l + 1, u, v), u, v)
    refused(lambda: _native.svd_residuals(ctx, inc, l, l + 1, u, v, np.ones(l + 1)), u, v)
    refused(lambda: _native.svd_residuals(ctx, inc, l, 4, u[:59], v, np.ones(4)))
    refused(lambda: _native.svd_start(ctx, 40, 0, 0, np.zeros((40, 0), np.float32)))
  finally:
    inc.close()
  # a sharded incidence
  shard = _native.Incidence(ctx, 60, 40, A.indptr, A.indices, _csr(A.T).indptr, _csr(A.T).indices, sharded=True)
  try:
    y = np.full((60, 8), 3.0, np.float32)
    with pytest.raises(AssertionError):
      _native.svd_half(ctx, shard, 0, 8, np.zeros((40, 8), np.float32), y)
    assert (y == 3).all()
  finally:
    shard.close()
  for kwargs in ({"k": 0}, {"k": 41}, {"k": 4, "n_iter": 0}, {"k": 4, "oversamples": -1},
                 {"k": 4, "tol": float("nan")}):
    with pytest.raises(AssertionError):
      TruncatedSVDDevice(A, **kwargs)


def _youtube():
  g = load_golden("algdist_youtube")
  node_ids, edge_ids = g["node_ids"], g["edge_ids"]
  return hypergraph_from_pairs(np.stack([node_ids[np.searchsorted(node_ids, g["pairs"][:, 0])],
                                         edge_ids[np.searchsorted(edge_ids, g["pairs"][:, 1])]], axis=1))


@pytest.mark.parametrize("dim", [8, 16])
def test_embed_svd_device_end_to_end(dim):
  import hypergraphembedding_b200 as H
  from hypergraphembedding_b200.hypergraph_util import compressed_incidence
  hg = _youtube()
  np.random.seed(0)
  state = np.random.get_state()
  emb = H.EmbedSVDDevice(hg, dim, seed=5)
  after = np.random.get_state()
  assert after[2] == state[2] and np.array_equal(after[1], state[1])
  assert emb.method_name == "SVD" and emb.dim == dim
  assert sorted(emb.node) == sorted(hg.node) and sorted(emb.edge) == sorted(hg.edge)
  node_ids, edge_ids, A = compressed_incidence(hg)
  xn = np.asarray([emb.node[int(i)].values for i in node_ids], dtype=np.float32)
  xe = np.asarray([emb.edge[int(i)].values for i in edge_ids], dtype=np.float32)
  U, s, Vt, _ = H.TruncatedSVDDevice(A, dim, seed=5)
  assert np.array_equal(xn.view(np.uint32), U.view(np.uint32))
  assert np.array_equal(xe.view(np.uint32), np.ascontiguousarray(Vt.T).view(np.uint32))
  live = s > 0
  assert live.any()
  assert np.allclose(np.linalg.norm(xn[:, live].astype(np.float64), axis=0), 1, atol=1e-4)
  assert np.allclose(np.linalg.norm(xe[:, live].astype(np.float64), axis=0), 1, atol=1e-4)
  assert H.EmbedSVDDevice not in H.EMBEDDING_OPTIONS.values()
