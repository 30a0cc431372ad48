"""Every device buffer a call allocates for itself is released on its error paths too.

HGE_FAIL_ALLOC_AT = n makes the n-th device allocation of a context after hge_ctx_reset_tuning
fail with HGE_ERR_NOMEM.  For n = 1, 2, ... each call below (with everything it needs built inside
the attempt) raises MemoryError until n passes its number of allocations; after every attempt,
once its objects are closed, the used memory of the device's default pool (which the library
allocates from with cudaMallocAsync) is back at what it was before, and the run that gets through
returns what a run without the countdown returns."""
import ctypes
import gc
import os

import numpy as np
import pytest
import scipy.sparse as sps

pytestmark = pytest.mark.gpu

ENV = "HGE_FAIL_ALLOC_AT"
USED_MEM_CURRENT = 7   # CU_MEMPOOL_ATTR_USED_MEM_CURRENT


class _Pool(object):
  def __init__(self, device):
    self.cu = ctypes.CDLL("libcuda.so.1")
    dev = ctypes.c_int()
    assert self.cu.cuDeviceGet(ctypes.byref(dev), device) == 0
    self.pool = ctypes.c_void_p()
    assert self.cu.cuDeviceGetDefaultMemPool(ctypes.byref(self.pool), dev) == 0

  def used(self):
    import torch
    torch.cuda.synchronize()
    v = ctypes.c_uint64(0)
    assert self.cu.cuMemPoolGetAttribute(self.pool, USED_MEM_CURRENT, ctypes.byref(v)) == 0
    return int(v.value)


def _graph(nodes=300, edges=80, per_edge=12, seed=0):
  rng = np.random.default_rng(seed)
  rows = np.concatenate([rng.choice(nodes, per_edge, replace=False) for _ in range(edges)])
  cols = np.repeat(np.arange(edges), per_edge)
  rows, cols = np.r_[rows, np.arange(nodes)], np.r_[cols, np.arange(nodes) % edges]   # no empty node
  A = sps.csr_matrix((np.ones(len(rows), dtype=bool), (rows, cols)), shape=(nodes, edges))
  A.sum_duplicates()
  A.sort_indices()
  return A


def _csr(m):
  m = sps.csr_matrix(m)
  return m.indptr.astype(np.int64), m.indices.astype(np.int32)


def _incidence(ctx, A, e2n=True):
  from hypergraphembedding_b200 import _native
  a = _csr(A)
  b = _csr(A.T) if e2n else (None, None)
  return _native.Incidence(ctx, A.shape[0], A.shape[1], a[0], a[1], b[0], b[1])


def _vectors(rows, R, seed):
  return np.random.default_rng(seed).standard_normal((rows, R)).astype(np.float32)


def _host(x):
  if x is None:
    return None
  if isinstance(x, (tuple, list)):
    return [_host(v) for v in x]
  if hasattr(x, "cpu"):
    return x.cpu().numpy()
  return np.asarray(x)


def _with_incidence(ctx, A, body, e2n=True):
  inc = _incidence(ctx, A, e2n)
  try:
    return body(inc)
  finally:
    inc.close()


def _cases(ctx):
  """name -> a call that builds what it needs, runs, closes its objects and returns host arrays"""
  import torch
  from hypergraphembedding_b200 import _native, synthetic
  from hypergraphembedding_b200.hg2v_sample import BooleanSamplesDevice
  from hypergraphembedding_b200.hg2v_model import Hg2vModel
  dev = torch.device("cuda", ctx.device)
  A = _graph()
  N, E = A.shape
  rng = np.random.default_rng(5)
  d_ptr, d_idx = (torch.from_numpy(v).to(dev) for v in _csr(A))
  F = sps.random(N, 40, density=0.2, format="csr", dtype=np.float32, random_state=7)
  feat = _native.FeatureCsr(F)
  feat_dev = feat.to_device(dev)
  # enough features per group that a 1 MB workspace takes several batches
  F_wide = sps.random(N, 1000, density=0.1, format="csr", dtype=np.float32, random_state=8)
  wide_dev = _native.FeatureCsr(F_wide).to_device(dev)
  pairs_n, pairs_e = rng.integers(0, N, 400), rng.integers(0, E, 400)
  t_nodes, t_edges = (torch.from_numpy(v.astype(np.int32)).to(dev) for v in (pairs_n, pairs_e))
  vectors = torch.from_numpy(_vectors(N, 8, 3)).to(dev)
  tiled = synthetic.power_law_hypergraph(20000, 200, 80000, seed=3, max_edge_size=4000)
  xn_t, xe_t = synthetic.legacy_initial_vectors(tiled.shape[0], tiled.shape[1], 32, seed=1)

  def incidence(e2n=True, device=False):
    def run():
      if device:
        inc = _native.Incidence(ctx, N, E, d_ptr, d_idx)
      else:
        inc = _incidence(ctx, A, e2n)
      try:
        return inc.nnz
      finally:
        inc.close()
    return run

  def algdist(B, xn0, xe0, iters, tile):
    def body(inc):
      xn, xe = xn0.copy(), xe0.copy()
      _native.algdist_run(ctx, inc, xn, xe, iters)
      return xn, xe

    def run():
      if tile:
        ctx.set_tile_mb(1, 0)   # 1 MB = 8192 rows of 32 floats: 3 tiles of the 20 000 nodes
      return _with_incidence(ctx, B, body)
    return run

  def on_incidence(body):
    return lambda: _with_incidence(ctx, A, body)

  def with_host_values(fn):
    values = _vectors(1, 500, 9).ravel()
    return lambda: fn(values.copy())

  def model(kind):
    m_rng = np.random.default_rng(6)
    feats = [m_rng.integers(1, (N if c in (0, 2, 4, 5) else E) + 1, 500).astype(np.int32) for c in range(8)]
    targets = [m_rng.random(500).astype(np.float32) for _ in range(3)]

    def run():
      m = Hg2vModel.seeded(N, E, 8, 2, "relu", "mean_squared_error", 11)
      try:
        if kind == "host":
          m.set_samples(feats, targets)
          m.fit_epoch(np.arange(m.num_samples)[::-1], 64)
        else:
          m.fit_device(BooleanSamplesDevice(A, 2, 4, neg_samples=1, seed=3, keep_on_device=True),
                       batch_size=64, epochs=2, seed=5, verbose=0)
        return m.weights()
      finally:
        m.close()
    return run

  def arena():
    a = _native.PeerArena(ctx, 0, 1, N, E, 8)
    try:
      a.open_peers(np.zeros(64, np.uint8))
    finally:
      a.close()

  xn3, xe3, xn4, xe4 = _vectors(N, 3, 1), _vectors(E, 3, 2), _vectors(N, 4, 1), _vectors(E, 4, 2)
  w_n2e = np.random.default_rng(4).random(A.nnz).astype(np.float32)
  ia, ib = rng.integers(0, N, 500), rng.integers(0, N, 500)
  groups = _native.CsrArrays(A.T.tocsr())
  samples = np.full(N, 3)
  return {
      "incidence_host": incidence(),
      "incidence_host_without_e2n": incidence(e2n=False),
      "incidence_device": incidence(device=True),
      "algdist_run": algdist(A, _vectors(N, 8, 1), _vectors(E, 8, 2), 3, False),
      "algdist_run_edge_tiles": algdist(tiled, xn_t, xe_t, 2, True),
      "incidence_l2_R3": on_incidence(lambda inc: _native.incidence_l2(ctx, inc, xn3, xe3, order=1)),
      "incidence_l2_R4": on_incidence(lambda inc: _native.incidence_l2(ctx, inc, xn4, xe4, order=0)),
      "pair_l2": lambda: _native.pair_l2(ctx, xn3, _vectors(N, 3, 7), ia, ib),
      "pair_l2_xb_is_xa": lambda: _native.pair_l2(ctx, xn3, xn3, ia, ib),
      "scale_transform": with_host_values(lambda v: _native.scale_transform(ctx, v, 0.25, want_minmax=True)),
      "scale_minmax": with_host_values(lambda v: _native.scale_minmax(ctx, v)),
      "scale_apply": with_host_values(lambda v: _native.scale_apply(ctx, v, 0.25, -1.0, 2.0)),
      "row_span": on_incidence(lambda inc: _native.row_span(ctx, inc, xn3, xe3, 1)),
      "same_type_prob": on_incidence(lambda inc: _native.same_type_prob(ctx, inc, 0, w_n2e, ia, ib)),
      "diff_type_prob": on_incidence(lambda inc: _native.diff_type_prob(ctx, inc, w_n2e, pairs_n, pairs_e)),
      "jaccard_rows": lambda: _native.jaccard_rows(ctx, feat, ia, ib),
      "jaccard_centroid": lambda: _native.jaccard_centroid(ctx, feat, groups, feat, pairs_n, pairs_e),
      "jaccard_centroid_grouped": on_incidence(lambda inc: _native.jaccard_centroid_grouped(
          ctx, inc, 1, wide_dev, wide_dev, t_nodes, t_edges, workspace_mb=1)),
      "jaccard_centroid_grouped_small": on_incidence(lambda inc: _native.jaccard_centroid_grouped(
          ctx, inc, 1, feat_dev, feat_dev, t_nodes, t_edges)),
      "sample_pairs_1": on_incidence(lambda inc: _native.sample_pairs_device(ctx, inc, 0, 1, 0, samples, 7, 1)),
      "sample_pairs_2": on_incidence(lambda inc: _native.sample_pairs_device(ctx, inc, 1, 2, 0, samples[:E], 7, 2)),
      "sample_pairs_3": on_incidence(lambda inc: _native.sample_pairs_device(ctx, inc, 0, 3, 0, samples, 7, 3)),
      "sample_pairs_negative": on_incidence(
          lambda inc: _native.sample_pairs_device(ctx, inc, 0, 1, 0, samples, 7, 6, negative=True)),
      "sample_neighbors": on_incidence(
          lambda inc: _native.sample_neighbors_device(ctx, inc, t_nodes, t_edges, 3, 7, 5, 0)),
      "shuffle_order": lambda: _native.shuffle_order(ctx, 3, 1, 1000),
      "hg2v_seeded_set_samples_fit_epoch": model("host"),
      "hg2v_seeded_fit_device": model("device"),
      "lp_svm_predict": on_incidence(lambda inc: _native.lp_svm_predict(ctx, inc, 1, vectors, t_nodes, t_edges,
                                                                         9)[:2]),
      "peer_arena_open_peers": arena,
  }


_CASES = {}


@pytest.fixture(scope="module")
def cases(gpu_ctx):
  import torch
  if torch.cuda.get_allocator_backend() != "native":
    pytest.skip("torch allocates from the same stream-ordered pool")
  if not _CASES:
    _CASES.update(_cases(gpu_ctx))
  return _CASES


NAMES = ["incidence_host", "incidence_host_without_e2n", "incidence_device", "algdist_run",
         "algdist_run_edge_tiles", "incidence_l2_R3", "incidence_l2_R4", "pair_l2", "pair_l2_xb_is_xa",
         "scale_transform", "scale_minmax", "scale_apply", "row_span", "same_type_prob", "diff_type_prob",
         "jaccard_rows", "jaccard_centroid", "jaccard_centroid_grouped", "jaccard_centroid_grouped_small",
         "sample_pairs_1", "sample_pairs_2", "sample_pairs_3", "sample_pairs_negative", "sample_neighbors",
         "shuffle_order", "hg2v_seeded_set_samples_fit_epoch", "hg2v_seeded_fit_device", "lp_svm_predict",
         "peer_arena_open_peers"]


def _set_countdown(ctx, n):
  if n:
    os.environ[ENV] = str(n)
  else:
    os.environ.pop(ENV, None)
  ctx.reset_tuning()


@pytest.mark.parametrize("name", NAMES)
def test_failed_allocations_release_every_buffer(name, cases, gpu_ctx):
  assert sorted(NAMES) == sorted(cases)
  call = cases[name]
  pool = _Pool(gpu_ctx.device)
  gc.collect()
  gc.disable()
  try:
    base = pool.used()
    _set_countdown(gpu_ctx, 0)
    want = _host(call())
    assert pool.used() == base, "%s leaks without a failure" % name
    n = 0
    while True:
      n += 1
      _set_countdown(gpu_ctx, n)
      try:
        got = _host(call())
      except MemoryError:
        assert pool.used() == base, "%s: %d bytes left after allocation %d failed" % (
            name, pool.used() - base, n)
        continue
      assert pool.used() == base
      break
  finally:
    _set_countdown(gpu_ctx, 0)
    gc.enable()
  assert n > 1, "%s allocates nothing" % name
  if name.startswith("hg2v"):
    # the epochs add duplicated rows' gradients with atomics: equal up to fp32 summation order
    for g, w in zip(got, want):
      assert np.allclose(g, w, rtol=0, atol=1e-6)
  elif want is not None:
    for g, w in zip(got if isinstance(got, list) else [got], want if isinstance(want, list) else [want]):
      assert np.array_equal(g, w, equal_nan=True), name
