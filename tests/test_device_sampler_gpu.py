"""BooleanSamplesDevice / AlgebraicDistanceSamplesDevice (csrc/hge_device_sampler.cu): bit-equal to
the numpy restatement (oracle/device_sampler_ref.py), structurally right at 100 000 nodes, and
independent of batching, chunking and the workspace budget."""
import numpy as np
import pytest
import scipy.sparse as sps

from conftest import load_golden
from oracle import device_sampler_ref as ref

pytestmark = pytest.mark.gpu

INDEX = ("left_node", "left_edge", "right_node", "right_edge", "neigh_node", "neigh_edge",
         "has_neighbors")
PROBS = ("nn_prob", "ee_prob", "ne_prob")


def _dense_csr(pairs):
  pairs = np.asarray(pairs)
  n = np.unique(pairs[:, 0], return_inverse=True)[1]
  e = np.unique(pairs[:, 1], return_inverse=True)[1]
  m = sps.csr_matrix((np.ones(len(n), dtype=bool), (n, e)), dtype=bool)
  m.sum_duplicates()
  m.sort_indices()
  return m


def _graphs():
  from hypergraphembedding_b200 import synthetic
  gadget = sps.block_diag([sps.csr_matrix(np.array([[1, 0, 0], [1, 1, 1], [0, 1, 0]], dtype=bool))] * 50,
                          format="csr")
  return {"youtube": _dense_csr(load_golden("boolean_youtube_s10")["pairs"]),
          "rand25": _dense_csr(load_golden("boolean_rand25")["pairs"]),
          "gadgets": gadget.astype(bool),
          "zipf2000": synthetic.zipf_hypergraph(2000, 1000, seed=8)}


def _same(got, want, probs=True):
  for f in INDEX + (PROBS if probs else ()):
    a, b = np.asarray(getattr(got, f) if not isinstance(got, dict) else got[f]), np.asarray(want[f])
    assert a.shape == b.shape, f
    if a.dtype.kind == "f":
      assert np.array_equal(a, b.astype(a.dtype), equal_nan=True), f
    else:
      assert np.array_equal(a.astype(np.int64), b.astype(np.int64)), f


@pytest.mark.parametrize("name", ["youtube", "rand25", "gadgets", "zipf2000"])
@pytest.mark.parametrize("neg", [0, 2])
def test_boolean_device_equals_the_restatement(name, neg):
  from hypergraphembedding_b200 import BooleanSamplesDevice
  A = _graphs()[name]
  out = BooleanSamplesDevice(A, 3, 7, neg_samples=neg, seed=1234)
  _same(out, ref.boolean_samples(A, 3, 7, neg_samples=neg, seed=1234))


def test_boolean_device_with_row_weights_equals_the_restatement():
  from hypergraphembedding_b200 import BooleanSamplesDevice
  A = _graphs()["zipf2000"]
  rng = np.random.default_rng(0)
  nw, ew = rng.random(A.shape[0]) * 2, rng.random(A.shape[1]) * 2
  out = BooleanSamplesDevice(A, 2, 5, neg_samples=3, node_weights=nw, edge_weights=ew, seed=9)
  _same(out, ref.boolean_samples(A, 2, 5, neg_samples=3, seed=9, node_weights=nw, edge_weights=ew))


def _vectors(A, R=6, seed=3):
  rng = np.random.default_rng(seed)
  return (rng.random((A.shape[0], R)).astype(np.float32), rng.random((A.shape[1], R)).astype(np.float32))


@pytest.mark.parametrize("name", ["youtube", "rand25", "gadgets", "zipf2000"])
def test_hobe_device_pairs_equal_the_restatement(name):
  from hypergraphembedding_b200 import AlgebraicDistanceSamplesDevice
  A = _graphs()[name]
  xn, xe = _vectors(A)
  timings = {}
  out = AlgebraicDistanceSamplesDevice(A, xn, xe, 4, 9, seed=77, timings=timings)
  _same(out, ref.hobe_pairs(A, 4, 9, seed=77), probs=False)
  assert set(timings) == {"pairs", "neighbours", "probabilities"}


def test_hobe_probabilities_equal_the_host_array_path():
  from hypergraphembedding_b200 import AlgebraicDistanceSamplesDevice
  from hypergraphembedding_b200.hg2v_sample import _Graph, _HobeWeights
  A = _graphs()["zipf2000"]
  xn, xe = _vectors(A)
  out = AlgebraicDistanceSamplesDevice(A, xn, xe, 3, 11, seed=5)
  w = _HobeWeights(_Graph.from_csr(A), xn, xe)
  try:
    nn = ~np.isnan(out.nn_prob)
    ee = ~np.isnan(out.ee_prob)
    ne = ~np.isnan(out.ne_prob)
    assert nn.sum() and ee.sum() and ne.sum() and (nn.sum() + ee.sum() + ne.sum()) == len(out)
    assert np.array_equal(out.nn_prob[nn], w.same_type(0, out.left_node[nn], out.right_node[nn]))
    assert np.array_equal(out.ee_prob[ee], w.same_type(1, out.left_edge[ee], out.right_edge[ee]))
    assert np.array_equal(out.ne_prob[ne], w.diff_type(out.left_node[ne], out.right_edge[ne]))
  finally:
    w.close()


@pytest.fixture(scope="module")
def zipf100k():
  from hypergraphembedding_b200 import synthetic
  return synthetic.zipf_hypergraph(100000, 50000, seed=2024)


def _check_rows(rows, cols, k, cand_ptr, cand_idx):
  """Every pair is a candidate of its row, rows ascending, columns ascending and distinct inside
  a row, min(k, n_r) pairs per row."""
  rows, cols = np.asarray(rows, np.int64), np.asarray(cols, np.int64)
  assert np.all(np.diff(rows) >= 0)
  same = np.diff(rows) == 0
  assert np.all(np.diff(cols)[same] > 0)
  n = np.diff(cand_ptr)
  assert np.array_equal(np.bincount(rows, minlength=len(n)), np.minimum(k, n))
  # membership: position of every column inside its row's sorted candidate list
  start, end = cand_ptr[rows], cand_ptr[rows + 1]
  key = rows * (1 << 32) + cols
  cand_rows = np.repeat(np.arange(len(n)), n)
  cand_key = cand_rows * (1 << 32) + cand_idx.astype(np.int64)
  at = np.searchsorted(cand_key, key)
  assert np.all(at < end) and np.all(at >= start) and np.array_equal(cand_key[at], key)


def test_structure_at_100k_nodes(zipf100k):
  from hypergraphembedding_b200 import _native
  from hypergraphembedding_b200.hg2v_sample import _Graph
  A = zipf100k
  g = _Graph.from_csr(A)
  ctx = _native.default_context()
  inc = g.incidence(ctx)
  try:
    for side, factors, mats, k in ((0, 2, (g.a, g.at), 20), (1, 2, (g.b, g.bt), 20),
                                   (0, 1, (g.a,), 3), (1, 1, (g.b,), 3),
                                   (0, 3, (g.a, g.at, g.a), 20), (1, 3, (g.b, g.bt, g.b), 20)):
      rows = g.num_nodes if side == 0 else g.num_edges
      cptr, cidx = _native.spgemm_rows(mats, np.arange(rows), sorted_rows=True)
      r, c = _native.sample_pairs_device(ctx, inc, side, factors, 0, np.full(rows, k), 42, 1)
      _check_rows(r.cpu().numpy(), c.cpu().numpy(), k, cptr, cidx)
  finally:
    inc.close()


def test_block_order_at_100k_nodes(zipf100k):
  from hypergraphembedding_b200 import BooleanSamplesDevice
  out = BooleanSamplesDevice(zipf100k, 2, 10, neg_samples=1, seed=3)
  N, E = zipf100k.shape
  kind = np.select([~np.isnan(out.nn_prob), ~np.isnan(out.ee_prob), ~np.isnan(out.ne_prob),
                    (out.left_node >= 0) & (out.right_node >= 0),
                    (out.left_edge >= 0) & (out.right_edge >= 0)], [0, 1, 2, 3, 4], 5)
  runs = kind[np.r_[True, kind[1:] != kind[:-1]]].tolist()
  assert runs == [0, 1, 2, 3, 4, 5]
  neg_ee = np.nonzero(kind == 4)[0]
  assert len(neg_ee) == 2 * E                      # the edge-edge negative block twice
  assert not np.array_equal(out.right_edge[neg_ee[:E]], out.right_edge[neg_ee[E:]])
  assert np.sum(kind == 5) == N + E


def _big_edge_graph(nodes=20000, small=500):
  """Every node in one giant edge and one small edge: every row of A * A^T expands to more than
  a megabyte of workspace entries, and so does every deduplicated row of (A * A^T) * A."""
  n = np.arange(nodes)
  rows = np.concatenate([n, n])
  cols = np.concatenate([np.zeros(nodes, np.int64), 1 + n % small])
  m = sps.csr_matrix((np.ones(len(rows), dtype=bool), (rows, cols)), shape=(nodes, small + 1))
  m.sort_indices()
  return m


@pytest.mark.parametrize("graph", ["big_edge", "zipf2000"])
def test_output_does_not_depend_on_the_workspace_budget(graph):
  from hypergraphembedding_b200 import _native
  from hypergraphembedding_b200.hg2v_sample import _Graph
  A = _big_edge_graph() if graph == "big_edge" else _graphs()["zipf2000"]
  g = _Graph.from_csr(A)
  ctx = _native.default_context()
  inc = g.incidence(ctx)
  try:
    for side, factors in ((0, 2), (1, 2), (0, 3), (1, 3)):
      rows = min(64, g.num_nodes if side == 0 else g.num_edges)
      k = np.arange(rows) % 40
      launches = ctx.launch_count
      a = _native.sample_pairs_device(ctx, inc, side, factors, 0, k, 7, 3)
      one_batch = ctx.launch_count - launches
      launches = ctx.launch_count
      b = _native.sample_pairs_device(ctx, inc, side, factors, 0, k, 7, 3, workspace_mb=1)
      tiny = ctx.launch_count - launches
      if graph == "big_edge" and side == 0:
        assert tiny > 8 * one_batch                # one row per batch
      for x, y in zip(a, b):
        assert np.array_equal(x.cpu().numpy(), y.cpu().numpy())
  finally:
    inc.close()


def test_results_are_reproducible_and_chunking_free():
  import hypergraphembedding_b200 as H
  A = _graphs()["zipf2000"]
  xn, xe = _vectors(A)
  state = np.random.get_state()
  one = H.BooleanSamplesDevice(A, 3, 6, neg_samples=2, seed=21)
  again = H.BooleanSamplesDevice(A, 3, 6, neg_samples=2, seed=21)
  parts = list(H.BooleanSamplesDevice(A, 3, 6, neg_samples=2, seed=21, chunk_rows=97, stream=True))
  assert len(parts) > 20
  for other in (again, H.SampleColumns.concatenate(parts)):
    _same(other, one.arrays())
  other_seed = H.BooleanSamplesDevice(A, 3, 6, neg_samples=2, seed=22)
  assert len(other_seed) != len(one) or not np.array_equal(other_seed.right_node, one.right_node)
  h1 = H.AlgebraicDistanceSamplesDevice(A, xn, xe, 3, 6, seed=21)
  h2 = H.SampleColumns.concatenate(list(H.AlgebraicDistanceSamplesDevice(A, xn, xe, 3, 6, seed=21,
                                                                         chunk_rows=101, stream=True)))
  _same(h2, h1.arrays())
  after = np.random.get_state()
  assert after[2] == state[2] and np.array_equal(after[1], state[1])


def test_trainer_accepts_the_output():
  import hypergraphembedding_b200 as H
  from conftest import hypergraph_from_pairs
  g = load_golden("hobe_youtube_s2")
  A = _dense_csr(g["pairs"])
  hg = hypergraph_from_pairs(np.stack(A.nonzero(), axis=1))
  out = H.AlgebraicDistanceSamplesDevice(A, g["xn"], g["xe"], int(g["k"]), 20, seed=1)
  feats, targets = H.SamplesToModelInput(out, int(g["k"]), weighted=False)
  model = H.UnweightedFloatModel(hg, 16, int(g["k"]))
  history = model.fit(feats, targets, batch_size=256, epochs=3, verbose=0)
  losses = history.history["loss"]
  assert len(losses) == 3 and np.all(np.isfinite(losses))


def test_errors():
  import hypergraphembedding_b200 as H
  from hypergraphembedding_b200 import _native
  from hypergraphembedding_b200.hg2v_sample import _Graph
  A = _graphs()["gadgets"].tolil()
  A[0, :] = False                                   # node 0 has no edges
  A = sps.csr_matrix(A)
  A.eliminate_zeros()
  # the negative node-edge block pairs node 0 with an edge: its neighbour draw has nothing to draw from
  with pytest.raises(ValueError, match="cannot be empty"):
    H.BooleanSamplesDevice(A, 2, 3, neg_samples=1)
  H.BooleanSamplesDevice(A, 0, 3, neg_samples=1)   # no draws, no error
  with pytest.raises(AssertionError):
    H.BooleanSamplesDevice(A, -1, 3)
  with pytest.raises(AssertionError):
    H.AlgebraicDistanceSamplesDevice(A, *_vectors(A), 2, -3)
  g = _Graph.from_csr(A)
  ctx = _native.default_context()
  inc = g.incidence(ctx)
  try:
    with pytest.raises(AssertionError, match="negative sample count"):
      _native.sample_pairs_device(ctx, inc, 0, 2, 0, np.array([2, -1, 2]), 0, 1)
    with pytest.raises(AssertionError):
      _native.sample_pairs_device(ctx, inc, 0, 4, 0, np.array([2]), 0, 1)
  finally:
    inc.close()
