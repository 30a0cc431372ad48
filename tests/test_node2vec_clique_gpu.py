"""node2vec on a weighted clique expansion on the GPU (csrc/hge_n2v_clique.cu) against
tests/n2v_clique_ref.py: walks and counts equal the restatement exactly on both sides for (p, q)
in {(1, 1), (0.25, 4), (4, 0.25)} and walk lengths 1, 2 and 80, on a graph with isolated vertices
and a node alone in its edge, on one edge of 120 000 members (whose node-side expansion is never
built) and around nodes in 4 097 edges (long adjacency tests); results are bit-identical run to
run; EmbedNode2VecCliqueDevice equals the fp32 restatement of the whole pipeline on both sides and
leaves the global RNGs alone; the planted-partition community AUC meets the float64 bar; and the
library refuses bad arguments."""
import random

import numpy as np
import pytest
import scipy.sparse as sps

import n2v_clique_ref as cref
from conftest import hypergraph_from_pairs
from oracle import node2vec_ref as ref
from test_node2vec_clique_host import AUC_BAR, QUALITY, community_labels, shape_graph
from test_node2vec_gpu import fast_math  # noqa: F401  (the device's __expf / __logf)

pytestmark = pytest.mark.gpu

PQ = [(1.0, 1.0), (0.25, 4.0), (4.0, 0.25)]


def _csr(rows, cols, shape):
  A = sps.csr_matrix((np.ones(len(rows), np.float32), (rows, cols)), shape=shape)
  A.sum_duplicates()
  A.sort_indices()
  A.data[:] = 1
  return A


def _star(members=120_000):
  """one edge of `members` nodes plus a small edge {0, 1, 2} and a pair {5, 6}"""
  rows = np.concatenate([np.arange(members), [0, 1, 2, 5, 6]])
  cols = np.concatenate([np.zeros(members, np.int64), [1, 1, 1, 2, 2]])
  return _csr(rows, cols, (members, 3))


def _hubs(edges=6145, seed=0):
  """node 0 in edges 0 .. 4096, node 1 in edges 2048 .. 6144 (4 097 each, 2 049 shared), and
  every edge has two to four other members drawn from 400 nodes"""
  rng = np.random.RandomState(seed)
  rows, cols = [], []
  for e in range(edges):
    if e <= 4096:
      rows.append(0), cols.append(e)
    if e >= 2048:
      rows.append(1), cols.append(e)
    others = 2 + rng.randint(400, size=rng.randint(2, 5))
    rows += others.tolist()
    cols += [e] * len(others)
  return _csr(np.asarray(rows), np.asarray(cols), (402, edges))


def _ctx():
  from hypergraphembedding_b200 import _native
  return _native, _native.default_context()


def _device_walks(A, side, num_walks, L, p, q, seed):
  import torch
  from hypergraphembedding_b200.algebraic_distance import make_incidence
  _native, ctx = _ctx()
  V = A.shape[side]
  walks = torch.empty((num_walks * V, L), dtype=torch.int32, device="cuda")
  counts = torch.empty(V, dtype=torch.int64, device="cuda")
  inc = make_incidence(A, ctx=ctx)
  try:
    _native.n2v_clique_walks(ctx, inc, side, num_walks, L, p, q, seed, walks, counts)
  finally:
    inc.close()
  return walks.cpu().numpy(), counts.cpu().numpy()


def _assert_exact(A, side, num_walks, L, p, q, seed):
  walks, counts = _device_walks(A, side, num_walks, L, p, q, seed)
  want_w, want_c = cref.clique_walks(A, side, num_walks, L, p, q, seed)
  assert np.array_equal(walks, want_w)
  assert np.array_equal(counts, want_c)
  return walks


@pytest.mark.parametrize("side", [0, 1])
@pytest.mark.parametrize("pq", PQ)
@pytest.mark.parametrize("L", [1, 2, 80])
def test_walks_exact(side, pq, L):
  A = shape_graph()
  walks = _assert_exact(A, side, 3, L, pq[0], pq[1], seed=11)
  V = A.shape[side]
  if L > 1:   # vertex 0 is isolated on both sides, vertex 1 only in a single-member edge
    assert np.all(walks[np.isin(np.arange(3 * V) % V, [0, 1]), 1:] == -1)


@pytest.mark.parametrize("side", [0, 1])
@pytest.mark.parametrize("pq", PQ)
def test_walks_exact_on_a_large_edge(side, pq):
  """node side: 120 000 walks through an edge whose expansion would hold 1.4e10 entries"""
  _assert_exact(_star(), side, 1, 6, pq[0], pq[1], seed=3)


@pytest.mark.parametrize("side", [0, 1])
@pytest.mark.parametrize("pq", PQ[1:])
def test_walks_exact_around_hubs(side, pq):
  A = _hubs()
  walks = _assert_exact(A, side, 2, 12, pq[0], pq[1], seed=5)
  if side == 0:
    assert np.sum(walks == 0) > 100 and np.sum(walks == 1) > 100


def test_reproducible():
  A = _hubs(seed=1)
  a = _device_walks(A, 0, 2, 30, 0.25, 4.0, 7)
  b = _device_walks(A, 0, 2, 30, 0.25, 4.0, 7)
  assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def _restated_tables(A, side, dim, walk_length, num_walks, window, negative, epochs, batch_pairs, seed, fast_math):
  exp, log = fast_math
  walks, counts = cref.clique_walks(A, side, num_walks, walk_length, 1.0, 1.0, seed)
  pairs = ref.pairs(walks, window, seed)
  cum = ref.noise_table(counts)
  tin, tout = ref.init_tables(seed, len(counts), dim)
  for e in range(epochs):
    ref.train32(tin, tout, pairs, cum, negative, seed, e, epochs, batch_pairs, exp=exp, log=log)
  return tin


def test_embed_end_to_end(fast_math):
  import hypergraphembedding_b200 as H
  from hypergraphembedding_b200.hypergraph_util import compressed_incidence
  A = shape_graph()
  A = A[np.diff(A.indptr) > 0][:, np.diff(A.tocsc().indptr) > 0].tocoo()   # a hypergraph has no empty rows
  hg = hypergraph_from_pairs(np.stack([A.row * 3 + 1, A.col * 5 + 2], axis=1))
  np.random.seed(0)
  random.seed(0)
  state, pystate = np.random.get_state(), random.getstate()
  emb = H.EmbedNode2VecCliqueDevice(hg, 16, walk_length=10, num_walks=2, window=4, epochs=2, seed=4)
  after = np.random.get_state()
  assert after[2] == state[2] and np.array_equal(after[1], state[1])
  assert random.getstate() == pystate
  assert emb.method_name == "N2V_CLIQUE" and emb.dim == 16
  assert sorted(emb.node) == sorted(hg.node) and sorted(emb.edge) == sorted(hg.edge)
  assert H.EmbedNode2VecCliqueDevice not in H.EMBEDDING_OPTIONS.values()
  node_ids, edge_ids, Ac = compressed_incidence(hg)
  xn = np.asarray([emb.node[int(i)].values for i in node_ids], dtype=np.float32)
  xe = np.asarray([emb.edge[int(i)].values for i in edge_ids], dtype=np.float32)
  kw = dict(dim=16, walk_length=10, num_walks=2, window=4, negative=5, epochs=2, batch_pairs=256)
  want_n = _restated_tables(Ac, 0, seed=4, fast_math=fast_math, **kw)
  want_e = _restated_tables(Ac, 1, seed=cref.edge_seed(4), fast_math=fast_math, **kw)
  assert np.array_equal(xn.view(np.uint32), want_n.view(np.uint32))
  assert np.array_equal(xe.view(np.uint32), want_e.view(np.uint32))


def test_timings_and_info():
  from hypergraphembedding_b200 import Node2VecCliqueDevice, Node2VecDevice
  A = shape_graph()
  t, tc = {}, {}
  _, info = Node2VecDevice(A, 8, walk_length=6, num_walks=1, epochs=1, timings=t)
  X, cinfo = Node2VecCliqueDevice(A, 8, side="edge", walk_length=6, num_walks=1, epochs=1, timings=tc)
  assert X.shape == (A.shape[1], 8) and X.dtype == np.float32
  assert set(cinfo) == set(info) and set(tc) == set(t)
  assert cinfo["num_walks"] == A.shape[1]


def test_quality_on_planted_partition():
  from hypergraphembedding_b200 import Node2VecCliqueDevice
  A = ref.planted_partition()
  kw = dict(QUALITY)
  dim = kw.pop("dim")
  for side, name in ((0, "node"), (1, "edge")):
    X, info = Node2VecCliqueDevice(A, dim, side=name, **kw)
    assert np.all(np.diff(info["losses"]) < 0)
    assert cref.community_auc(X, community_labels(side)) >= AUC_BAR[side]


def test_library_refusals():
  import torch
  from hypergraphembedding_b200.algebraic_distance import make_incidence
  _native, ctx = _ctx()
  A = shape_graph()
  walks = torch.empty((A.shape[0], 4), dtype=torch.int32, device="cuda")
  counts = torch.full((A.shape[0],), 7, dtype=torch.int64, device="cuda")
  inc = make_incidence(A, ctx=ctx)
  try:
    for args, match in (((2, 1, 4, 1.0, 1.0), "side"), ((-1, 1, 4, 1.0, 1.0), "side"),
                        ((0, 0, 4, 1.0, 1.0), "num_walks"), ((0, 1, 0, 1.0, 1.0), "walk_length"),
                        ((0, 1, 4, 0.0, 1.0), "p ="), ((0, 1, 4, 1.0, float("inf")), "q ="),
                        ((0, 1, 4, 1e-3, 1e3), "max / min")):
      with pytest.raises(AssertionError, match=match):
        _native.n2v_clique_walks(ctx, inc, *args, 0, walks, counts)
    assert torch.all(counts == 7)   # nothing ran
    rc = ctx.lib.hge_n2v_clique_walks(ctx.handle, inc.handle, 0, 1, 4, 1.0, 1.0, 0, None, _native.ptr(counts))
    assert rc == _native.HGE_ERR_INVALID and "NULL" in _native.last_error()
  finally:
    inc.close()
