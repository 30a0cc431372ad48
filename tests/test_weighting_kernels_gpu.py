"""The distance, span and HOBE-probability kernels of csrc/hge_weighting.cu at every lane width and
dispatch path, against the numpy restatements of oracle/weighting_ref.py.

One synthetic incidence serves every case.  Rows of both sides have the degrees of `DEGREES`
(empty, one float4 lane, warp and GP boundaries, the 2 048-incidence segments of
k_incidence_l2); 45 000 node rows give k_incidence_l2 more segments than warps; the node side's
mean degree selects k_same_type_prob<8>, the edge side's k_same_type_prob<32>.  The dimensions
cover every lanes-per-row class, R % 4 != 0 and one to eight 128-column slabs.

- Spans and probabilities are selections, equal to the restatement bit for bit.
- Distances on vectors of the dyadic grid {k / 16} are exact sums, so they equal
  sqrt(fp32(exact sum)) bit for bit; on random vectors they are held to the 1e-5 bar.
- Both orders of k_incidence_l2, k_pair_l2, host and device arrays, aligned and misaligned rows
  and a shared or copied second operand run the same chain of operations, so they are equal."""
import numpy as np
import pytest
import scipy.sparse as sps

from conftest import csr_from_pairs
from oracle import port
from oracle import weighting_ref as wref

pytestmark = pytest.mark.gpu

DEGREES = [0, 1, 3, 4, 5, 7, 8, 9, 31, 32, 33, 2047, 2048, 2049, 4096, 4097]
DIMS = [1, 3, 4, 5, 8, 9, 16, 17, 31, 32, 33, 64, 65, 127, 128, 129, 255, 257, 511, 1000, 1024]
LONG_PAIR_DIMS = {1, 5, 9, 17, 33, 257}     # one per lanes-per-row class, several slabs at 257
PAIR_COUNTS = [1, 31, 32, 33, 4097]
N, E = 45000, 5000
HUB = DEGREES.index(4097)                   # node in 4 097 edges
RTOL, ATOL_PER_SQRT_R = 1e-5, 1e-6


class Graph(object):

  def __init__(self):
    rng = np.random.default_rng(11)
    S = len(DEGREES)
    rows, cols = [], []
    for k, d in enumerate(DEGREES):   # node k: d of the ordinary edges
      rows.append(np.full(d, k))
      cols.append(S + rng.choice(E - S, d, replace=False))
    for k, d in enumerate(DEGREES):   # edge k: d of the ordinary nodes
      rows.append(S + rng.choice(N - S, d, replace=False))
      cols.append(np.full(d, k))
    reps = rng.integers(1, 5, N - S)  # every ordinary node in 1-4 ordinary edges
    rows.append(np.repeat(np.arange(S, N), reps))
    cols.append(S + rng.integers(0, E - S, int(reps.sum())))
    self.A = csr_from_pairs(np.stack([np.concatenate(rows), np.concatenate(cols)], 1), shape=(N, E))
    self.B = self.A.T.tocsr()
    self.B.sort_indices()
    self.ptr = (self.A.indptr.astype(np.int64), self.B.indptr.astype(np.int64))
    self.idx = (self.A.indices.astype(np.int32), self.B.indices.astype(np.int32))
    self.deg = (np.diff(self.ptr[0]), np.diff(self.ptr[1]))
    self.rows_a = np.repeat(np.arange(N), self.deg[0])
    # position in node -> edge order of every incidence in edge -> node order
    rows_b = np.repeat(np.arange(E), self.deg[1])
    self.b2a = np.searchsorted(self.rows_a.astype(np.int64) * E + self.idx[0],
                               self.idx[1].astype(np.int64) * E + rows_b)
    self.nnz = len(self.idx[0])


@pytest.fixture(scope="module")
def graph():
  return Graph()


@pytest.fixture(scope="module")
def inc(graph, gpu_ctx):
  from hypergraphembedding_b200 import _native
  g = graph
  handle = _native.Incidence(gpu_ctx, N, E, g.ptr[0], g.idx[0], g.ptr[1], g.idx[1])
  yield handle
  handle.close()


def _dev(a):
  import torch
  return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _host(t):
  return t.cpu().numpy()


def _misaligned(x):
  """The rows of x as a contiguous CUDA view whose first element is 4 bytes past a 16-byte
  boundary (R % 4 == 0 rows are then not float4-addressable in place)."""
  import torch
  base = torch.empty(x.size + 4, dtype=torch.float32, device="cuda")
  view = base[1:1 + x.size].view(*x.shape)
  view.copy_(torch.from_numpy(x))
  assert view.data_ptr() % 16 == 4 and view.is_contiguous()
  return view


def _dyadic(rng, rows, R):
  return (rng.integers(0, 16, (rows, R)) / 16).astype(np.float32)


def test_the_incidence_has_the_shapes_the_kernels_branch_on(graph):
  g = graph
  for side in (0, 1):
    assert list(g.deg[side][:len(DEGREES)]) == DEGREES
  assert (g.deg[0] > 0).sum() >= 40000
  assert g.deg[0][HUB] >= 3000
  # hge_same_type_prob: k_same_type_prob<8> at a mean degree <= 24, <32> above
  assert g.nnz / N <= 24 < g.nnz / E
  # k_incidence_l2 in node order: more segments of <= 2 048 incidences than the 16 * 148 * 8 warps
  assert ((g.deg[0] + 2047) // 2048).sum() > 16 * 148 * 8


@pytest.mark.parametrize("R", DIMS)
def test_distances_are_exact_on_dyadic_vectors(R, graph, inc, gpu_ctx):
  from hypergraphembedding_b200 import _native
  g = graph
  rng = np.random.default_rng(R)
  xn, xe = _dyadic(rng, N, R), _dyadic(rng, E, R)
  want = np.sqrt(wref.pair_sq_f64(xn, xe, g.rows_a, g.idx[0]).astype(np.float32))
  assert np.array_equal(_native.incidence_l2(gpu_ctx, inc, xn, xe, order=0), want)
  assert np.array_equal(_native.incidence_l2(gpu_ctx, inc, xn, xe, order=1), want[g.b2a])
  max_dist = np.float32(np.sqrt(R))
  want_w = (max_dist - want) / max_dist
  assert want_w.dtype == np.float32
  assert np.array_equal(_native.incidence_l2(gpu_ctx, inc, xn, xe, order=0, as_weight=True), want_w)
  assert np.array_equal(_native.incidence_l2(gpu_ctx, inc, xn, xe, order=1, as_weight=True),
                        want_w[g.b2a])
  counts = PAIR_COUNTS + ([1000003] if R in LONG_PAIR_DIMS else [])
  for n in counts:
    ia, ib = rng.integers(0, N, n), rng.integers(0, E, n)
    got = _native.pair_l2(gpu_ctx, xn, xe, ia, ib)
    assert np.array_equal(got, np.sqrt(wref.pair_sq_f64(xn, xe, ia, ib).astype(np.float32))), n


@pytest.mark.parametrize("R", DIMS)
def test_distances_on_random_vectors_and_across_call_forms(R, graph, inc, gpu_ctx):
  from hypergraphembedding_b200 import _native
  g = graph
  rng = np.random.default_rng(1000 + R)
  xn, xe = rng.random((N, R), dtype=np.float32), rng.random((E, R), dtype=np.float32)
  d64 = wref.incidence_l2_f64(g.ptr[0], g.idx[0], xn, xe)
  bar = RTOL * d64 + ATOL_PER_SQRT_R * np.sqrt(R)
  d0 = _native.incidence_l2(gpu_ctx, inc, xn, xe, order=0)
  assert np.all(np.abs(d0 - d64) <= bar)
  w = _native.incidence_l2(gpu_ctx, inc, xn, xe, order=0, as_weight=True)
  assert np.all(np.abs(w - wref.hobe_weight_f64(d64, R)) <= bar / np.sqrt(R) + 1e-7)
  # the same sq_diff chain and group_sum<LPR> tree in every form: equal bits
  assert np.array_equal(_native.incidence_l2(gpu_ctx, inc, xn, xe, order=1), d0[g.b2a])
  assert np.array_equal(_native.pair_l2(gpu_ctx, xn, xe, g.rows_a, g.idx[0]), d0)
  xn_d, xe_d = _dev(xn), _dev(xe)
  assert np.array_equal(_host(_native.incidence_l2(gpu_ctx, inc, xn_d, xe_d, order=0)), d0)
  assert np.array_equal(_host(_native.incidence_l2(gpu_ctx, inc, xn_d, xe_d, order=1, as_weight=True)),
                        _native.incidence_l2(gpu_ctx, inc, xn, xe, order=1, as_weight=True))
  if R % 4 == 0:
    assert np.array_equal(_host(_native.incidence_l2(gpu_ctx, inc, _misaligned(xn), xe_d, order=0)), d0)
    assert np.array_equal(_host(_native.incidence_l2(gpu_ctx, inc, xn_d, _misaligned(xe), order=1)),
                          d0[g.b2a])
  ia, ib = rng.integers(0, N, 4097).astype(np.int32), rng.integers(0, N, 4097).astype(np.int32)
  p = _native.pair_l2(gpu_ctx, xn, xn, ia, ib)
  p64 = wref.pair_l2_f64(xn, xn, ia, ib)
  assert np.all(np.abs(p - p64) <= RTOL * p64 + ATOL_PER_SQRT_R * np.sqrt(R))
  assert np.array_equal(_native.pair_l2(gpu_ctx, xn, xn.copy(), ia, ib), p)
  ia_d, ib_d = _dev(ia), _dev(ib)
  assert np.array_equal(_host(_native.pair_l2(gpu_ctx, xn_d, xn_d, ia_d, ib_d)), p)
  assert np.array_equal(_host(_native.pair_l2(gpu_ctx, xn_d, xn_d.clone(), ia_d, ib_d)), p)
  if R % 4 == 0:
    assert np.array_equal(_host(_native.pair_l2(gpu_ctx, _misaligned(xn), xn_d, ia_d, ib_d)), p)


def _spans_want(g, side, xn, xe):
  xs, xo = (xn, xe) if side == 0 else (xe, xn)
  return wref.row_span_f32(g.ptr[side], g.idx[side], xs, xo)


@pytest.mark.parametrize("R", DIMS)
def test_spans_are_exact(R, graph, inc, gpu_ctx):
  from hypergraphembedding_b200 import _native
  g = graph
  rng = np.random.default_rng(2000 + R)
  xn = rng.standard_normal((N, R), dtype=np.float32)
  xe = rng.standard_normal((E, R), dtype=np.float32)
  xn_d, xe_d = _dev(xn), _dev(xe)
  for side in (0, 1):
    want = _spans_want(g, side, xn, xe)
    got = _native.row_span(gpu_ctx, inc, xn, xe, side)
    assert np.array_equal(got, want), side
    assert np.all(got[g.deg[side] == 0] == 0) and np.all(got[g.deg[side] > 0] > 0)
    assert np.array_equal(_host(_native.row_span(gpu_ctx, inc, xn_d, xe_d, side)), want), side
    if R % 4 == 0:
      assert np.array_equal(_host(_native.row_span(gpu_ctx, inc, _misaligned(xn), _misaligned(xe), side)),
                            want), side


@pytest.mark.parametrize("R", [32, 200])
def test_compute_spans_gives_the_same_values(R, graph):
  from hypergraphembedding_b200 import ComputeSpans, Hypergraph, HypergraphEmbedding
  g = graph
  rng = np.random.default_rng(3000 + R)
  xn = rng.standard_normal((N, R), dtype=np.float32)
  xe = rng.standard_normal((E, R), dtype=np.float32)
  hg = Hypergraph()
  emb = HypergraphEmbedding()
  emb.dim = R
  for n in range(N):
    hg.node[n].edges.extend(g.idx[0][g.ptr[0][n]:g.ptr[0][n + 1]].tolist())
    emb.node[n].values.extend(xn[n].tolist())
  for e in range(E):
    hg.edge[e].nodes.extend(g.idx[1][g.ptr[1][e]:g.ptr[1][e + 1]].tolist())
    emb.edge[e].values.extend(xe[e].tolist())
  node2span, edge2span = ComputeSpans(hg, emb, run_in_parallel=False, disable_pbar=True)
  got_n = np.asarray([node2span[n] for n in range(N)], dtype=np.float32)
  got_e = np.asarray([edge2span[e] for e in range(E)], dtype=np.float32)
  assert np.array_equal(got_n, _spans_want(g, 0, xn, xe))
  assert np.array_equal(got_e, _spans_want(g, 1, xn, xe))


def _weights(rng, n):
  """fp32 weights, about a fifth of them negative, with zeros and many ties: half on a grid of
  eighths in [-0.5, 1], half normal around 0.5."""
  w = (rng.standard_normal(n) * 0.5 + 0.5).astype(np.float32)
  grid = rng.random(n) < 0.5
  w[grid] = rng.integers(-4, 9, int(grid.sum())) / 8
  return w


def _shared_pairs(ptr, idx, tptr, tidx, rows, rng):
  """For each given row r, a pair (r, s) with s a row that shares a column with r."""
  rows = rows[np.diff(ptr)[rows] > 0]
  col = idx[ptr[rows] + rng.integers(0, np.diff(ptr)[rows])]
  other = tidx[tptr[col] + rng.integers(0, np.diff(tptr)[col])]
  return rows, other


def _probability_pairs(g, side, rng, total=200003):
  """Every pair of special rows (both orders, i == j, empty rows, short against long), each
  special row with rows it shares a column with, then random rows with such partners and uniform
  pairs, `total` pairs in all."""
  ptr, idx, tptr, tidx = g.ptr[side], g.idx[side], g.ptr[1 - side], g.idx[1 - side]
  rows = len(ptr) - 1
  S = len(DEGREES)
  si, sj = np.meshgrid(np.arange(S), np.arange(S), indexing="ij")
  parts = [(si.ravel(), sj.ravel())]
  special = np.repeat(np.arange(S), 40)
  a, b = _shared_pairs(ptr, idx, tptr, tidx, special, rng)
  parts += [(a, b), (b, a)]
  a, b = _shared_pairs(ptr, idx, tptr, tidx, rng.integers(0, rows, 150000), rng)
  parts.append((a, b))
  used = sum(len(p[0]) for p in parts)
  parts.append(tuple(rng.integers(0, rows, (2, total - used))))
  pi = np.concatenate([p[0] for p in parts]).astype(np.int32)
  pj = np.concatenate([p[1] for p in parts]).astype(np.int32)
  assert len(pi) == total
  return pi, pj


def test_same_type_probabilities_are_exact(graph, inc, gpu_ctx):
  from hypergraphembedding_b200 import _native
  g = graph
  rng = np.random.default_rng(5)
  for side in (0, 1):
    w = _weights(rng, g.nnz)
    pi, pj = _probability_pairs(g, side, rng)
    want = wref.same_type_prob(g.ptr[side], g.idx[side], w, pi, pj)
    assert (want > 0).sum() > len(want) // 4 and (want == 0).sum() > len(want) // 10
    got = _native.same_type_prob(gpu_ctx, inc, side, w, pi, pj)
    assert np.array_equal(got, want), side
    got_d = _native.same_type_prob(gpu_ctx, inc, side, _dev(w), _dev(pi), _dev(pj))
    assert np.array_equal(_host(got_d), want), side


def test_both_group_widths_give_the_same_probabilities(gpu_ctx):
  """k_same_type_prob<32> on a small incidence whose sides have a mean degree above 24, and
  k_same_type_prob<8> on the same incidence with empty rows appended to both sides."""
  from hypergraphembedding_b200 import _native
  rng = np.random.default_rng(6)
  n, e, per_node = 200, 100, 30
  pairs = np.stack([np.repeat(np.arange(n), per_node),
                    np.concatenate([rng.choice(e, per_node, replace=False) for _ in range(n)])], 1)
  A = csr_from_pairs(pairs, shape=(n, e))
  B = A.T.tocsr()
  B.sort_indices()
  assert A.nnz / n > 24 and A.nnz / e > 24
  extra_n, extra_e = 100, 200
  A2 = sps.csr_matrix((A.data, A.indices, np.concatenate([A.indptr, np.full(extra_n, A.nnz)])),
                      shape=(n + extra_n, e + extra_e))
  B2 = sps.csr_matrix((B.data, B.indices, np.concatenate([B.indptr, np.full(extra_e, B.nnz)])),
                      shape=(e + extra_e, n + extra_n))
  assert A2.nnz / (n + extra_n) <= 24 and B2.nnz / (e + extra_e) <= 24
  inc32 = _native.Incidence(gpu_ctx, n, e, A.indptr, A.indices, B.indptr, B.indices)
  inc8 = _native.Incidence(gpu_ctx, n + extra_n, e + extra_e, A2.indptr, A2.indices, B2.indptr, B2.indices)
  try:
    for side, M, rows in ((0, A, n), (1, B, e)):
      w = _weights(rng, M.nnz)
      pi, pj = [a.ravel().astype(np.int32) for a in np.meshgrid(np.arange(rows), np.arange(rows))]
      want = wref.same_type_prob(M.indptr, M.indices, w, pi, pj)
      wide = _native.same_type_prob(gpu_ctx, inc32, side, w, pi, pj)
      narrow = _native.same_type_prob(gpu_ctx, inc8, side, w, pi, pj)
      assert np.array_equal(wide, want) and np.array_equal(narrow, want), side
      assert np.array_equal(wide.view(np.int32), narrow.view(np.int32)), side
  finally:
    inc32.close()
    inc8.close()


def test_diff_type_probabilities_are_exact(graph, inc, gpu_ctx):
  from hypergraphembedding_b200 import _native
  g = graph
  rng = np.random.default_rng(7)
  w_e2n = _weights(rng, g.nnz)
  S = len(DEGREES)
  big = np.flatnonzero(g.deg[1] >= 4097)
  assert len(big) > 0
  pn = [np.full(len(big), HUB), np.full(S, HUB), np.repeat(np.arange(S), S)]
  pe = [big, np.arange(S), np.tile(np.arange(S), S)]
  nodes = rng.integers(0, N, 30000)
  a, b = _shared_pairs(g.ptr[0], g.idx[0], g.ptr[1], g.idx[1], nodes, rng)   # node, co-member node
  pn.append(a)
  pe.append(g.idx[0][g.ptr[0][b] + rng.integers(0, g.deg[0][b])])             # an edge of that node
  pn.append(rng.integers(0, N, 10000))
  pe.append(rng.integers(0, E, 10000))
  pn, pe = np.concatenate(pn).astype(np.int32), np.concatenate(pe).astype(np.int32)
  want = wref.diff_type_prob(g.ptr[0], g.idx[0], g.ptr[1], g.idx[1], w_e2n, pn, pe)
  assert (want > 0).sum() > len(want) // 4
  assert np.array_equal(_native.diff_type_prob(gpu_ctx, inc, w_e2n, pn, pe), want)
  got_d = _native.diff_type_prob(gpu_ctx, inc, _dev(w_e2n), _dev(pn), _dev(pe))
  assert np.array_equal(_host(got_d), want)


def _signed_values(rng, n):
  v = rng.standard_normal(n).astype(np.float32)
  if n >= 4:
    v[1], v[2] = -0.0, 0.0
    v[0] = v.max() + 1      # the maximum first
    v[-1] = v.min() - 1     # the minimum last
  return v


def test_scale_transform_on_signed_values(gpu_ctx):
  from hypergraphembedding_b200 import _native
  rng = np.random.default_rng(8)
  for v in (_signed_values(rng, 5000003), _signed_values(rng, 1001), -np.abs(_signed_values(rng, 77)),
            np.full(1000, -3.25, np.float32)):
    for alpha in (0, 0.3, 1):
      want = np.asarray(port.alpha_scale(port.one_minus(port.zero_one_scale(v)), alpha), np.float32)
      got, mm = _native.scale_transform(gpu_ctx, v.copy(), alpha, want_minmax=True)
      assert np.array_equal(got, want), (len(v), alpha)
      assert (mm[0], mm[1]) == (v.min(), v.max())
      lo, hi = _native.scale_minmax(gpu_ctx, v)
      assert (lo, hi) == (float(v.min()), float(v.max()))
      assert np.array_equal(_native.scale_apply(gpu_ctx, v.copy(), alpha, lo, hi), want)
    got_d = _native.scale_transform(gpu_ctx, _dev(v), 0.3)
    assert np.array_equal(_host(got_d), np.asarray(port.alpha_scale(
        port.one_minus(port.zero_one_scale(v)), 0.3), np.float32))


def test_dimension_above_1024_is_refused(gpu_ctx):
  from hypergraphembedding_b200 import _native
  ptr, idx = np.asarray([0, 2, 3], np.int64), np.asarray([0, 1, 1], np.int32)
  small = _native.Incidence(gpu_ctx, 2, 2, ptr, idx)
  try:
    xn, xe = np.ones((2, 1025), np.float32), np.zeros((2, 1025), np.float32)
    launches = gpu_ctx.launch_count
    with pytest.raises(AssertionError, match="dimension 1025"):
      _native.incidence_l2(gpu_ctx, small, xn, xe)
    with pytest.raises(AssertionError, match="dimension 1025"):
      _native.pair_l2(gpu_ctx, xn, xe, [0, 1], [1, 0])
    with pytest.raises(AssertionError, match="dimension 1025"):
      _native.row_span(gpu_ctx, small, xn, xe, 0)
    assert gpu_ctx.launch_count == launches
    xn, xe = xn[:, :1024].copy(), xe[:, :1024].copy()
    assert np.array_equal(_native.incidence_l2(gpu_ctx, small, xn, xe), np.full(3, 32, np.float32))
    assert np.array_equal(_native.pair_l2(gpu_ctx, xn, xe, [0, 1], [1, 0]), np.full(2, 32, np.float32))
    assert np.array_equal(_native.row_span(gpu_ctx, small, xn, xe, 0), np.ones(2, np.float32))
  finally:
    small.close()


def test_pair_indices_out_of_range_are_refused(graph, inc, gpu_ctx):
  """-1 and exactly the row count, in each index array, from the host and from the device: each
  call raises before a kernel reads the index, and a valid call right after it succeeds."""
  from hypergraphembedding_b200 import _native
  g = graph
  rng = np.random.default_rng(9)
  x = rng.random((N, 8), dtype=np.float32)
  y = rng.random((E, 8), dtype=np.float32)
  w = [_weights(rng, g.nnz), _weights(rng, g.nnz)]
  ok_a, ok_b = np.asarray([0, N - 1, 5], np.int32), np.asarray([E - 1, 0, 7], np.int32)
  want_pair = _native.pair_l2(gpu_ctx, x, y, ok_a, ok_b)
  want_same = [wref.same_type_prob(g.ptr[s], g.idx[s], w[s], ok_b, ok_b[::-1].copy()) for s in (0, 1)]
  want_diff = wref.diff_type_prob(g.ptr[0], g.idx[0], g.ptr[1], g.idx[1], w[1], ok_a, ok_b)

  def bad(a, limit):
    out = []
    for v in (-1, limit):
      b = a.copy()
      b[1] = v
      out.append(b)
    return out

  for dev in (False, True):
    put = _dev if dev else (lambda a: a)
    get = _host if dev else (lambda a: a)
    calls = []
    for a in bad(ok_a, N):
      calls.append(lambda a=a: _native.pair_l2(gpu_ctx, put(x), put(y), put(a), put(ok_b)))
      calls.append(lambda a=a: _native.diff_type_prob(gpu_ctx, inc, put(w[1]), put(a), put(ok_b)))
    for b in bad(ok_b, E):
      calls.append(lambda b=b: _native.pair_l2(gpu_ctx, put(x), put(y), put(ok_a), put(b)))
      calls.append(lambda b=b: _native.diff_type_prob(gpu_ctx, inc, put(w[1]), put(ok_a), put(b)))
    for side, rows in ((0, N), (1, E)):
      for a in bad(ok_b, rows):
        calls.append(lambda a=a, s=side: _native.same_type_prob(gpu_ctx, inc, s, put(w[s]), put(a),
                                                                put(ok_b)))
        calls.append(lambda a=a, s=side: _native.same_type_prob(gpu_ctx, inc, s, put(w[s]), put(ok_b),
                                                                put(a)))
    for call in calls:
      with pytest.raises(AssertionError, match="outside"):
        call()
      assert np.array_equal(get(_native.pair_l2(gpu_ctx, put(x), put(y), put(ok_a), put(ok_b))), want_pair)
    for s in (0, 1):
      got = _native.same_type_prob(gpu_ctx, inc, s, put(w[s]), put(ok_b), put(ok_b[::-1].copy()))
      assert np.array_equal(get(got), want_same[s])
    assert np.array_equal(get(_native.diff_type_prob(gpu_ctx, inc, put(w[1]), put(ok_a), put(ok_b))),
                          want_diff)
