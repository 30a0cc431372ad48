"""WeightedJaccardSamplesDevice and the centroid factors: hge_jaccard_centroid (host arrays) and
hge_jaccard_centroid_grouped (device arrays, every budget) equal to each other and to the fp32
restatement of SparseWeightedJaccard / CentroidFromRows bit for bit on every pair; the range checks of
hge_jaccard_centroid and hge_jaccard_rows; the sampler's index and neighbour columns equal
to their numpy restatement (oracle/jaccard_device_ref.py), its probabilities and left / right weights
equal to the fp32 restatement of SparseWeightedJaccard / CentroidFromRows bit for bit (and to the
float64 one to the bars of tests/test_jaccard_samples_gpu.py); its result forms, the packing of its
kept blocks, the Embed*Device entry points of the Jaccard methods, the refusals, and a 100 000-node
run."""
import logging
import re

import numpy as np
import pytest
import scipy.sparse as sps

from conftest import hypergraph_from_pairs, load_golden
from oracle import jaccard_device_ref as jref
from test_device_sampler_gpu import _vectors
from test_jaccard_restatement import _centroid, _row, _signed_golden
from test_jaccard_samples_gpu import _features, _float64_restatement, _reference_loop

pytestmark = pytest.mark.gpu

GOLDEN = ["tiny_uniform", "rand25_uniform", "rand25_neighborhood", "rand25_distance", "youtube_s2_neighborhood"]
INDEX = ("left_node", "left_edge", "right_node", "right_edge", "neigh_node", "neigh_edge")
PROBS = ("nn_prob", "ee_prob", "ne_prob", "left_weight", "right_weight")
RTOL = 1e-5


def _golden_graph(name):
  """(incidence N x E, node features, edge features, golden dict) of a jaccard_* golden file."""
  g = load_golden("jaccard_" + name)
  NF, EF = _features(g, "n2f"), _features(g, "e2f")
  NF.sort_indices()
  EF.sort_indices()
  A = sps.csr_matrix((np.ones(len(g["pairs"]), dtype=bool), (g["pairs"][:, 0], g["pairs"][:, 1])),
                     shape=(NF.shape[0], EF.shape[0]))
  A.sort_indices()
  return A, NF, EF, g


def _dev(a):
  import torch
  from hypergraphembedding_b200 import _native
  return torch.as_tensor(np.ascontiguousarray(a, dtype=np.int32)).to(
      torch.device("cuda", _native.default_context().device))


def _scipy(feat):
  """The scipy CSR of a host FeatureCsr / CsrArrays: the rows exactly as the kernels read them."""
  data = feat.val if hasattr(feat, "val") else np.ones(len(feat.idx), np.float32)
  return sps.csr_matrix((data, feat.idx, feat.ptr), shape=feat.shape)


def _centroid_factors_equal_the_restatement(A, X, F, side, px, pg, budgets):
  """Both centroid entry points on the incidence A (groups: its edges for side 1, its nodes for
  side 0): hge_jaccard_centroid on host arrays with the group CSR given explicitly, and
  hge_jaccard_centroid_grouped on device arrays with the groups taken from the incidence, at every
  budget.  The outputs are bit-equal to each other and, on every pair, to the fp32 restatement of
  the reference (0 for a group without members)."""
  from hypergraphembedding_b200 import _native
  from hypergraphembedding_b200.hg2v_sample import _Graph
  ctx = _native.default_context()
  g = _Graph.from_csr(A)
  groups = g.b if side == 1 else g.a
  x, f = _native.FeatureCsr(X), _native.FeatureCsr(F)
  want = _native.jaccard_centroid(ctx, x, groups, f, px, pg)
  import torch
  dev = torch.device("cuda", ctx.device)
  xd, fd = x.to_device(dev), f.to_device(dev)
  inc = g.incidence(ctx)
  try:
    for mb in budgets:
      got = _native.jaccard_centroid_grouped(ctx, inc, side, xd, fd, _dev(px), _dev(pg), mb).cpu().numpy()
      assert got.dtype == np.float32 and np.array_equal(got, want), (side, mb)
  finally:
    inc.close()
  Xs, Fs, G = _scipy(x), _scipy(f), _scipy(groups)
  centroids, expect = {}, {}
  for i, key in enumerate(zip(np.asarray(px).tolist(), np.asarray(pg).tolist())):
    if key not in expect:
      a, grp = key
      if grp not in centroids:
        centroids[grp] = _centroid(G, grp, Fs) if G.indptr[grp + 1] > G.indptr[grp] else None
      c = centroids[grp]
      expect[key] = np.float32(0) if c is None else _reference_loop(*_row(Xs, a), *c)
    assert want[i] == expect[key], (side, i)
  return want


@pytest.mark.parametrize("name", GOLDEN)
def test_centroid_factors_equal_the_restatement_on_the_golden_graphs(name):
  A, NF, EF, _ = _golden_graph(name)
  N, E = A.shape
  rng = np.random.default_rng(11)
  nodes, edges = rng.integers(0, N, 3000), rng.integers(0, E, 3000)
  _centroid_factors_equal_the_restatement(A, NF, NF, 1, nodes, edges, (0, 1))
  _centroid_factors_equal_the_restatement(A, EF, EF, 0, edges, nodes, (0, 1))


def test_centroid_factors_on_signed_features_an_empty_group_and_a_group_above_the_budget():
  g, F, G = _signed_golden()
  G = sps.vstack([G, sps.csr_matrix((1, G.shape[1]), dtype=G.dtype)]).tocsr()     # the last group is empty
  G.sort_indices()
  assert np.diff(G.indptr)[-1] == 0 and (F.data < 0).any() and (F.data == 0).any()
  rng = np.random.default_rng(3)
  px = rng.integers(0, F.shape[0], 2000)
  pg = np.concatenate([rng.integers(0, G.shape[0], 1999), [G.shape[0] - 1]])
  # groups on the edge side (the incidence's edge -> node CSR is G), then on the node side (its node
  # -> edge CSR is G)
  want = _centroid_factors_equal_the_restatement(sps.csr_matrix(G.T), F, F, 1, px, pg, (0, 1))
  assert want[-1] == 0
  assert np.array_equal(_centroid_factors_equal_the_restatement(G, F, F, 0, px, pg, (0, 1)), want)
  # one group expands to 2400 x 40 entries: about 4.6 MB of workspace, more than a 1 MB budget
  # (its own batch) and than 4 MB (a batch of its own next to batches of small groups)
  big = sps.random(3000, 500, density=0.08, random_state=5, format="csr", dtype=np.float32)
  big.data -= 0.3
  inc = sps.random(3000, 60, density=0.02, random_state=6, format="csr", dtype=np.float32)
  inc = inc.tolil()
  inc[:2400, 7] = 1
  inc = sps.csr_matrix(inc, dtype=bool).astype(np.float32)
  inc.sort_indices()
  px = rng.integers(0, 3000, 5000)
  pg = np.concatenate([np.full(300, 7), rng.integers(0, 60, 4700)])
  _centroid_factors_equal_the_restatement(inc, big, big, 1, px, pg, (0, 1, 4))


@pytest.mark.parametrize("name", ["tiny_uniform", "rand25_uniform", "rand25_neighborhood"])
def test_sampler_equals_the_restatements(name):
  from hypergraphembedding_b200 import WeightedJaccardSamplesDevice
  A, NF, EF, g = _golden_graph(name)
  N, E = A.shape
  k, ns, seed = 3, 4, 17
  rng = np.random.default_rng(1)
  nw, ew = rng.random(N) * 2, rng.random(E) * 2
  want = jref.jaccard_pairs(A, k, ns, seed=seed, node_weights=nw, edge_weights=ew)
  out = WeightedJaccardSamplesDevice(A, NF, EF, k, ns, node_weights=nw, edge_weights=ew, seed=seed)
  arrays = out.arrays()
  for f in INDEX:
    assert np.array_equal(arrays[f].astype(np.int64), want[f].astype(np.int64)), f
  for chunk, mb in ((1, 0), (101, 1), (0, 1)):
    other = WeightedJaccardSamplesDevice(A, NF, EF, k, ns, node_weights=nw, edge_weights=ew, seed=seed,
                                         chunk_rows=chunk, workspace_mb=mb).arrays()
    for f in out.FIELDS:
      assert np.array_equal(other[f], arrays[f], equal_nan=arrays[f].dtype.kind == "f"), (f, chunk, mb)
  # fp32 restatement, record by record
  AT = sps.csr_matrix(A.T)
  AT.sort_indices()
  ln, rn, le, re_ = (arrays[f] for f in ("left_node", "right_node", "left_edge", "right_edge"))
  nn, ee, ne = (ln >= 0) & (rn >= 0), (le >= 0) & (re_ >= 0), (ln >= 0) & (re_ >= 0)
  assert nn.sum() and ee.sum() and ne.sum() and (nn | ee | ne).all()
  for f, mask in (("nn_prob", nn), ("ee_prob", ee), ("ne_prob", ne), ("left_weight", ne), ("right_weight", ne)):
    assert not np.isnan(arrays[f][mask]).any() and np.isnan(arrays[f][~mask]).all(), f
  for i in np.flatnonzero(nn):
    assert arrays["nn_prob"][i] == _reference_loop(*_row(NF, ln[i]), *_row(NF, rn[i])), i
  for i in np.flatnonzero(ee):
    assert arrays["ee_prob"][i] == _reference_loop(*_row(EF, le[i]), *_row(EF, re_[i])), i
  edge_c, node_c = {}, {}
  for i in np.flatnonzero(ne):
    if re_[i] not in edge_c:
      edge_c[re_[i]] = _centroid(AT, re_[i], NF)
    if ln[i] not in node_c:
      node_c[ln[i]] = _centroid(A, ln[i], EF)
    left = _reference_loop(*_row(NF, ln[i]), *edge_c[re_[i]])
    right = _reference_loop(*_row(EF, re_[i]), *node_c[ln[i]])
    assert arrays["left_weight"][i] == left and arrays["right_weight"][i] == right, i
    assert arrays["ne_prob"][i] == np.float32(left * right), i
  # and the float64 restatement to the bars of the host path
  truth = _float64_restatement(g, arrays)
  for f in PROBS:
    got, exact = np.nan_to_num(arrays[f]), np.nan_to_num(truth[f])
    assert np.all(np.abs(got - exact) <= RTOL * np.abs(exact) + 1e-5), (f, np.abs(got - exact).max())


def _zipf():
  """A 2000-node member of the zipf family with features of several values per row."""
  from hypergraphembedding_b200 import synthetic
  A = sps.csr_matrix(synthetic.zipf_hypergraph(2000, 1000, seed=8), dtype=np.float32)
  A.data[:] = 1
  NF = sps.csr_matrix(A.multiply((np.arange(A.shape[1]) % 7 + 1).astype(np.float32)[None, :]), dtype=np.float32)
  EF = sps.csr_matrix(A.T, dtype=np.float32)
  return A, NF, EF


def test_result_forms_weights_and_the_global_rng():
  import hypergraphembedding_b200 as H
  from test_hg2v_device_gpu import _same_columns
  A, NF, EF = _zipf()
  k = 3
  np.random.seed(4)
  state = np.random.get_state()
  timings = {}
  want = H.WeightedJaccardSamplesDevice(A, NF, EF, k, 5, seed=9, timings=timings)
  assert set(timings) == {"pairs", "neighbours", "probabilities"}
  kept = H.WeightedJaccardSamplesDevice(A, NF, EF, k, 5, seed=9, chunk_rows=97, keep_on_device=True)
  assert isinstance(kept, H.DeviceSampleColumns) and len(kept) == len(want)
  assert any(b.left_weight is not None and b.left_weight.is_cuda for b in kept.blocks)
  _same_columns(kept.to_host(), want)
  chunks = list(H.WeightedJaccardSamplesDevice(A, NF, EF, k, 5, seed=9, chunk_rows=301, stream=True))
  assert len(chunks) > 3
  _same_columns(H.SampleColumns.concatenate(chunks), want)
  with pytest.raises(AssertionError):
    H.WeightedJaccardSamplesDevice(A, NF, EF, k, 5, stream=True, keep_on_device=True)
  after = np.random.get_state()
  assert after[2] == state[2] and np.array_equal(after[1], state[1])
  # unit weights: the indices of the HOBE sampler at the same seed
  xn, xe = _vectors(A)
  hobe = H.AlgebraicDistanceSamplesDevice(A, xn, xe, k, 5, seed=9)
  for f in INDEX:
    assert np.array_equal(getattr(hobe, f), getattr(want, f)), f
  # row weights: int(w * num_samples) per row, as the reference
  nw = np.linspace(0, 2, A.shape[0])
  got = H.WeightedJaccardSamplesDevice(A, NF, EF, k, 5, node_weights=nw, seed=9)
  ref = jref.jaccard_pairs(A, k, 5, seed=9, node_weights=nw)
  for f in INDEX:
    assert np.array_equal(getattr(got, f).astype(np.int64), ref[f].astype(np.int64)), f


def test_packing_the_kept_blocks_equals_samples_to_model_input():
  import hypergraphembedding_b200 as H
  from hypergraphembedding_b200.hg2v_model import Hg2vModel
  from test_hg2v_device_gpu import _same_model_input
  A, NF, EF = _zipf()
  k = 3
  host = H.WeightedJaccardSamplesDevice(A, NF, EF, k, 6, seed=5)
  dev = H.WeightedJaccardSamplesDevice(A, NF, EF, k, 6, seed=5, keep_on_device=True)
  model = Hg2vModel.seeded(A.shape[0], A.shape[1], 8, k, "relu", "mean_squared_error", 3)
  try:
    history = model.fit_device(dev, batch_size=256, epochs=0, seed=1)
    assert history.history["loss"] == [] and dev.blocks == []
    assert model.num_samples == len(host)
    _same_model_input(model.samples(), H.SamplesToModelInput(host, k, weighted=False))
  finally:
    model.close()


def _fixture():
  g = load_golden("algdist_youtube")
  node_ids, edge_ids = g["node_ids"], g["edge_ids"]
  return hypergraph_from_pairs(np.stack([node_ids[np.searchsorted(node_ids, g["pairs"][:, 0])],
                                         edge_ids[np.searchsorted(edge_ids, g["pairs"][:, 1])]], axis=1))


@pytest.mark.parametrize("method", ["EmbedHg2vAdjJaccardDevice", "EmbedHg2vNeighborhoodWeightedJaccardDevice"])
def test_embed_device_end_to_end_on_the_fixture(method, caplog, monkeypatch):
  import hypergraphembedding_b200 as H
  from hypergraphembedding_b200.hg2v_model import Hg2vModel
  hg = _fixture()
  buffers = []
  set_samples = Hg2vModel.set_device_samples

  def spy(self, samples):
    set_samples(self, samples)
    buffers.append(self.samples())

  monkeypatch.setattr(Hg2vModel, "set_device_samples", spy)
  np.random.seed(0)
  state = np.random.get_state()
  with caplog.at_level(logging.INFO):
    emb = getattr(H, method)(hg, 8, num_samples=20, epochs=3, seed=5)
  getattr(H, method)(hg, 8, num_samples=20, epochs=1, seed=5)
  after = np.random.get_state()
  assert after[2] == state[2] and np.array_equal(after[1], state[1])
  assert len(buffers) == 2
  for a, b in zip(buffers[0][0] + buffers[0][1], buffers[1][0] + buffers[1][1]):
    assert np.array_equal(a, b)          # the sample buffer depends on the seed only
  assert emb.method_name == {"EmbedHg2vAdjJaccardDevice": "HG2V_ADJ_JAC",
                             "EmbedHg2vNeighborhoodWeightedJaccardDevice": "HG2V_NEIGH_JAC"}[method]
  assert emb.dim == 8
  assert sorted(emb.node) == sorted(hg.node) and sorted(emb.edge) == sorted(hg.edge)
  xn = np.asarray([emb.node[i].values for i in sorted(emb.node)])
  assert xn.shape == (len(hg.node), 8) and np.isfinite(xn).all()
  losses = [float(x) for x in re.findall(r"Epoch \d+/\d+ - loss: ([0-9.eE+-]+)", caplog.text)]
  assert len(losses) >= 2 and losses[-1] < losses[0], losses
  assert getattr(H, method) not in H.EMBEDDING_OPTIONS.values()


def test_refusals_leave_the_context_usable():
  import hypergraphembedding_b200 as H
  from hypergraphembedding_b200 import _native
  from hypergraphembedding_b200.hg2v_sample import _Graph
  A, NF, EF = _zipf()
  with pytest.raises(AssertionError):
    H.WeightedJaccardSamplesDevice(A, NF[:-1], EF, 3, 5)
  with pytest.raises(AssertionError):
    H.WeightedJaccardSamplesDevice(A, NF, EF[:-1], 3, 5)
  ctx = _native.default_context()
  import torch
  dev = torch.device("cuda", ctx.device)
  nfd = _native.FeatureCsr(NF).to_device(dev)
  g = _Graph.from_csr(A)
  inc = g.incidence(ctx)
  try:
    px, pg = _dev(np.arange(10)), _dev(np.arange(10))
    out = torch.empty(10, dtype=torch.float32, device=dev)

    def call(px, pg, side=1, f=nfd):
      return ctx.lib.hge_jaccard_centroid_grouped(
          ctx.handle, inc.handle, side, _native.ptr(nfd.ptr), _native.ptr(nfd.idx), _native.ptr(nfd.val),
          nfd.shape[0], int(nfd.idx.shape[0]), _native.ptr(f.ptr), _native.ptr(f.idx), _native.ptr(f.val),
          f.shape[0], int(f.idx.shape[0]), _native.ptr(px), _native.ptr(pg), int(px.shape[0]), 0,
          _native.ptr(out))

    bad_g = pg.clone()
    bad_g[7] = A.shape[1]
    assert call(px, bad_g) == _native.HGE_ERR_INVALID and "group" in _native.last_error()
    bad_x = px.clone()
    bad_x[3] = -1
    assert call(bad_x, pg) == _native.HGE_ERR_INVALID
    assert call(px, pg, side=0) == _native.HGE_ERR_INVALID     # F has node rows, the members are edges
    assert call(px, pg, side=2) == _native.HGE_ERR_INVALID
    # the context still works
    got = _native.jaccard_centroid_grouped(ctx, inc, 1, nfd, nfd, px, pg).cpu().numpy()
    want = _native.jaccard_centroid(ctx, _native.FeatureCsr(NF), g.b, _native.FeatureCsr(NF), np.arange(10),
                                    np.arange(10))
    assert np.array_equal(got, want)
  finally:
    inc.close()


def test_centroid_and_rows_refuse_out_of_range_pairs_on_host_and_device_arrays():
  """hge_jaccard_centroid and hge_jaccard_rows check every pair index before a kernel reads it: a
  row or group outside the matrix is HGE_ERR_INVALID on host and on device arrays, as are 2^31
  centroid pairs (refused before any array is read), and the context gives the restatement's
  values afterwards."""
  import torch
  from hypergraphembedding_b200 import _native
  A, NF, _ = _zipf()
  N, E = A.shape
  ctx = _native.default_context()
  dev = torch.device("cuda", ctx.device)
  feat = _native.FeatureCsr(NF)
  groups = _native.CsrArrays(sps.csr_matrix(A.T))     # edges with their nodes
  on = {False: (feat, groups.ptr, groups.idx),
        True: (feat.to_device(dev), torch.from_numpy(groups.ptr).to(dev), torch.from_numpy(groups.idx).to(dev))}
  P = _native.ptr

  def centroid(px, pg, on_device, n=None):
    f, gp, gi = on[on_device]
    px, pg = (_dev(px), _dev(pg)) if on_device else (_native._as_i32(px), _native._as_i32(pg))
    out = torch.empty(len(px), device=dev) if on_device else np.empty(len(px), np.float32)
    return ctx.lib.hge_jaccard_centroid(
        ctx.handle, P(f.ptr), P(f.idx), P(f.val), N, len(f.idx), P(gp), P(gi), E, len(gi), P(f.ptr), P(f.idx),
        P(f.val), N, len(f.idx), P(px), P(pg), len(px) if n is None else n, P(out),
        _native.MEM_DEVICE if on_device else _native.MEM_HOST)

  ok = np.arange(10)
  for on_device in (False, True):
    for bad in (-1, N):
      px = ok.copy()
      px[3] = bad
      assert centroid(px, ok, on_device) == _native.HGE_ERR_INVALID and "row" in _native.last_error()
    for bad in (-1, E):
      pg = ok.copy()
      pg[7] = bad
      assert centroid(ok, pg, on_device) == _native.HGE_ERR_INVALID and "group" in _native.last_error()
  assert centroid(ok, ok, False, n=1 << 31) == _native.HGE_ERR_INVALID
  for on_device in (False, True):
    fr = on[on_device][0]
    arr = _dev if on_device else np.asarray
    for bad in (-1, N):
      bad_i = ok.copy()
      bad_i[5] = bad
      with pytest.raises(AssertionError, match="outside"):
        _native.jaccard_rows(ctx, fr, arr(bad_i), arr(ok))
      with pytest.raises(AssertionError, match="outside"):
        _native.jaccard_rows(ctx, fr, arr(ok), arr(bad_i))
  # the context still works
  Fs = _scipy(feat)
  pi, pj = np.arange(10), np.arange(10)[::-1]
  want = np.asarray([_reference_loop(*_row(Fs, a), *_row(Fs, b)) for a, b in zip(pi, pj)], np.float32)
  assert np.array_equal(_native.jaccard_rows(ctx, feat, pi, pj), want)
  assert np.array_equal(_native.jaccard_rows(ctx, on[True][0], _dev(pi), _dev(pj)).cpu().numpy(), want)
  _centroid_factors_equal_the_restatement(A, NF, NF, 1, ok, ok, (0,))


def test_sampler_at_100k_nodes_with_a_small_budget():
  import hypergraphembedding_b200 as H
  from hypergraphembedding_b200 import synthetic
  from hypergraphembedding_b200.hg2v_sample import _Graph
  A = synthetic.zipf_hypergraph(100000, 50000, seed=2024)
  g = _Graph.from_csr(A)
  NF = sps.csr_matrix(g.A, dtype=np.float32)
  EF = sps.csr_matrix(g.B, dtype=np.float32)
  NF.data[:] = 1
  EF.data[:] = 1
  want = H.WeightedJaccardSamplesDevice(g, NF, EF, 5, 8, seed=3)
  got = H.WeightedJaccardSamplesDevice(g, NF, EF, 5, 8, seed=3, workspace_mb=16, chunk_rows=40000)
  assert len(want) > 1000000
  for f in want.FIELDS:
    a, b = getattr(got, f), getattr(want, f)
    assert np.array_equal(a, b, equal_nan=a.dtype.kind == "f"), f
  # a strided subset of the node-edge factors against the fp32 restatement (groups: the edge's
  # nodes are EF's pattern, the node's edges NF's)
  ne = np.flatnonzero((want.left_node >= 0) & (want.right_edge >= 0))
  for i in ne[::len(ne) // 300]:
    n, e = want.left_node[i], want.right_edge[i]
    assert want.left_weight[i] == _reference_loop(*_row(NF, n), *_centroid(EF, e, NF)), i
    assert want.right_weight[i] == _reference_loop(*_row(EF, e), *_centroid(NF, n, EF)), i
