"""The relaxation on the GPU equals oracle/sweep_ref.py (its fp32 restatement in the device's
operation order) bit for bit: xn, xe and the per-sweep min / max as uint32, signed zeros included.

The graph gives node rows and edge rows every degree where the schedule changes shape: 1-5, 7, 8
(where a light row's own slot falls on a step boundary), 127-129 (light / long at the default),
255, 256, 1023-1025 and 2049 (chunk boundaries; 65 chunks with chunk = 32).  R covers every lane
width (1 .. 32 lanes per row), inactive lanes, R % 4 != 0 and 1 .. 3 column slabs.  When a full
run disagrees, test_stepwise_halves says which half does first."""
import numpy as np
import pytest

from oracle import sweep_ref as sr

pytestmark = pytest.mark.gpu

SPECIAL_DEGREES = [1, 2, 3, 4, 5, 7, 8, 127, 128, 129, 255, 256, 1023, 1024, 1025, 2049]
R_VALUES = [1, 2, 3, 4, 5, 8, 9, 16, 17, 31, 32, 33, 64, 65, 128, 129, 200, 257]
INPUTS = ("uniform", "signed", "wide")
TUNINGS = [None, (1, 32), (255, 64), (8, 32)]      # (light_max_deg, chunk); None: the defaults


def bipartite_with_degrees(node_deg, edge_deg, rng):
  """N x E bool CSR (sorted indices) with exactly these row and column degrees: edges by
  descending degree each take the nodes with the most incidences left (Gale-Ryser greedy), ties
  broken at random; node and edge labels shuffled afterwards."""
  import scipy.sparse as sps
  node_deg = np.asarray(node_deg, np.int64)
  edge_deg = np.asarray(edge_deg, np.int64)
  assert node_deg.sum() == edge_deg.sum()
  left = node_deg.astype(np.float64) + rng.random(len(node_deg)) * 0.5
  rows, cols = [], []
  for e in np.argsort(-edge_deg, kind="stable"):
    d = int(edge_deg[e])
    pick = np.argpartition(-left, d - 1)[:d]
    assert (left[pick] >= 1).all(), "degree sequences are not bipartite-graphical"
    left[pick] -= 1
    rows.append(pick)
    cols.append(np.full(d, e))
  rows, cols = np.concatenate(rows), np.concatenate(cols)
  pn, pe = rng.permutation(len(node_deg)), rng.permutation(len(edge_deg))
  A = sps.csr_matrix((np.ones(len(rows), bool), (pn[rows], pe[cols])), shape=(len(node_deg), len(edge_deg)))
  A.sort_indices()
  assert A.nnz == len(rows)
  return A


def special_graph(seed=0, n=2600):
  rng = np.random.default_rng(seed)
  filler = rng.integers(1, 7, n - len(SPECIAL_DEGREES))
  node_deg = np.concatenate([SPECIAL_DEGREES, filler])
  edge_deg = np.concatenate([SPECIAL_DEGREES, rng.permutation(filler)])
  return bipartite_with_degrees(node_deg, edge_deg, rng)


def vectors(kind, n, R, rng):
  if kind == "uniform":
    return rng.random((n, R)).astype(np.float32)
  if kind == "signed":
    x = (rng.random((n, R)) * 2 - 1).astype(np.float32)
    z = rng.random((n, R)) < 0.1
    x[z] = np.where(rng.random(int(z.sum())) < 0.5, np.float32(0.0), np.float32(-0.0))
    return x
  mag = 10.0 ** rng.uniform(-3, 3, (n, R))
  return (mag * np.where(rng.random((n, R)) < 0.5, -1, 1)).astype(np.float32)


def assert_bits(got, want, what):
  got = np.ascontiguousarray(got, np.float32).view(np.uint32)
  want = np.ascontiguousarray(want, np.float32).view(np.uint32)
  assert got.shape == want.shape, what
  bad = np.argwhere(got != want)
  assert len(bad) == 0, "%s: %d words differ, first at %s: %#x, restated %#x" % (
      what, len(bad), tuple(bad[0]), got[tuple(bad[0])], want[tuple(bad[0])])


@pytest.fixture(scope="module")
def graph():
  A = special_graph()
  return A, sr.Incidence.from_csr(A)


def _inputs(A, R, kind, seed):
  rng = np.random.default_rng(seed)
  return vectors(kind, A.shape[0], R, rng), vectors(kind, A.shape[1], R, rng)


def _tuned(ctx, tuning, blocks_per_sm=0):
  ctx.reset_tuning()
  light, chunk = tuning or (0, 0)
  ctx.set_tuning(light, chunk, blocks_per_sm)


CASES = [(R, (1, 2, 20)[i % 3], INPUTS[(i // 3 + i) % 3]) for i, R in enumerate(R_VALUES)]


@pytest.mark.parametrize("R,sweeps,kind", CASES)
def test_run_from_host_arrays(R, sweeps, kind, graph, gpu_ctx):
  from hypergraphembedding_b200 import algebraic_distance as ad
  A, ref = graph
  xn0, xe0 = _inputs(A, R, kind, R)
  want_n, want_e, want_mm = sr.relax(ref, xn0, xe0, sweeps)
  inc = ad.make_incidence(A, ctx=gpu_ctx)
  try:
    xn, xe = xn0.copy(), xe0.copy()
    lohi = np.zeros((sweeps, 2, R), np.float32)
    ad.relax(inc, xn, xe, sweeps, lohi=lohi)
  finally:
    inc.close()
  assert_bits(lohi, want_mm, "lohi")
  assert_bits(xn, want_n, "xn")
  assert_bits(xe, want_e, "xe")


@pytest.mark.parametrize("tuning", TUNINGS)
@pytest.mark.parametrize("R", [3, 33, 129])
def test_tunings_and_pieces(tuning, R, graph, gpu_ctx):
  """Every (light_max_deg, chunk) the restatement is told about, and 1, 3 or 32 blocks per SM
  (different pieces, same order): the same bits as the restatement."""
  from hypergraphembedding_b200 import algebraic_distance as ad
  A, ref = graph
  light, chunk = tuning or (sr.DEFAULT_LIGHT_MAX, sr.DEFAULT_CHUNK)
  xn0, xe0 = _inputs(A, R, "signed", 100 + R)
  sweeps = 3
  want_n, want_e, want_mm = sr.relax(ref, xn0, xe0, sweeps, light_max=light, chunk=chunk)
  try:
    for bps in (1, 3, 32):
      _tuned(gpu_ctx, tuning, bps)
      inc = ad.make_incidence(A, ctx=gpu_ctx)
      try:
        xn, xe = xn0.copy(), xe0.copy()
        lohi = np.zeros((sweeps, 2, R), np.float32)
        ad.relax(inc, xn, xe, sweeps, lohi=lohi)
      finally:
        inc.close()
      assert_bits(lohi, want_mm, "lohi, %d blocks per SM" % bps)
      assert_bits(xn, want_n, "xn, %d blocks per SM" % bps)
      assert_bits(xe, want_e, "xe, %d blocks per SM" % bps)
  finally:
    gpu_ctx.reset_tuning()


@pytest.mark.parametrize("kind", ["wide", "signed"])
def test_device_arrays_and_the_one_call_path(kind, graph, gpu_ctx):
  """hge_algdist_run on device tensors, hge_algdist_run_csr with one orientation from host and
  from device arrays: the restatement's bits on each."""
  import torch
  from hypergraphembedding_b200 import _native
  from hypergraphembedding_b200 import algebraic_distance as ad
  from hypergraphembedding_b200.hypergraph_util import csr_arrays
  A, ref = graph
  R, sweeps = 17, 20
  xn0, xe0 = _inputs(A, R, kind, 7)
  want_n, want_e, want_mm = sr.relax(ref, xn0, xe0, sweeps)
  inc = ad.make_incidence(A, ctx=gpu_ctx)
  try:
    xn, xe = torch.from_numpy(xn0.copy()).cuda(), torch.from_numpy(xe0.copy()).cuda()
    lohi = np.zeros((sweeps, 2, R), np.float32)
    ad.relax(inc, xn, xe, sweeps, lohi=lohi)
    torch.cuda.synchronize()
  finally:
    inc.close()
  assert_bits(lohi, want_mm, "device run: lohi")
  assert_bits(xn.cpu().numpy(), want_n, "device run: xn")
  assert_bits(xe.cpu().numpy(), want_e, "device run: xe")
  a_ptr, a_idx = csr_arrays(A)
  for device in (False, True):
    lohi = np.zeros((sweeps, 2, R), np.float32)
    if device:
      dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
      xn, xe = dev(xn0), dev(xe0)
      _native.algdist_run_csr(gpu_ctx, A.shape[0], A.shape[1], dev(a_ptr.astype(np.int64)),
                              dev(a_idx.astype(np.int32)), xn, xe, sweeps, lohi=lohi)
      torch.cuda.synchronize()
      xn, xe = xn.cpu().numpy(), xe.cpu().numpy()
    else:
      xn, xe = xn0.copy(), xe0.copy()
      _native.algdist_run_csr(gpu_ctx, A.shape[0], A.shape[1], a_ptr, a_idx, xn, xe, sweeps, lohi=lohi)
    assert_bits(lohi, want_mm, "run_csr (device %s): lohi" % device)
    assert_bits(xn, want_n, "run_csr (device %s): xn" % device)
    assert_bits(xe, want_e, "run_csr (device %s): xe" % device)


def _minmax(state, sweep, ld, R):
  import torch
  from hypergraphembedding_b200.distributed import _CudaView
  view = torch.as_tensor(_CudaView(state.minmax_ptr(sweep), (2, ld), "<i4"), device="cuda")
  torch.cuda.synchronize()
  return sr.dec(view.cpu().numpy()[:, :R].copy())


@pytest.mark.parametrize("R", [5, 32, 129])
def test_stepwise_halves(R, graph, gpu_ctx):
  """load -> node_half(0) -> store(0, ...) pins the node half alone; then edge_half(0) ->
  store(0, ...) and sweep 1 through the map of sweep 0."""
  from hypergraphembedding_b200 import _native
  from hypergraphembedding_b200 import algebraic_distance as ad
  A, ref = graph
  xn0, xe0 = _inputs(A, R, "signed", 300 + R)
  st_ref = sr.Relaxation(ref, R)
  st_ref.load(xn0, xe0)
  inc = ad.make_incidence(A, ctx=gpu_ctx)
  try:
    st = _native.AlgDistState(gpu_ctx, inc, R, 2)
    try:
      st.load(xn0, xe0)
      xn, xe = np.empty_like(xn0), np.empty_like(xe0)
      st.node_half(0)
      st_ref.node_half(0)
      st.store(0, xn, xe)
      want_n, want_e = st_ref.store(0)
      assert_bits(xn, want_n, "node half 0: xn")
      assert_bits(xe, want_e, "node half 0: xe (untouched)")
      assert_bits(_minmax(st, 0, st.ld, R), st_ref.lohi()[0], "node half 0: min / max")
      st.edge_half(0)
      st_ref.edge_half(0)
      st.store(0, xn, xe)
      want_n, want_e = st_ref.store(0)
      assert_bits(xe, want_e, "edge half 0: xe")
      assert_bits(_minmax(st, 0, st.ld, R), st_ref.lohi()[0], "sweep 0: min / max")
      st.node_half(1)
      st_ref.node_half(1)
      st.store(0, xn, xe)
      want_n, want_e = st_ref.store(0)
      assert_bits(xn, want_n, "node half 1: xn")
      st.edge_half(1)
      st_ref.edge_half(1)
      st.store(2, xn, xe)
      want_n, want_e = st_ref.store(2)
      assert_bits(xn, want_n, "sweep 1, rescaled: xn")
      assert_bits(xe, want_e, "sweep 1, rescaled: xe")
      assert_bits(_minmax(st, 1, st.ld, R), st_ref.lohi()[1], "sweep 1: min / max")
    finally:
      st.close()
  finally:
    inc.close()


def tiled_graph(seed=1, n=20000, e=300):
  """Every node in one or two edges; edge sizes from 1 to 9000, so that the member lists of the
  large edges cross the tile boundaries with sub-ranges that are light, long and multi-chunk."""
  import scipy.sparse as sps
  rng = np.random.default_rng(seed)
  sizes = np.concatenate([[9000, 5000, 2049, 1025, 300, 129, 128, 127], rng.integers(1, 9, e - 8)])
  w = sizes / sizes.sum()
  rows = np.concatenate([np.arange(n), rng.integers(0, n, n // 2), rng.integers(0, n, e)])
  cols = np.concatenate([rng.choice(e, n + n // 2, p=w), np.arange(e)])
  A = sps.csr_matrix((np.ones(len(rows), bool), (rows, cols)), shape=(n, e))
  A.sum_duplicates()
  A.sort_indices()
  return A


@pytest.mark.parametrize("R", [32, 129])
def test_node_range_tiles(R, gpu_ctx):
  """The edge half in node-range tiles (set_tile_mb(1, 0): 8192 rows at R = 32, 1985 at
  R = 129): per-tile schedules over the sub-ranges, raw sums added tile by tile, then
  k_edge_finalize -- the restatement's bits."""
  from hypergraphembedding_b200 import algebraic_distance as ad
  A = tiled_graph()
  ref = sr.Incidence.from_csr(A)
  tile_rows = (1 << 20) // (((R + 3) & ~3) * 4)
  assert A.shape[0] > 2 * tile_rows
  xn0, xe0 = _inputs(A, R, "signed", 500 + R)
  sweeps = 3
  want_n, want_e, want_mm = sr.relax(ref, xn0, xe0, sweeps, edge_path=("tiled", tile_rows))
  try:
    gpu_ctx.set_tile_mb(1, 0)
    inc = ad.make_incidence(A, ctx=gpu_ctx)
    try:
      xn, xe = xn0.copy(), xe0.copy()
      lohi = np.zeros((sweeps, 2, R), np.float32)
      ad.relax(inc, xn, xe, sweeps, lohi=lohi)
    finally:
      inc.close()
  finally:
    gpu_ctx.reset_tuning()
  assert_bits(lohi, want_mm, "tiled: lohi")
  assert_bits(xn, want_n, "tiled: xn")
  assert_bits(xe, want_e, "tiled: xe")


@pytest.mark.parametrize("num_slices", [1, 3])
def test_sharded_single_rank(num_slices, graph, gpu_ctx):
  """One shard holding every node: edge_sums / finish_sharded, then per sweep node_half,
  edge_partial and edge_finalize for every slice -- the restatement's sharded path."""
  import torch
  from hypergraphembedding_b200 import _native
  from hypergraphembedding_b200.hypergraph_util import csr_arrays
  A, ref = graph
  R, sweeps = 31, 3
  B = A.T.tocsr()
  B.sort_indices()
  a_ptr, a_idx = csr_arrays(A)
  b_ptr, b_idx = csr_arrays(B)
  xn0, xe0 = _inputs(A, R, "wide", 900 + num_slices)
  want_n, want_e, want_mm = sr.relax(ref, xn0, xe0, sweeps, edge_path=("sharded", num_slices))
  inc = _native.Incidence(gpu_ctx, A.shape[0], A.shape[1], a_ptr, a_idx, b_ptr, b_idx, sharded=True,
                          num_slices=num_slices)
  try:
    inc.edge_sums()                 # one rank: the all-reduce of these is the identity
    inc.finish_sharded()
    st = _native.AlgDistState(gpu_ctx, inc, R, sweeps)
    try:
      partial = torch.zeros((A.shape[1], st.ld), dtype=torch.float32, device="cuda")
      torch.cuda.synchronize()        # the library's stream need not be torch's
      st.load(xn0, xe0)
      for t in range(sweeps):
        st.node_half(t)
        for k in range(num_slices):
          st.edge_partial(t, k, partial)
        for k in range(num_slices):
          st.edge_finalize(t, k, partial)
      mm = np.stack([_minmax(st, t, st.ld, R) for t in range(sweeps)])
      xn, xe = np.empty_like(xn0), np.empty_like(xe0)
      st.store(sweeps, xn, xe)
    finally:
      st.close()
  finally:
    inc.close()
  assert_bits(mm, want_mm, "sharded: lohi")
  assert_bits(xn, want_n, "sharded: xn")
  assert_bits(xe, want_e, "sharded: xe")
