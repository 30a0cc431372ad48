"""node2vec on the GPU (csrc/hge_n2v.cu) against oracle/node2vec_ref.py: walks, pairs (the windows
are visible through them) and negatives equal the restatement exactly for (p, q) in {(1, 1),
(0.25, 4), (4, 0.25)}, walk_length 1 and 80, isolated vertices and an edge of 120 000 members;
the input and output tables equal the fp32 restatement as uint32 after every epoch at dim 1 to 256
(every lane class), several batch sizes and a hub row named hundreds of times in one batch, with
__expf / __logf taken from the device; results are bit-identical run to run and for other plan
sizes; EmbedNode2VecDevice works end to end and leaves the global RNGs alone; and held-out
incidences of a planted-partition hypergraph are ranked above non-incidences."""
import ctypes
import random
import subprocess

import numpy as np
import pytest
import scipy.sparse as sps

from conftest import hypergraph_from_pairs
from oracle import node2vec_ref as ref

pytestmark = pytest.mark.gpu

_HELPER_SRC = r"""
#include <cuda_runtime.h>

__global__ void k_fast_math(const float* __restrict__ in, float* __restrict__ out, long long n, int which) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = which ? __logf(in[i]) : __expf(in[i]);
}

extern "C" int n2v_test_fast_math(const float* in, float* out, long long n, int which, cudaStream_t stream) {
  const long long blocks = (n + 255) / 256;
  if (n > 0) k_fast_math<<<(unsigned)(blocks < 4096 ? blocks : 4096), 256, 0, stream>>>(in, out, n, which);
  return (int)cudaGetLastError();
}
"""

PQ = [(1.0, 1.0), (0.25, 4.0), (4.0, 0.25)]


@pytest.fixture(scope="module")
def fast_math(tmp_path_factory):
  """(exp, log): the device's __expf / __logf, from a helper built with the library's nvcc and flags."""
  import torch
  from hypergraphembedding_b200 import _native, build
  tmp = tmp_path_factory.mktemp("n2v_fast_math")
  src, lib = tmp / "fast_math.cu", tmp / "libfast_math.so"
  src.write_text(_HELPER_SRC)
  run = subprocess.run([build.find_nvcc()] + build.NVCC_FLAGS + ["-shared", "-o", str(lib), str(src)],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
  assert run.returncode == 0, run.stdout
  fn = ctypes.CDLL(str(lib)).n2v_test_fast_math
  fn.restype = ctypes.c_int
  fn.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int, ctypes.c_void_p]
  dev = torch.device("cuda", _native.default_context().device)

  def call(x, which):
    x = np.ascontiguousarray(x, dtype=np.float32)
    a = torch.from_numpy(x.reshape(-1)).to(dev)
    out = torch.empty_like(a)
    with torch.cuda.device(dev):
      assert fn(a.data_ptr(), out.data_ptr(), a.numel(), which, torch.cuda.current_stream(dev).cuda_stream) == 0
    return out.cpu().numpy().reshape(x.shape)

  return (lambda x: call(x, 0)), (lambda x: call(x, 1))


def _csr(A):
  A = sps.csr_matrix(A, dtype=np.float32)
  A.sum_duplicates()
  A.sort_indices()
  return A


def _random_graph(N=60, E=25, density=0.12, seed=0):
  """random incidence with an isolated node (row 0) and an isolated edge (column 0)"""
  A = sps.random(N, E, density=density, random_state=seed, format="lil")
  A[0, :] = 0
  A[:, 0] = 0
  A = _csr(A)
  A.data[:] = 1
  A.eliminate_zeros()
  return A


def _star(members=120_000):
  """one edge of `members` nodes plus a small second edge"""
  rows = np.concatenate([np.arange(members), [0, 1, 2]])
  cols = np.concatenate([np.zeros(members, np.int64), [1, 1, 1]])
  return _csr(sps.csr_matrix((np.ones(len(rows)), (rows, cols)), shape=(members, 2)))


def _hub(N=300):
  """one edge holding every node, plus small edges: the hub edge is in about half of all pairs"""
  rows = list(range(N)) + [i for i in range(0, N, 3)] + [i for i in range(1, N, 5)]
  cols = [0] * N + [1 + (i // 3) % 7 for i in range(0, N, 3)] + [8 + (i // 5) % 4 for i in range(1, N, 5)]
  return _csr(sps.csr_matrix((np.ones(len(rows)), (rows, cols)), shape=(N, 12)))


def _ctx():
  from hypergraphembedding_b200 import _native
  return _native, _native.default_context()


def _device_walks(A, num_walks, L, p, q, seed):
  import torch
  from hypergraphembedding_b200.algebraic_distance import make_incidence
  _native, ctx = _ctx()
  V = sum(A.shape)
  walks = torch.empty((num_walks * V, L), dtype=torch.int32, device="cuda")
  counts = torch.empty(V, dtype=torch.int64, device="cuda")
  inc = make_incidence(A, ctx=ctx)
  try:
    _native.n2v_walks(ctx, inc, num_walks, L, p, q, seed, walks, counts)
  finally:
    inc.close()
  return walks, counts


def _device_pairs(walks, window, seed):
  import torch
  _native, ctx = _ctx()
  P = _native.n2v_pairs(ctx, walks, window, seed)
  pairs = torch.empty((P, 2), dtype=torch.int32, device="cuda")
  assert _native.n2v_pairs(ctx, walks, window, seed, pairs) == P
  return pairs


@pytest.mark.parametrize("pq", PQ)
@pytest.mark.parametrize("L", [1, 2, 80])
def test_walks_pairs_negatives_exact(pq, L):
  import torch
  A = _random_graph()
  p, q = pq
  walks, counts = _device_walks(A, 3, L, p, q, seed=11)
  want_w, want_c = ref.walks(A, 3, L, p, q, 11)
  assert np.array_equal(walks.cpu().numpy(), want_w)
  assert np.array_equal(counts.cpu().numpy(), want_c)
  V = sum(A.shape)
  assert np.all(want_w[np.arange(3 * V) % V == 0, 1:] == -1)   # node 0 is isolated
  for window in (1, 5):
    pairs = _device_pairs(walks, window, seed=12)
    want_p = ref.pairs(want_w, window, 12)
    assert np.array_equal(pairs.cpu().numpy(), want_p)
  _native, ctx = _ctx()
  cum = ref.noise_table(want_c)
  P = len(want_p)
  for epoch in (0, 3):
    out = torch.empty((P, 5), dtype=torch.int32, device="cuda")
    _native.n2v_negatives(ctx, P, torch.from_numpy(cum).cuda(), 5, 13, epoch, out)
    assert np.array_equal(out.cpu().numpy(), ref.negatives(cum, P, 5, 13, epoch))


@pytest.mark.parametrize("pq", PQ)
def test_walks_binary_search_of_a_large_edge(pq):
  A = _star()
  walks, counts = _device_walks(A, 1, 6, pq[0], pq[1], seed=3)
  want_w, want_c = ref.walks(A, 1, 6, pq[0], pq[1], 3)
  assert np.array_equal(walks.cpu().numpy(), want_w)
  assert np.array_equal(counts.cpu().numpy(), want_c)


def _train_case(A, dim, batch, epochs, fast_math, seed=5, negative=5, plan_bytes=0, num_walks=1, L=10, window=3):
  """device and fp32 restatement side by side; every epoch's tables compared as uint32"""
  import torch
  _native, ctx = _ctx()
  walks, counts = _device_walks(A, num_walks, L, 1.0, 1.0, seed)
  pairs = _device_pairs(walks, window, seed)
  cum_h = ref.noise_table(counts.cpu().numpy())
  cum = torch.from_numpy(cum_h).cuda()
  V = sum(A.shape)
  tin = torch.empty((V, dim), dtype=torch.float32, device="cuda")
  tout = torch.empty_like(tin)
  _native.n2v_init(ctx, seed, tin, tout)
  rin, rout = ref.init_tables(seed, V, dim)
  assert np.array_equal(tin.cpu().numpy().view(np.uint32), rin.view(np.uint32))
  assert not tout.cpu().numpy().any()
  pairs_h = pairs.cpu().numpy()
  exp, log = fast_math
  losses = []
  for e in range(epochs):
    loss = _native.n2v_train_epoch(ctx, tin, tout, pairs, cum, negative, seed, e, epochs, batch, 0.025, 1e-4,
                                   plan_bytes)
    want = ref.train32(rin, rout, pairs_h, cum_h, negative, seed, e, epochs, batch, exp=exp, log=log)
    assert np.array_equal(tin.cpu().numpy().view(np.uint32), rin.view(np.uint32)), "in table, epoch %d" % e
    assert np.array_equal(tout.cpu().numpy().view(np.uint32), rout.view(np.uint32)), "out table, epoch %d" % e
    assert loss == want, (e, loss, want)
    losses.append(loss)
  return tin.cpu().numpy(), tout.cpu().numpy(), losses, len(pairs_h)


@pytest.mark.parametrize("dim", [1, 7, 32, 33, 64, 65, 100, 128, 129, 200, 256])
def test_tables_exact_every_lane_class(dim, fast_math):
  _train_case(_random_graph(), dim, 97, 2, fast_math)


@pytest.mark.parametrize("batch", [1, 50, 256, 4096])
def test_tables_exact_with_hub_rows(batch, fast_math):
  """the hub edge is named hundreds of times in one batch (the ordered reduction needs no bound)"""
  A = _hub()
  _native, ctx = _ctx()
  walks, _ = _device_walks(A, 1, 10, 1.0, 1.0, 5)
  pairs = _device_pairs(walks, 3, 5).cpu().numpy()
  hub = A.shape[0]   # vertex of edge 0
  if batch >= 256:
    assert max(np.sum(pairs[i:i + batch] == hub) for i in range(0, len(pairs), batch)) >= 100
  _train_case(A, 48, batch, 2, fast_math, num_walks=1)


def test_reproducible_across_runs_and_plan_sizes(fast_math):
  A = _random_graph(seed=3)
  a = _train_case(A, 40, 64, 2, fast_math)
  b = _train_case(A, 40, 64, 2, fast_math, plan_bytes=1)        # one batch per chunk
  c = _train_case(A, 40, 64, 2, fast_math, plan_bytes=200_000)  # a few batches per chunk
  for other in (b, c):
    assert np.array_equal(a[0].view(np.uint32), other[0].view(np.uint32))
    assert np.array_equal(a[1].view(np.uint32), other[1].view(np.uint32))
    assert a[2] == other[2]


def test_no_negatives(fast_math):
  _train_case(_random_graph(), 16, 33, 2, fast_math, negative=0)


def test_library_refusals():
  import torch
  _native, ctx = _ctx()
  walks, counts = _device_walks(_random_graph(), 1, 4, 1.0, 1.0, 0)
  with pytest.raises(AssertionError, match="window"):
    _native.n2v_pairs(ctx, walks, 0, 0)
  pairs = _device_pairs(walks, 2, 0)
  with pytest.raises(AssertionError, match="room"):
    _native.n2v_pairs(ctx, walks, 2, 0, pairs[:-1].contiguous())
  V = counts.shape[0]
  tin = torch.zeros((V, 300), dtype=torch.float32, device="cuda")
  with pytest.raises(AssertionError, match="dimension"):
    _native.n2v_init(ctx, 0, tin, tin.clone())
  cum = torch.from_numpy(ref.noise_table(counts.cpu().numpy())).cuda()
  t = torch.zeros((V, 8), dtype=torch.float32, device="cuda")
  with pytest.raises(AssertionError, match="epoch"):
    _native.n2v_train_epoch(ctx, t, t.clone(), pairs, cum, 5, 0, 3, 3, 16, 0.025, 1e-4)
  with pytest.raises(AssertionError, match="batch_pairs"):
    _native.n2v_train_epoch(ctx, t, t.clone(), pairs, cum, 5, 0, 0, 1, 0, 0.025, 1e-4)


def test_embed_end_to_end():
  import hypergraphembedding_b200 as H
  from hypergraphembedding_b200.hypergraph_util import compressed_incidence
  A = _random_graph(N=40, E=15, density=0.2, seed=7).tocoo()
  hg = hypergraph_from_pairs(np.stack([A.row * 3 + 1, A.col * 5 + 2], axis=1))
  np.random.seed(0)
  random.seed(0)
  state, pystate = np.random.get_state(), random.getstate()
  emb = H.EmbedNode2VecDevice(hg, 16, walk_length=10, num_walks=2, epochs=2, seed=4)
  after = np.random.get_state()
  assert after[2] == state[2] and np.array_equal(after[1], state[1])
  assert random.getstate() == pystate
  assert emb.method_name == "N2V" and emb.dim == 16
  assert sorted(emb.node) == sorted(hg.node) and sorted(emb.edge) == sorted(hg.edge)
  node_ids, edge_ids, Ac = compressed_incidence(hg)
  X, info = H.Node2VecDevice(Ac, 16, walk_length=10, num_walks=2, epochs=2, seed=4)
  xn = np.asarray([emb.node[int(i)].values for i in node_ids], dtype=np.float32)
  xe = np.asarray([emb.edge[int(i)].values for i in edge_ids], dtype=np.float32)
  assert np.array_equal(xn.view(np.uint32), X[:len(node_ids)].view(np.uint32))
  assert np.array_equal(xe.view(np.uint32), X[len(node_ids):].view(np.uint32))
  assert len(info["losses"]) == 2 and info["num_pairs"] > 0
  assert H.EmbedNode2VecDevice not in H.EMBEDDING_OPTIONS.values()


# The float64 restatement at the same settings (d 128, 10 walks of 20, batch 64, 256 or 4096)
# reaches AUC 0.811 (DESIGN section 9.12).
AUC_BAR = 0.80


def test_quality_on_planted_partition():
  from hypergraphembedding_b200 import Node2VecDevice
  train, score = ref.held_out_auc(ref.planted_partition(seed=1), seed=2)
  X, info = Node2VecDevice(train, 128, walk_length=20, num_walks=10, seed=0)
  assert np.all(np.diff(info["losses"]) < 0)
  assert score(X) >= AUC_BAR
