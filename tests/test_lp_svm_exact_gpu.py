"""hge_lp_svm_predict bit for bit against its numpy restatement (oracle/lp_svm_ref.py).  For every
named owner the device's training set equals `ref.training_sets`, its coef, rho and SMO iteration
count equal `ref.solve` on that set, and every link's decision value equals
`ref.decision_device_order`; the kernel entries' exp is taken from the device's own expf (a helper
built with the library's compiler and flags), so nothing is compared to a tolerance.

Cases: training-set sizes on both sides of the warp / CTA solver boundary (32 / 33) and of the CTA's
stride (256 / 257) next to a ~3 000-point owner in one call, d from 1 to 200, C / gamma / tol off
their defaults, degenerate geometry (vectors shared by members and non-members, or nearly shared so
that K rounds to 1, identical points, points too far apart for K to be non-zero off the diagonal), a 1 MB workspace budget, and a sample
of owners of a 100 000-node graph.  The restatement's branch counters, summed over the file, show
that every branch of the solver ran in a case that compared equal."""
import ctypes
import subprocess

import numpy as np
import pytest
import scipy.sparse as sps

from oracle import lp_svm_ref as ref

pytestmark = pytest.mark.gpu

_EXPF_SRC = r"""
#include <cuda_runtime.h>
#include <math.h>

__global__ void k_expf(const float* __restrict__ in, float* __restrict__ out, long long n) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = expf(in[i]);
}

extern "C" int lp_svm_test_expf(const float* in, float* out, long long n, cudaStream_t stream) {
  const long long blocks = (n + 255) / 256;
  if (n > 0) k_expf<<<(unsigned)(blocks < 4096 ? blocks : 4096), 256, 0, stream>>>(in, out, n);
  return (int)cudaGetLastError();
}
"""

# branch counters of every restated owner of the file (test_every_branch_was_compared reads them)
TRACE = {}
_TRACED = set()


@pytest.fixture(scope="module")
def device_exp(tmp_path_factory):
  """fp32 array -> the device's expf of it.  The helper is compiled by the library's nvcc with its
  flags (no fast math), so its expf is the sequence rbf() inlines."""
  import torch
  from hypergraphembedding_b200 import _native, build
  tmp = tmp_path_factory.mktemp("expf")
  src, lib = tmp / "expf.cu", tmp / "libexpf.so"
  src.write_text(_EXPF_SRC)
  run = subprocess.run([build.find_nvcc()] + build.NVCC_FLAGS + ["-shared", "-o", str(lib), str(src)],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
  assert run.returncode == 0, run.stdout
  fn = ctypes.CDLL(str(lib)).lp_svm_test_expf
  fn.restype = ctypes.c_int
  fn.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_longlong, ctypes.c_void_p]
  dev = torch.device("cuda", _native.default_context().device)

  def exp(x):
    x = np.ascontiguousarray(x, dtype=np.float32)
    a = torch.from_numpy(x.reshape(-1)).to(dev)
    out = torch.empty_like(a)
    with torch.cuda.device(dev):
      assert fn(a.data_ptr(), out.data_ptr(), a.numel(), torch.cuda.current_stream(dev).cuda_stream) == 0
    return out.cpu().numpy().reshape(x.shape)

  return exp


def _vectors(rows, d, seed):
  rng = np.random.RandomState(seed)
  return (rng.randn(rows, d) * 0.5 * np.sqrt(32.0 / d)).astype(np.float32)


def _graph(members, items, per_edge):
  """N x E incidence CSR whose owners (edges when `per_edge`, else nodes) 0, 1, ... have the member
  lists `members` among `items` items."""
  pairs = np.asarray([(o, i) for o, ms in enumerate(members) for i in ms], dtype=np.int64).reshape(-1, 2)
  M = sps.csr_matrix((np.ones(len(pairs), dtype=bool), (pairs[:, 0], pairs[:, 1])), shape=(len(members), items))
  M = sps.csr_matrix(M.T if per_edge else M)
  M.sum_duplicates()
  M.sort_indices()
  return M


def _owners(sizes, items, seed):
  """random member lists of the given sizes among `items` items"""
  rng = np.random.RandomState(seed)
  return [np.sort(rng.choice(items, m, replace=False)) for m in sizes]


def _links(owners, items, per_edge, per_owner, seed):
  """(node, edge) rows: `per_owner` random items for each owner in `owners`"""
  rng = np.random.RandomState(seed)
  o = np.repeat(np.asarray(owners, dtype=np.int64), per_owner)
  i = rng.randint(0, items, len(o))
  return np.stack([i, o] if per_edge else [o, i], axis=1)


def _members(A, per_edge):
  M = sps.csr_matrix(A.T if per_edge else A)
  M.sort_indices()
  return M.indptr.astype(np.int64), M.indices.astype(np.int64)


def _bits(a):
  return np.asarray(a, dtype=np.float64).view(np.int64)


def _predict(A, X, links, per_edge, seed, C, gamma, tol, workspace_mb):
  """the public entry point: keep, decision (host arrays) and the model"""
  import torch
  from hypergraphembedding_b200 import _native
  from hypergraphembedding_b200.hg2v_sample import _Graph
  ctx = _native.default_context()
  dev = torch.device("cuda", ctx.device)
  items, owners = (links[:, 0], links[:, 1]) if per_edge else (links[:, 1], links[:, 0])
  as_i32 = lambda a: torch.as_tensor(np.asarray(a, dtype=np.int32)).to(dev)
  inc = _Graph.from_csr(A).incidence(ctx)
  try:
    keep, decision, capped, model = _native.lp_svm_predict(
        ctx, inc, 1 if per_edge else 0, torch.as_tensor(X).to(dev), as_i32(items), as_i32(owners), seed, C, gamma,
        tol, workspace_mb, return_model=True)
  finally:
    inc.close()
  assert capped == 0
  return keep.cpu().numpy(), decision.cpu().numpy(), model


def _check(exp, A, X, links, per_edge, seed=1, C=1.0, gamma=0.1, tol=1e-3, workspace_mb=0, test=None):
  """every named owner's model and every link's decision bit-equal to the restatement; returns the
  training-set size of each named owner"""
  X = np.asarray(X, dtype=np.float32)
  keep, decision, model = _predict(A, X, links, per_edge, seed, C, gamma, tol, workspace_mb)
  mptr, midx = _members(A, per_edge)
  owner_col, item_col = (1, 0) if per_edge else (0, 1)
  named = np.unique(links[:, owner_col])
  assert model.owner_ids.tolist() == named.tolist()
  phase = ref.PHASE_LP_EDGE_OWNERS if per_edge else ref.PHASE_LP_NODE_OWNERS
  sets = ref.training_sets(mptr, midx, X.shape[0], named, seed, phase)
  sizes = []
  for u, o in enumerate(named.tolist()):
    lo, hi = int(model.offset[u]), int(model.offset[u + 1])
    pts = model.point_ids[lo:hi]
    mem, neg = sets[o]
    assert pts.tolist() == mem.tolist() + neg.tolist(), o
    n, m = len(pts), int(mptr[o + 1] - mptr[o])
    sizes.append(n)
    if n:
      y = np.r_[np.ones(len(mem)), -np.ones(len(neg))]
      alpha, rho, it = ref.solve(X[pts], y, C, gamma, tol, exp=exp, trace=TRACE)
      coef = y * alpha
    else:
      coef, rho, it = np.zeros(0), (np.inf if m == 0 else -np.inf), 0
    got = model.coef[lo:hi]
    what = "owner %d (n %d, m %d): device %d iterations, rho %r; restated %d, %r" % (
        o, n, m, model.iterations[u], model.rho[u], it, rho)
    assert model.iterations[u] == it, what
    bad = np.nonzero(_bits(got) != _bits(coef))[0]
    assert len(bad) == 0, "%s; coef differs at %d points, first %d: %r vs %r" % (
        what, len(bad), bad[0], got[bad[0]], coef[bad[0]])
    assert _bits(model.rho[u]) == _bits(rho), what
    sel = np.nonzero(links[:, owner_col] == o)[0]
    want = ref.decision_device_order(X[pts], coef, rho, X[links[sel, item_col]], gamma, exp)
    bad = np.nonzero(_bits(decision[sel]) != _bits(want))[0]
    assert len(bad) == 0, "%s; decision differs at %d of %d links, first %r vs %r" % (
        what, len(bad), len(sel), decision[sel][bad[0]], want[bad[0]])
    assert np.array_equal(keep[sel], want > 0), what
  if test:
    _TRACED.add(test)
  return sizes


def test_device_expf_is_an_exp(device_exp):
  """the helper computes exp: within CUDA's documented 2 ulp of expf wherever the result is normal"""
  x = np.concatenate([np.linspace(-104, 0, 200001), -np.random.RandomState(0).rand(10000) * 20]).astype(np.float32)
  got = device_exp(x)
  want = np.exp(x.astype(np.float64))
  normal = want >= np.finfo(np.float32).tiny
  ulp = np.spacing(want.astype(np.float32)).astype(np.float64)
  assert np.all(np.abs(got - want)[normal] <= 2 * ulp[normal])
  assert np.all((got[~normal] >= 0) & (got[~normal] < np.finfo(np.float32).tiny))
  print("device expf: %d of %d arguments differ from numpy's exp; %d subnormal results" % (
      np.count_nonzero(got != ref.exp32(x)), len(x), np.count_nonzero((got > 0) & ~normal)))


# (items, member counts, d): owners of n = 3M points when N - M >= 2M, else of N points
_LAYOUTS = [
    (3003, [0, 1, 10, 11, 85, 1001, 3003], 32),   # n 0, 3, 30, 33, 255, 3003, 0
    (257, [1, 11, 85, 86, 200], 3),                # n 3, 33, 255, 257, 257
    (256, [10, 86, 128, 255], 1),                  # n 30, 256, 256, 256
    (33, [1, 11, 32], 33),                         # n 3, 33, 33
    (32, [11, 20, 31], 200),                       # n 32, 32, 32
    (31, [1, 11, 15, 30], 32),                     # n 3, 31, 31, 31
    (2, [1, 1, 0, 2], 3),                          # n 2, 2, 0, 0
    (1200, [400, 700], 200),                       # n 1200, 1200: the transposed gather at d = 200
]


@pytest.mark.parametrize("per_edge", [True, False])
@pytest.mark.parametrize("layout", range(len(_LAYOUTS)))
def test_sizes_at_the_path_boundaries(device_exp, layout, per_edge):
  items, counts, d = _LAYOUTS[layout]
  A = _graph(_owners(counts, items, layout), items, per_edge)
  X = _vectors(items, d, 10 + layout)
  links = _links(range(len(counts)), items, per_edge, 12, layout)
  sizes = _check(device_exp, A, X, links, per_edge, seed=layout, test="sizes")
  want = [0 if m in (0, items) else m + min(items - m, 2 * m) for m in counts]
  assert sizes == want


# (C, gamma, tol, d); gamma = 10 at d = 32 sends most entries to zero and some to subnormals
_PARAMETERS = [
    (0.05, 0.1, 1e-3, 32),
    (50.0, 0.1, 1e-6, 8),
    (1.0, 1e-4, 1e-3, 32),
    (0.05, 1e-4, 1e-6, 3),
    (1.0, 10.0, 1e-1, 32),
    (50.0, 10.0, 1e-6, 32),
    (1.0, 0.1, 1e-1, 3),
]


@pytest.mark.parametrize("per_edge", [True, False])
@pytest.mark.parametrize("C,gamma,tol,d", _PARAMETERS)
def test_parameters(device_exp, C, gamma, tol, d, per_edge):
  items, counts = 600, [1, 5, 10, 40, 150, 400]
  A = _graph(_owners(counts, items, 20), items, per_edge)
  X = _vectors(items, d, 21)
  links = _links(range(len(counts)), items, per_edge, 20, 22)
  _check(device_exp, A, X, links, per_edge, seed=23, C=C, gamma=gamma, tol=tol, test="parameters")


def _geometry(kind):
  """(items, member counts, vectors)"""
  rng = np.random.RandomState(30)
  if kind == "palette":   # 3 distinct rows: members and non-members share vectors
    return 300, [1, 4, 10, 20, 50, 100, 200], rng.randn(3, 3).astype(np.float32)[rng.randint(0, 3, 300)]
  if kind == "near":
    # the palette moved by ~1e-4: K rounds to exactly 1 inside a cluster (quad = 0) while the
    # gradients differ, so TAU, not the tie-break, decides which of the cluster is chosen
    X = rng.randn(3, 3)[rng.randint(0, 3, 300)] + rng.randn(300, 3) * 1e-4
    return 300, [1, 4, 10, 20, 50, 100, 200], X.astype(np.float32)
  if kind == "identical":
    return 100, [1, 5, 10, 20, 40, 70], np.full((100, 4), 0.7, np.float32)
  # at least 40 apart: gamma 0.1 * 1600 puts K below the smallest subnormal off the diagonal
  return 200, [1, 5, 10, 50, 120], (40.0 * rng.permutation(200)).astype(np.float32)[:, None]


@pytest.mark.parametrize("per_edge", [True, False])
@pytest.mark.parametrize("kind", ["palette", "near", "identical", "far"])
def test_degenerate_geometry(device_exp, kind, per_edge):
  items, counts, X = _geometry(kind)
  A = _graph(_owners(counts, items, 31), items, per_edge)
  links = _links(range(len(counts)), items, per_edge, 16, 32)
  _check(device_exp, A, X, links, per_edge, seed=33, test="geometry")
  if kind == "far":
    assert np.all(ref.kernel(X, X, 0.1, device_exp) == np.eye(items, dtype=np.float32))


@pytest.mark.parametrize("per_edge", [True, False])
def test_workspace_budget_of_1_mb(device_exp, per_edge):
  # 24 + 4 d = 156 bytes a point: 1 800 + 2 100 + 2 400 points in one batch, 2 700 + 3 000 in another
  items, counts, d = 3000, [600, 700, 800, 900, 1000], 33
  A = _graph(_owners(counts, items, 40), items, per_edge)
  X = _vectors(items, d, 41)
  links = _links(range(len(counts)), items, per_edge, 20, 42)
  sizes = _check(device_exp, A, X, links, per_edge, seed=43, workspace_mb=1, test="budget")
  assert sum(sizes) * (24 + 4 * d) > 1 << 20 and min(sizes) * (24 + 4 * d) < 1 << 19


@pytest.mark.parametrize("per_edge", [True, False])
def test_sample_of_a_100k_node_graph(device_exp, per_edge):
  from hypergraphembedding_b200 import synthetic
  A = synthetic.zipf_hypergraph(100000, 50000, seed=2024)
  mptr, _ = _members(A, per_edge)
  items = A.shape[0] if per_edge else A.shape[1]
  m = np.diff(mptr)
  n = np.where((m == 0) | (m == items), 0, m + np.minimum(items - m, 2 * m))
  largest = np.argsort(n, kind="stable")[-20:]
  rng = np.random.RandomState(50)
  owners = np.union1d(largest, rng.choice(len(m), 200, replace=False))
  X = _vectors(items, 32, 51)
  links = _links(owners, items, per_edge, 4, 52)
  sizes = _check(device_exp, A, X, links, per_edge, seed=3, test="zipf")
  assert max(sizes) > 1000


def test_every_branch_was_compared():
  """the restatement's branch counters over the owners compared above: bit-equality covered each"""
  cases = {"sizes", "parameters", "geometry", "budget", "zipf"}
  if _TRACED != cases:
    pytest.skip("counts branches over the whole file; ran only %s" % sorted(_TRACED))
  missed = [k for k in ref.TRACE_KEYS if not TRACE.get(k)]
  assert not missed, (missed, TRACE)
