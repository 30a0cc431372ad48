"""k_hg2v_epoch (csrc/hge_hg2v_train.cu) bit for bit against its fp32 restatement
(oracle/hg2v_train_ref.py): the node and edge tables after EVERY epoch compared as uint32, signed
zeros included, so that a failure names the first bad epoch; the epoch loss within M * 2^-52
relative (the per-warp double sums meet in unordered atomics).  __expf and __logf are taken from
the device itself (a helper built with the library's compiler and flags).

The inputs are what makes bits comparable: samples come in batch-aligned groups in which every
(table, row) is named at most twice among the gradient targets (ln, rn, nn_i on the node side, le,
re, ne_i on the edge side), so every gradient element receives at most two atomic contributions
and its value does not depend on their order.  Double hits are built on purpose: inside one sample
(ln == rn, rn == nn_i, le == re), and across samples of one CTA, of different CTAs and of different
clusters; the padding row 0 is named in at most two columns of a group.  Epoch orders permute the
whole groups and the samples inside each group; the short last group stays last.

Geometry: every instance DPL 1, 2, 4, 8 with partial and full column slots and both dispatch
boundaries (dim 1 .. 256), k on both sides of the preload limit (8 / 9 at dim <= 32) and k = 14
(cols = 32), all four (activation, loss) pairs, batches 1 .. 4096 with ragged last batches, cluster
caps 0 .. 3, samples and orders from host and device memory.  Values: uniform +-0.7 rows, wide rows
(sigmoid saturates to 1.0f, relu outputs far above 1), dyadic rows (dot products exactly 0 and 1),
rows with subnormal entries (subnormal contributions), targets 0, 1 and 1e-8 among random ones.
The restatement's boundary counters, summed over the file, show each boundary was compared.

Runtime: the restatement is numpy on the host and dominates; the file takes 37 s on one NVIDIA
B200 (1000 W power limit)."""
import ctypes
import subprocess

import numpy as np
import pytest

from oracle import hg2v_train_ref as ref

pytestmark = pytest.mark.gpu

_HELPER_SRC = r"""
#include <cuda_runtime.h>

__global__ void k_fast_math(const float* __restrict__ in, float* __restrict__ out, long long n, int which) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = which ? __logf(in[i]) : __expf(in[i]);
}

extern "C" int hg2v_test_fast_math(const float* in, float* out, long long n, int which, cudaStream_t stream) {
  const long long blocks = (n + 255) / 256;
  if (n > 0) k_fast_math<<<(unsigned)(blocks < 4096 ? blocks : 4096), 256, 0, stream>>>(in, out, n, which);
  return (int)cudaGetLastError();
}
"""

ACT = {"sigmoid": 0, "relu": 1}
LOSS = {"kld": 0, "mse": 1}
TRACE = {}
_TRACED = set()


@pytest.fixture(scope="module")
def fast_math(tmp_path_factory):
  """(exp, log): fp32 array -> the device's __expf / __logf of it, from a helper compiled by the
  library's nvcc with its flags into pytest's temporary directory."""
  import torch
  from hypergraphembedding_b200 import _native, build
  tmp = tmp_path_factory.mktemp("hg2v_fast_math")
  src, lib = tmp / "fast_math.cu", tmp / "libfast_math.so"
  src.write_text(_HELPER_SRC)
  run = subprocess.run([build.find_nvcc()] + build.NVCC_FLAGS + ["-shared", "-o", str(lib), str(src)],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
  assert run.returncode == 0, run.stdout
  fn = ctypes.CDLL(str(lib)).hg2v_test_fast_math
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


def test_device_fast_math_is_exp_and_log(fast_math):
  """The helper computes exp and log within the CUDA Programming Guide's bounds for the intrinsics:
  __expf 2 + floor(|1.173 x|) ulp; __logf 2^-21.41 absolute on [0.5, 2], 3 ulp elsewhere."""
  exp, log = fast_math
  x = np.concatenate([np.linspace(-87, 88, 200001), np.random.RandomState(0).randn(10000) * 10]).astype(np.float32)
  got = exp(x).astype(np.float64)
  want = np.exp(x.astype(np.float64))
  normal = want >= np.finfo(np.float32).tiny
  ulp = np.spacing(want.astype(np.float32)).astype(np.float64)
  bound = (2 + np.floor(np.abs(1.173 * x.astype(np.float64)))) * ulp
  assert np.all(np.abs(got - want)[normal] <= bound[normal])
  y = np.concatenate([np.geomspace(1e-37, 1e37, 200001), np.random.RandomState(1).rand(10000) * 1.5 + 0.5])
  y = y.astype(np.float32)
  got = log(y).astype(np.float64)
  want = np.log(y.astype(np.float64))
  near = (y >= 0.5) & (y <= 2)
  assert np.all(np.abs(got - want)[near] <= 2 ** -21.41)
  ulp = np.spacing(np.abs(want).astype(np.float32)).astype(np.float64)
  assert np.all(np.abs(got - want)[~near] <= 3 * ulp[~near])


# ---- inputs -------------------------------------------------------------------------------------

def _make_equal(V, a, b):
  """V[b] = V[a] keeping every value at most twice: swap the other copy of V[a] into b."""
  r = V[a]
  other = [p for p in zip(*np.nonzero(V == r)) if p != a]
  if other:
    q = other[0]
    V[q], V[b] = V[b], V[q]
  else:
    V[b] = r


def _group_slots(rng, g, k, rows):
  """[g, 2 + k] row ids, each of 1 .. rows at most twice, with in-sample double hits (columns 0
  and 1, 1 and 2) and row 0 in at most two slots."""
  V = rng.permutation(np.tile(np.arange(1, rows + 1), 2))[:g * (2 + k)].reshape(g, 2 + k)
  for s in rng.choice(g, max(1, g // 16), replace=False):
    if k and rng.random() < 0.5:
      _make_equal(V, (s, 1), (s, 2 + rng.integers(k)))
    else:
      _make_equal(V, (s, 0), (s, 1))
  for _ in range(rng.integers(0, 3)):
    V[rng.integers(g), rng.integers(2 + k)] = 0
  assert np.bincount(V[V > 0], minlength=1).max() <= 2 and np.count_nonzero(V == 0) <= 2
  return V


def _table(rng, rows, dim, values):
  if values == "uniform":
    return rng.uniform(-0.7, 0.7, (rows, dim)).astype(np.float32)
  T = rng.uniform(-0.7, 0.7, (rows, dim))
  kind = rng.integers(0, 10, rows)
  wide = kind < 2                                  # sigmoid saturates, relu far above 1
  T[wide] = rng.uniform(-1, 1, (np.count_nonzero(wide), dim)) * 2.0 ** rng.integers(1, 5, (np.count_nonzero(wide), 1))
  dyadic = (kind >= 2) & (kind < 5)                # exact 0 and 1 dot products
  T[dyadic] = rng.choice([-1.0, -0.5, 0.0, 0.5, 1.0], (np.count_nonzero(dyadic), dim))
  sub = kind == 5                                  # some entries subnormal
  mask = sub[:, None] & (rng.random((rows, dim)) < 0.5)
  T[mask] = rng.uniform(-1, 1, np.count_nonzero(mask)) * 2.0 ** -130
  return T.astype(np.float32)


def _problem(seed, dim, k, batch, M, values):
  """(N0, E0, feats [4 + 2k][M] int32, targets [3][M] float32, groups): samples of group q are
  q * batch .. min(M, (q + 1) * batch) - 1."""
  rng = np.random.default_rng(seed)
  g = min(batch, M)
  rows = (g * (2 + k) + 1) // 2 + 2
  feats = np.zeros((4 + 2 * k, M), np.int32)
  groups = []
  for first in range(0, M, batch):
    n = min(batch, M - first)
    node = _group_slots(rng, n, k, rows)             # ln, rn, nn_0 ..
    edge = _group_slots(rng, n, k, rows)             # re, le, ne_0 ..
    sl = slice(first, first + n)
    feats[0, sl], feats[2, sl] = node[:, 0], node[:, 1]
    feats[3, sl], feats[1, sl] = edge[:, 0], edge[:, 1]
    feats[4:4 + k, sl] = node[:, 2:].T
    feats[4 + k:, sl] = edge[:, 2:].T
    groups.append(np.arange(first, first + n))
  t = rng.random((3, M))
  special = rng.random((3, M)) < 0.3
  t[special] = rng.choice([0.0, 1.0, 1e-8], np.count_nonzero(special))
  return (_table(rng, rows + 1, dim, values), _table(rng, rows + 1, dim, values), feats,
          t.astype(np.float32), groups)


def _order(rng, groups):
  """whole full groups permuted, samples permuted inside each; a short last group stays last"""
  full = [q for q in groups if len(q) == len(groups[0])]
  tail = groups[len(full):]
  return np.concatenate([rng.permutation(full[i]) for i in rng.permutation(len(full))] +
                        [rng.permutation(q) for q in tail]).astype(np.int32)


# ---- device -------------------------------------------------------------------------------------

class _Model(object):
  def __init__(self, N0, E0, k, activation, loss):
    from hypergraphembedding_b200 import _native
    self.ctx = _native.default_context()
    self.lib = self.ctx.lib
    self.shape = N0.shape, E0.shape
    self.handle = _native.c_vp()
    _native.check(self.lib.hge_hg2v_create(self.ctx.handle, N0.shape[0], E0.shape[0], N0.shape[1], k,
                                           ACT[activation], LOSS[loss], _native.ptr(N0), _native.ptr(E0),
                                           _native.MEM_HOST, ctypes.byref(self.handle)))

  def set_samples(self, feats, targets, mem):
    from hypergraphembedding_b200 import _native
    f, t = np.ascontiguousarray(feats), np.ascontiguousarray(targets)
    if mem == _native.MEM_DEVICE:
      f, t = _on_device(f), _on_device(t)
    _native.check(self.lib.hge_hg2v_set_samples(self.handle, _native.ptr(f), _native.ptr(t), feats.shape[1], mem))

  def epoch(self, order, batch, mem):
    from hypergraphembedding_b200 import _native
    o = np.ascontiguousarray(order, dtype=np.int32)
    if mem == _native.MEM_DEVICE:
      o = _on_device(o)
    loss = ctypes.c_double()
    _native.check(self.lib.hge_hg2v_fit_epoch(self.handle, _native.ptr(o), int(batch), mem, ctypes.byref(loss)))
    return loss.value, int(self.lib.hge_hg2v_last_clusters(self.handle))

  def weights(self):
    from hypergraphembedding_b200 import _native
    N = np.empty(self.shape[0], np.float32)
    E = np.empty(self.shape[1], np.float32)
    _native.check(self.lib.hge_hg2v_get_weights(self.handle, _native.ptr(N), _native.ptr(E), _native.MEM_HOST))
    return N, E

  def close(self):
    self.lib.hge_hg2v_destroy(self.handle)


def _on_device(a):
  import torch
  from hypergraphembedding_b200 import _native
  return torch.from_numpy(a).to(torch.device("cuda", _native.default_context().device))


def _first_difference(got, want):
  bad = np.argwhere(got.view(np.uint32) != want.view(np.uint32))
  if len(bad) == 0:
    return None
  r, c = bad[0]
  return "%d elements differ, first at row %d column %d: %r (0x%08x) vs %r (0x%08x)" % (
      len(bad), r, c, got[r, c], got.view(np.uint32)[r, c], want[r, c], want.view(np.uint32)[r, c])


def _train(fast_math, seed, dim, k, activation, loss, batch, M, values, epochs=3, cap=0, mem=0, test=None):
  """Trains on the device and in the restatement, comparing after every epoch.  Returns the
  device's tables per epoch and the clusters of each launch."""
  from hypergraphembedding_b200 import _native
  exp, log = fast_math
  N0, E0, feats, targets, groups = _problem(seed, dim, k, batch, M, values)
  rng = np.random.default_rng(seed + 1)
  orders = [_order(rng, groups) for _ in range(epochs)]
  trainer = ref.Trainer(N0, E0, k, activation, loss, exp=exp, log=log, trace=TRACE)
  ctx = _native.default_context()
  model = _Model(N0, E0, k, activation, loss)
  history = []
  try:
    ctx.set_trainer_clusters(cap)
    model.set_samples(feats, targets, mem)
    for e, order in enumerate(orders):
      got_loss, clusters = model.epoch(order, batch, mem)
      with np.errstate(over="ignore", divide="ignore", invalid="ignore"):
        want_loss = trainer.epoch(feats, targets, order, batch, clusters=clusters)
      N, E = model.weights()
      for name, got, want in (("node", N, trainer.N), ("edge", E, trainer.E)):
        diff = _first_difference(got, want)
        assert diff is None, "epoch %d (of %d), %s table, %d clusters: %s" % (e, epochs, name, clusters, diff)
      assert abs(got_loss - want_loss) <= M * 2.0 ** -52 * abs(want_loss), (e, got_loss, want_loss)
      history.append((N, E, clusters))
  finally:
    ctx.reset_tuning()
    model.close()
  assert np.any(history[-1][0] != N0) and np.any(history[-1][1] != E0)    # and it did train
  if test:
    _TRACED.add(test)
  return history


# (dim, k, activation, loss, batch, M): each dim 1 .. 256 boundary, each k, each pair, each batch
_GEOMETRY = [
    (1, 0, "sigmoid", "kld", 1, 24),
    (5, 1, "relu", "mse", 31, 100),
    (31, 8, "relu", "kld", 32, 100),
    (32, 9, "sigmoid", "mse", 100, 250),
    (32, 14, "relu", "mse", 256, 600),
    (1, 14, "sigmoid", "kld", 257, 600),
    (33, 7, "sigmoid", "kld", 257, 600),
    (48, 2, "relu", "kld", 300, 700),
    (64, 13, "sigmoid", "mse", 1000, 2300),
    (65, 8, "relu", "mse", 256, 520),
    (96, 0, "sigmoid", "kld", 100, 230),
    (128, 1, "relu", "kld", 4096, 8300),
    (129, 2, "sigmoid", "mse", 32, 100),
    (200, 9, "relu", "mse", 1000, 2100),
    (255, 7, "sigmoid", "kld", 300, 650),
    (256, 14, "sigmoid", "mse", 4096, 4200),
    (256, 0, "relu", "kld", 31, 70),
    (5, 8, "sigmoid", "kld", 1000, 2300),
]


@pytest.mark.parametrize("values", ["uniform", "mixed"])
@pytest.mark.parametrize("dim,k,activation,loss,batch,M", _GEOMETRY)
def test_epochs_match_the_restatement_bit_for_bit(fast_math, dim, k, activation, loss, batch, M, values):
  _train(fast_math, 1000 * dim + 10 * k + batch % 7, dim, k, activation, loss, batch, M, values, test="geometry")


@pytest.mark.parametrize("dim,k,activation,loss", [(16, 3, "relu", "mse"), (40, 9, "sigmoid", "kld")])
def test_cluster_caps_give_identical_bits(fast_math, dim, k, activation, loss):
  """Caps 0 .. 3 on batches of 1000 (four clusters wanted): every cap equals the restatement at its
  own cluster count, and all are the same bits.  Uniform values keep every row-0 contribution
  normal, where the CTA split cannot change a bit (checked in the restatement too)."""
  runs = [_train(fast_math, 7 + dim, dim, k, activation, loss, 1000, 2300, "uniform", cap=cap, test="caps")
          for cap in (0, 1, 2, 3)]
  assert [r[0][2] for r in runs][1:] == [1, 2, 3] and runs[0][0][2] >= 3
  for r in runs[1:]:
    for (n, e, _), (n0, e0, _) in zip(r, runs[0]):
      assert np.array_equal(n.view(np.uint32), n0.view(np.uint32))
      assert np.array_equal(e.view(np.uint32), e0.view(np.uint32))


@pytest.mark.parametrize("dim,k,batch,M", [(32, 8, 300, 700), (200, 13, 100, 250)])
def test_device_samples_and_orders_give_the_same_bits(fast_math, dim, k, batch, M):
  from hypergraphembedding_b200 import _native
  host = _train(fast_math, 3 + k, dim, k, "relu", "kld", batch, M, "mixed", mem=_native.MEM_HOST, test="mem")
  dev = _train(fast_math, 3 + k, dim, k, "relu", "kld", batch, M, "mixed", mem=_native.MEM_DEVICE, test="mem")
  for (n, e, _), (n0, e0, _) in zip(dev, host):
    assert np.array_equal(n.view(np.uint32), n0.view(np.uint32))
    assert np.array_equal(e.view(np.uint32), e0.view(np.uint32))


def test_every_boundary_was_compared():
  """The restatement's counters over the cases above: each boundary occurred in a compared epoch."""
  if _TRACED != {"geometry", "caps", "mem"}:
    pytest.skip("counts boundaries over the whole file; ran only %s" % sorted(_TRACED))
  missed = [key for key in ref.TRACE_KEYS if not TRACE.get(key)]
  assert not missed, (missed, TRACE)
