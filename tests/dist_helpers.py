"""Test infrastructure for the multi-rank relaxation: a numpy stand-in for the per-rank kernels
(same protocol as hypergraphembedding_b200.distributed.NativeOps: Y rows are kept un-rescaled,
the previous sweep's affine map is applied lazily, min / max travel as order-preserving int32
encodings of fp32) and the worker functions the spawn-based tests run."""
import os

import numpy as np
import scipy.sparse as sps


def enc(x):
  i = np.asarray(x, dtype=np.float32).view(np.int32)
  return i ^ ((i >> 31) & 0x7fffffff)


def dec(i):
  i = np.asarray(i, dtype=np.int32)
  return (i ^ ((i >> 31) & 0x7fffffff)).view(np.float32)


class NumpyOps(object):

  def __init__(self, A_local, R, iterations, num_slices):
    import torch
    self.torch = torch
    self.A = sps.csr_matrix(A_local).astype(np.float64)
    self.B = self.A.T.tocsr()
    node_deg = np.diff(self.A.indptr)
    if np.any(node_deg == 0):
      raise ZeroDivisionError("a local node has no incidence")
    self.w_n = 1.0 / node_deg
    self.R, self.E = R, self.A.shape[1]
    self.iterations = iterations
    self.bounds = [self.E * k // num_slices for k in range(num_slices + 1)]
    self.ld = R
    self._deg = torch.from_numpy(np.diff(self.B.indptr).astype(np.int32))
    self._wsum = torch.from_numpy(np.asarray(self.B @ self.w_n, dtype=np.float64))

  def edge_sums(self):
    return self._deg, self._wsum

  def finish(self):
    self.w_e = 1.0 / self._deg.numpy().astype(np.float64)
    self.inv_s_n = 1.0 / (self.A @ self.w_e)
    self.inv_s_e = (1.0 / self._wsum.numpy()).astype(np.float32).astype(np.float64)
    mm = np.empty((max(1, self.iterations), 2, self.R), dtype=np.int32)
    mm[:, 0] = np.iinfo(np.int32).max
    mm[:, 1] = np.iinfo(np.int32).min
    self.mm = self.torch.from_numpy(mm)

  def new_partial_buffer(self):
    return self.torch.zeros((self.E, self.R), dtype=self.torch.float32)

  def slice_range(self, k):
    return self.bounds[k], self.bounds[k + 1]

  def load(self, xn, xe):
    self.xn = np.asarray(xn, dtype=np.float64).copy()
    self.xe = np.asarray(xe, dtype=np.float64).copy()

  def _affine(self, t):
    if t == 0:
      return np.zeros(self.R), np.ones(self.R)
    m = self.mm[t - 1].numpy()
    lo, hi = dec(m[0]).astype(np.float64), dec(m[1]).astype(np.float64)
    return lo, 1.0 / (hi - lo)

  def _track(self, t, x):
    m = self.mm[t].numpy()
    m[0] = np.minimum(m[0], enc(x.min(axis=0)))
    m[1] = np.maximum(m[1], enc(x.max(axis=0)))

  def node_half(self, t):
    lo, inv = self._affine(t)
    own = (self.xn - lo) * inv
    edges = (self.xe - lo) * inv
    self.xn = 0.5 * (own + (self.A @ (edges * self.w_e[:, None])) * self.inv_s_n[:, None])
    self._track(t, self.xn)

  def edge_partial(self, t, k, partial):
    r0, r1 = self.slice_range(k)
    sums = self.B[r0:r1] @ (self.xn * self.w_n[:, None])
    partial[r0:r1] = self.torch.from_numpy(sums.astype(np.float32))

  def edge_finalize(self, t, k, partial):
    r0, r1 = self.slice_range(k)
    lo, inv = self._affine(t)
    own = (self.xe[r0:r1] - lo) * inv
    total = partial[r0:r1].numpy().astype(np.float64)
    self.xe[r0:r1] = 0.5 * (own + total * self.inv_s_e[r0:r1, None])
    self._track(t, self.xe[r0:r1])

  def minmax(self, t):
    return self.mm[t]

  def store(self, sweeps_done, xn, xe):
    lo, inv = self._affine(sweeps_done)
    xn[...] = ((self.xn - lo) * inv).astype(xn.dtype)
    xe[...] = ((self.xe - lo) * inv).astype(xe.dtype)

  def close(self):
    pass


def make_graph(seed, n, e, nnz):
  rng = np.random.default_rng(seed)
  rows = np.concatenate([rng.integers(0, n, nnz), np.arange(n), rng.integers(0, n, e)])
  cols = np.concatenate([rng.integers(0, e, nnz), rng.integers(0, e, n), np.arange(e)])
  m = sps.csr_matrix((np.ones(len(rows), dtype=bool), (rows, cols)), shape=(n, e), dtype=bool)
  m.sum_duplicates()
  m.sort_indices()
  return m


def worker(rank, world, port, backend, graph_args, R, iters, slices, out_dir, use_native,
           comm="nccl", tile_mb=0):
  """Runs the sharded relaxation on one rank and writes its node block to out_dir.  tile_mb > 0
  forces node-range tiles of that many MB on the rank's context, whatever the edge sizes."""
  os.environ["MASTER_ADDR"] = "127.0.0.1"
  os.environ["MASTER_PORT"] = str(port)
  import torch
  import torch.distributed as dist
  from hypergraphembedding_b200 import distributed as hd
  if use_native:
    torch.cuda.set_device(rank % torch.cuda.device_count())
  dist.init_process_group(backend=backend, rank=rank, world_size=world)
  try:
    A = make_graph(*graph_args)
    rng = np.random.default_rng(123)
    xn0 = rng.random((A.shape[0], R)).astype(np.float32)
    xe0 = rng.random((A.shape[1], R)).astype(np.float32)
    A_loc, r0, r1 = hd.local_shard(A, rank, world)
    if tile_mb:
      from hypergraphembedding_b200 import _native
      _native.default_context().set_tile_mb(tile_mb, 0)
    relax = hd.ShardedRelaxation(A_loc, R, iters, num_slices=slices, comm=comm,
                                 ops_factory=None if use_native else NumpyOps)
    assert relax.use_p2p == (comm == "p2p")
    if use_native:
      xn = torch.from_numpy(xn0[r0:r1].copy()).cuda()
      xe = torch.from_numpy(xe0.copy()).cuda()
      relax.run(xn, xe)
      torch.cuda.synchronize()
      xn, xe = xn.cpu().numpy(), xe.cpu().numpy()
      if relax.use_p2p:
        # a second relaxation of the same shape re-uses the pooled exchange arena
        relax.close()
        relax = hd.ShardedRelaxation(A_loc, R, iters, num_slices=slices, comm=comm)
        assert len(hd._ARENA_POOL) == 1 and len(list(hd._ARENA_POOL.values())[0]) == 1
        xn2 = torch.from_numpy(xn0[r0:r1].copy()).cuda()
        xe2 = torch.from_numpy(xe0.copy()).cuda()
        relax.run(xn2, xe2)
        torch.cuda.synchronize()
        assert np.array_equal(xn2.cpu().numpy(), xn) and np.array_equal(xe2.cpu().numpy(), xe)
    else:
      xn, xe = xn0[r0:r1].copy(), xe0.copy()
      relax.run(xn, xe)
    relax.close()
    hd.release_peer_arenas(dist)
    assert not hd._ARENA_POOL
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), xn=xn, xe=xe, r0=r0, r1=r1)
  finally:
    dist.destroy_process_group()


class NumpyPairOps(object):
  """numpy stand-in for the pair-distance kernels behind distributed.sharded_pair_weights."""

  def pair_l2(self, xa, xb, ia, ib):
    d = np.asarray(xa, np.float64)[ia] - np.asarray(xb, np.float64)[ib]
    return np.sqrt((d * d).sum(1)).astype(np.float32)

  def minmax(self, d):
    return (float(d.min()), float(d.max())) if len(d) else (float("inf"), float("-inf"))

  def apply(self, d, alpha, lo, hi):
    d = np.asarray(d, dtype=np.float32)
    span = np.float32(hi) - np.float32(lo)
    scaled = np.ones_like(d) if span == 0 else (d - np.float32(lo)) / span
    return (np.float32(alpha) + np.float32(1 - alpha) * (np.float32(1) - scaled)).astype(np.float32)


def pair_worker(rank, world, port, backend, seed, num_pairs, alpha, out_dir, use_native):
  """Weights of this rank's slice of a pair list (distributed.sharded_pair_weights)."""
  os.environ["MASTER_ADDR"] = "127.0.0.1"
  os.environ["MASTER_PORT"] = str(port)
  import torch
  import torch.distributed as dist
  from hypergraphembedding_b200 import distributed as hd
  if use_native:
    torch.cuda.set_device(rank % torch.cuda.device_count())
  dist.init_process_group(backend=backend, rank=rank, world_size=world)
  try:
    rng = np.random.default_rng(seed)
    xa = rng.random((500, 12)).astype(np.float32)
    xb = rng.random((300, 12)).astype(np.float32)
    ia = rng.integers(0, 500, num_pairs).astype(np.int32)
    ib = rng.integers(0, 300, num_pairs).astype(np.int32)
    lo, hi = num_pairs * rank // world, num_pairs * (rank + 1) // world
    if rank == world - 1 and world > 1:
      lo = hi                                    # one rank without pairs must not break the bounds
    w = hd.sharded_pair_weights(xa, xb, ia[lo:hi], ib[lo:hi], alpha,
                                ops=None if use_native else NumpyPairOps())
    np.savez(os.path.join(out_dir, "pairs%d.npz" % rank), w=np.asarray(w), lo=lo, hi=hi)
  finally:
    dist.destroy_process_group()


def failure_worker(rank, world, port, backend, graph_args, out_dir):
  """A node without incidences on the LAST rank only: every rank must raise (the same
  ZeroDivisionError the reference raises) instead of one raising and the others waiting in the
  next collective."""
  os.environ["MASTER_ADDR"] = "127.0.0.1"
  os.environ["MASTER_PORT"] = str(port)
  import datetime
  import torch.distributed as dist
  from hypergraphembedding_b200 import distributed as hd
  dist.init_process_group(backend=backend, rank=rank, world_size=world,
                          timeout=datetime.timedelta(seconds=60))
  outcome = "no error"
  try:
    A = make_graph(*graph_args).tolil()
    A[A.shape[0] - 3, :] = 0                      # lives in the last rank's block
    A = sps.csr_matrix(A)
    A.eliminate_zeros()
    A_loc, r0, r1 = hd.local_shard(A, rank, world)
    try:
      hd.ShardedRelaxation(A_loc, 4, 2, ops_factory=NumpyOps)
    except ZeroDivisionError as exc:
      outcome = "ZeroDivisionError: %s" % exc
    except Exception as exc:      # noqa: BLE001
      outcome = "%s: %s" % (type(exc).__name__, exc)
    with open(os.path.join(out_dir, "outcome%d.txt" % rank), "w") as f:
      f.write(outcome)
  finally:
    dist.destroy_process_group()
