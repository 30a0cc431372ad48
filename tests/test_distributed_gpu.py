"""Sharded relaxation with the real kernels: world_size 1 over NCCL on one GPU must equal the
single-GPU path; with >= 2 GPUs, 2 ranks must equal it too."""
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import dist_helpers
from oracle import port

pytestmark = pytest.mark.gpu


def _free_port():
  s = socket.socket()
  s.bind(("127.0.0.1", 0))
  p = s.getsockname()[1]
  s.close()
  return p


def _check(tmp_path, world, graph_args, R, iters):
  A = dist_helpers.make_graph(*graph_args)
  rng = np.random.default_rng(123)
  xn0 = rng.random((A.shape[0], R)).astype(np.float32)
  xe0 = rng.random((A.shape[1], R)).astype(np.float32)
  ref_xn, ref_xe = port.algdist_vectorised(A, A.T.tocsr(), xn0, xe0, iters)
  got_xn = np.zeros_like(ref_xn)
  for r in range(world):
    z = np.load(tmp_path / ("rank%d.npz" % r))
    got_xn[int(z["r0"]):int(z["r1"])] = z["xn"]
    assert np.abs(z["xe"] - ref_xe).max() < 2e-5
  assert np.abs(got_xn - ref_xn).max() < 2e-5


@pytest.mark.parametrize("slices,comm", [(1, "nccl"), (4, "nccl"), (1, "p2p")])
def test_one_rank(tmp_path, slices, comm):
  graph_args = (9, 20000, 700, 150000)
  mp.spawn(dist_helpers.worker,
           args=(1, _free_port(), "nccl", graph_args, 32, 8, slices, str(tmp_path), True, comm),
           nprocs=1, join=True)
  _check(tmp_path, 1, graph_args, 32, 8)


@pytest.mark.parametrize("world", [1, 2])
def test_peer_memory_sweep_with_node_range_tiles(tmp_path, world):
  """The shard's edge gather in node-range tiles (1 MB tiles forced on every worker's context):
  partial sums accumulated per tile, then pushed to their owners."""
  if torch.cuda.device_count() < world:
    pytest.skip("needs %d GPUs" % world)
  graph_args = (12, 60000, 800, 400000)
  mp.spawn(dist_helpers.worker,
           args=(world, _free_port(), "nccl", graph_args, 32, 6, 1, str(tmp_path), True, "p2p", 1),
           nprocs=world, join=True)
  _check(tmp_path, world, graph_args, 32, 6)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("comm,R", [("nccl", 32), ("p2p", 32), ("p2p", 10)])
def test_two_ranks(tmp_path, comm, R):
  """2 ranks on 2 GPUs; the peer-memory exchange and the NCCL exchange give the oracle's result."""
  graph_args = (10, 30000, 900, 250000)
  mp.spawn(dist_helpers.worker,
           args=(2, _free_port(), "nccl", graph_args, R, 8, 4 if comm == "nccl" else 1,
                 str(tmp_path), True, comm),
           nprocs=2, join=True)
  _check(tmp_path, 2, graph_args, R, 8)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_ranks_p2p_is_reproducible(tmp_path):
  graph_args = (11, 20000, 500, 200000)
  outs = []
  for rep in range(2):
    d = tmp_path / ("rep%d" % rep)
    d.mkdir()
    mp.spawn(dist_helpers.worker,
             args=(2, _free_port(), "nccl", graph_args, 32, 6, 1, str(d), True, "p2p"),
             nprocs=2, join=True)
    outs.append([np.load(d / ("rank%d.npz" % r)) for r in range(2)])
  for r in range(2):
    assert np.array_equal(outs[0][r]["xn"], outs[1][r]["xn"])
    assert np.array_equal(outs[0][r]["xe"], outs[1][r]["xe"])
