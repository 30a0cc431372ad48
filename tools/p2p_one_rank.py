"""The peer-memory sweep on ONE rank (world size 1: every push goes to the rank's own staging
block), for the phase split of a p2p sweep without a second GPU:

    python tools/p2p_one_rank.py
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402
from bench import WORKLOADS, build_workload  # noqa: E402
from hypergraphembedding_b200 import _native, synthetic  # noqa: E402
from hypergraphembedding_b200 import distributed as hd  # noqa: E402


def main():
  os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
  os.environ.setdefault("MASTER_PORT", "29877")
  dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", 0))
  spec = WORKLOADS["c2"]
  A, B = build_workload(spec)
  R, sweeps = spec["R"], spec["sweeps"]
  ctx = _native.default_context(0)
  xn0, xe0 = synthetic.legacy_initial_vectors(A.shape[0], A.shape[1], R, seed=0)
  relax = hd.ShardedRelaxation(A, R, sweeps, comm="p2p", ctx=ctx, B_local=B)
  assert relax.use_p2p
  xn, xe = torch.from_numpy(xn0).cuda(), torch.from_numpy(xe0).cuda()
  for rep in range(3):
    relax.ops.load(xn, xe)
    relax.ops.arena.set_timing(True)
    for t in range(sweeps):
      relax.sweep(t)
    ms5, n = relax.ops.arena.phase_ms()
    relax.ops.arena.set_timing(False)
  print(json.dumps({"sweeps": n,
                    "phases_ms": dict(zip(("node_half", "gather", "barrier_a", "reduce", "barrier_b"),
                                          [round(v, 4) for v in ms5]))}), flush=True)
  relax.close()
  hd.release_peer_arenas(dist)
  dist.destroy_process_group()


if __name__ == "__main__":
  main()
