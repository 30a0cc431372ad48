"""node2vec on the GPU (hypergraphembedding_b200.node2vec):

  walks     config 2 (synthetic.power_law_hypergraph(1 000 000, 500 000, 10 000 000, seed=1234)),
            10 walks of 80 vertices per vertex, p = q = 1: CUDA-event milliseconds of
            hge_n2v_walks and walks / s (its pair set, about 10^10 pairs, does not fit the device).
  pipeline  synthetic.power_law_hypergraph(100 000, 50 000, 1 000 000), d = 128, one walk of 80
            vertices per vertex and one epoch (the other settings at their defaults): milliseconds of
            the walks, the pairs and the training (which includes building the per-chunk plan), the
            training rate in pairs / s, and the table bytes a pair gathers, computed from shapes: the
            coefficient step reads in[c] and S rows of out, the delta step S rows of out and S rows
            of in (S = 1 + negative), 4 d bytes each, so (1 + 3 S) 4 d bytes before any row repeats.
  host      the numpy walk restatement (oracle/node2vec_ref.py) at 1/100 of config 2
            (power_law_hypergraph(10 000, 5 000, 100 000)), one walk of 80 vertices per vertex: wall
            seconds on the host's cores.  A host number, not a GPU number.

The GPU's name and power limit are read in the same run.

    python tools/n2v_bench.py --out DIR
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from device_sampler_bench import gpu_info  # noqa: E402


def walks_only(A, num_walks, L):
  import torch
  from hypergraphembedding_b200 import _native
  from hypergraphembedding_b200.algebraic_distance import make_incidence
  ctx = _native.default_context()
  V = sum(A.shape)
  walks = torch.empty((num_walks * V, L), dtype=torch.int32, device="cuda")
  counts = torch.empty(V, dtype=torch.int64, device="cuda")
  inc = make_incidence(A, ctx=ctx)
  try:
    _native.n2v_walks(ctx, inc, 1, 2, 1.0, 1.0, 0, walks[:V], counts)   # warm-up
    runs = []
    for _ in range(3):
      a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      a.record()
      _native.n2v_walks(ctx, inc, num_walks, L, 1.0, 1.0, 0, walks, counts)
      b.record()
      b.synchronize()
      runs.append(a.elapsed_time(b))
  finally:
    inc.close()
  ms = float(np.median(runs))
  return {"num_walks": num_walks * V, "walk_length": L, "ms_runs": runs, "ms": ms,
          "walks_per_s": num_walks * V / (ms / 1e3), "steps_per_s": num_walks * V * (L - 1) / (ms / 1e3)}


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--out", required=True)
  args = ap.parse_args()
  os.makedirs(args.out, exist_ok=True)
  import scipy.sparse as sps
  from hypergraphembedding_b200 import synthetic
  from hypergraphembedding_b200.node2vec import Node2VecDevice
  from oracle import node2vec_ref as ref

  def csr(A):
    A = sps.csr_matrix(A, dtype=np.float32)
    A.sum_duplicates()
    A.sort_indices()
    return A

  result = {"gpu": gpu_info()}
  A = csr(synthetic.power_law_hypergraph(1_000_000, 500_000, 10_000_000, seed=1234))
  result["walks_config2"] = walks_only(A, 10, 80)
  print(json.dumps(result["walks_config2"]), flush=True)
  del A

  A = csr(synthetic.power_law_hypergraph(100_000, 50_000, 1_000_000))
  Node2VecDevice(A, 128, walk_length=10, num_walks=1, epochs=1)   # warm-up
  d, negative = 128, 5
  t = {}
  t0 = time.perf_counter()
  X, info = Node2VecDevice(A, d, walk_length=80, num_walks=1, epochs=1, negative=negative, timings=t)
  wall = time.perf_counter() - t0
  P, S = info["num_pairs"], negative + 1
  result["pipeline"] = {"num_nodes": A.shape[0], "num_edges": A.shape[1], "incidences": int(A.nnz), "dim": d,
                        "num_walks": info["num_walks"], "walk_length": 80, "epochs": 1,
                        "batch_pairs": info["batch_pairs"], "num_pairs": P, "losses": info["losses"].tolist(),
                        "wall_s": wall, **t, "train_pairs_per_s": P / (t["train_ms"] / 1e3),
                        "gathered_bytes_per_pair": (1 + 3 * S) * 4 * d, "finite": bool(np.isfinite(X).all())}
  print(json.dumps(result["pipeline"]), flush=True)

  B = csr(synthetic.power_law_hypergraph(10_000, 5_000, 100_000))
  t0 = time.perf_counter()
  ref.walks(B, 1, 80, 1.0, 1.0, 0)
  host_s = time.perf_counter() - t0
  result["host_numpy_walks_1_100"] = {"num_walks": sum(B.shape), "walk_length": 80, "wall_s": host_s,
                                      "walks_per_s": sum(B.shape) / host_s, "note": "host CPU, numpy"}
  print(json.dumps(result["host_numpy_walks_1_100"]), flush=True)
  with open(os.path.join(args.out, "n2v_bench.json"), "w") as f:
    json.dump(result, f, indent=1)


if __name__ == "__main__":
  main()
