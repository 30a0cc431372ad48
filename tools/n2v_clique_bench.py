"""node2vec on the weighted clique expansions on the GPU (hypergraphembedding_b200.node2vec,
Node2VecCliqueDevice; DESIGN section 9.13):

  walks        config 2 (synthetic.power_law_hypergraph(1 000 000, 500 000, 10 000 000, seed=1234)),
               10 walks of 80 vertices per vertex, node side and edge side, (p, q) = (1, 1) and
               (0.25, 4): CUDA-event milliseconds of hge_n2v_clique_walks (the row prefix included),
               walks / s and accepted steps / s.
  pipeline     node side of synthetic.power_law_hypergraph(100 000, 50 000, 1 000 000), d = 128,
               one walk of 80 vertices per vertex, one epoch (the other settings at their defaults):
               milliseconds of the walks, the pairs and the training.
  expansion    the entries a materialized expansion would hold, from shapes: sum over edges of
               |e| (|e| - 1) (node side) and over nodes of d (d - 1) (edge side), directed entries
               counted with multiplicity, and the largest row weight S(v), for both graphs above.
  proposals    the mean proposals per accepted step, counted by the numpy restatement
               (tests/n2v_clique_ref.py) at 1/100 of config 2 (power_law_hypergraph(10 000, 5 000,
               100 000)), one walk of 80 per vertex.  A host count, not a GPU number.

The GPU's name and power limit are read in the same run.

    python tools/n2v_clique_bench.py --out DIR
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from device_sampler_bench import gpu_info  # noqa: E402

PQ = [(1.0, 1.0), (0.25, 4.0)]


def csr(A):
  import scipy.sparse as sps
  A = sps.csr_matrix(A, dtype=np.float32)
  A.sum_duplicates()
  A.sort_indices()
  return A


def expansion_sizes(A):
  """entries of both materialized expansions and the largest S(v) of each side, from shapes"""
  deg_n = np.diff(A.indptr).astype(np.int64)
  size_e = np.bincount(A.indices, minlength=A.shape[1]).astype(np.int64)
  s_node = np.bincount(np.repeat(np.arange(A.shape[0]), deg_n), weights=(size_e - 1)[A.indices],
                       minlength=A.shape[0])
  s_edge = np.bincount(A.indices, weights=(deg_n - 1)[np.repeat(np.arange(A.shape[0]), deg_n)],
                       minlength=A.shape[1])
  return {"num_nodes": A.shape[0], "num_edges": A.shape[1], "incidences": int(A.nnz),
          "node_side_entries": int(np.sum(size_e * (size_e - 1))), "edge_side_entries": int(np.sum(deg_n * (deg_n - 1))),
          "max_row_weight_node_side": int(s_node.max()), "max_row_weight_edge_side": int(s_edge.max())}


def walks_only(A, side, num_walks, L, p, q):
  import torch
  from hypergraphembedding_b200 import _native
  from hypergraphembedding_b200.algebraic_distance import make_incidence
  ctx = _native.default_context()
  V = A.shape[side]
  walks = torch.empty((num_walks * V, L), dtype=torch.int32, device="cuda")
  counts = torch.empty(V, dtype=torch.int64, device="cuda")
  inc = make_incidence(A, ctx=ctx)
  try:
    _native.n2v_clique_walks(ctx, inc, side, 1, 2, p, q, 0, walks[:V], counts)   # warm-up
    runs = []
    for _ in range(3):
      a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      a.record()
      _native.n2v_clique_walks(ctx, inc, side, num_walks, L, p, q, 0, walks, counts)
      b.record()
      b.synchronize()
      runs.append(a.elapsed_time(b))
    steps = int((walks[:, 1:] >= 0).sum().item())
  finally:
    inc.close()
  ms = float(np.median(runs))
  return {"side": ["node", "edge"][side], "p": p, "q": q, "num_walks": num_walks * V, "walk_length": L,
          "ms_runs": runs, "ms": ms, "walks_per_s": num_walks * V / (ms / 1e3), "steps": steps,
          "steps_per_s": steps / (ms / 1e3)}


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--out", required=True)
  args = ap.parse_args()
  os.makedirs(args.out, exist_ok=True)
  from hypergraphembedding_b200 import synthetic
  from hypergraphembedding_b200.node2vec import Node2VecCliqueDevice
  import n2v_clique_ref as cref

  result = {"gpu": gpu_info(), "walks_config2": []}
  A = csr(synthetic.power_law_hypergraph(1_000_000, 500_000, 10_000_000, seed=1234))
  result["expansion_config2"] = expansion_sizes(A)
  for side in (0, 1):
    for p, q in PQ:
      result["walks_config2"].append(walks_only(A, side, 10, 80, p, q))
      print(json.dumps(result["walks_config2"][-1]), flush=True)
  del A

  A = csr(synthetic.power_law_hypergraph(100_000, 50_000, 1_000_000, seed=1234))
  result["expansion_pipeline_graph"] = expansion_sizes(A)
  Node2VecCliqueDevice(A, 128, side="node", walk_length=10, num_walks=1, epochs=1)   # warm-up
  t = {}
  X, info = Node2VecCliqueDevice(A, 128, side="node", walk_length=80, num_walks=1, epochs=1, timings=t)
  result["pipeline_node_side"] = {"num_nodes": A.shape[0], "num_edges": A.shape[1], "incidences": int(A.nnz),
                                  "dim": 128, "num_walks": info["num_walks"], "walk_length": 80, "epochs": 1,
                                  "batch_pairs": info["batch_pairs"], "num_pairs": info["num_pairs"],
                                  "losses": info["losses"].tolist(), **t,
                                  "train_pairs_per_s": info["num_pairs"] / (t["train_ms"] / 1e3),
                                  "finite": bool(np.isfinite(X).all())}
  print(json.dumps(result["pipeline_node_side"]), flush=True)

  B = csr(synthetic.power_law_hypergraph(10_000, 5_000, 100_000, seed=1234))
  result["host_proposals_1_100"] = []
  for side in (0, 1):
    for p, q in ((0.25, 4.0), (4.0, 0.25)):
      st = {}
      cref.clique_walks(B, side, 1, 80, p, q, 0, stats=st)
      result["host_proposals_1_100"].append({"side": ["node", "edge"][side], "p": p, "q": q, **st,
                                             "proposals_per_step": st["proposals"] / st["steps"],
                                             "note": "host count, numpy restatement"})
      print(json.dumps(result["host_proposals_1_100"][-1]), flush=True)
  with open(os.path.join(args.out, "n2v_clique_bench.json"), "w") as f:
    json.dump(result, f, indent=1)


if __name__ == "__main__":
  main()
