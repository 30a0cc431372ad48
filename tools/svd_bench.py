"""The truncated SVD on the GPU (hypergraphembedding_b200.svd) on config 2
(synthetic.power_law_hypergraph(1 000 000, 500 000, 10 000 000, seed=1234)), k = 32 and 128:

  device    n_iter = 5 (the default) and 20 from the seeded start (seed 0), device working arrays:
            wall seconds of the whole call (start to residuals, ended by the residuals' read-back),
            then a second run with per-iteration timing: wall milliseconds per iteration, CUDA-event
            milliseconds of the two products (SpMM), the two f64 Gram matrices and the two
            row-times-matrix steps, and the host milliseconds of the two eigh steps; the half calls'
            remainder (Gram read-back, synchronisation) is wall - the rest.  Both runs must agree
            bit for bit.  The final residuals ||A v_i - s_i u_i|| / s_1 and Ritz values.
  host      at 1/100 scale (10 000 nodes, 5 000 edges, 100 000 incidences) on the host's cores:
            scipy.sparse.linalg.svds (ARPACK, k singular triplets to its default tolerance) and
            scikit-learn's randomized_svd (n_iter 5, 10 oversamples, the same algorithm family in
            float64), wall seconds each.  These are host numbers, not GPU numbers.

The GPU's name and power limit are read in the same run.

    python tools/svd_bench.py --out DIR
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

KS = (32, 128)
ITERS = (5, 20)


def device_runs(ctx, inc, k):
  from hypergraphembedding_b200.svd import truncated_svd
  truncated_svd(ctx, inc, k, 1)   # warm-up: modules, pool
  out = {}
  for n_iter in ITERS:
    ctx.sync()
    t0 = time.perf_counter()
    U, s, V, info = truncated_svd(ctx, inc, k, n_iter)
    wall = time.perf_counter() - t0
    U, V = U.cpu().numpy(), V.cpu().numpy()
    per = []
    U2, s2, V2, info2 = truncated_svd(ctx, inc, k, n_iter, timings=per)
    same = bool(np.array_equal(U.view(np.uint32), U2.cpu().numpy().view(np.uint32)) and
                np.array_equal(V.view(np.uint32), V2.cpu().numpy().view(np.uint32)) and
                np.array_equal(s, s2) and np.array_equal(info["residuals"], info2["residuals"]))
    mean = {key: float(np.mean([p[key] for p in per])) for key in per[0]}
    mean["half_calls_remainder"] = mean["wall"] - sum(mean[key] for key in ("spmm", "gram", "rowmat", "eigh_host"))
    out["n_iter_%d" % n_iter] = {
        "block_width": info["block_width"], "wall_s": wall, "timed_run_bit_identical": same,
        "ms_per_iteration_timed_run": mean, "per_iteration_ms": per,
        "residuals": info["residuals"].tolist(), "singular_values": s.tolist(),
        "ritz_change_last_iteration": (np.abs(info["ritz_values"][-1][:k] - info["ritz_values"][-2][:k]).max()
                                       / s[0]) if n_iter > 1 else None,
    }
    print(json.dumps({"k": k, "n_iter": n_iter, "wall_s": wall, "per_iteration_ms": mean, "bit_identical": same,
                      "max_residual": float(info["residuals"].max())}), flush=True)
  return out


def host_side(k):
  import scipy.sparse.linalg as spla
  from sklearn.utils.extmath import randomized_svd
  from hypergraphembedding_b200 import synthetic
  A = synthetic.power_law_hypergraph(10000, 5000, 100000, seed=1234).astype(np.float64)
  out = {"graph": [int(A.shape[0]), int(A.shape[1]), int(A.nnz)], "host_cores": os.cpu_count()}
  t0 = time.perf_counter()
  spla.svds(A, k=k, random_state=0)
  out["scipy_svds_s"] = time.perf_counter() - t0
  t0 = time.perf_counter()
  randomized_svd(A, k, n_oversamples=10, n_iter=5, random_state=0)
  out["sklearn_randomized_svd_n_iter_5_s"] = time.perf_counter() - t0
  return out


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--out", required=True)
  args = ap.parse_args()
  import torch
  from hypergraphembedding_b200 import _native, synthetic
  from hypergraphembedding_b200.algebraic_distance import make_incidence
  torch.cuda.init()
  result = {"gpu": gpu_info(), "workload": "config 2: power_law_hypergraph(1000000, 500000, 10000000, seed=1234)"}
  A = synthetic.power_law_hypergraph(1000000, 500000, 10000000, seed=1234)
  A.sort_indices()
  N, E = A.shape
  result["graph"] = {"nodes": N, "edges": E, "nnz": int(A.nnz), "max_node_degree": int(np.diff(A.indptr).max()),
                     "max_edge_size": int(np.bincount(A.indices, minlength=E).max())}
  ctx = _native.default_context()
  inc = make_incidence(A, ctx=ctx)
  try:
    for k in KS:
      result["k%d" % k] = {"device": device_runs(ctx, inc, k)}
  finally:
    inc.close()
  for k in KS:
    result["k%d" % k]["host_1_100_scale"] = host_side(k)
    print(json.dumps({"k": k, "host": result["k%d" % k]["host_1_100_scale"]}), flush=True)
  os.makedirs(args.out, exist_ok=True)
  with open(os.path.join(args.out, "svd_bench.json"), "w") as f:
    json.dump(result, f, indent=1)


if __name__ == "__main__":
  main()
