"""The non-negative factorization on the GPU (hge_nmf_fit) on config 2
(synthetic.power_law_hypergraph(1 000 000, 500 000, 10 000 000, seed=1234)), k = 32 and 128:

  runs      50 iterations at tol = 0, and the default stop (max_iter 200, tol 1e-4), from the seeded
            start (seed 0): wall seconds (ended by the fit's own synchronise), iterations, and from a
            second run with CUDA events per phase the milliseconds per iteration of the products
            (SpMM), the Gram matrices and the coordinate-descent passes; the products' algorithmic
            bytes over their time (per iteration both products read every incidence's column id and
            gathered row and write every output row: 2 nnz (4 + 4 ld) + 4 ld (N + E) + 8 (N + E + 2),
            ld = k rounded up to a multiple of 4);
  sweep     the relaxation's half-sweeps at R = k on the same graph (hge_algdist_node_half /
            _edge_half, CUDA events over 10 sweeps after 2 warm-up sweeps), for comparison only;
  parity    at k = 32 (--parity): the first two iterations compared bit for bit with
            oracle/nmf_ref.py's fp32 restatement at full size (W, H, violations);
  sklearn   scikit-learn's NMF(solver="cd") from the same kind of start on the 1/100-scale member of
            the family (10 000 nodes, 5 000 edges, 100 000 incidences) on the host's cores.

The GPU's name and power limit are read in the same run.

    python tools/nmf_bench.py --out DIR [--parity]
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
FIXED_ITERS = 50


def spmm_bytes(N, E, nnz, k):
  ld = (k + 3) & ~3
  return 2 * nnz * (4 + 4 * ld) + 4 * ld * (N + E) + 8 * (N + E + 2)


def fit(ctx, inc, W0, Ht0, max_iter, tol, timed):
  from hypergraphembedding_b200 import _native
  W, Ht = W0.clone(), Ht0.clone()
  ms = np.zeros(3) if timed else None
  ctx.sync()
  t0 = time.perf_counter()
  it, viols = _native.nmf_fit(ctx, inc, W, Ht, max_iter, tol, phase_ms=ms)
  wall = time.perf_counter() - t0
  return W, Ht, it, viols, wall, ms


def device_runs(A, k, ctx, inc):
  import torch
  from hypergraphembedding_b200.nmf import seeded_start
  N, E = A.shape
  W0, Ht0 = seeded_start(N, E, A.nnz, k, 0)
  W0, Ht0 = torch.from_numpy(W0).cuda(), torch.from_numpy(Ht0).cuda()
  fit(ctx, inc, W0, Ht0, 2, 0.0, False)   # warm-up: modules, pool
  out = {}
  for name, max_iter, tol in (("fixed_50", FIXED_ITERS, 0.0), ("default_stop", 200, 1e-4)):
    _, _, it, viols, wall, _ = fit(ctx, inc, W0, Ht0, max_iter, tol, False)
    _, _, it2, viols2, _, ms = fit(ctx, inc, W0, Ht0, max_iter, tol, True)
    assert it2 == it and np.array_equal(viols, viols2)
    per = ms / it
    out[name] = {
        "max_iter": max_iter, "tol": tol, "n_iter": it, "wall_s": wall, "ms_per_iteration": wall * 1e3 / it,
        "timed_ms_per_iteration": {"spmm": per[0], "gram": per[1], "cd": per[2]},
        "spmm_algorithmic_GBps": spmm_bytes(N, E, A.nnz, k) / (per[0] * 1e-3) / 1e9,
        "violation_first_last": [float(viols[0]), float(viols[-1])],
    }
  return out, (W0, Ht0)


def half_sweep(ctx, inc, N, E, R):
  import torch
  from hypergraphembedding_b200 import _native
  st = _native.AlgDistState(ctx, inc, R, 12)
  try:
    rng = np.random.default_rng(0)
    st.load(rng.random((N, R), dtype=np.float32), rng.random((E, R), dtype=np.float32))
    for s in range(2):
      st.node_half(s)
      st.edge_half(s)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    node = edge = 0.0
    for s in range(2, 12):
      ev[0].record()
      st.node_half(s)
      ev[1].record()
      st.edge_half(s)
      ev[2].record()
      ev[2].synchronize()
      node += ev[0].elapsed_time(ev[1])
      edge += ev[1].elapsed_time(ev[2])
    return {"R": R, "node_half_ms": node / 10, "edge_half_ms": edge / 10}
  finally:
    st.close()


def parity(A, ctx, inc, W0, Ht0):
  import scipy.sparse as sps
  from oracle import nmf_ref as ref
  W, Ht, it, viols, _, _ = fit(ctx, inc, W0, Ht0, 2, 0.0, False)
  B = sps.csr_matrix(A.T)
  B.sort_indices()
  t0 = time.perf_counter()
  rW, rHt, rit, rviols = ref.fit32(A.indptr, A.indices, B.indptr, B.indices, W0.cpu().numpy(), Ht0.cpu().numpy(),
                                   2, 0.0)
  return {"iterations": 2, "k": int(W0.shape[1]), "restatement_s": time.perf_counter() - t0,
          "W_bit_exact": bool(np.array_equal(W.cpu().numpy().view(np.uint32), rW.view(np.uint32))),
          "H_bit_exact": bool(np.array_equal(Ht.cpu().numpy().view(np.uint32), rHt.view(np.uint32))),
          "violations_equal": bool(it == rit and np.array_equal(viols, rviols))}


def sklearn_side(k):
  import warnings
  from sklearn.decomposition import non_negative_factorization
  from hypergraphembedding_b200 import synthetic
  from oracle import nmf_ref as ref
  from hypergraphembedding_b200.nmf import start_scale
  A = synthetic.power_law_hypergraph(10000, 5000, 100000, seed=1234).astype(np.float64)
  N, E = A.shape
  W0, Ht0 = ref.start(N, E, k, 0, start_scale(N, E, A.nnz, k))
  out = {"graph": [N, E, int(A.nnz)], "host_cores": os.cpu_count()}
  for name, max_iter, tol in (("fixed_50", FIXED_ITERS, 0.0), ("default_stop", 200, 1e-4)):
    t0 = time.perf_counter()
    with warnings.catch_warnings():
      warnings.simplefilter("ignore")
      _, _, it = non_negative_factorization(A, W=W0.astype(np.float64), H=Ht0.T.astype(np.float64), n_components=k,
                                            init="custom", solver="cd", max_iter=max_iter, tol=tol)
    wall = time.perf_counter() - t0
    out[name] = {"n_iter": int(it), "wall_s": wall, "ms_per_iteration": wall * 1e3 / it}
  return out


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--out", required=True)
  ap.add_argument("--parity", action="store_true")
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
      runs, start = device_runs(A, k, ctx, inc)
      result["k%d" % k] = {"device": runs, "half_sweep_at_R_eq_k": half_sweep(ctx, inc, N, E, k)}
      if args.parity and k == 32:
        result["k%d" % k]["parity"] = parity(A, ctx, inc, *start)
      else:
        result["k%d" % k]["parity"] = "not measured"
      print(json.dumps({"k": k, **result["k%d" % k]}), flush=True)
  finally:
    inc.close()
  for k in KS:
    result["k%d" % k]["sklearn_1_100_scale"] = sklearn_side(k)
    print(json.dumps({"k": k, "sklearn": result["k%d" % k]["sklearn_1_100_scale"]}), flush=True)
  os.makedirs(args.out, exist_ok=True)
  with open(os.path.join(args.out, "nmf_bench.json"), "w") as f:
    json.dump(result, f, indent=1)


if __name__ == "__main__":
  main()
