"""Times the node and edge half-sweeps of the built library on one bench workload (config 2 by
default) and reports its error on the youtube golden.  Prints one JSON line.

    python tools/time_variant.py [WORKLOAD [LIGHT_MAX_DEG CHUNK BLOCKS_PER_SM]]
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402
from bench import WORKLOADS, build_workload  # noqa: E402
from conftest import csr_from_pairs, incidence_distances, load_golden  # noqa: E402
from hypergraphembedding_b200 import _native, synthetic  # noqa: E402
from hypergraphembedding_b200 import algebraic_distance as ad  # noqa: E402


def golden_error(ctx):
  g = load_golden("algdist_youtube")
  r = np.searchsorted(g["node_ids"], g["pairs"][:, 0])
  c = np.searchsorted(g["edge_ids"], g["pairs"][:, 1])
  A = csr_from_pairs(np.stack([r, c], 1), shape=(len(g["node_ids"]), len(g["edge_ids"])))
  xn, xe = synthetic.legacy_initial_vectors(A.shape[0], A.shape[1], int(g["dim"]), int(g["seed"]))
  inc = ad.make_incidence(A, ctx=ctx)
  ad.relax(inc, xn, xe, int(g["iters"]))
  inc.close()
  d, dr = incidence_distances(A, xn, xe), incidence_distances(A, g["xn"], g["xe"])
  bound = 1e-5 * dr + 1e-6 * np.sqrt(10)
  return dict(dist_abs=float(np.abs(d - dr).max()), dist_vs_bound=float((np.abs(d - dr) / bound).max()),
              coord_abs=float(max(np.abs(xn - g["xn"]).max(), np.abs(xe - g["xe"]).max())))


def main():
  workload = sys.argv[1] if len(sys.argv) > 1 else "c2"
  tuning = [int(v) for v in sys.argv[2:5]] if len(sys.argv) >= 5 else None
  spec = WORKLOADS[workload]
  ctx = _native.default_context(0)
  if tuning:
    ctx.set_tuning(*tuning)
  out = dict(tuning=tuning)
  out.update(golden_error(ctx))
  A, B = build_workload(spec)
  N, E = A.shape
  R, sweeps = spec["R"], spec["sweeps"]
  xn0, xe0 = synthetic.legacy_initial_vectors(N, E, R, seed=0)
  inc = ad.make_incidence(A, B, ctx=ctx)
  xn, xe = torch.from_numpy(xn0).cuda(), torch.from_numpy(xe0).cuda()
  st = _native.AlgDistState(ctx, inc, R, sweeps)
  times = []
  for rep in range(4):
    st.load(xn, xe)
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(2 * sweeps + 1)]
    evs[0].record()
    for t in range(sweeps):
      st.node_half(t)
      evs[2 * t + 1].record()
      st.edge_half(t)
      evs[2 * t + 2].record()
    torch.cuda.synchronize()
    if rep:
      times.append([evs[i].elapsed_time(evs[i + 1]) for i in range(2 * sweeps)])
  t = np.asarray(times)
  out.update(node_ms=float(t[:, 0::2].mean()), edge_ms=float(t[:, 1::2].mean()),
             sweep_ms=float(t.sum(axis=1).mean() / sweeps))
  bytes_sweep = 2 * A.nnz * (4 * R + 4) + 2 * (N + E) * 4 * R
  out["alg_GBps"] = bytes_sweep / (out["sweep_ms"] * 1e-3) / 1e9
  print(json.dumps(out), flush=True)


if __name__ == "__main__":
  main()
