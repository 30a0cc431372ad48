"""Device sampler (BooleanSamplesDevice / AlgebraicDistanceSamplesDevice) against the bit-exact host
replay (BooleanSamplesCsr / AlgebraicDistanceSamplesCsr) on the same inputs, in one process:

  * HOBE on the 100 000-node config-4-family graph of tests/golden/hobe_scale.npz (R 10, k 5,
    20 samples per row);
  * FOBE on the 100 000- and 1 000 000-node members of the config-4 family (k 5, 200 samples);
  * FOBE on the full 10 M-node config 4, streamed in chunks of 262 144 rows.

Reports records/s, two-factor expansion entries/s (the A * A^T and B * B^T rows the device
expands: sum of squared edge sizes plus sum of squared node degrees) and the phase split, with
the GPU's name and power limit read in the same run.  Every timed call ends in a device
synchronise (the result is on the host).

    python tools/device_sampler_bench.py --out DIR [--skip-full] [--reps 2]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
  import torch
  info = {"name": torch.cuda.get_device_name(0)}
  try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    info["power_limit_and_max_sm_clock"] = q[0] if q else None
  except (OSError, subprocess.SubprocessError) as exc:
    info["power_limit_and_max_sm_clock"] = "unavailable: %s" % exc
  return info


def expansion_entries(A):
  """Entries the device writes for the two-factor rows: sum_e |e|^2 (node rows of A * A^T) plus
  sum_n deg(n)^2 (edge rows of B * B^T)."""
  deg_n = np.diff(A.indptr).astype(np.int64)
  deg_e = np.bincount(A.indices, minlength=A.shape[1]).astype(np.int64)
  return int((deg_e * deg_e).sum() + (deg_n * deg_n).sum())


def best(fn, reps):
  times, out = [], None
  for _ in range(reps):
    t = time.perf_counter()
    out = fn()
    times.append(time.perf_counter() - t)
  return min(times), times, out


def hobe(reps):
  import hypergraphembedding_b200 as H
  from hypergraphembedding_b200 import synthetic
  g = np.load(os.path.join(ROOT, "tests", "golden", "hobe_scale.npz"))
  A = synthetic.zipf_hypergraph(int(g["nodes"]), int(g["edges"]), seed=int(g["graph_seed"]))
  xn, xe = synthetic.legacy_initial_vectors(A.shape[0], A.shape[1], int(g["R"]), seed=int(g["vec_seed"]))
  k, s = int(g["k"]), int(g["num_samples"])
  H.AlgebraicDistanceSamplesDevice(A, xn, xe, k, s, seed=1)             # warm-up: modules, pools
  dev_t = {}
  dev_s, dev_all, out = best(lambda: H.AlgebraicDistanceSamplesDevice(A, xn, xe, k, s, seed=1,
                                                                     timings=dev_t), reps)
  n_dev = len(out)
  del out
  rep_t = {}

  def replay():
    np.random.seed(int(g["seed"]))
    return H.AlgebraicDistanceSamplesCsr(A, xn, xe, k, s, timings=rep_t)

  rep_s, rep_all, out = best(replay, reps)
  n_rep = len(out)
  return {"graph": "zipf_hypergraph(%d, %d, seed=%d)" % (A.shape[0], A.shape[1], int(g["graph_seed"])),
          "nnz": int(A.nnz), "k": k, "num_samples": s,
          "device": {"records": n_dev, "seconds": dev_s, "all_seconds": dev_all, "samples_per_s": n_dev / dev_s,
                     "expanded_2f_entries_per_s": expansion_entries(A) / dev_s, "phases_last_run": dev_t},
          "replay": {"records": n_rep, "seconds": rep_s, "all_seconds": rep_all, "samples_per_s": n_rep / rep_s,
                     "phases_last_run": rep_t}}


def fobe_device_split(A, k, s, chunk_rows):
  """Seconds of the device calls alone (pairs, neighbour arrays, results left on the device)."""
  from hypergraphembedding_b200 import _native
  from hypergraphembedding_b200.hg2v_sample import _DeviceSampler, _Graph
  g = _Graph.from_csr(A)
  ctx = _native.default_context()
  inc = g.incidence(ctx)
  try:
    d = _DeviceSampler(g, ctx, inc, k, 1, chunk_rows)
    node_s, edge_s = np.full(g.num_nodes, s, np.int32), np.full(g.num_edges, s, np.int32)
    for side, samples, phase in ((0, node_s, _native.PHASE_NN), (1, edge_s, _native.PHASE_EE)):
      for _ in d.pairs(side, 2, samples, phase):
        pass
    for _ in d.node_edge(node_s, edge_s, 1, (_native.PHASE_NE, _native.PHASE_EN, _native.PHASE_NEIGHBORS)):
      pass
    return d.spent
  finally:
    inc.close()


def fobe(A, label, reps, stream=False, with_replay=True):
  import hypergraphembedding_b200 as H
  from hypergraphembedding_b200.hg2v_sample import _Graph
  k, s = 5, 200
  chunk = 262144 if stream else 0

  def count(result):
    if not stream:
      return len(result)
    return sum(len(part) for part in result)

  count(H.BooleanSamplesDevice(A, k, s, seed=1, chunk_rows=chunk, stream=stream))   # warm-up
  dev_s, dev_all, n_dev = best(lambda: count(H.BooleanSamplesDevice(A, k, s, seed=1, chunk_rows=chunk,
                                                                    stream=stream)), reps)
  split = fobe_device_split(A, k, s, chunk)
  out = {"graph": label, "nodes": int(A.shape[0]), "edges": int(A.shape[1]), "nnz": int(A.nnz), "k": k,
         "num_samples": s, "chunk_rows": chunk,
         "device": {"records": n_dev, "seconds": dev_s, "all_seconds": dev_all, "samples_per_s": n_dev / dev_s,
                    "expanded_2f_entries_per_s": expansion_entries(A) / dev_s,
                    "phases": {"device_pairs_s": split["pairs"], "device_neighbours_s": split["neighbours"],
                               "host_columns_s": max(0.0, dev_s - split["pairs"] - split["neighbours"])}}}
  if with_replay:
    graph = _Graph.from_csr(A)

    def replay():
      np.random.seed(0)
      return count(H.BooleanSamplesCsr(graph, k, s, chunk_rows=chunk, stream=stream))

    rep_s, rep_all, n_rep = best(replay, 1 if stream else reps)
    out["replay"] = {"records": n_rep, "seconds": rep_s, "all_seconds": rep_all, "samples_per_s": n_rep / rep_s}
  return out


def main():
  ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
  ap.add_argument("--out", required=True, help="directory for device_sampler_bench.json")
  ap.add_argument("--reps", type=int, default=2)
  ap.add_argument("--skip-full", action="store_true", help="leave out the 10 M-node config 4")
  args = ap.parse_args()
  import torch
  assert torch.cuda.is_available(), "the device sampler needs a CUDA device"
  from hypergraphembedding_b200 import synthetic
  os.makedirs(args.out, exist_ok=True)
  result = {"gpu": gpu_info(), "host_threads": os.cpu_count()}
  result["hobe_100k"] = hobe(args.reps)
  print(json.dumps(result["hobe_100k"]), flush=True)
  for n, e in ((100000, 50000), (1000000, 500000)):
    A = synthetic.zipf_hypergraph(n, e, seed=2024)
    key = "fobe_%dk" % (n // 1000)
    result[key] = fobe(A, "zipf_hypergraph(%d, %d, seed=2024)" % (n, e), args.reps)
    print(json.dumps(result[key]), flush=True)
  if not args.skip_full:
    t = time.perf_counter()
    A = synthetic.zipf_hypergraph(10000000, 5000000, seed=2024)
    gen_s = time.perf_counter() - t
    result["fobe_config4"] = fobe(A, "config 4: zipf_hypergraph(10000000, 5000000, seed=2024)", 1,
                                  stream=True)
    result["fobe_config4"]["generate_s"] = gen_s
    print(json.dumps(result["fobe_config4"]), flush=True)
  path = os.path.join(args.out, "device_sampler_bench.json")
  with open(path, "w") as f:
    json.dump(result, f, indent=1)
  print("wrote", path)


if __name__ == "__main__":
  main()
