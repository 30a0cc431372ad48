"""The Jaccard methods (HG2V_ADJ_JAC / HG2V_NEIGH_JAC) on device-resident samples, on the 100 000- and
1 000 000-node members of the config-4 family (zipf_hypergraph(n, n / 2, seed=2024)), k 5, 200
samples, dimension 32, 2 epochs at batch 256, uniform and neighbourhood (alpha 0) features:

  (a) the new path end to end: features on the host (UniformWeight / WeightByNeighborhood restated on
      the CSR), WeightedJaccardSamplesDevice(keep_on_device=True) with its pairs / neighbours /
      probabilities split, packing into the model's buffer, 2 training epochs (fit_device); peak
      device memory in torch's allocator and in the device's default stream-ordered pool;
  (b) at 100 000 nodes only, the existing EmbedHg2vAdjJaccard / EmbedHg2vNeighborhoodWeightedJaccard
      on the same graph built as a proto (proto construction timed separately).

Every timed step ends in a device synchronise.  The GPU's name and power limit are read in the
same run.

    python tools/jaccard_device_bench.py --out DIR
"""
import argparse
import ctypes
import json
import os
import sys
import time

import numpy as np
import scipy.sparse as sps

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from device_sampler_bench import gpu_info  # noqa: E402
from hg2v_device_bench import PoolStats, peaks, reset_peaks, rss_gb  # noqa: E402

K, SAMPLES, DIM, EPOCHS, BATCH, SEED = 5, 200, 32, 2, 256, 1


def sync_time(fn):
  import torch
  torch.cuda.synchronize()
  t = time.perf_counter()
  out = fn()
  torch.cuda.synchronize()
  return time.perf_counter() - t, out


def features(A, kind):
  """UniformWeight / WeightByNeighborhood(alpha 0) of the hypergraph whose ToCsrMatrix is A."""
  from hypergraphembedding_b200.hg2v_weighting import _scaled_row
  A = sps.csr_matrix(A, dtype=np.float32)
  B = A.T.tocsr()
  B.sort_indices()
  if kind == "uniform":
    return A, B
  deg_n = np.diff(A.indptr)
  deg_e = np.diff(B.indptr)
  node_row = _scaled_row(dict(enumerate(deg_n.tolist())), 0)
  edge_row = _scaled_row(dict(enumerate(deg_e.tolist())), 0)
  return sps.csr_matrix(A.multiply(edge_row), dtype=np.float32), sps.csr_matrix(B.multiply(node_row),
                                                                                dtype=np.float32)


def new_path(A, kind, pool):
  import torch
  import hypergraphembedding_b200 as H
  from hypergraphembedding_b200 import _native
  from hypergraphembedding_b200.hg2v_model import Hg2vModel
  from hypergraphembedding_b200.hg2v_sample import _Graph
  reset_peaks(pool)
  out = {"features": kind}
  t = time.perf_counter()
  NF, EF = features(A, kind)
  g = _Graph.from_csr(A)
  out["host_features_s"] = time.perf_counter() - t
  timings = {}
  out["sample_s"], samples = sync_time(lambda: H.WeightedJaccardSamplesDevice(
      g, NF, EF, K, SAMPLES, seed=SEED, timings=timings, keep_on_device=True))
  out["sample_split_s"] = timings
  out["records"] = len(samples)
  model = Hg2vModel.seeded(g.num_nodes, g.num_edges, DIM, K, "relu", "mean_squared_error", SEED)
  try:
    out["pack_s"], _ = sync_time(lambda: model.set_device_samples(samples))
    # the epochs of fit_device on the packed buffer: shuffle on the device, then one training launch
    order = torch.empty(max(model.num_samples, 1), dtype=torch.int32,
                        device=torch.device("cuda", model.ctx.device))[:model.num_samples]
    out["epoch_s"], out["losses"] = [], []
    for epoch in range(EPOCHS):
      loss = ctypes.c_double(0.0)

      def one_epoch():
        _native.shuffle_order(model.ctx, SEED, epoch, model.num_samples, out=order)
        _native.check(model.ctx.lib.hge_hg2v_fit_epoch(model.handle, _native.ptr(order), BATCH,
                                                       _native.MEM_DEVICE, ctypes.byref(loss)))

      dt, _ = sync_time(one_epoch)
      out["epoch_s"].append(dt)
      out["losses"].append(loss.value)
  finally:
    model.close()
  out["total_s"] = out["host_features_s"] + out["sample_s"] + out["pack_s"] + sum(out["epoch_s"])
  out["peak_device"] = peaks(pool)
  return out


def proto_from_csr(A):
  from hypergraphembedding_b200 import Hypergraph
  hg = Hypergraph()
  A = sps.csr_matrix(A)
  B = A.T.tocsr()
  B.sort_indices()
  for n in range(A.shape[0]):
    hg.node[n].edges.extend(A.indices[A.indptr[n]:A.indptr[n + 1]].tolist())
  for e in range(B.shape[0]):
    hg.edge[e].nodes.extend(B.indices[B.indptr[e]:B.indptr[e + 1]].tolist())
  return hg


def existing_path(hg, kind, pool):
  import hypergraphembedding_b200 as H
  reset_peaks(pool)
  np.random.seed(SEED)
  fn = H.EmbedHg2vAdjJaccard if kind == "uniform" else H.EmbedHg2vNeighborhoodWeightedJaccard
  dt, emb = sync_time(lambda: fn(hg, DIM, num_neighbors=K, num_samples=SAMPLES, batch_size=BATCH, epochs=EPOCHS,
                                 disable_pbar=True))
  return {"features": kind, "total_s": dt, "method_name": emb.method_name, "peak_device": peaks(pool)}


def main():
  ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
  ap.add_argument("--out", required=True, help="directory for jaccard_device_bench.json")
  ap.add_argument("--sizes", default="100000,1000000", help=argparse.SUPPRESS)   # rehearsal at small sizes
  args = ap.parse_args()
  import torch
  assert torch.cuda.is_available(), "the benchmark needs a CUDA device"
  from hypergraphembedding_b200 import synthetic
  os.makedirs(args.out, exist_ok=True)
  pool = PoolStats()
  result = {"gpu": gpu_info(), "host_threads": os.cpu_count(), "k": K, "num_samples": SAMPLES,
            "dimension": DIM, "epochs": EPOCHS, "batch": BATCH, "runs": []}
  # warm-up: modules, memory pools, cub tuning of every kernel the paths launch
  small = synthetic.zipf_hypergraph(20000, 10000, seed=1)
  new_path(small, "uniform", pool)
  existing_path(proto_from_csr(small), "uniform", pool)
  for n in (int(x) for x in args.sizes.split(",")):
    A = synthetic.zipf_hypergraph(n, n // 2, seed=2024)
    run = {"graph": "zipf_hypergraph(%d, %d, seed=2024)" % (n, n // 2), "nnz": int(A.nnz), "new": []}
    for kind in ("uniform", "neighborhood"):
      run["new"].append(new_path(A, kind, pool))
      print(json.dumps(run["new"][-1]), flush=True)
    if n <= 100000:
      t = time.perf_counter()
      hg = proto_from_csr(A)
      run["proto_build_s"] = time.perf_counter() - t
      run["existing"] = [existing_path(hg, kind, pool) for kind in ("uniform", "neighborhood")]
      print(json.dumps(run["existing"]), flush=True)
      del hg
    run["host_peak_rss_gb"] = rss_gb()
    result["runs"].append(run)
  result["gpu_after"] = gpu_info()
  path = os.path.join(args.out, "jaccard_device_bench.json")
  with open(path, "w") as f:
    json.dump(result, f, indent=1)
  print("wrote", path)


if __name__ == "__main__":
  main()
