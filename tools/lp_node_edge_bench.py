"""The node-edge link classifier on the GPU (hge_lp_node_edge_train / _predict) on the graphs, links and
embeddings of tools/lp_svm_bench.py (zipf_hypergraph(n, n / 2, seed=2024), n in {20 000, 100 000,
1 000 000}, 10 % of the connections hidden, FOBE d = 32):

  device   NodeEdgeClassifierDevice's kernels with the defaults (hidden 64, 10 epochs, batch 256,
           lr 0.01): set-up (training set + initialisation) and per-epoch seconds, each ended by a
           device synchronise, samples/s, microseconds per batch, the predict call over the links,
           the peak of the device's default memory pool, per-epoch losses, accuracy and F1;
  context  PersonalizedEdgeClassifierPredictionDevice (the per-edge SVCs) on the same links: time,
           accuracy and F1;
  host     at 20 000 nodes only, the restatement's model in torch on the CPU (fp32) on the same
           training set and epoch orders: time and accuracy.

The GPU's name and power limit are read in the same run.

    python tools/lp_node_edge_bench.py --out DIR
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
from hg2v_device_bench import PoolStats  # noqa: E402
from lp_svm_bench import SEED, embed, hook_links, metrics, numpy_links  # noqa: E402

HIDDEN, EPOCHS, BATCH, LR = 64, 10, 256, 0.01


def device_side(R, xn, xe, links, good, bad, pool):
  import torch
  from hypergraphembedding_b200 import _native
  from hypergraphembedding_b200.hg2v_sample import _Graph
  ctx = _native.default_context()
  dev = torch.device("cuda", ctx.device)
  Xn, Xe = torch.from_numpy(xn).to(dev), torch.from_numpy(xe).to(dev)
  nodes = torch.from_numpy(links[:, 0].astype(np.int32)).to(dev)
  edges = torch.from_numpy(links[:, 1].astype(np.int32)).to(dev)
  inc = _Graph.from_csr(R).incidence(ctx)
  try:
    w, _ = _native.lp_node_edge_train(ctx, inc, Xn, Xe, SEED, HIDDEN, 1, BATCH, LR)   # warm-up
    _native.lp_node_edge_predict(ctx, Xn, Xe, w, nodes, edges)
    torch.cuda.synchronize()
    pool.reset()
    split = {}
    t = time.perf_counter()
    w, losses = _native.lp_node_edge_train(ctx, inc, Xn, Xe, SEED, HIDDEN, EPOCHS, BATCH, LR, timings=split)
    torch.cuda.synchronize()
    train_s = time.perf_counter() - t
    t = time.perf_counter()
    _, keep = _native.lp_node_edge_predict(ctx, Xn, Xe, w, nodes, edges)
    torch.cuda.synchronize()
    predict_s = time.perf_counter() - t
    peak = pool.high()
    M = 2 * inc.nnz
  finally:
    inc.close()
  keep = keep.cpu().numpy()
  epoch_s = float(np.mean(split["epochs"]))
  out = {"samples": M, "batches_per_epoch": -(-M // BATCH), "train_s": train_s, "setup_s": split["setup"],
         "epoch_s": split["epochs"], "samples_per_s": M / epoch_s, "us_per_batch": epoch_s / -(-M // BATCH) * 1e6,
         "predict_s": predict_s, "links": int(len(links)), "pool_peak_gb": peak / 1e9, "losses": losses.tolist()}
  out.update(metrics(links[keep], good, bad))
  return out


def svc_side(R, xn, links, good, bad):
  import torch
  from hypergraphembedding_b200 import evaluation_util as ev
  ev.PersonalizedClassifierPredictionDevice(R, xn, links, True, seed=SEED)   # warm-up
  torch.cuda.synchronize()
  t = time.perf_counter()
  keep = ev.PersonalizedClassifierPredictionDevice(R, xn, links, True, seed=SEED)
  out = {"s": time.perf_counter() - t}
  out.update(metrics(links[keep], good, bad))
  return out


def host_side(R, xn, xe, links, good, bad):
  """the model of oracle/lp_node_edge_ref.py in torch (CPU, fp32) on the device's training set and orders"""
  import torch
  from oracle import lp_node_edge_ref as ref
  t = time.perf_counter()
  nodes, edges, labels = ref.training_set(R.indptr, R.indices, R.shape[1], SEED)
  orders = [ref.shuffle_order(SEED, e, len(nodes)) for e in range(EPOCHS)]
  prm = [torch.tensor(w, requires_grad=True) for w in ref.init_weights(SEED, xn.shape[1], HIDDEN)]
  opt = torch.optim.Adagrad(prm, lr=LR, eps=1e-7, initial_accumulator_value=0)
  Xn, Xe = torch.from_numpy(xn), torch.from_numpy(xe)
  N, E, Y = torch.from_numpy(nodes), torch.from_numpy(edges), torch.from_numpy(labels.astype(np.float32))
  setup = time.perf_counter() - t
  t = time.perf_counter()
  for order in orders:
    order = torch.from_numpy(order)
    for first in range(0, len(order), BATCH):
      s = order[first:first + BATCH]
      x = torch.cat([Xn[N[s]], Xe[E[s]]], dim=1)
      z = torch.relu(x @ prm[0] + prm[1]) @ prm[2] + prm[3][0]
      loss = torch.nn.functional.binary_cross_entropy_with_logits(z, Y[s])
      opt.zero_grad()
      loss.backward()
      opt.step()
  train_s = time.perf_counter() - t
  with torch.no_grad():
    x = torch.cat([Xn[torch.from_numpy(links[:, 0])], Xe[torch.from_numpy(links[:, 1])]], dim=1)
    p = torch.sigmoid(torch.relu(x @ prm[0] + prm[1]) @ prm[2] + prm[3][0]).numpy()
  out = {"setup_s": setup, "train_s": train_s, "threads": torch.get_num_threads()}
  out.update(metrics(links[p > 0.5], good, bad))
  return out


def main():
  ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
  ap.add_argument("--out", required=True, help="directory for lp_node_edge_bench.json")
  ap.add_argument("--sizes", default="20000,100000,1000000", help=argparse.SUPPRESS)
  args = ap.parse_args()
  import torch
  from hypergraphembedding_b200 import synthetic
  torch.zeros(1, device="cuda")   # the driver is initialised before the pool is looked up
  pool = PoolStats()
  result = {"gpu": gpu_info(), "model": {"hidden": HIDDEN, "epochs": EPOCHS, "batch": BATCH, "lr": LR},
            "runs": []}
  for size in [int(s) for s in args.sizes.split(",")]:
    A = synthetic.zipf_hypergraph(size, size // 2, seed=2024)
    run = {"nodes": size, "edges": size // 2, "incidences": int(A.nnz)}
    R, _, good, bad = hook_links(A) if size <= 20000 else numpy_links(A)
    R.sort_indices()
    run["hidden_links"] = int(len(good))
    xn, xe = embed(R)
    links = np.concatenate([bad, good])
    run["device"] = device_side(R, xn, xe, links, good, bad, pool)
    run["LP_EDGE_CLASSIFIERS_device"] = svc_side(R, xn, links, good, bad)
    if size <= 20000:
      run["host_torch_cpu"] = host_side(R, xn, xe, links, good, bad)
    print(size, json.dumps(run), flush=True)
    result["runs"].append(run)
  os.makedirs(args.out, exist_ok=True)
  with open(os.path.join(args.out, "lp_node_edge_bench.json"), "w") as f:
    json.dump(result, f, indent=1)


if __name__ == "__main__":
  main()
