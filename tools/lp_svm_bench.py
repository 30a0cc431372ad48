"""The personalized link-prediction classifiers on the GPU (hge_lp_svm_predict) on the config-4 family
(zipf_hypergraph(n, n / 2, seed=2024)), n in {20 000, 100 000, 1 000 000}:

  links      10 % of the connections hidden and as many sampled non-connections: through the
             reference hooks (RemoveRandomConnections / SampleMissingConnections on a proto, Python's
             `random` seeded) at 20 000 nodes, a seeded numpy equivalent above that;
  embedding  FOBE on the reduced graph (BooleanSamplesDevice, k 5, 200 samples, dimension 32,
             2 epochs at batch 4 096, seeded), the tables read back;
  device     PersonalizedClassifierPredictionDevice on both sides: the call, its grouping / negatives
             / solve / predict split (each ended by a device synchronise), SMO iterations (median,
             p99, max), owners at the iteration cap, the peak of the device's default memory pool,
             accuracy and F1;
  host       at 20 000 nodes only, LP_EDGE_CLASSIFIERS / LP_NODE_CLASSIFIERS (scikit-learn) on the
             same links and embedding: time, accuracy and F1.  They draw other negatives, so the
             metrics are close, not equal.

The GPU's name and power limit are read in the same run.

    python tools/lp_svm_bench.py --out DIR
"""
import argparse
import json
import os
import random
import sys
import time

import numpy as np
import scipy.sparse as sps

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from device_sampler_bench import gpu_info  # noqa: E402
from hg2v_device_bench import PoolStats  # noqa: E402

K, SAMPLES, DIM, EPOCHS, BATCH, SEED, REMOVAL = 5, 200, 32, 2, 4096, 1, 0.1


def proto(A):
  from hypergraphembedding_b200 import Hypergraph
  hg = Hypergraph()
  A = sps.csr_matrix(A)
  B = A.T.tocsr()
  for n in range(A.shape[0]):
    hg.node[n].edges.extend(A.indices[A.indptr[n]:A.indptr[n + 1]].tolist())
  for e in range(A.shape[1]):
    hg.edge[e].nodes.extend(B.indices[B.indptr[e]:B.indptr[e + 1]].tolist())
  return hg


def hook_links(A):
  """(reduced CSR, reduced proto, good, bad) through the reference hooks"""
  from hypergraphembedding_b200 import evaluation_util as ev
  from hypergraphembedding_b200.hypergraph_util import ToCsrMatrix
  hg = proto(A)
  random.seed(2024)
  reduced, good = ev.RemoveRandomConnections(hg, REMOVAL)
  bad = ev.SampleMissingConnections(hg, len(good))
  R = sps.csr_matrix(ToCsrMatrix(reduced), shape=A.shape)
  return R, reduced, np.asarray(good, dtype=np.int64), np.asarray(bad, dtype=np.int64)


def numpy_links(A):
  """RemoveRandomConnections / SampleMissingConnections restated on the CSR with a seeded numpy
  generator: connections visited in a random order, each dropped with probability 0.1 unless it is
  its node's or its edge's last; as many distinct non-connections drawn uniformly."""
  rng = np.random.RandomState(2024)
  C = A.tocoo()
  n, e = C.row.astype(np.int64), C.col.astype(np.int64)
  left_n, left_e = np.bincount(n, minlength=A.shape[0]), np.bincount(e, minlength=A.shape[1])
  drop = np.zeros(len(n), dtype=bool)
  coin = rng.rand(len(n)) < REMOVAL
  for i in rng.permutation(len(n)).tolist():
    if coin[i] and left_n[n[i]] > 1 and left_e[e[i]] > 1:
      drop[i] = True
      left_n[n[i]] -= 1
      left_e[e[i]] -= 1
  good = np.stack([n[drop], e[drop]], axis=1)
  R = sps.csr_matrix((np.ones(int((~drop).sum()), dtype=bool), (n[~drop], e[~drop])), shape=A.shape)
  R.sort_indices()
  present = set((n * A.shape[1] + e).tolist())
  bad = set()
  while len(bad) < len(good):
    cand = rng.randint(0, A.shape[0], len(good)) * A.shape[1] + rng.randint(0, A.shape[1], len(good))
    bad.update(c for c in cand.tolist() if c not in present)
  bad = np.asarray(sorted(bad)[:len(good)], dtype=np.int64)
  return R, None, good, np.stack([bad // A.shape[1], bad % A.shape[1]], axis=1)


def embed(R):
  """FOBE tables of the reduced graph (rows of the nodes / edges)"""
  import hypergraphembedding_b200 as H
  from hypergraphembedding_b200.hg2v_model import Hg2vModel
  samples = H.BooleanSamplesDevice(R, K, SAMPLES, seed=SEED, keep_on_device=True)
  model = Hg2vModel.seeded(R.shape[0], R.shape[1], DIM, K, "sigmoid", "kullback_leibler_divergence", SEED)
  try:
    model.fit_device(samples, batch_size=BATCH, epochs=EPOCHS, seed=SEED, verbose=0)
    node, edge = model.weights()
  finally:
    model.close()
  return node[1:R.shape[0] + 1], edge[1:R.shape[1] + 1]


def metrics(kept, good, bad):
  from hypergraphembedding_b200 import evaluation_util as ev
  m = ev.CalculateCommunityPredictionMetrics([tuple(l) for l in kept], [tuple(l) for l in good.tolist()],
                                             [tuple(l) for l in bad.tolist()])
  return {"accuracy": m.accuracy, "f1": m.f1, "true_pos": m.num_true_pos, "false_pos": m.num_false_pos}


def device_side(R, xn, xe, links, good, bad, per_edge, pool):
  import torch
  from hypergraphembedding_b200 import _native
  from hypergraphembedding_b200.hg2v_sample import _Graph
  g = _Graph.from_csr(R)
  ctx = _native.default_context()
  dev = torch.device("cuda", ctx.device)
  X = torch.from_numpy(xn if per_edge else xe).to(dev)
  items = torch.from_numpy((links[:, 0] if per_edge else links[:, 1]).astype(np.int32)).to(dev)
  owners = torch.from_numpy((links[:, 1] if per_edge else links[:, 0]).astype(np.int32)).to(dev)
  inc = g.incidence(ctx)
  try:
    _native.lp_svm_predict(ctx, inc, 1 if per_edge else 0, X, items, owners, SEED)   # warm-up
    torch.cuda.synchronize()
    pool.reset()
    t = time.perf_counter()
    keep, _, capped = _native.lp_svm_predict(ctx, inc, 1 if per_edge else 0, X, items, owners, SEED)
    torch.cuda.synchronize()
    total = time.perf_counter() - t
    peak = pool.high()
    split = {}
    _, _, _, model = _native.lp_svm_predict(ctx, inc, 1 if per_edge else 0, X, items, owners, SEED,
                                            return_model=True, timings=split)
  finally:
    inc.close()
  keep = keep.cpu().numpy()
  it = model.iterations[np.diff(model.offset) > 0]
  n = np.diff(model.offset)
  out = {"s": total, "phases_s": split, "named_owners": int(len(model.owner_ids)),
         "trained_owners": int(len(it)), "training_points": int(model.offset[-1]),
         "largest_owner_points": int(n.max(initial=0)), "owners_at_cap": int(capped),
         "smo_iterations": {"median": float(np.median(it)) if len(it) else 0,
                            "p99": float(np.percentile(it, 99)) if len(it) else 0, "max": int(it.max(initial=0))},
         "pool_peak_gb": peak / 1e9}
  out.update(metrics(links[keep], good, bad))
  return out


def host_side(reduced, xn, xe, links, good, bad, per_edge):
  from hypergraphembedding_b200 import HypergraphEmbedding, evaluation_util as ev
  emb = HypergraphEmbedding()
  emb.dim = DIM
  for i, v in enumerate(xn.tolist()):
    emb.node[i].values.extend(v)
  for i, v in enumerate(xe.tolist()):
    emb.edge[i].values.extend(v)
  fn = ev.PersonalizedEdgeClassifierPrediction if per_edge else ev.PersonalizedNodeClassifierPrediction
  random.seed(7)
  t = time.perf_counter()
  kept = fn(reduced, emb, [tuple(l) for l in links.tolist()])
  out = {"s": time.perf_counter() - t}
  out.update(metrics(np.asarray(kept, dtype=np.int64).reshape(-1, 2), good, bad))
  return out


def main():
  ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
  ap.add_argument("--out", required=True, help="directory for lp_svm_bench.json")
  ap.add_argument("--sizes", default="20000,100000,1000000", help=argparse.SUPPRESS)
  args = ap.parse_args()
  import torch
  from hypergraphembedding_b200 import synthetic
  torch.zeros(1, device="cuda")   # the driver is initialised before the pool is looked up
  pool = PoolStats()
  result = {"gpu": gpu_info(), "runs": []}
  for size in [int(s) for s in args.sizes.split(",")]:
    A = synthetic.zipf_hypergraph(size, size // 2, seed=2024)
    run = {"nodes": size, "edges": size // 2, "incidences": int(A.nnz)}
    t = time.perf_counter()
    R, reduced, good, bad = hook_links(A) if size <= 20000 else numpy_links(A)
    run["links_s"] = time.perf_counter() - t
    run["hidden_links"] = int(len(good))
    t = time.perf_counter()
    xn, xe = embed(R)
    run["embedding_s"] = time.perf_counter() - t
    links = np.concatenate([bad, good])
    for name, per_edge in (("LP_EDGE_CLASSIFIERS", True), ("LP_NODE_CLASSIFIERS", False)):
      run[name] = {"device": device_side(R, xn, xe, links, good, bad, per_edge, pool)}
      if reduced is not None:
        run[name]["host"] = host_side(reduced, xn, xe, links, good, bad, per_edge)
      print(name, size, json.dumps(run[name]), flush=True)
    result["runs"].append(run)
  os.makedirs(args.out, exist_ok=True)
  with open(os.path.join(args.out, "lp_svm_bench.json"), "w") as f:
    json.dump(result, f, indent=1)


if __name__ == "__main__":
  main()
