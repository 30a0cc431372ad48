"""hypergraph2vec training on device-resident samples (BooleanSamplesDevice(keep_on_device=True) ->
Hg2vModel.seeded -> fit_device) against the existing path on the same graph
(BooleanSamplesDevice -> SamplesToModelInput -> Hg2vModel.fit), in one process:

  * FOBE on the 1 000 000-node member of the config-4 family (zipf_hypergraph(1000000, 500000,
    seed=2024), k 5, 200 samples: about 108 M records), dimension 32, 2 epochs at batch 256 and
    at batch 4 096;
  * with --full, the new path on config 4 itself (10 M nodes, about 1.08e9 records) at batch
    4 096: its times and peak memory, or the HGE_ERR_NOMEM the library returns when the set does
    not fit.

New path, timed: sampling, packing into the model's buffer (append kernels, release of the raw
blocks), then per epoch the shuffle (hge_shuffle_order) and the training launch.  Existing path,
timed: sampling (columns copied to the host), packing (SamplesToModelInput), upload
(set_samples: stack, host range check, copy), then per epoch the host shuffle (np.random.shuffle)
and the training call (host range check of the order, upload, launch).  Every timed step ends in
a device synchronise.  Also reported: peak device memory (torch's allocator, which holds the raw
blocks, and the device's default stream-ordered pool, which holds the library's buffers), host
peak RSS after each path, the per-epoch losses, and the GPU's name and power limit.

    python tools/hg2v_device_bench.py --out DIR [--full]
"""
import argparse
import ctypes
import json
import os
import resource
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from device_sampler_bench import gpu_info  # noqa: E402

K, SAMPLES, DIM, EPOCHS, SEED = 5, 200, 32, 2, 1


class PoolStats(object):
  """Used-memory high-water mark of the device's default memory pool (the library allocates with
  cudaMallocAsync from it), read through the driver API."""

  USED_MEM_HIGH = 8   # CU_MEMPOOL_ATTR_USED_MEM_HIGH

  def __init__(self, device=0):
    self.cu = ctypes.CDLL("libcuda.so.1")
    dev = ctypes.c_int()
    assert self.cu.cuDeviceGet(ctypes.byref(dev), device) == 0
    self.pool = ctypes.c_void_p()
    assert self.cu.cuDeviceGetDefaultMemPool(ctypes.byref(self.pool), dev) == 0

  def reset(self):
    zero = ctypes.c_uint64(0)
    self.cu.cuMemPoolSetAttribute(self.pool, self.USED_MEM_HIGH, ctypes.byref(zero))

  def high(self):
    v = ctypes.c_uint64(0)
    self.cu.cuMemPoolGetAttribute(self.pool, self.USED_MEM_HIGH, ctypes.byref(v))
    return int(v.value)


def reset_peaks(pool):
  import torch
  torch.cuda.synchronize()
  torch.cuda.reset_peak_memory_stats()
  pool.reset()


def peaks(pool):
  import torch
  torch.cuda.synchronize()
  return {"torch_allocated_gb": torch.cuda.max_memory_allocated() / 1e9, "pool_used_gb": pool.high() / 1e9}


def rss_gb():
  return resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 1e6   # ru_maxrss is in kB on Linux


def timed(fn):
  import torch
  torch.cuda.synchronize()
  t = time.perf_counter()
  out = fn()
  torch.cuda.synchronize()
  return time.perf_counter() - t, out


def new_path(A, batch, pool, chunk_rows=0):
  """Sampling, packing, then per epoch shuffle + train, as fit_device runs them."""
  import torch
  import hypergraphembedding_b200 as H
  from hypergraphembedding_b200 import _native
  from hypergraphembedding_b200.hg2v_model import Hg2vModel
  reset_peaks(pool)
  out = {"batch": batch}
  model = Hg2vModel.seeded(A.shape[0], A.shape[1], DIM, K, "sigmoid", "kullback_leibler_divergence", SEED)
  try:
    out["sampling_s"], samples = timed(lambda: H.BooleanSamplesDevice(A, K, SAMPLES, seed=SEED,
                                                                      chunk_rows=chunk_rows,
                                                                      keep_on_device=True))
    out["records"] = len(samples)
    out["raw_blocks_gb"] = torch.cuda.memory_allocated() / 1e9
    out["pack_s"], _ = timed(lambda: model.set_device_samples(samples))
    del samples
    order = torch.empty(model.num_samples, dtype=torch.int32, device="cuda")
    out["epochs"] = []
    for epoch in range(EPOCHS):
      shuffle_s, _ = timed(lambda: _native.shuffle_order(model.ctx, SEED, epoch, model.num_samples, out=order))
      loss = ctypes.c_double()
      train_s, _ = timed(lambda: _native.check(model.ctx.lib.hge_hg2v_fit_epoch(
          model.handle, _native.ptr(order), batch, _native.MEM_DEVICE, ctypes.byref(loss))))
      out["epochs"].append({"shuffle_s": shuffle_s, "train_s": train_s, "loss": loss.value})
    del order
  finally:
    model.close()
  out["total_s"] = out["sampling_s"] + out["pack_s"] + sum(e["shuffle_s"] + e["train_s"] for e in out["epochs"])
  out["peak_device"] = peaks(pool)
  return out


class _Ids(object):
  """The id ranges Hg2vModel's constructor reads from a hypergraph."""

  def __init__(self, nodes, edges):
    self.node, self.edge = range(nodes), range(edges)


def existing_path(A, batches, pool):
  """BooleanSamplesDevice -> SamplesToModelInput -> set_samples + per epoch np.random.shuffle and
  fit_epoch, as Hg2vModel.fit runs them; the sampling and packing are shared by the batch sizes."""
  import hypergraphembedding_b200 as H
  from hypergraphembedding_b200.hg2v_model import Hg2vModel
  reset_peaks(pool)
  out = {}
  out["sampling_s"], cols = timed(lambda: H.BooleanSamplesDevice(A, K, SAMPLES, seed=SEED))
  out["records"] = len(cols)
  out["pack_s"], (feats, targets) = timed(lambda: H.SamplesToModelInput(cols, K, weighted=False))
  del cols
  out["runs"] = []
  np.random.seed(SEED)
  for batch in batches:
    run = {"batch": batch}
    model = Hg2vModel(_Ids(A.shape[0], A.shape[1]), DIM, K, "sigmoid", "kullback_leibler_divergence")
    try:
      run["upload_s"], _ = timed(lambda: model.set_samples(feats, targets))
      run["epochs"] = []
      for _ in range(EPOCHS):
        index = np.arange(model.num_samples)
        shuffle_s, _ = timed(lambda: np.random.shuffle(index))
        train_s, loss = timed(lambda: model.fit_epoch(index, batch))
        run["epochs"].append({"shuffle_s": shuffle_s, "train_s": train_s, "loss": loss})
    finally:
      model.close()
    run["total_s"] = out["sampling_s"] + out["pack_s"] + run["upload_s"] + sum(
        e["shuffle_s"] + e["train_s"] for e in run["epochs"])
    out["runs"].append(run)
  out["peak_device"] = peaks(pool)
  return out


def main():
  ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
  ap.add_argument("--out", required=True, help="directory for hg2v_device_bench.json")
  ap.add_argument("--full", action="store_true", help="also try the new path on config 4 (10 M nodes)")
  ap.add_argument("--nodes", type=int, default=1000000, help=argparse.SUPPRESS)   # rehearsal at small sizes
  args = ap.parse_args()
  import torch
  assert torch.cuda.is_available(), "the benchmark needs a CUDA device"
  from hypergraphembedding_b200 import synthetic
  os.makedirs(args.out, exist_ok=True)
  pool = PoolStats()
  result = {"gpu": gpu_info(), "host_threads": os.cpu_count(), "k": K, "num_samples": SAMPLES,
            "dimension": DIM, "epochs": EPOCHS}
  n, e = args.nodes, args.nodes // 2
  A = synthetic.zipf_hypergraph(n, e, seed=2024)
  result["graph"] = "zipf_hypergraph(%d, %d, seed=2024)" % (n, e)
  # warm-up: modules, memory pools, cub tuning of every kernel both paths launch
  small = synthetic.zipf_hypergraph(20000, 10000, seed=1)
  new_path(small, 256, pool)
  new_path(small, 4096, pool)
  existing_path(small, [256], pool)
  result["new"] = []
  for batch in (256, 4096):
    result["new"].append(new_path(A, batch, pool))
    print(json.dumps(result["new"][-1]), flush=True)
  result["new_host_peak_rss_gb"] = rss_gb()
  result["existing"] = existing_path(A, [256, 4096], pool)
  print(json.dumps(result["existing"]), flush=True)
  result["existing_host_peak_rss_gb"] = rss_gb()
  del A
  if args.full:
    from hypergraphembedding_b200 import _native
    t = time.perf_counter()
    A = synthetic.zipf_hypergraph(10000000, 5000000, seed=2024)
    full = {"graph": "config 4: zipf_hypergraph(10000000, 5000000, seed=2024)",
            "generate_s": time.perf_counter() - t}
    try:
      full.update(new_path(A, 4096, pool, chunk_rows=262144))
    except MemoryError as exc:     # HGE_ERR_NOMEM from the library
      full["nomem"] = str(exc) or _native.last_error()
    except torch.cuda.OutOfMemoryError as exc:
      full["nomem"] = "torch: %s" % exc
    full["host_peak_rss_gb"] = rss_gb()
    result["full_config4"] = full
    print(json.dumps(full), flush=True)
  path = os.path.join(args.out, "hg2v_device_bench.json")
  with open(path, "w") as f:
    json.dump(result, f, indent=1)
  print("wrote", path)


if __name__ == "__main__":
  main()
