"""ctypes binding of libhge_b200.so (include/hge_b200.h).

There is deliberately no fallback here: if the shared library is missing or no CUDA
device is usable, the first call raises.  Build the library with
``python -m hypergraphembedding_b200.build`` (or ``__graft_entry__.build()``).
"""
import ctypes
import os
import threading

import numpy as np

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "libhge_b200.so")

HGE_OK = 0
HGE_ERR_INVALID = -1
HGE_ERR_CUDA = -2
HGE_ERR_EMPTY_ROW = -3
HGE_ERR_NOMEM = -4
HGE_ERR_UNSUPPORTED = -5
MEM_HOST = 0
MEM_DEVICE = 1

c_i32p = ctypes.POINTER(ctypes.c_int32)
c_i64p = ctypes.POINTER(ctypes.c_int64)
c_u32p = ctypes.POINTER(ctypes.c_uint32)
c_f32p = ctypes.POINTER(ctypes.c_float)
c_f64p = ctypes.POINTER(ctypes.c_double)
c_vp = ctypes.c_void_p


class NativeLibraryMissing(ImportError):
  pass


class NativeError(RuntimeError):
  pass


_lib = None
_lock = threading.Lock()

# name -> (restype, argtypes); checked against include/hge_b200.h by tests/test_abi.py
SIGNATURES = {
    "hge_version": (ctypes.c_int, []),
    "hge_last_error": (ctypes.c_char_p, []),
    "hge_ctx_create": (ctypes.c_int, [ctypes.c_int, c_vp, ctypes.POINTER(c_vp)]),
    "hge_ctx_destroy": (ctypes.c_int, [c_vp]),
    "hge_ctx_set_stream": (ctypes.c_int, [c_vp, c_vp]),
    "hge_ctx_sync": (ctypes.c_int, [c_vp]),
    "hge_ctx_set_tuning": (ctypes.c_int, [c_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "hge_ctx_reset_tuning": (ctypes.c_int, [c_vp]),
    "hge_ctx_set_tile_mb": (ctypes.c_int, [c_vp, ctypes.c_int, ctypes.c_int]),
    "hge_ctx_set_trainer_clusters": (ctypes.c_int, [c_vp, ctypes.c_int]),
    "hge_ctx_launch_count": (ctypes.c_int64, [c_vp]),
    "hge_incidence_create": (ctypes.c_int, [c_vp, ctypes.c_int32, ctypes.c_int32, c_vp, c_vp, c_vp,
                                            c_vp, ctypes.c_int, ctypes.POINTER(c_vp)]),
    "hge_incidence_destroy": (ctypes.c_int, [c_vp]),
    "hge_incidence_nnz": (ctypes.c_int64, [c_vp]),
    "hge_algdist_run": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, ctypes.c_int, ctypes.c_int,
                                       ctypes.c_int, c_vp]),
    "hge_algdist_run_csr": (ctypes.c_int, [c_vp, ctypes.c_int32, ctypes.c_int32, c_vp, c_vp, c_vp, c_vp, c_vp,
                                           c_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_vp]),
    "hge_column_rescale": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int64, c_vp, ctypes.c_int64, ctypes.c_int,
                                          ctypes.c_int]),
    "hge_algdist_create": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int, ctypes.c_int,
                                          ctypes.POINTER(c_vp)]),
    "hge_algdist_destroy": (ctypes.c_int, [c_vp]),
    "hge_algdist_load": (ctypes.c_int, [c_vp, c_vp, c_vp, ctypes.c_int]),
    "hge_algdist_node_half": (ctypes.c_int, [c_vp, ctypes.c_int]),
    "hge_algdist_edge_half": (ctypes.c_int, [c_vp, ctypes.c_int]),
    "hge_algdist_edge_partial": (ctypes.c_int, [c_vp, ctypes.c_int, ctypes.c_int, c_vp]),
    "hge_algdist_edge_finalize": (ctypes.c_int, [c_vp, ctypes.c_int, ctypes.c_int, c_vp]),
    "hge_incidence_create_sharded": (ctypes.c_int, [c_vp, ctypes.c_int32, ctypes.c_int32, c_vp,
                                                    c_vp, c_vp, c_vp, ctypes.c_int, ctypes.c_int,
                                                    ctypes.POINTER(c_vp)]),
    "hge_incidence_edge_sums": (ctypes.c_int, [c_vp, ctypes.POINTER(c_vp), ctypes.POINTER(c_vp)]),
    "hge_incidence_finish_sharded": (ctypes.c_int, [c_vp]),
    "hge_incidence_slice_range": (ctypes.c_int, [c_vp, ctypes.c_int, c_i32p, c_i32p]),
    "hge_algdist_minmax_ptr": (ctypes.c_int, [c_vp, ctypes.c_int, ctypes.POINTER(c_vp)]),
    "hge_algdist_ld": (ctypes.c_int, [c_vp]),
    "hge_algdist_store": (ctypes.c_int, [c_vp, ctypes.c_int, c_vp, c_vp, ctypes.c_int]),
    "hge_p2p_create": (ctypes.c_int, [c_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int32, ctypes.c_int32,
                                      ctypes.c_int, ctypes.POINTER(c_vp)]),
    "hge_p2p_export": (ctypes.c_int, [c_vp, c_vp]),
    "hge_p2p_open_peers": (ctypes.c_int, [c_vp, c_vp]),
    "hge_p2p_check": (ctypes.c_int, [c_vp]),
    "hge_p2p_phase_ms": (ctypes.c_int, [c_vp, c_vp, c_vp]),
    "hge_p2p_set_timing": (ctypes.c_int, [c_vp, ctypes.c_int]),
    "hge_p2p_close_peers": (ctypes.c_int, [c_vp]),
    "hge_p2p_destroy": (ctypes.c_int, [c_vp]),
    "hge_algdist_attach_p2p": (ctypes.c_int, [c_vp, c_vp]),
    "hge_algdist_sweep_p2p": (ctypes.c_int, [c_vp, ctypes.c_int]),
    "hge_incidence_l2": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, ctypes.c_int, ctypes.c_int,
                                        ctypes.c_int, c_vp, ctypes.c_int]),
    "hge_pair_l2": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int64, c_vp, ctypes.c_int64, ctypes.c_int,
                                   c_vp, c_vp, ctypes.c_int64, c_vp, ctypes.c_int]),
    "hge_scale_transform": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int64, ctypes.c_double, c_vp,
                                           ctypes.c_int]),
    "hge_scale_minmax": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int64, c_vp, ctypes.c_int]),
    "hge_scale_apply": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int64, ctypes.c_double, ctypes.c_float,
                                       ctypes.c_float, ctypes.c_int]),
    "hge_row_span": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, ctypes.c_int, ctypes.c_int, c_vp,
                                    ctypes.c_int]),
    "hge_same_type_prob": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int, c_vp, c_vp, c_vp,
                                          ctypes.c_int64, c_vp, ctypes.c_int]),
    "hge_diff_type_prob": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, ctypes.c_int64, c_vp,
                                          ctypes.c_int]),
    "hge_jaccard_rows": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, ctypes.c_int64, ctypes.c_int64, c_vp,
                                        c_vp, ctypes.c_int64, c_vp, ctypes.c_int]),
    "hge_jaccard_centroid": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, ctypes.c_int64, ctypes.c_int64,
                                            c_vp, c_vp, ctypes.c_int64, ctypes.c_int64, c_vp, c_vp,
                                            c_vp, ctypes.c_int64, ctypes.c_int64, c_vp, c_vp,
                                            ctypes.c_int64, c_vp, ctypes.c_int]),
    "hge_jaccard_centroid_grouped": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int, c_vp, c_vp, c_vp, ctypes.c_int64,
                                                    ctypes.c_int64, c_vp, c_vp, c_vp, ctypes.c_int64,
                                                    ctypes.c_int64, c_vp, c_vp, ctypes.c_int64, ctypes.c_int64,
                                                    c_vp]),
    "hge_hg2v_create": (ctypes.c_int, [c_vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int, ctypes.c_int,
                                       ctypes.c_int, ctypes.c_int, c_vp, c_vp, ctypes.c_int,
                                       ctypes.POINTER(c_vp)]),
    "hge_hg2v_destroy": (ctypes.c_int, [c_vp]),
    "hge_hg2v_set_samples": (ctypes.c_int, [c_vp, c_vp, c_vp, ctypes.c_int64, ctypes.c_int]),
    "hge_hg2v_fit_epoch": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int, ctypes.c_int,
                                          ctypes.POINTER(ctypes.c_double)]),
    "hge_hg2v_get_weights": (ctypes.c_int, [c_vp, c_vp, c_vp, ctypes.c_int]),
    "hge_hg2v_last_clusters": (ctypes.c_int, [c_vp]),
    "hge_hg2v_create_seeded": (ctypes.c_int, [c_vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int, ctypes.c_int,
                                              ctypes.c_int, ctypes.c_int, ctypes.c_uint64, ctypes.POINTER(c_vp)]),
    "hge_hg2v_reserve_samples": (ctypes.c_int, [c_vp, ctypes.c_int64]),
    "hge_hg2v_append_samples": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, ctypes.c_int,
                                               ctypes.c_float, ctypes.c_int64]),
    "hge_hg2v_get_samples": (ctypes.c_int, [c_vp, c_vp, c_vp, ctypes.c_int]),
    "hge_shuffle_order": (ctypes.c_int, [c_vp, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int64, c_vp,
                                         ctypes.c_int]),
    "hge_lp_svm_predict": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int, c_vp, ctypes.c_int, c_vp, c_vp, ctypes.c_int64,
                                          ctypes.c_uint64, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                                          ctypes.c_int64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                          ctypes.c_int64, c_vp]),
    "hge_lp_node_edge_train": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, ctypes.c_int, ctypes.c_int, ctypes.c_uint64,
                                              ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_float, c_vp, c_vp,
                                              c_vp, c_vp, c_vp, c_vp]),
    "hge_lp_node_edge_samples": (ctypes.c_int, [c_vp, c_vp, ctypes.c_uint64, ctypes.c_int, c_vp, c_vp, c_vp]),
    "hge_lp_node_edge_predict": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int64, c_vp, ctypes.c_int64, ctypes.c_int,
                                                ctypes.c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, ctypes.c_int64, c_vp,
                                                c_vp]),
    "hge_nmf_init": (ctypes.c_int, [c_vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int, ctypes.c_uint64,
                                    ctypes.c_float, c_vp, c_vp, ctypes.c_int]),
    "hge_nmf_fit": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int, c_vp, c_vp,
                                   ctypes.c_int, ctypes.c_double, ctypes.c_int, ctypes.POINTER(ctypes.c_int), c_vp,
                                   c_vp]),
    "hge_svd_start": (ctypes.c_int, [c_vp, ctypes.c_int32, ctypes.c_int, ctypes.c_uint64, c_vp, ctypes.c_int]),
    "hge_svd_half": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int, ctypes.c_int32, ctypes.c_int32, ctypes.c_int, c_vp,
                                    c_vp, c_vp, ctypes.c_int, c_vp]),
    "hge_svd_rowmat": (ctypes.c_int, [c_vp, ctypes.c_int64, ctypes.c_int, ctypes.c_int, c_vp, c_vp, c_vp,
                                      ctypes.c_int]),
    "hge_svd_flip": (ctypes.c_int, [c_vp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int, ctypes.c_int, c_vp, c_vp,
                                    ctypes.c_int]),
    "hge_svd_residuals": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int, ctypes.c_int,
                                         c_vp, c_vp, c_vp, c_vp, ctypes.c_int]),
    "hge_n2v_walks": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_double,
                                     ctypes.c_uint64, c_vp, c_vp]),
    "hge_n2v_pairs": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_uint64, c_vp,
                                     ctypes.c_int64, ctypes.POINTER(ctypes.c_int64)]),
    "hge_n2v_negatives": (ctypes.c_int, [c_vp, ctypes.c_int64, c_vp, ctypes.c_int32, ctypes.c_int, ctypes.c_uint64,
                                         ctypes.c_int, c_vp]),
    "hge_n2v_init": (ctypes.c_int, [c_vp, ctypes.c_int32, ctypes.c_int, ctypes.c_uint64, c_vp, c_vp]),
    "hge_n2v_train_epoch": (ctypes.c_int, [c_vp, ctypes.c_int32, ctypes.c_int, c_vp, c_vp, c_vp, ctypes.c_int64,
                                           c_vp, ctypes.c_int, ctypes.c_uint64, ctypes.c_int, ctypes.c_int,
                                           ctypes.c_int, ctypes.c_double, ctypes.c_double, ctypes.c_int64,
                                           ctypes.POINTER(ctypes.c_double)]),
    "hge_n2v_clique_walks": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double,
                                            ctypes.c_double, ctypes.c_uint64, c_vp, c_vp]),
    "hge_mt19937_random_raw":(ctypes.c_int, [c_vp, ctypes.c_int64, c_vp]),
    "hge_mt19937_interval": (ctypes.c_int, [c_vp, ctypes.c_uint32, ctypes.c_int64, c_vp]),
    "hge_spgemm_rows": (ctypes.c_int, [ctypes.c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                       ctypes.c_int32, ctypes.c_int32, c_vp, ctypes.c_int64,
                                       ctypes.c_int, c_vp, c_vp, ctypes.c_int64]),
    "hge_sample_adj_rows": (ctypes.c_int, [ctypes.c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                           ctypes.c_int32, ctypes.c_int32, c_vp, ctypes.c_int64,
                                           c_vp, ctypes.c_int, ctypes.c_int, c_vp, c_vp, c_vp,
                                           ctypes.c_int64, ctypes.POINTER(ctypes.c_int64)]),
    "hge_sampler_set_threads": (ctypes.c_int, [ctypes.c_int]),
    "hge_hypergraph_parse": (ctypes.c_int, [c_vp, ctypes.c_size_t, ctypes.POINTER(c_vp)]),
    "hge_hypergraph_destroy": (ctypes.c_int, [c_vp]),
    "hge_hypergraph_sizes": (ctypes.c_int, [c_vp, c_vp]),
    "hge_hypergraph_arrays": (ctypes.c_int, [c_vp] * 9),
    "hge_hypergraph_compress": (ctypes.c_int, [c_vp] * 8),
    "hge_embedding_wire_size": (ctypes.c_int, [c_vp, ctypes.c_int64, c_vp, ctypes.c_int64,
                                               ctypes.c_int32, ctypes.c_int32, ctypes.c_char_p,
                                               ctypes.POINTER(ctypes.c_size_t)]),
    "hge_embedding_write": (ctypes.c_int, [c_vp, ctypes.c_int64, c_vp, c_vp, ctypes.c_int64, c_vp,
                                           ctypes.c_int32, ctypes.c_int32, ctypes.c_char_p, c_vp,
                                           ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t)]),
    "hge_embedding_parse": (ctypes.c_int, [c_vp, ctypes.c_size_t, ctypes.POINTER(c_vp)]),
    "hge_embedding_destroy": (ctypes.c_int, [c_vp]),
    "hge_embedding_sizes": (ctypes.c_int, [c_vp, c_vp, ctypes.POINTER(ctypes.c_int32)]),
    "hge_embedding_arrays": (ctypes.c_int, [c_vp] * 7),
    "hge_sample_neighbors": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, ctypes.c_int64,
                                            ctypes.c_int, c_vp, c_vp, c_vp]),
    "hge_sample_pairs_device": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int32,
                                               ctypes.c_int32, c_vp, ctypes.c_int, ctypes.c_uint64,
                                               ctypes.c_uint32, ctypes.c_int64, c_vp, c_vp,
                                               ctypes.c_int64, ctypes.POINTER(ctypes.c_int64),
                                               ctypes.c_int]),
    "hge_sample_neighbors_device": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, ctypes.c_int64, ctypes.c_int,
                                                   ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int64,
                                                   c_vp, c_vp, ctypes.c_int]),
}


def load_library():
  """Loads libhge_b200.so once.  Raises NativeLibraryMissing when it has not been built."""
  global _lib
  with _lock:
    if _lib is not None:
      return _lib
    if not os.path.exists(LIB_PATH):
      raise NativeLibraryMissing(
          "%s is missing: build it with `python -m hypergraphembedding_b200.build`. "
          "hypergraphembedding_b200 has no CPU or PyTorch fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
      fn = getattr(lib, name)  # AttributeError if the .so is stale
      fn.restype = restype
      fn.argtypes = argtypes
    _lib = lib
    return lib


def last_error():
  msg = load_library().hge_last_error()
  return msg.decode("utf-8", "replace") if msg else ""


def check(rc, what=""):
  """Maps a status code to the exception the reference would raise at that point."""
  if rc == HGE_OK:
    return
  msg = "%s%s" % (what + ": " if what else "", last_error())
  if rc == HGE_ERR_INVALID:
    raise AssertionError(msg)           # the reference validates with assert
  if rc == HGE_ERR_EMPTY_ROW:
    raise ZeroDivisionError(msg)        # algebraic_distance.py:49 divides 0/0
  if rc == HGE_ERR_NOMEM:
    raise MemoryError(msg)
  raise NativeError("%s (status %d)" % (msg, rc))


def ptr(x):
  """Address of a numpy array / torch tensor / None as a void pointer."""
  if x is None:
    return None
  if isinstance(x, np.ndarray):
    assert x.flags["C_CONTIGUOUS"], "array must be C-contiguous"
    return x.ctypes.data_as(c_vp)
  if hasattr(x, "data_ptr"):
    assert x.is_contiguous(), "tensor must be contiguous"
    return c_vp(x.data_ptr())
  if isinstance(x, int):
    return c_vp(x)
  raise TypeError("cannot take the address of %r" % type(x))


def is_device(x):
  return hasattr(x, "is_cuda") and x.is_cuda


class Context(object):
  """One hge_ctx per (device, stream)."""

  def __init__(self, device=0, stream=None):
    self.lib = load_library()
    self.device = int(device)
    handle = c_vp()
    stream_ptr = c_vp(int(stream)) if stream else None
    check(self.lib.hge_ctx_create(self.device, stream_ptr, ctypes.byref(handle)), "hge_ctx_create")
    self.handle = handle
    self._stream = int(stream) if stream else 0

  def set_stream(self, stream):
    check(self.lib.hge_ctx_set_stream(self.handle, c_vp(int(stream)) if stream else None))
    self._stream = int(stream) if stream else 0

  def bind_torch_stream(self):
    """Queues this context's work on torch's CURRENT stream of the device (a no-op while that
    is the stream already bound; switching drains the old one).  Callers that interleave torch
    collectives or kernels with library calls (distributed.py) rely on stream order, which only
    holds when both sides use the same stream -- e.g. inside ``with torch.cuda.stream(s):``."""
    try:
      import torch
    except ImportError:
      return
    if not torch.cuda.is_initialized():
      return
    current = int(torch.cuda.current_stream(self.device).cuda_stream)
    if current != getattr(self, "_stream", 0):
      self.set_stream(current)

  def set_tuning(self, light_max_deg=0, chunk=0, blocks_per_sm=0):
    check(self.lib.hge_ctx_set_tuning(self.handle, light_max_deg, chunk, blocks_per_sm))

  def set_tile_mb(self, tile_mb, min_rows_mb=1024):
    check(self.lib.hge_ctx_set_tile_mb(self.handle, int(tile_mb), int(min_rows_mb)))

  def set_trainer_clusters(self, max_clusters):
    """Cap on the clusters of one hypergraph2vec training launch (0: what fits the device)."""
    check(self.lib.hge_ctx_set_trainer_clusters(self.handle, int(max_clusters)))

  def reset_tuning(self):
    """Every schedule / kernel / tile knob back to the library's defaults."""
    check(self.lib.hge_ctx_reset_tuning(self.handle))

  def sync(self):
    check(self.lib.hge_ctx_sync(self.handle), "hge_ctx_sync")

  @property
  def launch_count(self):
    return int(self.lib.hge_ctx_launch_count(self.handle))

  def close(self):
    if getattr(self, "handle", None):
      self.lib.hge_ctx_destroy(self.handle)
      self.handle = None

  def __del__(self):
    try:
      self.close()
    except Exception:
      pass


_default_ctx = {}


def default_context(device=None):
  """Process-wide context of the current torch device, bound to torch's current stream of that
  device at every call (the legacy default stream when torch has not initialised CUDA)."""
  stream = None
  if device is None:
    device = 0
    try:
      import torch
      if torch.cuda.is_available():
        device = torch.cuda.current_device()
    except ImportError:
      pass
  key = int(device)
  ctx = _default_ctx.get(key)
  if ctx is None:
    ctx = Context(key, stream)
    _default_ctx[key] = ctx
  ctx.bind_torch_stream()
  return ctx


def _as_i64(a):
  return np.ascontiguousarray(a, dtype=np.int64)


def _as_i32(a):
  return np.ascontiguousarray(a, dtype=np.int32)


class Incidence(object):
  """Device-resident incidence (hge_incidence): int32 CSR of node->edge and edge->node.  With
  `sharded=True` it is one shard of a node-partitioned hypergraph: all-reduce the arrays
  returned by `edge_sums()` over the shards, then call `finish_sharded()`."""

  def __init__(self, ctx, num_nodes, num_edges, n2e_ptr, n2e_idx, e2n_ptr=None, e2n_idx=None,
               sharded=False, num_slices=1):
    """e2n_ptr / e2n_idx None: the library builds the edge -> node orientation on the device."""
    self.ctx = ctx
    self.num_nodes = int(num_nodes)
    self.num_edges = int(num_edges)
    device = is_device(n2e_idx)
    assert (e2n_ptr is None) == (e2n_idx is None)
    if device:
      keep = (n2e_ptr, n2e_idx, e2n_ptr, e2n_idx)   # borrowed by the library
      import torch
      assert n2e_ptr.dtype == torch.int64 and n2e_idx.dtype == torch.int32
      assert e2n_ptr is None or (e2n_ptr.dtype == torch.int64 and e2n_idx.dtype == torch.int32)
    elif e2n_ptr is None:
      keep = (_as_i64(n2e_ptr), _as_i32(n2e_idx), None, None)
    else:
      keep = (_as_i64(n2e_ptr), _as_i32(n2e_idx), _as_i64(e2n_ptr), _as_i32(e2n_idx))
    self._keep = keep
    handle = c_vp()
    self.num_slices = int(num_slices)
    if not sharded:
      check(ctx.lib.hge_incidence_create(ctx.handle, self.num_nodes, self.num_edges, ptr(keep[0]),
                                         ptr(keep[1]), ptr(keep[2]), ptr(keep[3]),
                                         MEM_DEVICE if device else MEM_HOST, ctypes.byref(handle)),
            "hge_incidence_create")
    else:
      check(ctx.lib.hge_incidence_create_sharded(
          ctx.handle, self.num_nodes, self.num_edges, ptr(keep[0]), ptr(keep[1]), ptr(keep[2]),
          ptr(keep[3]), self.num_slices, MEM_DEVICE if device else MEM_HOST, ctypes.byref(handle)),
            "hge_incidence_create_sharded")
    self.handle = handle
    self.nnz_n2e = int(keep[1].shape[0])
    self.nnz_e2n = int(keep[3].shape[0]) if keep[3] is not None else self.nnz_n2e
    if not device:
      self._keep = None  # the library copied the arrays

  @property
  def nnz(self):
    return int(self.ctx.lib.hge_incidence_nnz(self.handle))

  def nnz_of(self, order):
    return self.nnz_n2e if order == 0 else self.nnz_e2n

  def edge_sums(self):
    """(device pointer to int32 [E] local edge degrees, device pointer to f64 [E] local weight
    sums) of a pending shard; all-reduce both in place, then finish_sharded()."""
    deg, wsum = c_vp(), c_vp()
    check(self.ctx.lib.hge_incidence_edge_sums(self.handle, ctypes.byref(deg), ctypes.byref(wsum)),
          "hge_incidence_edge_sums")
    return deg.value, wsum.value

  def finish_sharded(self):
    check(self.ctx.lib.hge_incidence_finish_sharded(self.handle), "hge_incidence_finish_sharded")

  def slice_range(self, slice_index):
    r0, r1 = ctypes.c_int32(), ctypes.c_int32()
    check(self.ctx.lib.hge_incidence_slice_range(self.handle, slice_index, ctypes.byref(r0),
                                                 ctypes.byref(r1)), "hge_incidence_slice_range")
    return r0.value, r1.value

  def close(self):
    if getattr(self, "handle", None):
      self.ctx.lib.hge_incidence_destroy(self.handle)
      self.handle = None

  def __del__(self):
    try:
      self.close()
    except Exception:
      pass


def algdist_run(ctx, inc, xn, xe, iterations, lohi=None):
  """hge_algdist_run on numpy (host) or torch CUDA (device) fp32 [rows, R] arrays, in place."""
  device = is_device(xn)
  assert device == is_device(xe)
  R = int(xn.shape[1])
  assert tuple(xn.shape) == (inc.num_nodes, R) and tuple(xe.shape) == (inc.num_edges, R)
  if not device:
    assert xn.dtype == np.float32 and xe.dtype == np.float32
  if lohi is not None:
    assert lohi.dtype == np.float32 and lohi.shape == (iterations, 2, R)
  check(ctx.lib.hge_algdist_run(ctx.handle, inc.handle, ptr(xn), ptr(xe), R, int(iterations),
                                MEM_DEVICE if device else MEM_HOST, ptr(lohi)), "hge_algdist_run")
  return xn, xe


def algdist_run_csr(ctx, num_nodes, num_edges, n2e_ptr, n2e_idx, xn, xe, iterations, e2n_ptr=None,
                    e2n_idx=None, lohi=None):
  """hge_algdist_run_csr: incidence set-up + relaxation in one call on host (numpy) or device
  (torch CUDA) arrays, in place; int64 row pointers, int32 sorted column ids."""
  device = is_device(xn)
  assert device == is_device(xe) == is_device(n2e_idx)
  assert (e2n_ptr is None) == (e2n_idx is None)
  R = int(xn.shape[1])
  assert tuple(xn.shape) == (num_nodes, R) and tuple(xe.shape) == (num_edges, R)
  if not device:
    assert xn.dtype == np.float32 and xe.dtype == np.float32
    n2e_ptr, n2e_idx = _as_i64(n2e_ptr), _as_i32(n2e_idx)
    if e2n_ptr is not None:
      e2n_ptr, e2n_idx = _as_i64(e2n_ptr), _as_i32(e2n_idx)
  if lohi is not None:
    assert lohi.dtype == np.float32 and lohi.shape == (iterations, 2, R)
  check(ctx.lib.hge_algdist_run_csr(ctx.handle, int(num_nodes), int(num_edges), ptr(n2e_ptr), ptr(n2e_idx),
                                    ptr(e2n_ptr), ptr(e2n_idx), ptr(xn), ptr(xe), R, int(iterations),
                                    MEM_DEVICE if device else MEM_HOST, ptr(lohi)), "hge_algdist_run_csr")
  return xn, xe


class AlgDistState(object):
  """Stepwise relaxation (hge_algdist_*), device pointers only."""

  def __init__(self, ctx, inc, R, max_iterations):
    self.ctx, self.inc, self.R = ctx, inc, int(R)
    handle = c_vp()
    check(ctx.lib.hge_algdist_create(ctx.handle, inc.handle, self.R, int(max_iterations),
                                     ctypes.byref(handle)), "hge_algdist_create")
    self.handle = handle
    self.ld = int(ctx.lib.hge_algdist_ld(handle))

  def load(self, xn, xe):
    mem = MEM_DEVICE if is_device(xn) else MEM_HOST
    check(self.ctx.lib.hge_algdist_load(self.handle, ptr(xn), ptr(xe), mem), "hge_algdist_load")

  def node_half(self, sweep):
    check(self.ctx.lib.hge_algdist_node_half(self.handle, sweep), "hge_algdist_node_half")

  def edge_half(self, sweep):
    check(self.ctx.lib.hge_algdist_edge_half(self.handle, sweep), "hge_algdist_edge_half")

  def edge_partial(self, sweep, slice_index, partial):
    check(self.ctx.lib.hge_algdist_edge_partial(self.handle, sweep, slice_index, ptr(partial)),
          "hge_algdist_edge_partial")

  def edge_finalize(self, sweep, slice_index, partial):
    check(self.ctx.lib.hge_algdist_edge_finalize(self.handle, sweep, slice_index, ptr(partial)),
          "hge_algdist_edge_finalize")

  def attach_p2p(self, arena):
    check(self.ctx.lib.hge_algdist_attach_p2p(self.handle, arena.handle), "hge_algdist_attach_p2p")

  def sweep_p2p(self, sweep):
    check(self.ctx.lib.hge_algdist_sweep_p2p(self.handle, sweep), "hge_algdist_sweep_p2p")

  def minmax_ptr(self, sweep):
    out = c_vp()
    check(self.ctx.lib.hge_algdist_minmax_ptr(self.handle, sweep, ctypes.byref(out)))
    return out.value

  def store(self, sweeps_done, xn, xe):
    mem = MEM_DEVICE if is_device(xn) else MEM_HOST
    check(self.ctx.lib.hge_algdist_store(self.handle, sweeps_done, ptr(xn), ptr(xe), mem),
          "hge_algdist_store")

  def close(self):
    if getattr(self, "handle", None):
      self.ctx.lib.hge_algdist_destroy(self.handle)
      self.handle = None

  def __del__(self):
    try:
      self.close()
    except Exception:
      pass


# ---------------------------------------------------------------------------------------------
# distances / weights / probabilities
# ---------------------------------------------------------------------------------------------


def _mem(*arrays):
  dev = [is_device(a) for a in arrays if a is not None]
  assert all(dev) or not any(dev), "mixing host and device arrays in one call"
  return MEM_DEVICE if dev and dev[0] else MEM_HOST


def _f32(a):
  if is_device(a):
    return a
  return np.ascontiguousarray(a, dtype=np.float32)


def _new_like(ref, n, dtype=np.float32):
  if is_device(ref):
    import torch
    return torch.empty(int(n), dtype=torch.float32 if dtype == np.float32 else torch.int32,
                       device=ref.device)
  return np.empty(int(n), dtype=dtype)


def incidence_l2(ctx, inc, xn, xe, order=0, as_weight=False, nnz=None):
  """Per-incidence L2 distance (or HOBE weight) in node->edge (order 0) / edge->node (1) order."""
  xn, xe = _f32(xn), _f32(xe)
  R = int(xn.shape[1])
  out = _new_like(xn, inc.nnz_of(order) if nnz is None else nnz)
  check(ctx.lib.hge_incidence_l2(ctx.handle, inc.handle, ptr(xn), ptr(xe), R, int(order),
                                 1 if as_weight else 0, ptr(out), _mem(xn, xe)), "hge_incidence_l2")
  return out


def pair_l2(ctx, xa, xb, ia, ib):
  xa, xb = _f32(xa), _f32(xb)
  if not is_device(ia):
    ia, ib = _as_i32(ia), _as_i32(ib)
  n = int(ia.shape[0])
  out = _new_like(xa, n)
  check(ctx.lib.hge_pair_l2(ctx.handle, ptr(xa), int(xa.shape[0]), ptr(xb), int(xb.shape[0]),
                            int(xa.shape[1]), ptr(ia), ptr(ib), n, ptr(out), _mem(xa, xb, ia, ib)),
        "hge_pair_l2")
  return out


def scale_transform(ctx, values, alpha, want_minmax=False):
  """In place alpha + (1 - alpha) * (1 - zero_one(values)); asserts 0 <= alpha <= 1."""
  mm = np.zeros(2, dtype=np.float32) if want_minmax else None
  check(ctx.lib.hge_scale_transform(ctx.handle, ptr(values), int(values.shape[0]), float(alpha),
                                    ptr(mm), _mem(values)), "hge_scale_transform")
  return (values, mm) if want_minmax else values


def scale_minmax(ctx, values):
  mm = np.zeros(2, dtype=np.float32)
  check(ctx.lib.hge_scale_minmax(ctx.handle, ptr(values), int(values.shape[0]), ptr(mm), _mem(values)),
        "hge_scale_minmax")
  return float(mm[0]), float(mm[1])


def scale_apply(ctx, values, alpha, lo, hi):
  check(ctx.lib.hge_scale_apply(ctx.handle, ptr(values), int(values.shape[0]), float(alpha), float(lo),
                                float(hi), _mem(values)), "hge_scale_apply")
  return values


def row_span(ctx, inc, xn, xe, side):
  xn, xe = _f32(xn), _f32(xe)
  out = _new_like(xn, inc.num_nodes if side == 0 else inc.num_edges)
  check(ctx.lib.hge_row_span(ctx.handle, inc.handle, ptr(xn), ptr(xe), int(xn.shape[1]), int(side),
                             ptr(out), _mem(xn, xe)), "hge_row_span")
  return out


def same_type_prob(ctx, inc, side, w, pi, pj):
  if not is_device(pi):
    pi, pj = _as_i32(pi), _as_i32(pj)
  out = _new_like(w, int(pi.shape[0]))
  check(ctx.lib.hge_same_type_prob(ctx.handle, inc.handle, int(side), ptr(w), ptr(pi), ptr(pj),
                                   int(pi.shape[0]), ptr(out), _mem(w, pi, pj)), "hge_same_type_prob")
  return out


def diff_type_prob(ctx, inc, w_e2n, pn, pe):
  if not is_device(pn):
    pn, pe = _as_i32(pn), _as_i32(pe)
  out = _new_like(w_e2n, int(pn.shape[0]))
  check(ctx.lib.hge_diff_type_prob(ctx.handle, inc.handle, ptr(w_e2n), ptr(pn), ptr(pe),
                                   int(pn.shape[0]), ptr(out), _mem(w_e2n, pn, pe)),
        "hge_diff_type_prob")
  return out


class FeatureCsr(object):
  """(int64 ptr, int32 sorted idx, fp32 val, shape) of a scipy sparse feature matrix, host."""

  def __init__(self, matrix):
    import scipy.sparse as sps
    m = sps.csr_matrix(matrix, dtype=np.float32)
    if not m.has_canonical_format:
      m = m.copy()
      m.sum_duplicates()
    self.shape = m.shape
    self.ptr = np.ascontiguousarray(m.indptr, dtype=np.int64)
    self.idx = np.ascontiguousarray(m.indices, dtype=np.int32)
    self.val = np.ascontiguousarray(m.data, dtype=np.float32)

  def to_device(self, device):
    """The same matrix with its three arrays uploaded as CUDA tensors to `device`."""
    import torch
    d = FeatureCsr.__new__(FeatureCsr)
    d.shape = self.shape
    d.ptr, d.idx, d.val = (torch.from_numpy(a).to(device) for a in (self.ptr, self.idx, self.val))
    return d


def jaccard_rows(ctx, feat, pi, pj):
  """J(F[pi], F[pj]): a numpy fp32 array for host index arrays, a CUDA tensor for int32 CUDA
  tensors (then `feat` must be FeatureCsr.to_device)."""
  if not is_device(pi):
    pi, pj = _as_i32(pi), _as_i32(pj)
  n = int(pi.shape[0])
  out = _new_like(pi, n)
  check(ctx.lib.hge_jaccard_rows(ctx.handle, ptr(feat.ptr), ptr(feat.idx), ptr(feat.val),
                                 feat.shape[0], int(feat.idx.shape[0]), ptr(pi), ptr(pj), n, ptr(out),
                                 _mem(feat.ptr, pi, pj)), "hge_jaccard_rows")
  return out


def jaccard_centroid(ctx, x, groups, feat, px, pg):
  """J(X[px], mean of the rows F[t], t in G[pg]) for host arrays; `groups` is a CsrArrays."""
  px, pg = _as_i32(px), _as_i32(pg)
  assert x.shape[1] == feat.shape[1]
  assert groups.shape[1] == feat.shape[0]
  out = np.empty(len(px), dtype=np.float32)
  if x is feat:
    xa = (feat.ptr, feat.idx, feat.val)
  else:
    xa = (x.ptr, x.idx, x.val)
  check(ctx.lib.hge_jaccard_centroid(
      ctx.handle, ptr(xa[0]), ptr(xa[1]), ptr(xa[2]), x.shape[0], len(xa[1]), ptr(groups.ptr),
      ptr(groups.idx), groups.shape[0], len(groups.idx), ptr(feat.ptr), ptr(feat.idx), ptr(feat.val),
      feat.shape[0], len(feat.idx), ptr(px), ptr(pg), len(px), ptr(out), MEM_HOST),
        "hge_jaccard_centroid")
  return out


def jaccard_centroid_grouped(ctx, inc, group_side, x, feat, px, pg, workspace_mb=0):
  """hge_jaccard_centroid_grouped: J(X[px], mean of F over the members of group pg) with the groups
  taken from the incidence (group_side 1: edges and their nodes, 0: nodes and their edges).  x and
  feat are FeatureCsr.to_device, px / pg int32 CUDA tensors; returns an fp32 CUDA tensor."""
  import torch
  n = int(px.shape[0])
  assert int(pg.shape[0]) == n
  assert x.shape[1] == feat.shape[1]
  out = torch.empty(max(n, 1), dtype=torch.float32, device=px.device)[:n]
  check(ctx.lib.hge_jaccard_centroid_grouped(
      ctx.handle, inc.handle, int(group_side), ptr(x.ptr), ptr(x.idx), ptr(x.val), x.shape[0],
      int(x.idx.shape[0]), ptr(feat.ptr), ptr(feat.idx), ptr(feat.val), feat.shape[0],
      int(feat.idx.shape[0]), ptr(px.contiguous()), ptr(pg.contiguous()), n, int(workspace_mb), ptr(out)),
        "hge_jaccard_centroid_grouped")
  return out


# ---------------------------------------------------------------------------------------------
# host-side sampling (numpy legacy RNG replay)
# ---------------------------------------------------------------------------------------------


class LegacyRngState(object):
  """The process-global numpy RandomState as the 625-word buffer the library advances."""

  def __init__(self):
    st = np.random.get_state()
    assert st[0] == "MT19937"
    self._rest = (st[3], st[4])
    self.buf = np.empty(625, dtype=np.uint32)
    self.buf[:624] = st[1]
    self.buf[624] = st[2]

  def copy(self):
    other = LegacyRngState.__new__(LegacyRngState)
    other._rest = self._rest
    other.buf = self.buf.copy()
    return other

  def commit(self):
    """Writes the advanced state back so later np.random calls continue the same stream."""
    np.random.set_state(("MT19937", self.buf[:624].copy(), int(self.buf[624])) + self._rest)


class CsrArrays(object):
  """(int64 ptr, int32 idx, shape) of a canonical boolean CSR on the host."""

  def __init__(self, matrix):
    import scipy.sparse as sps
    m = sps.csr_matrix(matrix)
    self.shape = m.shape
    self.ptr = np.ascontiguousarray(m.indptr, dtype=np.int64)
    self.idx = np.ascontiguousarray(m.indices, dtype=np.int32)


def _factors(mats):
  args = []
  for m in list(mats) + [None] * (3 - len(mats)):
    args += [ptr(m.ptr) if m is not None else None, ptr(m.idx) if m is not None else None]
  kind = len(mats) - 1
  mid_cols = mats[1].shape[1] if kind >= 1 else 0
  out_cols = mats[-1].shape[1]
  return kind, args, int(mid_cols), int(out_cols)


def spgemm_rows(mats, rows, sorted_rows=False):
  """Rows of mats[0] (* mats[1] (* mats[2])) in scipy's stored order (or sorted)."""
  lib = load_library()
  kind, args, mid_cols, out_cols = _factors(mats)
  rows = _as_i32(rows)
  out_ptr = np.zeros(len(rows) + 1, dtype=np.int64)
  check(lib.hge_spgemm_rows(kind, *args, mid_cols, out_cols, ptr(rows), len(rows),
                            1 if sorted_rows else 0, ptr(out_ptr), None, 0), "hge_spgemm_rows")
  out_idx = np.empty(int(out_ptr[-1]), dtype=np.int32)
  check(lib.hge_spgemm_rows(kind, *args, mid_cols, out_cols, ptr(rows), len(rows),
                            1 if sorted_rows else 0, ptr(out_ptr), ptr(out_idx), len(out_idx)),
        "hge_spgemm_rows")
  return out_ptr, out_idx


def sample_adj_rows(mats, rows, samples_per_row, state, replace=False, negative=False):
  """_sample_adj_matrix over mats[0] (* mats[1] (* mats[2])): returns (row, col) int32 arrays."""
  lib = load_library()
  kind, args, mid_cols, out_cols = _factors(mats)
  rows = _as_i32(rows)
  samples = _as_i32(samples_per_row)
  assert len(samples) == len(rows)
  assert len(samples) > 0
  cap = int(samples.astype(np.int64).sum())
  out_row = np.empty(cap, dtype=np.int32)
  out_col = np.empty(cap, dtype=np.int32)
  count = ctypes.c_int64(0)
  check(lib.hge_sample_adj_rows(kind, *args, mid_cols, out_cols, ptr(rows), len(rows), ptr(samples),
                                1 if replace else 0, 1 if negative else 0, ptr(state.buf),
                                ptr(out_row), ptr(out_col), cap, ctypes.byref(count)),
        "hge_sample_adj_rows")
  return out_row[:count.value], out_col[:count.value]


def sample_neighbors(n2e, e2n, nodes, edges, k, state):
  lib = load_library()
  nodes, edges = _as_i32(nodes), _as_i32(edges)
  m = len(nodes)
  nbr_e = np.empty((m, k), dtype=np.int32)
  nbr_n = np.empty((m, k), dtype=np.int32)
  rc = lib.hge_sample_neighbors(ptr(n2e.ptr), ptr(n2e.idx), ptr(e2n.ptr), ptr(e2n.idx), ptr(nodes),
                                ptr(edges), m, int(k), ptr(state.buf), ptr(nbr_e), ptr(nbr_n))
  if rc == HGE_ERR_INVALID and "cannot be empty" in last_error():
    raise ValueError("'a' cannot be empty unless no samples are taken")
  check(rc, "hge_sample_neighbors")
  return nbr_e, nbr_n


# ---------------------------------------------------------------------------------------------
# device sampling (Philox streams, csrc/hge_device_sampler.cu)
# ---------------------------------------------------------------------------------------------

# phase constants of csrc/hge_philox.cuh (HgePhase)
PHASE_NN, PHASE_EE, PHASE_NE, PHASE_EN, PHASE_NEIGHBORS = 1, 2, 3, 4, 5
PHASE_NEG_NN, PHASE_NEG_EE, PHASE_NEG_EE_AGAIN, PHASE_NEG_NE, PHASE_NEG_EN = 6, 7, 8, 9, 10
PHASE_NEG_NEIGHBORS = 11
PHASE_SHUFFLE, PHASE_INIT_NODES, PHASE_INIT_EDGES = 12, 13, 14
PHASE_LP_EDGE_OWNERS, PHASE_LP_NODE_OWNERS = 15, 16


def sample_pairs_device(ctx, inc, side, factors, row0, samples, seed, phase, negative=False,
                        workspace_mb=0):
  """hge_sample_pairs_device over rows [row0, row0 + len(samples)): (row, col) int32 CUDA tensors."""
  import torch
  dev = torch.device("cuda", ctx.device)
  k = torch.as_tensor(_as_i32(samples)).to(dev)
  cap = int(np.asarray(samples, dtype=np.int64).clip(min=0).sum())
  out_row = torch.empty(max(cap, 1), dtype=torch.int32, device=dev)
  out_col = torch.empty(max(cap, 1), dtype=torch.int32, device=dev)
  count = ctypes.c_int64(0)
  check(ctx.lib.hge_sample_pairs_device(ctx.handle, inc.handle, int(side), int(factors), int(row0),
                                        int(row0) + len(k), ptr(k), 1 if negative else 0,
                                        int(seed) & 0xFFFFFFFFFFFFFFFF, int(phase), int(workspace_mb),
                                        ptr(out_row), ptr(out_col), cap, ctypes.byref(count), MEM_DEVICE),
        "hge_sample_pairs_device")
  return out_row[:count.value], out_col[:count.value]


def sample_neighbors_device(ctx, inc, nodes, edges, k, seed, phase, first_index):
  """hge_sample_neighbors_device on int32 CUDA tensors: ([m, k] edges of the nodes, [m, k] nodes
  of the edges) as CUDA tensors."""
  import torch
  m = int(nodes.shape[0])
  nbr_e = torch.empty((m, int(k)), dtype=torch.int32, device=nodes.device)
  nbr_n = torch.empty((m, int(k)), dtype=torch.int32, device=nodes.device)
  rc = ctx.lib.hge_sample_neighbors_device(ctx.handle, inc.handle, ptr(nodes.contiguous()),
                                           ptr(edges.contiguous()), m, int(k),
                                           int(seed) & 0xFFFFFFFFFFFFFFFF, int(phase), int(first_index),
                                           ptr(nbr_e), ptr(nbr_n), MEM_DEVICE)
  if rc == HGE_ERR_INVALID and "cannot be empty" in last_error():
    raise ValueError("'a' cannot be empty unless no samples are taken")
  check(rc, "hge_sample_neighbors_device")
  return nbr_e, nbr_n


def shuffle_order(ctx, seed, epoch, n, out=None):
  """hge_shuffle_order: the seeded permutation of [0, n) of one epoch as an int32 CUDA tensor
  (written into `out` when given)."""
  import torch
  if out is None:
    out = torch.empty(max(int(n), 1), dtype=torch.int32, device=torch.device("cuda", ctx.device))[:int(n)]
  assert out.dtype == torch.int32 and out.is_cuda and int(out.shape[0]) == int(n)
  check(ctx.lib.hge_shuffle_order(ctx.handle, int(seed) & 0xFFFFFFFFFFFFFFFF, int(epoch), int(n), ptr(out),
                                  MEM_DEVICE), "hge_shuffle_order")
  return out


class LpSvmModel(object):
  """The classifiers of one hge_lp_svm_predict call, on the host: named owners in ascending id with
  their rho, SMO iterations and first training point (offset, U + 1 entries), and per training point
  its item id and alpha_i y_i.  capped = owners that hit the iteration cap."""

  def __init__(self, owner_ids, rho, iterations, offset, point_ids, coef, capped):
    self.owner_ids, self.rho, self.iterations, self.offset = owner_ids, rho, iterations, offset
    self.point_ids, self.coef, self.capped = point_ids, coef, capped


def lp_svm_predict(ctx, inc, owner_side, vectors, items, owners, seed, C=1.0, gamma=0.1, tol=1e-3,
                   workspace_mb=0, return_model=False, timings=None):
  """hge_lp_svm_predict on CUDA tensors: vectors fp32 [num items, d], items / owners int32 [L].
  Returns (keep bool [L], decision fp64 [L], owners at the iteration cap) as CUDA tensors and an
  int, plus an LpSvmModel when `return_model`.  `timings` (a dict) receives the seconds of the
  grouping, negatives, solve and predict phases, each ended by a synchronise."""
  import torch
  dev = vectors.device
  L = int(items.shape[0])
  assert int(owners.shape[0]) == L and vectors.dim() == 2 and vectors.dtype == torch.float32
  assert items.dtype == torch.int32 and owners.dtype == torch.int32
  keep = torch.empty(max(L, 1), dtype=torch.uint8, device=dev)[:L]
  decision = torch.empty(max(L, 1), dtype=torch.float64, device=dev)[:L]
  counts = np.zeros(3, dtype=np.int64)
  phase = np.zeros(4, dtype=np.float64) if timings is not None else None
  model = [None] * 6
  cap = 0
  if return_model:
    cap = 3 * max(inc.nnz_of(0), inc.nnz_of(1))   # an owner trains on at most 3 x its members
    model = [torch.empty(max(L, 1), dtype=torch.int32, device=dev), torch.empty(max(L, 1), dtype=torch.float64, device=dev),
             torch.empty(max(L, 1), dtype=torch.int64, device=dev), torch.empty(L + 1, dtype=torch.int64, device=dev),
             torch.empty(max(cap, 1), dtype=torch.int32, device=dev), torch.empty(max(cap, 1), dtype=torch.float64, device=dev)]
  vectors = vectors.contiguous()
  check(ctx.lib.hge_lp_svm_predict(ctx.handle, inc.handle, int(owner_side), ptr(vectors), int(vectors.shape[1]),
                                   ptr(items.contiguous()), ptr(owners.contiguous()), L,
                                   int(seed) & 0xFFFFFFFFFFFFFFFF, float(C), float(gamma), float(tol),
                                   int(workspace_mb), ptr(keep), ptr(decision), ptr(counts),
                                   *[ptr(m) for m in model], cap, ptr(phase)), "hge_lp_svm_predict")
  if timings is not None:
    timings.update(zip(("grouping", "negatives", "solve", "predict"), (phase / 1e3).tolist()))
  U, T, capped = (int(v) for v in counts)
  out = (keep.bool(), decision, capped)
  if return_model:
    host = [m.cpu().numpy() for m in model]
    out += (LpSvmModel(host[0][:U], host[1][:U], host[2][:U], host[3][:U + 1], host[4][:T], host[5][:T],
                       capped),)
  return out


def lp_node_edge_train(ctx, inc, xn, xe, seed, hidden=64, epochs=10, batch_size=256, lr=0.01, eps=1e-7,
                       timings=None):
  """hge_lp_node_edge_train on fp32 CUDA tensors xn [N, d], xe [E, d]: ((W1 [2d, hidden], b1 [hidden],
  w2 [hidden], b2 [1]) as CUDA tensors, per-epoch losses as a numpy array).  `timings` (a dict)
  receives the seconds of the set-up and of each epoch, each ended by a synchronise."""
  import torch
  assert xn.dim() == 2 and xe.dim() == 2 and xn.dtype == torch.float32 and xe.dtype == torch.float32
  assert xn.shape[1] == xe.shape[1], "node and edge vectors must have the same length"
  d, dev = int(xn.shape[1]), xn.device
  W1 = torch.empty((max(2 * d, 1), max(int(hidden), 1)), dtype=torch.float32, device=dev)
  b1 = torch.empty(max(int(hidden), 1), dtype=torch.float32, device=dev)
  w2 = torch.empty(max(int(hidden), 1), dtype=torch.float32, device=dev)
  b2 = torch.empty(1, dtype=torch.float32, device=dev)
  losses = np.zeros(max(int(epochs), 1), dtype=np.float64)
  phase = np.zeros(1 + max(int(epochs), 0), dtype=np.float64) if timings is not None else None
  xn, xe = xn.contiguous(), xe.contiguous()
  check(ctx.lib.hge_lp_node_edge_train(ctx.handle, inc.handle, ptr(xn), ptr(xe), d, int(hidden),
                                       int(seed) & 0xFFFFFFFFFFFFFFFF, int(epochs), int(batch_size), float(lr),
                                       float(eps), ptr(W1), ptr(b1), ptr(w2), ptr(b2), ptr(losses), ptr(phase)),
        "hge_lp_node_edge_train")
  if timings is not None:
    timings["setup"] = float(phase[0]) / 1e3
    timings["epochs"] = (phase[1:] / 1e3).tolist()
  return (W1, b1, w2, b2), losses[:max(int(epochs), 0)]


def lp_node_edge_samples(ctx, inc, seed, epochs):
  """hge_lp_node_edge_samples: (sample nodes [2 nnz], sample edges [2 nnz], orders [epochs, 2 nnz]) as
  int32 CUDA tensors."""
  import torch
  dev = torch.device("cuda", ctx.device)
  M = 2 * inc.nnz
  sn = torch.empty(max(M, 1), dtype=torch.int32, device=dev)
  se = torch.empty(max(M, 1), dtype=torch.int32, device=dev)
  orders = torch.empty((max(int(epochs), 1), max(M, 1)), dtype=torch.int32, device=dev)
  check(ctx.lib.hge_lp_node_edge_samples(ctx.handle, inc.handle, int(seed) & 0xFFFFFFFFFFFFFFFF, int(epochs),
                                         ptr(sn), ptr(se), ptr(orders)), "hge_lp_node_edge_samples")
  return sn[:M], se[:M], orders[:int(epochs), :M]


def lp_node_edge_predict(ctx, xn, xe, weights, nodes, edges):
  """hge_lp_node_edge_predict on CUDA tensors: xn [N, d], xe [E, d] fp32, weights (W1, b1, w2, b2),
  nodes / edges int32 [L].  Returns (probability fp32 [L], keep bool [L]) as CUDA tensors."""
  import torch
  W1, b1, w2, b2 = (w.contiguous() for w in weights)
  assert xn.dim() == 2 and xe.dim() == 2 and xn.shape[1] == xe.shape[1]
  assert xn.dtype == torch.float32 and xe.dtype == torch.float32
  assert nodes.dtype == torch.int32 and edges.dtype == torch.int32 and nodes.shape == edges.shape
  d, L, dev = int(xn.shape[1]), int(nodes.shape[0]), xn.device
  prob = torch.empty(max(L, 1), dtype=torch.float32, device=dev)[:L]
  keep = torch.empty(max(L, 1), dtype=torch.uint8, device=dev)[:L]
  xn, xe = xn.contiguous(), xe.contiguous()
  check(ctx.lib.hge_lp_node_edge_predict(ctx.handle, ptr(xn), int(xn.shape[0]), ptr(xe), int(xe.shape[0]), d,
                                         int(W1.shape[1]), ptr(W1), ptr(b1), ptr(w2), ptr(b2),
                                         ptr(nodes.contiguous()), ptr(edges.contiguous()), L, ptr(prob), ptr(keep)),
        "hge_lp_node_edge_predict")
  return prob, keep.bool()


def _factor_pair(W, Ht, k):
  mem = _mem(W, Ht)
  if mem == MEM_HOST:
    assert isinstance(W, np.ndarray) and isinstance(Ht, np.ndarray)
    assert W.dtype == np.float32 and Ht.dtype == np.float32
  else:
    import torch
    assert W.dtype == torch.float32 and Ht.dtype == torch.float32
  assert W.ndim == 2 and Ht.ndim == 2 and W.shape[1] == k and Ht.shape[1] == k, "factors must be [N, k], [E, k]"
  return mem


def nmf_init(ctx, num_nodes, num_edges, k, seed, scale, W, Ht):
  """hge_nmf_init into fp32 W [num_nodes, k] and Ht [num_edges, k] (numpy, or CUDA tensors)."""
  mem = _factor_pair(W, Ht, k)
  assert tuple(W.shape) == (num_nodes, k) and tuple(Ht.shape) == (num_edges, k)
  check(ctx.lib.hge_nmf_init(ctx.handle, int(num_nodes), int(num_edges), int(k), int(seed) & 0xFFFFFFFFFFFFFFFF,
                             float(scale), ptr(W), ptr(Ht), mem), "hge_nmf_init")
  return W, Ht


def nmf_fit(ctx, inc, W, Ht, max_iter, tol, phase_ms=None):
  """hge_nmf_fit in place on fp32 W [N, k] and Ht [E, k] (numpy, or CUDA tensors): (n_iter,
  violations [n_iter] float64).  phase_ms: optional float64 [3] numpy array."""
  k = int(W.shape[1]) if W.ndim == 2 else 0
  mem = _factor_pair(W, Ht, k)
  n_iter = ctypes.c_int(0)
  viol = np.zeros(max(1, int(max_iter)), dtype=np.float64)
  if phase_ms is not None:
    assert phase_ms.dtype == np.float64 and phase_ms.shape == (3,)
  check(ctx.lib.hge_nmf_fit(ctx.handle, inc.handle, int(W.shape[0]), int(Ht.shape[0]), k, ptr(W), ptr(Ht),
                            int(max_iter), float(tol), mem, ctypes.byref(n_iter), ptr(viol), ptr(phase_ms)),
        "hge_nmf_fit")
  return n_iter.value, viol[:n_iter.value].copy()


def svd_ld(l):
  """Row stride of the truncated SVD's dense arrays: l rounded up to a multiple of 4."""
  return (int(l) + 3) & ~3


def _svd_dense(*arrays):
  mem = _mem(*arrays)
  for a in arrays:
    if mem == MEM_HOST:
      assert isinstance(a, np.ndarray) and a.dtype == np.float32, "host arrays must be float32 numpy arrays"
    else:
      import torch
      assert a.dtype == torch.float32, "device arrays must be float32 tensors"
    assert a.ndim == 2, "dense arrays must be [rows, ld]"
  return mem


def svd_start(ctx, num_edges, l, seed, omega):
  """hge_svd_start into fp32 omega [num_edges, svd_ld(l)] (numpy, or a CUDA tensor)."""
  mem = _svd_dense(omega)
  assert tuple(omega.shape) == (int(num_edges), svd_ld(l)), "omega must be [E, ld]"
  check(ctx.lib.hge_svd_start(ctx.handle, int(num_edges), int(l), int(seed) & 0xFFFFFFFFFFFFFFFF, ptr(omega), mem),
        "hge_svd_start")
  return omega


def svd_half(ctx, inc, side, l, x, y, phase_ms=None):
  """hge_svd_half: y = A x (side 0) or A^T x (side 1) in place, returns the f64 Gram matrix
  y^T y [l, l] (numpy).  x, y: fp32 [rows, svd_ld(l)], both numpy or both CUDA tensors.  phase_ms:
  optional float64 [2] numpy array (product, Gram milliseconds)."""
  mem = _svd_dense(x, y)
  nodes, edges = (y.shape[0], x.shape[0]) if side == 0 else (x.shape[0], y.shape[0])
  gram = np.empty((int(l), int(l)), dtype=np.float64)
  if phase_ms is not None:
    assert phase_ms.dtype == np.float64 and phase_ms.shape == (2,)
  check(ctx.lib.hge_svd_half(ctx.handle, inc.handle, int(side), int(nodes), int(edges), int(l), ptr(x), ptr(y),
                             ptr(gram), mem, ptr(phase_ms)), "hge_svd_half")
  return gram


def svd_rowmat(ctx, l, y, m, out):
  """hge_svd_rowmat: out = y m in place; y, out fp32 [rows, svd_ld(l)] (numpy or CUDA tensors),
  m fp32 [l, cols] numpy."""
  mem = _svd_dense(y, out)
  m = np.ascontiguousarray(m, dtype=np.float32)
  assert m.ndim == 2 and m.shape[0] == int(l), "m must be [l, cols]"
  assert y.shape[0] == out.shape[0], "y and out must have the same rows"
  check(ctx.lib.hge_svd_rowmat(ctx.handle, int(y.shape[0]), int(l), int(m.shape[1]), ptr(y), ptr(m), ptr(out), mem),
        "hge_svd_rowmat")
  return out


def svd_flip(ctx, l, k, u, v):
  """hge_svd_flip in place on fp32 u [N, svd_ld(l)] and v [E, svd_ld(l)]."""
  mem = _svd_dense(u, v)
  check(ctx.lib.hge_svd_flip(ctx.handle, int(u.shape[0]), int(v.shape[0]), int(l), int(k), ptr(u), ptr(v), mem),
        "hge_svd_flip")
  return u, v


def svd_residuals(ctx, inc, l, k, u, v, sigma):
  """hge_svd_residuals: ||A v_i - sigma_i u_i|| / sigma_0 for i < k as a float64 numpy array."""
  mem = _svd_dense(u, v)
  sigma = np.ascontiguousarray(sigma, dtype=np.float64)
  assert sigma.shape == (int(k),)
  resid = np.zeros(int(k), dtype=np.float64)
  check(ctx.lib.hge_svd_residuals(ctx.handle, inc.handle, int(u.shape[0]), int(v.shape[0]), int(l), int(k), ptr(u),
                                  ptr(v), ptr(sigma), ptr(resid), mem), "hge_svd_residuals")
  return resid


class PeerArena(object):
  """hge_p2p: the IPC-shared exchange arena of one shard."""

  def __init__(self, ctx, rank, world, num_local_nodes, num_edges, ld):
    self.ctx = ctx
    handle = c_vp()
    check(ctx.lib.hge_p2p_create(ctx.handle, rank, world, num_local_nodes, num_edges, ld,
                                 ctypes.byref(handle)), "hge_p2p_create")
    self.handle = handle
    self.world = world

  def export(self):
    buf = np.zeros(64, dtype=np.uint8)
    check(self.ctx.lib.hge_p2p_export(self.handle, ptr(buf)), "hge_p2p_export")
    return buf

  def open_peers(self, handles):
    handles = np.ascontiguousarray(handles, dtype=np.uint8).reshape(self.world, 64)
    check(self.ctx.lib.hge_p2p_open_peers(self.handle, ptr(handles)), "hge_p2p_open_peers")

  def check(self):
    check(self.ctx.lib.hge_p2p_check(self.handle), "hge_p2p_check")

  def set_timing(self, on):
    check(self.ctx.lib.hge_p2p_set_timing(self.handle, int(bool(on))), "hge_p2p_set_timing")

  def phase_ms(self):
    """(mean ms per sweep of [node half, gather + push, barrier A, reduce + all-gather, barrier B],
    sweeps averaged over) since the last call; records only while set_timing(True) is on."""
    out = np.zeros(5, dtype=np.float64)
    n = ctypes.c_int(0)
    check(self.ctx.lib.hge_p2p_phase_ms(self.handle, ptr(out), ctypes.byref(n)), "hge_p2p_phase_ms")
    return out.tolist(), int(n.value)

  def close_peers(self):
    if getattr(self, "handle", None):
      self.ctx.lib.hge_p2p_close_peers(self.handle)

  def close(self):
    if getattr(self, "handle", None):
      self.ctx.lib.hge_p2p_destroy(self.handle)
      self.handle = None


# ---- node2vec (csrc/hge_n2v.cu); every array is a CUDA tensor -------------------------------------

def _cuda(*arrays):
  assert all(is_device(a) and a.is_contiguous() for a in arrays), "node2vec arrays must be contiguous CUDA tensors"


def n2v_walks(ctx, inc, num_walks, walk_length, p, q, seed, walks, counts):
  """hge_n2v_walks into int32 walks [num_walks V, walk_length] and int64 counts [V]."""
  _cuda(walks, counts)
  check(ctx.lib.hge_n2v_walks(ctx.handle, inc.handle, int(num_walks), int(walk_length), float(p), float(q),
                              int(seed) & 0xFFFFFFFFFFFFFFFF, ptr(walks), ptr(counts)), "hge_n2v_walks")


def n2v_pairs(ctx, walks, window, seed, pairs=None):
  """hge_n2v_pairs: the pair count, and with `pairs` (int32 [P, 2]) the pairs themselves."""
  _cuda(walks)
  n = ctypes.c_int64()
  cap = 0
  if pairs is not None:
    _cuda(pairs)
    cap = int(pairs.shape[0])
  check(ctx.lib.hge_n2v_pairs(ctx.handle, ptr(walks), int(walks.shape[0]), int(walks.shape[1]), int(window),
                              int(seed) & 0xFFFFFFFFFFFFFFFF, ptr(pairs), cap, ctypes.byref(n)), "hge_n2v_pairs")
  return int(n.value)


def n2v_negatives(ctx, num_pairs, cum, negative, seed, epoch, out):
  """hge_n2v_negatives into int32 out [num_pairs, negative]; cum is the int64 noise table [V + 1]."""
  _cuda(cum, out)
  check(ctx.lib.hge_n2v_negatives(ctx.handle, int(num_pairs), ptr(cum), int(cum.shape[0]) - 1, int(negative),
                                  int(seed) & 0xFFFFFFFFFFFFFFFF, int(epoch), ptr(out)), "hge_n2v_negatives")


def n2v_init(ctx, seed, tin, tout):
  """hge_n2v_init on fp32 tables [V, dim]."""
  _cuda(tin, tout)
  check(ctx.lib.hge_n2v_init(ctx.handle, int(tin.shape[0]), int(tin.shape[1]), int(seed) & 0xFFFFFFFFFFFFFFFF,
                             ptr(tin), ptr(tout)), "hge_n2v_init")


def n2v_train_epoch(ctx, tin, tout, pairs, cum, negative, seed, epoch, epochs, batch_pairs, alpha, min_alpha,
                    plan_bytes=0):
  """hge_n2v_train_epoch in place on tin / tout; returns the epoch loss."""
  _cuda(tin, tout, pairs, cum)
  loss = ctypes.c_double()
  check(ctx.lib.hge_n2v_train_epoch(ctx.handle, int(tin.shape[0]), int(tin.shape[1]), ptr(tin), ptr(tout),
                                    ptr(pairs), int(pairs.shape[0]), ptr(cum), int(negative),
                                    int(seed) & 0xFFFFFFFFFFFFFFFF, int(epoch), int(epochs), int(batch_pairs),
                                    float(alpha), float(min_alpha), int(plan_bytes), ctypes.byref(loss)),
        "hge_n2v_train_epoch")
  return float(loss.value)


def n2v_clique_walks(ctx, inc, side, num_walks, walk_length, p, q, seed, walks, counts):
  """hge_n2v_clique_walks on side 0 (nodes) or 1 (edges) into int32 walks [num_walks V,
  walk_length] and int64 counts [V]."""
  _cuda(walks, counts)
  check(ctx.lib.hge_n2v_clique_walks(ctx.handle, inc.handle, int(side), int(num_walks), int(walk_length), float(p),
                                     float(q), int(seed) & 0xFFFFFFFFFFFFFFFF, ptr(walks), ptr(counts)),
        "hge_n2v_clique_walks")
