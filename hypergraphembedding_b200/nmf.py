"""Non-negative factorization of a hypergraph's node-edge incidence on the GPU: the NMF baseline
embedder the reference compares HOBE against (embedding.py:110-261 of the reference, which runs
scikit-learn's ``NMF(dim)``).

``NonNegativeFactorizationDevice`` runs scikit-learn's coordinate-descent solver (``solver="cd"``,
Frobenius loss, no regularization, ``shuffle=False``) in libhge_b200.so (csrc/hge_nmf.cu, DESIGN
section 9.10).  The reference's default start (``init="nndsvda"``) draws numpy's global RNG; the
start here is seeded instead, in the style of ``init="random"`` (see ``seeded_start``), or given by
the caller as scikit-learn's ``init="custom"`` takes it.
"""
import numpy as np
import scipy.sparse as sps

from . import _native
from .algebraic_distance import make_incidence


def start_scale(num_nodes, num_edges, nnz, k):
  """2 avg with avg = sqrt(nnz / (N E k)) computed in float64 and rounded to float32: the seeded
  start is uniform on [0, 2 avg), so its mean is scikit-learn's init="random" scale."""
  avg = np.float32(np.sqrt(float(nnz) / (float(num_nodes) * float(num_edges) * float(k))))
  return np.float32(2) * avg


def seeded_start(num_nodes, num_edges, nnz, k, seed=0):
  """(W [N, k], Ht [E, k]) float32: element (r, c) = scale * ((w >> 8) 2^-24), w = word c of the
  Philox stream of row r in phase 20 (W) or 21 (Ht) of `seed` (hge_nmf_init)."""
  ctx = _native.default_context()
  W = np.empty((int(num_nodes), int(k)), dtype=np.float32)
  Ht = np.empty((int(num_edges), int(k)), dtype=np.float32)
  _native.nmf_init(ctx, num_nodes, num_edges, k, seed, start_scale(num_nodes, num_edges, nnz, k), W, Ht)
  return W, Ht


def NonNegativeFactorizationDevice(incidence, k, W=None, H=None, seed=0, max_iter=200, tol=1e-4):
  """A ~ W H for the N x E incidence pattern `incidence` (scipy sparse; every stored entry counts as
  1), 1 <= k <= 256.  Returns (W [N, k], H [k, E], n_iter) as float32 numpy arrays, in the shapes
  of scikit-learn's ``non_negative_factorization``.  W and H given together are the start
  (scikit-learn's init="custom"); otherwise the seeded start of `seed`.  numpy's global RNG is
  neither read nor advanced."""
  A = sps.csr_matrix(incidence)
  N, E = A.shape
  assert (W is None) == (H is None), "give both W and H, or neither"
  ctx = _native.default_context()
  inc = make_incidence(A, ctx=ctx)
  try:
    if W is None:
      W0, Ht0 = seeded_start(N, E, inc.nnz, k, seed)
    else:
      W0 = np.array(W, dtype=np.float32, order="C")
      Ht0 = np.ascontiguousarray(np.asarray(H, dtype=np.float32).T)
      assert W0.shape == (N, k) and Ht0.shape == (E, k), \
          "start of shapes %s, %s for a %d x %d incidence and k = %d" % (W0.shape, Ht0.T.shape, N, E, k)
    n_iter, _ = _native.nmf_fit(ctx, inc, W0, Ht0, max_iter, tol)
  finally:
    inc.close()
  return W0, np.ascontiguousarray(Ht0.T), n_iter
