"""Numpy restatement of the personalized link-prediction classifiers of csrc/hge_lp_svm.cu: each
owner's training set (members, then negatives drawn by Floyd's algorithm over the positions of its
ascending non-member list from the Philox streams of oracle/device_sampler_ref.py) and libsvm's
dual C-SVC solver as the kernel runs it (WSS3, no shrinking, fp32 kernel entries with the squared
distance summed sequentially over the components, fp64 gradient and alpha, ties to the largest
index, rho as calculate_rho).

Test infrastructure only.
"""
import numpy as np

from oracle.device_sampler_ref import Streams

PHASE_LP_EDGE_OWNERS, PHASE_LP_NODE_OWNERS = 15, 16
TAU = 1e-12


def training_sets(mptr, midx, items, owners, seed, phase):
  """{owner: (members, negatives)} (ascending int64 ids) of the owners `owners` of the member CSR
  (mptr, midx) over `items` items; degenerate owners (no member, or every item a member) get two
  empty arrays.  Floyd's steps run for all owners at once."""
  owners = np.unique(np.asarray(owners, dtype=np.int64))
  mptr = np.asarray(mptr, dtype=np.int64)
  midx = np.asarray(midx, dtype=np.int64)
  m = mptr[owners + 1] - mptr[owners]
  others = items - m
  k = np.where((m == 0) | (others == 0), 0, np.minimum(others, 2 * m))
  pos = {int(o): [] for o in owners}
  draw = np.nonzero((k > 0) & (k < others))[0]
  st = Streams(seed, phase, owners[draw])
  taken = set()
  for s in range(int(k[draw].max(initial=0))):
    act = np.nonzero(s < k[draw])[0]
    j = others[draw[act]] - k[draw[act]] + s
    t = st.below(act, j + 1)
    for a, jj, tt in zip(act.tolist(), j.tolist(), t.tolist()):
      o = int(owners[draw[a]])
      v = jj if (o, tt) in taken else tt
      taken.add((o, v))
      pos[o].append(v)
  out = {}
  for o, mm, kk, nn in zip(owners.tolist(), m.tolist(), k.tolist(), others.tolist()):
    members = midx[mptr[o]:mptr[o + 1]]
    if kk == 0:
      out[o] = (np.zeros(0, np.int64), np.zeros(0, np.int64))
      continue
    p = np.arange(nn, dtype=np.int64) if kk == nn else np.sort(np.asarray(pos[o], dtype=np.int64))
    out[o] = (members.copy(), nonmember_ids(members, p))
  return out


def nonmember_ids(members, positions):
  """Id of each position of the ascending list of the ids that are not in `members` (sorted)."""
  members = np.asarray(members, dtype=np.int64)
  c = np.searchsorted(members - np.arange(len(members)), positions, side="right")
  return positions + c


def kernel(A, B, gamma):
  """fp32 K(a, b) = exp(-gamma ||a - b||^2) of every row pair, the squared distance summed in
  component order, each operation rounded to fp32."""
  A = np.asarray(A, dtype=np.float32)
  B = np.asarray(B, dtype=np.float32)
  s = np.zeros((len(A), len(B)), dtype=np.float32)
  for c in range(A.shape[1]):
    t = A[:, c][:, None] - B[:, c][None, :]
    s = s + t * t
  return np.exp(np.float32(-gamma) * s).astype(np.float32)


def solve(X, y, C=1.0, gamma=0.1, tol=1e-3, max_iter=None):
  """(alpha, rho, iterations) of libsvm's C-SVC dual on points X with labels y in {+1, -1}."""
  y = np.asarray(y, dtype=np.float64)
  n = len(y)
  Q = (kernel(X, X, gamma) * np.where(y[:, None] == y[None, :], 1, -1).astype(np.float32)).astype(np.float32)
  G = np.full(n, -1.0)
  A = np.zeros(n)
  cap = max(10000000, 100 * n) if max_iter is None else max_iter
  idx = np.arange(n)
  it = 0
  while it < cap:
    up = np.where(y > 0, A < C, A > 0)
    if not up.any():
      break
    v = np.where(up, -(y * G), -np.inf)
    Gmax = v.max()
    i = int(idx[v == Gmax][-1])
    Qi = Q[i].astype(np.float64)
    low = np.where(y > 0, A > 0, A < C)
    g2 = np.where(low, y * G, -np.inf).max()
    grad_diff = Gmax + y * G
    cand = low & (grad_diff > 0)
    if not cand.any():
      break
    quad = 2.0 - y * ((2.0 * y[i]) * Qi)
    quad = np.where(quad > 0, quad, TAU)
    obj = np.where(cand, -(grad_diff * grad_diff) / quad, np.inf)
    omin = obj.min()
    j = int(idx[obj == omin][-1])
    if Gmax + g2 < tol:
      break
    Qj = Q[j].astype(np.float64)
    ai, aj = _step(y[i], y[j], G[i], G[j], A[i], A[j], Q[i, j], C)
    dai, daj = ai - A[i], aj - A[j]
    G = G + (Qi * dai + Qj * daj)
    A[i], A[j] = ai, aj
    it += 1
  return A, _rho(y, G, A, C), it


def _step(yi, yj, Gi, Gj, ai, aj, Qij, C):
  two_q = float(np.float32(2) * np.float32(Qij))
  if yi != yj:
    quad = 2.0 + two_q
    quad = quad if quad > 0 else TAU
    delta = (-Gi - Gj) / quad
    diff = ai - aj
    ai, aj = ai + delta, aj + delta
    if diff > 0:
      if aj < 0:
        aj, ai = 0.0, diff
    elif ai < 0:
      ai, aj = 0.0, -diff
    if diff > 0:
      if ai > C:
        ai, aj = C, C - diff
    elif aj > C:
      aj, ai = C, C + diff
  else:
    quad = 2.0 - two_q
    quad = quad if quad > 0 else TAU
    delta = (Gi - Gj) / quad
    total = ai + aj
    ai, aj = ai - delta, aj + delta
    if total > C:
      if ai > C:
        ai, aj = C, total - C
    elif aj < 0:
      aj, ai = 0.0, total
    if total > C:
      if aj > C:
        aj, ai = C, total - C
    elif ai < 0:
      ai, aj = 0.0, total
  return ai, aj


def _rho(y, G, A, C):
  yG = y * G
  upper, lower = A >= C, A <= 0
  free = ~upper & ~lower
  if free.any():
    return sum(yG[free].tolist(), 0.0) / int(free.sum())   # sequential, in index order
  ub = np.min(yG[(upper & (y < 0)) | (lower & (y > 0))], initial=np.inf)
  lb = np.max(yG[(upper & (y > 0)) | (lower & (y < 0))], initial=-np.inf)
  return float((ub + lb) / 2)


def kkt_gap(X, y, coef, C=1.0, gamma=0.1):
  """max over I_up of -y G + max over I_low of y G, G = Q alpha - 1 recomputed in fp64 from the fp32
  kernel entries and alpha = y * coef."""
  y = np.asarray(y, dtype=np.float64)
  A = np.asarray(coef, dtype=np.float64) * y
  Q = kernel(X, X, gamma).astype(np.float64) * np.outer(y, y)
  G = Q @ A - 1.0
  up = np.where(y > 0, A < C, A > 0)
  low = np.where(y > 0, A > 0, A < C)
  return float(np.max(-(y * G)[up], initial=-np.inf) + np.max((y * G)[low], initial=-np.inf))


def decision(X, coef, rho, Z, gamma=0.1):
  """sum_i coef_i K(x_i, z) - rho for every row z of Z."""
  return kernel(Z, X, gamma).astype(np.float64) @ np.asarray(coef, dtype=np.float64) - rho
