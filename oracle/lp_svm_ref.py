"""Numpy restatement of the personalized link-prediction classifiers of csrc/hge_lp_svm.cu: each
owner's training set (members, then negatives drawn by Floyd's algorithm over the positions of its
ascending non-member list from the Philox streams of oracle/device_sampler_ref.py) and libsvm's
dual C-SVC solver as the kernel runs it (WSS3, no shrinking, fp32 kernel entries with the squared
distance summed sequentially over the components, fp64 gradient and alpha, ties to the largest
index, rho as calculate_rho), and k_predict's decision values in the kernel's summation order.

Every operation is IEEE fp32 / fp64 as the kernel performs it, except exp: nothing makes numpy's
exp round as the device's expf does, so `exp` (default: numpy's) lets a caller supply the device's
values, and with them the restatement is bit-exact.

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


def exp32(x):
  """numpy's exp of an fp32 array, in fp32 (the default `exp` hook)."""
  return np.exp(np.asarray(x, dtype=np.float32)).astype(np.float32)


def kernel(A, B, gamma, exp=exp32):
  """fp32 K(a, b) = exp(-gamma ||a - b||^2) of every row pair, the squared distance summed in
  component order, each operation rounded to fp32.  `exp` maps the fp32 argument array to fp32."""
  A = np.asarray(A, dtype=np.float32)
  B = np.asarray(B, dtype=np.float32)
  s = np.zeros((len(A), len(B)), dtype=np.float32)
  for c in range(A.shape[1]):
    t = A[:, c][:, None] - B[:, c][None, :]
    s = s + t * t
  return np.asarray(exp(np.float32(-gamma) * s), dtype=np.float32)


TRACE_KEYS = (
    "select_tau",        # a WSS3 candidate's quad <= 0, TAU used
    "step_tau",          # the update's quad <= 0, TAU used
    "ne_free", "ne_lo_j", "ne_lo_i", "ne_hi_i", "ne_hi_j",   # y_i != y_j: no clip, or which clip
    "eq_free", "eq_hi_i", "eq_lo_j", "eq_hi_j", "eq_lo_i",   # y_i == y_j
    "tie_i",             # more than one index attains Gmax
    "tie_j",             # more than one candidate attains the least objective
    "rho_free",          # rho from the free alphas
    "rho_bounds",        # no free alpha: rho = (ub + lb) / 2
    "stop_empty",        # stop: no I_up member or no WSS3 candidate left
    "stop_tol",          # stop: max_up -yG + max_low yG < tol
)


def _count(trace, key, k=1):
  if trace is not None:
    trace[key] = trace.get(key, 0) + int(k)


def solve(X, y, C=1.0, gamma=0.1, tol=1e-3, max_iter=None, exp=exp32, trace=None):
  """(alpha, rho, iterations) of libsvm's C-SVC dual on points X with labels y in {+1, -1}.
  `trace` (a dict) has the TRACE_KEYS branch counters added to it."""
  y = np.asarray(y, dtype=np.float64)
  n = len(y)
  Q = (kernel(X, X, gamma, exp) * np.where(y[:, None] == y[None, :], 1, -1).astype(np.float32)).astype(np.float32)
  G = np.full(n, -1.0)
  A = np.zeros(n)
  cap = max(10000000, 100 * n) if max_iter is None else max_iter
  idx = np.arange(n)
  it = 0
  while it < cap:
    up = np.where(y > 0, A < C, A > 0)
    if not up.any():
      _count(trace, "stop_empty")
      break
    v = np.where(up, -(y * G), -np.inf)
    Gmax = v.max()
    top = idx[v == Gmax]
    _count(trace, "tie_i", len(top) > 1)
    i = int(top[-1])
    Qi = Q[i].astype(np.float64)
    low = np.where(y > 0, A > 0, A < C)
    g2 = np.where(low, y * G, -np.inf).max()
    grad_diff = Gmax + y * G
    cand = low & (grad_diff > 0)
    if not cand.any():
      _count(trace, "stop_empty")
      break
    quad = 2.0 - y * ((2.0 * y[i]) * Qi)
    _count(trace, "select_tau", np.count_nonzero(cand & ~(quad > 0)))
    quad = np.where(quad > 0, quad, TAU)
    obj = np.where(cand, -(grad_diff * grad_diff) / quad, np.inf)
    omin = obj.min()
    best = idx[obj == omin]
    if Gmax + g2 < tol:
      _count(trace, "stop_tol")
      break
    _count(trace, "tie_j", len(best) > 1)
    j = int(best[-1])
    Qj = Q[j].astype(np.float64)
    ai, aj = _step(y[i], y[j], G[i], G[j], A[i], A[j], Q[i, j], C, trace)
    dai, daj = ai - A[i], aj - A[j]
    G = G + (Qi * dai + Qj * daj)
    A[i], A[j] = ai, aj
    it += 1
  return A, _rho(y, G, A, C, trace), it


def _step(yi, yj, Gi, Gj, ai, aj, Qij, C, trace=None):
  two_q = float(np.float32(2) * np.float32(Qij))
  clips = []
  if yi != yj:
    quad = 2.0 + two_q
    if quad <= 0:
      quad = TAU
      _count(trace, "step_tau")
    delta = (-Gi - Gj) / quad
    diff = ai - aj
    ai, aj = ai + delta, aj + delta
    if diff > 0:
      if aj < 0:
        aj, ai = 0.0, diff
        clips.append("ne_lo_j")
    elif ai < 0:
      ai, aj = 0.0, -diff
      clips.append("ne_lo_i")
    if diff > 0:
      if ai > C:
        ai, aj = C, C - diff
        clips.append("ne_hi_i")
    elif aj > C:
      aj, ai = C, C + diff
      clips.append("ne_hi_j")
  else:
    quad = 2.0 - two_q
    if quad <= 0:
      quad = TAU
      _count(trace, "step_tau")
    delta = (Gi - Gj) / quad
    total = ai + aj
    ai, aj = ai - delta, aj + delta
    if total > C:
      if ai > C:
        ai, aj = C, total - C
        clips.append("eq_hi_i")
    elif aj < 0:
      aj, ai = 0.0, total
      clips.append("eq_lo_j")
    if total > C:
      if aj > C:
        aj, ai = C, total - C
        clips.append("eq_hi_j")
    elif ai < 0:
      ai, aj = 0.0, total
      clips.append("eq_lo_i")
  for key in clips or ["ne_free" if yi != yj else "eq_free"]:
    _count(trace, key)
  return ai, aj


def _rho(y, G, A, C, trace=None):
  yG = y * G
  upper, lower = A >= C, A <= 0
  free = ~upper & ~lower
  if free.any():
    _count(trace, "rho_free")
    # sequential, in index order, as calculate_rho's sum_free += yG (not Python's sum(), which
    # compensates its float sums since 3.12)
    total = 0.0
    for v in yG[free].tolist():
      total += v
    return total / int(free.sum())
  _count(trace, "rho_bounds")
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


def decision(X, coef, rho, Z, gamma=0.1, exp=exp32):
  """sum_i coef_i K(x_i, z) - rho for every row z of Z."""
  return kernel(Z, X, gamma, exp).astype(np.float64) @ np.asarray(coef, dtype=np.float64) - rho


def decision_device_order(X, coef, rho, Z, gamma=0.1, exp=exp32):
  """decision() summed as k_predict sums it, one warp per z: lane l adds the terms
  fl64(coef_t * K(x_t, z)) of t = l, l + 32, ... in order, skipping coef_t == 0; then for o = 16, 8,
  4, 2, 1 every lane adds lane l ^ o's sum to its own; lane 0's sum minus rho.  No points: -rho."""
  coef = np.asarray(coef, dtype=np.float64)
  Z = np.asarray(Z, dtype=np.float32)
  lanes = np.zeros((32, len(Z)))
  if len(coef):
    K = kernel(X, Z, gamma, exp).astype(np.float64)
    for r in range(0, len(coef), 32):
      c, k = coef[r:r + 32], K[r:r + 32]
      s = lanes[:len(c)]
      lanes[:len(c)] = np.where((c != 0)[:, None], s + c[:, None] * k, s)
  for o in (16, 8, 4, 2, 1):
    lanes = lanes + lanes[np.arange(32) ^ o]
  return lanes[0] - rho
