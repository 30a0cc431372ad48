"""Numpy restatement of the fp32 hypergraph2vec epoch kernel k_hg2v_epoch (csrc/hge_hg2v_train.cu)
in the device's own operation order: the tables after every epoch bit for bit, signed zeros
included, on inputs where every table row receives at most two gradient contributions per batch.
tests/test_hg2v_train_ref_host.py pins it on the CPU (against the float64 Keras restatement
oracle/hg2v_model_ref.py, and on hand-built batches), tests/test_hg2v_train_exact_gpu.py compares
the kernel with it.

Why an exact restatement is possible at all: the only unordered operations are the float atomics
that sum duplicated rows' gradients.  fp32 addition is commutative, so a gradient element that
receives at most two contributions in a batch gets the same bits in any order (0 + a, then a + b).
With heavier duplication the order is a race and only oracle/hg2v_model_ref.py's tolerance applies;
this file then sums in one fixed order of its own.

What the compiler made of the source is part of the order.  Read from `cuobjdump -sass` of all four
instances k_hg2v_epoch<1>, <2>, <4>, <8> built with build.NVCC_FLAGS (no fast math, no FTZ flag);
the four agree on every point below:
- dot<DPL>: per lane s = FFMA(a[j], b[j], s) for j ascending from s = +0 (FFMA with RZ, not FMUL),
  over column lane + 32 j; columns >= dim enter as 0 and still take their FFMA, which matters for
  the sign of zero.  The preload path (DPL 1, k <= 8) forms the neighbour dots with an FMUL.
- warp_sum: five FADDs of rounded values behind SHFL.BFLY 16, 8, 4, 2, 1; no contraction.
- sigmoid: 1 / (1 + __expf(-z)) with a correctly rounded reciprocal (MUFU.RCP + FFMA fix-up and
  a slow path); __expf is taken through the `exp` hook.  relu: FMNMX(z, +0).
- KL: yc / pc and -yc / pc IEEE divisions (FCHK + slow path), yc * __logf(yc / pc) with __logf
  through the `log` hook; the gradient is zero unless 1e-7 <= p <= 1.
- MSE: the node_edge residual is CONTRACTED: d = FFMA(A, B, -y), so p_ne = A * B is never rounded
  on that path (KL still rounds p_ne = FMUL(A, B)).  node_node / edge_edge: FADD p - y.  Then
  loss d * d, gradient d + d.
- coefficients as written, left to right, one FMUL each: d_nn = (g_nn * inv_bs) * act'(z_nn),
  da = (((g_ne * inv_bs) * B) * inv_k) * act'(za); inv_k = 1 / k and inv_bs = 1 / bs in fp32;
  sigmoid' = p * (1 - p).
- gLn = d_nn * Rn, then FFMA(da_i, nb_i, gLn) for i ascending; a neighbour with da_i == 0 takes
  neither that FFMA nor its own row's contribution.  Likewise gRe on the edge side.
- gradient atomics to rows != 0: ATOMG.E.ADD.F32.FTZ.RN -- subnormal inputs and results flush to
  sign-preserving zero.
- row 0 (the padding row, s_g0): a shared-memory CAS loop (ATOMS.CAST.SPIN) around a plain FADD, so
  subnormals are kept; after phase 1 each CTA adds its sum to the global gradient with the FTZ
  atomic, and only where it is non-zero.  Two subnormal row-0 contributions therefore give
  different bits in one CTA than in two, and this file MODELS that split: sample position p of a
  batch runs on warp p mod (clusters * 256), in CTA warp // 32, with `clusters` the launch's
  cluster count (Hg2vModel.last_clusters).
- Adagrad on elements with g != 0 only: acc = FFMA(g, g, acc) (the float64 oracle rounds twice);
  then p - (lr * g) / (sqrt(acc) + eps), FMUL, IEEE sqrt (MUFU.RSQ + fix-up), FADD, IEEE division,
  FADD; lr = 0.01f, eps = 1e-7f.  The gradient element is then cleared.
- epoch loss: per sample (double(l_nn) + double(l_ee)) + double(l_ne) of fp32 losses, summed in
  double in an order the atomics decide (here: sample order), divided by M.

numpy cannot round __expf / __logf as the device does; `exp` and `log` are hooks (fp32 array in,
fp32 array out).  The defaults are numpy in fp32, so on the CPU the restatement is exact up to
those two functions.

Test infrastructure only."""
import numpy as np

from oracle.sweep_ref import fma32

F32 = np.float32
LR = F32(0.01)
EPS = F32(1e-7)
KL_EPS = F32(1e-7)
TINY = np.finfo(F32).tiny
WARPS_PER_CTA = 32
WARPS_PER_CLUSTER = 256
PRELOAD_MAX_K = 8
_XOR = [np.arange(32) ^ off for off in (16, 8, 4, 2, 1)]


def exp32(x):
  return np.exp(np.asarray(x, F32)).astype(F32)


def log32(x):
  return np.log(np.asarray(x, F32)).astype(F32)


def ftz(x):
  """Subnormal -> zero of the same sign (the FTZ float atomics)."""
  x = np.asarray(x, F32)
  return np.where(np.abs(x) < TINY, np.copysign(F32(0), x), x).astype(F32)


def lanes_per_dim(dim):
  """DPL of the instance hge_hg2v_fit_epoch launches: columns per lane, 1, 2, 4 or 8."""
  dpl = (int(dim) + 31) // 32
  return 1 if dpl <= 1 else 2 if dpl <= 2 else 4 if dpl <= 4 else 8


def warp_sum(v):
  """[..., 32] lane values -> [...]: the xor butterfly 16 .. 1; all lanes end equal."""
  for x in _XOR:
    v = v + v[..., x]
  return v[..., 0]


def _lanes(rows, dpl):
  """[m, dim] rows -> [m, dpl, 32]: element (j, lane) is column lane + 32 j, 0 beyond dim."""
  m, dim = rows.shape
  out = np.zeros((m, dpl * 32), F32)
  out[:, :dim] = rows
  return out.reshape(m, dpl, 32)


def _dot(a, b):
  """dot<DPL>: [m, dpl, 32] x2 -> [m]"""
  s = np.zeros(a.shape[:1] + a.shape[2:], F32)
  for j in range(a.shape[1]):
    s = fma32(a[:, j], b[:, j], s)
  return warp_sum(s)


def _activate(z, kind, exp):
  if kind == "sigmoid":
    return F32(1) / (F32(1) + exp(-z))
  return np.where(z > 0, z, F32(0)).astype(F32)


def _activate_grad(z, p, kind):
  if kind == "sigmoid":
    return p * (F32(1) - p)
  return np.where(z > 0, F32(1), F32(0)).astype(F32)


def _loss_grad(p, y, kind, log, fused=None):
  """(per-sample loss, d loss / d p), fp32.  `fused` = (A, B): the MSE residual is FFMA(A, B, -y)."""
  if kind == "kld":
    yc = np.minimum(np.maximum(y, KL_EPS), F32(1))
    pc = np.minimum(np.maximum(p, KL_EPS), F32(1))
    inside = (p >= KL_EPS) & (p <= F32(1))
    return yc * log(yc / pc), np.where(inside, -yc / pc, F32(0)).astype(F32)
  d = fma32(fused[0], fused[1], -y) if fused is not None else p - y
  return d * d, d + d


def _scatter_ftz(g, rows, vals):
  """g[rows[i]] = ftz(g[rows[i]] + ftz(vals[i])), one contribution at a time in a fixed order."""
  if len(rows) == 0:
    return
  order = np.argsort(rows, kind="stable")
  rows, vals = rows[order], vals[order]
  start = np.r_[0, np.flatnonzero(np.diff(rows)) + 1]
  rank = np.arange(len(rows)) - np.repeat(start, np.diff(np.r_[start, len(rows)]))
  for r in range(int(rank.max()) + 1):
    sel = rank == r
    g[rows[sel]] = ftz(g[rows[sel]] + ftz(vals[sel]))


TRACE_KEYS = ("relu_z_zero", "sigmoid_p_one", "kl_p_below_eps", "kl_p_above_one", "kl_p_one",
              "target_zero", "target_one", "target_1e-8", "subnormal_contribution", "da_zero_skip",
              "row0_one_cta_pair", "row0_two_cta_pair", "grad_zero_element")


def _count(trace, key, n):
  if trace is not None:
    trace[key] = trace.get(key, 0) + int(n)


class Trainer(object):
  """The state of one hge_hg2v_model: fp32 tables, Adagrad accumulators and gradient tables.

  activation "sigmoid" / "relu", loss "kld" / "mse" (hg2v_model_ref's names)."""

  def __init__(self, N, E, k, activation, loss, exp=exp32, log=log32, trace=None):
    self.N, self.E = np.array(N, F32), np.array(E, F32)
    self.accN, self.accE = np.zeros_like(self.N), np.zeros_like(self.E)
    self.gN, self.gE = np.zeros_like(self.N), np.zeros_like(self.E)
    self.k, self.activation, self.loss = int(k), activation, loss
    self.exp, self.log = exp, log
    self.trace = trace      # dict: counts of the boundary cases met (TRACE_KEYS), or None
    self.dim = self.N.shape[1]
    self.dpl = lanes_per_dim(self.dim)

  def epoch(self, feats, targets, order, batch_size, clusters=1):
    """One hge_hg2v_fit_epoch: feats [4 + 2k][M] int, targets [3][M], order [M].  Returns the
    epoch loss (sum of the per-sample losses / M)."""
    feats = np.asarray(feats, np.int64)
    targets = np.asarray(targets, F32)
    order = np.asarray(order, np.int64)
    M = len(order)
    total = 0.0
    for first in range(0, M, batch_size):
      sel = order[first:first + batch_size]
      total += self.batch(feats[:, sel], targets[:, sel], clusters)
    return total / M

  def batch(self, f, t, clusters=1):
    """Phase 1 and phase 2 of one batch (f [cols][bs], t [3][bs]); returns the summed loss."""
    k, dpl, kind, exp = self.k, self.dpl, self.activation, self.exp
    bs = f.shape[1]
    inv_bs = F32(1) / F32(bs)
    inv_k = F32(1) / F32(k) if k else F32(0)
    ln, le, rn, re = f[0], f[1], f[2], f[3]
    nbn, nbe = f[4:4 + k].T, f[4 + k:4 + 2 * k].T          # [bs, k]
    Ln, Rn = _lanes(self.N[ln], dpl), _lanes(self.N[rn], dpl)
    Le, Re = _lanes(self.E[le], dpl), _lanes(self.E[re], dpl)
    z_nn, z_ee = _dot(Ln, Rn), _dot(Le, Re)
    p_nn, p_ee = _activate(z_nn, kind, exp), _activate(z_ee, kind, exp)
    XN = [_lanes(self.N[nbn[:, i]], dpl) for i in range(k)]
    XE = [_lanes(self.E[nbe[:, i]], dpl) for i in range(k)]
    if dpl == 1 and k <= PRELOAD_MAX_K:
      za = [warp_sum(X[:, 0] * Ln[:, 0]) for X in XN]
      zb = [warp_sum(X[:, 0] * Re[:, 0]) for X in XE]
    else:
      za = [_dot(X, Ln) for X in XN]
      zb = [_dot(X, Re) for X in XE]
    a_lane = np.zeros((bs, 32), F32)
    b_lane = np.zeros((bs, 32), F32)
    for i in range(k):
      a_lane[:, i] = _activate(za[i], kind, exp)
      b_lane[:, i] = _activate(zb[i], kind, exp)
    A, B = warp_sum(a_lane) * inv_k, warp_sum(b_lane) * inv_k
    l_nn, g_nn = _loss_grad(p_nn, t[0], self.loss, self.log)
    l_ee, g_ee = _loss_grad(p_ee, t[1], self.loss, self.log)
    l_ne, g_ne = _loss_grad(A * B, t[2], self.loss, self.log, fused=(A, B))
    loss = float(np.sum((l_nn.astype(np.float64) + l_ee.astype(np.float64)) + l_ne.astype(np.float64)))
    d_nn = g_nn * inv_bs * _activate_grad(z_nn, p_nn, kind)
    d_ee = g_ee * inv_bs * _activate_grad(z_ee, p_ee, kind)
    ne_bs = g_ne * inv_bs
    da = [ne_bs * B * inv_k * _activate_grad(za[i], a_lane[:, i], kind) for i in range(k)]
    db = [ne_bs * A * inv_k * _activate_grad(zb[i], b_lane[:, i], kind) for i in range(k)]
    gLn = d_nn[:, None, None] * Rn
    gRe = d_ee[:, None, None] * Le
    rowsN, valsN, rowsE, valsE = [ln, rn], [gLn, d_nn[:, None, None] * Ln], [re, le], [gRe, d_ee[:, None, None] * Re]
    pos = np.arange(bs)
    posN, posE = [pos, pos], [pos, pos]
    for i in range(k):
      on = da[i] != 0
      gLn = np.where(on[:, None, None], fma32(da[i][:, None, None], XN[i], gLn), gLn)
      rowsN.append(nbn[on, i])
      valsN.append(da[i][on, None, None] * Ln[on])
      posN.append(pos[on])
      on = db[i] != 0
      gRe = np.where(on[:, None, None], fma32(db[i][:, None, None], XE[i], gRe), gRe)
      rowsE.append(nbe[on, i])
      valsE.append(db[i][on, None, None] * Re[on])
      posE.append(pos[on])
    valsN[0], valsE[0] = gLn, gRe
    tr = self.trace
    if tr is not None:
      zs = [z_nn, z_ee] + za + zb
      ps = [p_nn, p_ee] + [a_lane[:, i] for i in range(k)] + [b_lane[:, i] for i in range(k)]
      if kind == "relu":
        _count(tr, "relu_z_zero", sum(np.count_nonzero(z == 0) for z in zs))
      else:
        _count(tr, "sigmoid_p_one", sum(np.count_nonzero(p == 1) for p in ps))
      if self.loss == "kld":
        for p in (p_nn, p_ee, A * B):
          _count(tr, "kl_p_below_eps", np.count_nonzero(p < KL_EPS))
          _count(tr, "kl_p_above_one", np.count_nonzero(p > 1))
          _count(tr, "kl_p_one", np.count_nonzero(p == 1))
      _count(tr, "target_zero", np.count_nonzero(t == 0))
      _count(tr, "target_one", np.count_nonzero(t == 1))
      _count(tr, "target_1e-8", np.count_nonzero(t == F32(1e-8)))
      _count(tr, "da_zero_skip", sum(np.count_nonzero(d == 0) for d in da + db))
    cta = (pos % (clusters * WARPS_PER_CLUSTER)) // WARPS_PER_CTA
    for P, acc, g, rows, vals, at in ((self.N, self.accN, self.gN, rowsN, valsN, posN),
                                      (self.E, self.accE, self.gE, rowsE, valsE, posE)):
      rows = np.concatenate(rows)
      vals = np.concatenate(vals).reshape(len(rows), -1)[:, :self.dim]
      at = cta[np.concatenate(at)]
      zero = rows == 0
      if tr is not None:
        sub = (vals != 0) & (np.abs(vals) < TINY)
        _count(tr, "subnormal_contribution", np.count_nonzero(sub))
        if np.count_nonzero(zero) == 2:
          _count(tr, "row0_one_cta_pair" if at[zero][0] == at[zero][1] else "row0_two_cta_pair", 1)
      _scatter_ftz(g, rows[~zero], vals[~zero])
      # row 0: a plain (non-FTZ) sum per CTA, then one FTZ atomic per CTA where that sum is non-zero
      s0 = np.zeros((int(cta.max()) + 1, self.dim), F32)
      order = np.argsort(at[zero], kind="stable")
      for c, v in zip(at[zero][order], vals[zero][order]):
        s0[c] = s0[c] + v
      for c in np.unique(at[zero]):
        g[0] = np.where(s0[c] != 0, ftz(g[0] + ftz(s0[c])), g[0])
      # phase 2: Adagrad on the rows the batch named, elements with g != 0
      touched = np.unique(rows if len(rows) else np.zeros(0, np.int64))
      gv, av, pv = g[touched], acc[touched], P[touched]
      upd = gv != 0
      _count(tr, "grad_zero_element", np.count_nonzero(~upd))
      a2 = fma32(gv, gv, av)
      p2 = pv - (LR * gv) / (np.sqrt(a2) + EPS)
      acc[touched] = np.where(upd, a2, av)
      P[touched] = np.where(upd, p2, pv)
      g[touched] = np.where(upd, F32(0), gv)
    return loss
