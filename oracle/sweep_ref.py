"""Numpy restatement of the fp32 algebraic-distance relaxation of csrc/hge_algdist.cu and
csrc/hge_sweep.cu in the device's own operation order: xn, xe and the per-sweep min / max the
kernels should produce bit for bit, signed zeros included.  tests/test_sweep_ref_host.py pins it
on the CPU, tests/test_sweep_exact_gpu.py compares the kernels with it.

Why an exact restatement is possible (DESIGN section 6):
- every row sum is a sequence of single IEEE fp32 additions (add.rn.f32x2) in an order fixed by
  the gather stream (csrc/hge_schedule.cu), not by the grid: pieces and block counts move work
  between warps, never incidences between sums;
- long rows go through a fixed group butterfly and a Kahan hand-off in chunk order;
- everything else is one IEEE operation at a time: explicit fmaf, __frcp_rn, IEEE division,
  f64 sums rounded once to fp32.  build.NVCC_FLAGS has no fast-math, FTZ or prec-div flag.

What the compiler made of the source is part of the order.  Read from `cuobjdump -sass` of the
sm_100a build (the PTX alone is not enough: ptxas contracts a PTX mul.f32 + sub.f32 pair):
- k_sweep's finish: FMUL inv*hd, FMUL inv*hs (node half), then the two FFMA as written; no other
  contraction.  Prologue: inv = rcp.rn(hi - lo), c3 = h * (lo * inv).
- k_load_rows: FMUL x * rcp.rn(deg).
- k_store_rows: with a map, `y * deg - lo` is ONE FFMA (y, deg, -lo) (PTX: mul.f32 + sub.f32,
  fused by ptxas), then an IEEE division by (hi - lo).  Without a map: FMUL y * deg.
- k_edge_finalize: `0.5f * (own + raw * invs)` is contracted, and differently on the two paths:
  sweep 0 (no map): FMUL raw*invs, FFMA (y, deg, that), FMUL 0.5 -- `own = y * deg` is never
  rounded on its own; later sweeps: FMUL own = y*deg, FMUL -lo*inv, FFMA (inv, own, that),
  FFMA (raw, invs, that), FMUL 0.5.
- k_invert: rcp.rn.f64 then cvt.rn.f32.f64.

Out of scope: the peer-memory push mode (kSweepPush) and the NCCL path at more than one rank.

Test infrastructure only."""
import numpy as np

DEFAULT_LIGHT_MAX = 128     # hge_core.cu: ctx->light_max_deg
DEFAULT_CHUNK = 1024        # hge_core.cu: ctx->chunk
WSUM_LONG = 512             # hge_algdist.cu: kWsumLong
F32 = np.float32


# ---- single fp32 operations ------------------------------------------------------------------

def fma32(a, b, c):
  """Correctly rounded fp32 fma(a, b, c), elementwise.  a * b is exact in f64 (24 + 24 bits);
  TwoSum gives s + e == a * b + c exactly; rounding s to odd in f64 (53 >= 2 * 24 + 2 bits) and
  then once to fp32 rounds the exact sum correctly.  Zero signs follow IEEE: an exact zero sum is
  +0 unless both addends are -0, as in f64."""
  a, b, c = np.broadcast_arrays(np.asarray(a, F32), np.asarray(b, F32), np.asarray(c, F32))
  p = a.astype(np.float64) * b.astype(np.float64)
  c64 = c.astype(np.float64)
  with np.errstate(invalid="ignore", over="ignore"):
    s = p + c64
    bp = s - p
    e = (p - (s - bp)) + (c64 - bp)
    odd = (s.view(np.int64) & 1) != 0
    bump = (e != 0) & ~odd & np.isfinite(s)
    s = np.where(bump, np.nextafter(s, np.where(e > 0, np.inf, -np.inf)), s)
  return s.astype(F32)


def rcp32(d):
  """__frcp_rn: the correctly rounded fp32 reciprocal."""
  return F32(1) / np.asarray(d, F32)


def enc(x):
  """hge_enc: fp32 -> int32 in the order -NaN < -inf < ... < -0 < +0 < ... < +inf."""
  i = np.asarray(x, F32).view(np.int32)
  return i ^ ((i >> 31) & 0x7fffffff)


def dec(i):
  i = np.asarray(i, np.int32)
  return (i ^ ((i >> 31) & 0x7fffffff)).view(F32)


def lanes_per_row(R):
  """hge_algdist_create: lanes per row = next power of two >= ld / 4, at most 32."""
  ld4 = ((R + 3) & ~3) // 4
  lpr = 1
  while lpr < ld4 and lpr < 32:
    lpr <<= 1
  return lpr


def groups_of(R):
  return 32 // lanes_per_row(R)


# ---- set-up -------------------------------------------------------------------------------------

def _bfly(v, axis_len, stop=None):
  """In-place xor butterfly over axis -2 (lanes): v_l <- v_l + v_{l ^ m}, m = 1, 2, 4, ..."""
  m = 1
  n = axis_len if stop is None else stop
  while m < n:
    v = v + v[..., np.arange(axis_len) ^ m, :]
    m <<= 1
  return v


def weight_sums(ptr, idx, other_deg):
  """wsum[r] = sum over the row of 1 / other_deg, f64, in the order of k_row_wsum (rows of at most
  512 incidences: 8 lanes at stride 8, then xor 4, 2, 1) and k_row_wsum_long (longer rows: 4
  accumulators per thread at stride 256, (s0 + s1) + (s2 + s3), warp butterfly 16 .. 1, then the 8
  warp partials added in order)."""
  ptr = np.asarray(ptr, np.int64)
  idx = np.asarray(idx, np.int64)
  w = 1.0 / np.asarray(other_deg, np.float64)[idx]
  deg = np.diff(ptr)
  rows = len(deg)
  out = np.zeros(rows, np.float64)
  short = np.nonzero(deg <= WSUM_LONG)[0]
  if len(short):
    s = np.zeros((len(short), 8), np.float64)
    b, d = ptr[short], deg[short]
    for k in range(0, int(d.max(initial=0)), 8):
      p = k + np.arange(8)[None, :]
      valid = p < d[:, None]
      vals = np.where(valid, w[np.where(valid, b[:, None] + p, 0)], 0.0)
      s = np.where(valid, s + vals, s)
    for off in (4, 2, 1):
      s = s + s[:, np.arange(8) ^ off]
    out[short] = s[:, 0]
  for r in np.nonzero(deg > WSUM_LONG)[0]:
    wr = w[ptr[r]:ptr[r + 1]]
    e = len(wr)
    lane_sum = np.zeros(256, np.float64)
    for t in range(256):
      s4 = [0.0, 0.0, 0.0, 0.0]
      p = t
      while p + 3 * 256 < e:
        for q in range(4):
          s4[q] = s4[q] + wr[p + q * 256]
        p += 4 * 256
      while p < e:
        s4[0] = s4[0] + wr[p]
        p += 256
      lane_sum[t] = (s4[0] + s4[1]) + (s4[2] + s4[3])
    v = lane_sum.reshape(8, 32)
    for off in (16, 8, 4, 2, 1):
      v = v + v[:, np.arange(32) ^ off]
    t = 0.0
    for wp in v[:, 0]:
      t = t + wp
    out[r] = t
  return out


class Incidence(object):
  """Both orientations of an N x E incidence (int64 row pointers, int32 column ids sorted inside
  every row) and what hge_incidence_create derives from them: degrees and invs = fp32(1 / wsum)."""

  def __init__(self, n2e_ptr, n2e_idx, e2n_ptr, e2n_idx):
    self.n_ptr = np.asarray(n2e_ptr, np.int64)
    self.n_idx = np.asarray(n2e_idx, np.int64)
    self.e_ptr = np.asarray(e2n_ptr, np.int64)
    self.e_idx = np.asarray(e2n_idx, np.int64)
    self.N, self.E = len(self.n_ptr) - 1, len(self.e_ptr) - 1
    self.n_deg = np.diff(self.n_ptr)
    self.e_deg = np.diff(self.e_ptr)
    if (self.n_deg == 0).any() or (self.e_deg == 0).any():
      raise ZeroDivisionError("a row without incidences")
    self.e_invs = (1.0 / weight_sums(self.e_ptr, self.e_idx, self.n_deg)).astype(F32)
    self.n_invs = (1.0 / weight_sums(self.n_ptr, self.n_idx, self.e_deg)).astype(F32)

  @classmethod
  def from_csr(cls, A):
    """From a scipy N x E CSR with sorted indices (the edge -> node side is its transpose)."""
    B = A.T.tocsr()
    B.sort_indices()
    return cls(A.indptr, A.indices, B.indptr, B.indices)


# ---- gathered sums ------------------------------------------------------------------------------

def row_sums(begin, end, idx, Y, light_max, chunk, G):
  """Gathered sums sum_{p in [begin[r], end[r])} Y[idx[p]] of k_sweep, fp32 [rows, R].

  Light rows (degree <= light_max): one lane group adds the rows one at a time in CSR order
  from +0 (the padding adds the zero row, which changes nothing: such a sum is never -0).
  Long rows: chunks of `chunk` incidences; incidence j of a chunk is summed by group
  (j // 4) % G in increasing j, the groups are combined by the xor butterfly of reduce_groups
  and group 0's value is the chunk's sum.  With several chunks, group g Kahan-sums the chunk sums
  k = g (mod G) in increasing k (kahan_add4), takes tot - comp, and the butterfly runs again."""
  begin = np.asarray(begin, np.int64)
  end = np.asarray(end, np.int64)
  Y = np.asarray(Y, F32)
  R = Y.shape[1]
  deg = end - begin
  out = np.zeros((len(deg), R), F32)
  # light rows, by descending degree so that "degree > k" is a prefix
  light = np.nonzero(deg <= light_max)[0]
  light = light[np.argsort(-deg[light], kind="stable")]
  ld_ = deg[light]
  acc = np.zeros((len(light), R), F32)
  for k in range(int(ld_.max(initial=0))):
    n = int(np.searchsorted(-ld_, -k, side="left"))   # rows with degree > k
    acc[:n] += Y[idx[begin[light[:n]] + k]]
  out[light] = acc
  heavy = np.nonzero(deg > light_max)[0]
  if len(heavy) == 0:
    return out
  # every chunk of every long row at once: [chunks, G, R] group sums
  nch = (deg[heavy] + chunk - 1) // chunk
  ch_row = np.repeat(np.arange(len(heavy)), nch)
  ch_k = np.concatenate([np.arange(c) for c in nch])
  ch_beg = begin[heavy][ch_row] + ch_k * chunk
  ch_cnt = np.minimum(chunk, deg[heavy][ch_row] - ch_k * chunk)
  order = np.argsort(-ch_cnt, kind="stable")
  cnt_sorted = ch_cnt[order]
  V = np.zeros((len(order), G, R), F32)
  for j in range(int(cnt_sorted[0])):
    n = int(np.searchsorted(-cnt_sorted, -j, side="left"))
    V[:n, (j // 4) % G] += Y[idx[ch_beg[order[:n]] + j]]
  V = _bfly(V, G)
  chunk_sum = np.empty((len(order), R), F32)
  chunk_sum[order] = V[:, 0]
  first = np.concatenate([[0], np.cumsum(nch)[:-1]])
  for h, r in enumerate(heavy):
    sums = chunk_sum[first[h]:first[h] + nch[h]]
    if nch[h] == 1:
      out[r] = sums[0]
      continue
    tot = np.zeros((G, R), F32)
    comp = np.zeros((G, R), F32)
    for k in range(int(nch[h])):
      g = k % G
      y = sums[k] - comp[g]
      t = tot[g] + y
      comp[g] = (t - tot[g]) - y
      tot[g] = t
    out[r] = _bfly((tot - comp)[None], G)[0, 0]
  return out


# ---- the two halves -----------------------------------------------------------------------------

def _prologue(mm_prev, R, h):
  """k_sweep's per-column constants: inv = 1 / (hi - lo), c3 = h * (lo * inv); lo = 0, inv = 1
  without a map (sweep 0)."""
  if mm_prev is None:
    return np.ones(R, F32), np.zeros(R, F32)
  lo, hi = mm_prev
  inv = F32(1) / (hi - lo)
  return inv, F32(h) * (lo * inv)


def finish_rows(deg, invs, yown, acc, mm_prev, node):
  """finish_row of k_sweep (kSweepNode / kSweepEdge): returns (x, y = x * rcp(deg))."""
  R = acc.shape[1]
  inv, c3 = _prologue(mm_prev, R, 1.0 if node else 0.5)
  degf = np.asarray(deg, F32)[:, None]
  hd = F32(0.5) * degf
  hs = F32(0.5) * np.asarray(invs, F32)[:, None]
  if node:
    inner = fma32(inv[None] * hs, acc, -c3[None])
  else:
    inner = fma32(hs, acc, -c3[None])
  x = fma32(inv[None] * hd, yown, inner)
  return x, x * rcp32(degf)


def edge_finalize(deg, invs, y_old, raw, mm_prev):
  """k_edge_finalize (tiled and sharded edge halves) as compiled: returns (x, y)."""
  degf = np.asarray(deg, F32)[:, None]
  invs = np.asarray(invs, F32)[:, None]
  if mm_prev is None:
    # 0.5f * (y * deg + raw * invs): FMUL raw*invs, FFMA(y, deg, .) -- own is not rounded alone
    x = F32(0.5) * fma32(y_old, degf, raw * invs)
  else:
    lo, hi = mm_prev
    inv = F32(1) / (hi - lo)
    own = fma32(inv[None], y_old * degf, (-lo * inv)[None])
    x = F32(0.5) * fma32(raw, invs, own)
  return x, x * rcp32(degf)


def _minmax(x):
  e = enc(x)
  return e.min(axis=0), e.max(axis=0)


class Relaxation(object):
  """State of hge_algdist: Y rows (yn, ye) and the encoded per-sweep min / max slots.

  edge_path: "untiled" (kSweepEdge), ("tiled", tile_rows) (node-range tiles, kSweepRawAdd, then
  k_edge_finalize) or ("sharded", num_slices) (one rank: kSweepRaw per slice, then
  k_edge_finalize per slice; slices do not change the sums, so num_slices only names the path)."""

  def __init__(self, inc, R, light_max=DEFAULT_LIGHT_MAX, chunk=DEFAULT_CHUNK, edge_path="untiled"):
    self.inc, self.R = inc, int(R)
    self.light_max, self.chunk = int(light_max), int(chunk)
    self.G = groups_of(self.R)
    self.edge_path = edge_path
    self.mm = []          # per sweep: [2, R] int32 (hge_enc of min, max)
    if isinstance(edge_path, tuple) and edge_path[0] == "tiled":
      tile_rows = int(edge_path[1])
      tiles = (inc.N + tile_rows - 1) // tile_rows
      # k_tile_offsets: first member >= t * tile_rows in every edge (members are sorted)
      self.tile_pos = np.empty((tiles + 1, inc.E), np.int64)
      for t in range(tiles + 1):
        for e in range(inc.E):
          b, en = inc.e_ptr[e], inc.e_ptr[e + 1]
          if t == 0:
            self.tile_pos[t, e] = b
          elif t == tiles:
            self.tile_pos[t, e] = en
          else:
            self.tile_pos[t, e] = b + np.searchsorted(inc.e_idx[b:en], t * tile_rows, side="left")

  def load(self, xn, xe):
    """k_load_rows: Y = x * rcp(deg)."""
    self.yn = np.asarray(xn, F32) * rcp32(self.inc.n_deg)[:, None]
    self.ye = np.asarray(xe, F32) * rcp32(self.inc.e_deg)[:, None]
    self.mm = []

  def _map(self, sweep):
    if sweep == 0:
      return None
    e = self.mm[sweep - 1]
    return dec(e[0]), dec(e[1])

  def node_half(self, sweep):
    inc = self.inc
    assert len(self.mm) == sweep
    acc = row_sums(inc.n_ptr[:-1], inc.n_ptr[1:], inc.n_idx, self.ye, self.light_max, self.chunk, self.G)
    x, self.yn = finish_rows(inc.n_deg, inc.n_invs, self.yn, acc, self._map(sweep), node=True)
    self.mm.append(np.stack(_minmax(x)))

  def edge_half(self, sweep):
    inc = self.inc
    mm_prev = self._map(sweep)
    if self.edge_path == "untiled":
      acc = row_sums(inc.e_ptr[:-1], inc.e_ptr[1:], inc.e_idx, self.yn, self.light_max, self.chunk, self.G)
      x, self.ye = finish_rows(inc.e_deg, inc.e_invs, self.ye, acc, mm_prev, node=False)
    elif self.edge_path[0] == "tiled":
      raw = np.zeros((inc.E, self.R), F32)
      for t in range(self.tile_pos.shape[0] - 1):
        raw = raw + row_sums(self.tile_pos[t], self.tile_pos[t + 1], inc.e_idx, self.yn, self.light_max,
                             self.chunk, self.G)
      x, self.ye = edge_finalize(inc.e_deg, inc.e_invs, self.ye, raw, mm_prev)
    else:
      raw = row_sums(inc.e_ptr[:-1], inc.e_ptr[1:], inc.e_idx, self.yn, self.light_max, self.chunk, self.G)
      x, self.ye = edge_finalize(inc.e_deg, inc.e_invs, self.ye, raw, mm_prev)
    lo, hi = _minmax(x)
    m = self.mm[sweep]
    m[0] = np.minimum(m[0], lo)
    m[1] = np.maximum(m[1], hi)

  def store(self, sweeps_done):
    """k_store_rows as compiled: x = y * deg without a map; with the map of the last sweep
    fma(y, deg, -lo) / (hi - lo) (ptxas fuses the PTX mul + sub)."""
    out = []
    for y, deg in ((self.yn, self.inc.n_deg), (self.ye, self.inc.e_deg)):
      degf = np.asarray(deg, F32)[:, None]
      if sweeps_done == 0:
        out.append(y * degf)
      else:
        lo, hi = self._map(sweeps_done)
        out.append(fma32(y, degf, -lo[None]) / (hi - lo)[None])
    return out[0], out[1]

  def lohi(self):
    """[sweeps, 2, R] fp32 as hge_algdist_run returns it."""
    return np.stack([dec(m) for m in self.mm]) if self.mm else np.zeros((0, 2, self.R), F32)


def relax(inc, xn, xe, iterations, light_max=DEFAULT_LIGHT_MAX, chunk=DEFAULT_CHUNK, edge_path="untiled"):
  """hge_algdist_run: (xn, xe, lohi) after `iterations` sweeps."""
  st = Relaxation(inc, np.asarray(xn).shape[1], light_max, chunk, edge_path)
  st.load(xn, xe)
  if iterations == 0:
    return np.asarray(xn, F32).copy(), np.asarray(xe, F32).copy(), st.lohi()
  for t in range(iterations):
    st.node_half(t)
    st.edge_half(t)
  xn2, xe2 = st.store(iterations)
  return xn2, xe2, st.lohi()
