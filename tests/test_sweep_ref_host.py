"""CPU checks of oracle/sweep_ref.py, the restatement of the relaxation kernels in their own
fp32 operation order:
- its exact fp32 fma against rational arithmetic;
- the relaxation it restates against the f64 port (oracle/port.py) at the 1e-5 bar;
- hand-built rows whose last bit shows the summation order it claims (lane groups, butterfly,
  Kahan hand-off over the chunks, tile boundaries)."""
from fractions import Fraction

import numpy as np
import pytest

from conftest import csr_from_pairs, incidence_distances, load_golden
from oracle import sweep_ref as sr

F32 = np.float32


def _round_f32(q):
  """Fraction -> nearest fp32 (ties to even), by bisection over the ordered fp32 bit patterns."""
  if q == 0:
    return F32(0.0)
  sign = -1 if q < 0 else 1
  a = abs(q)
  lo, hi = 0, 0x7f800000          # a lies in [value(lo), value(hi)]
  while hi - lo > 1:
    mid = (lo + hi) // 2
    if Fraction(float(np.uint32(mid).view(F32))) <= a:
      lo = mid
    else:
      hi = mid
  vlo, vhi = Fraction(float(np.uint32(lo).view(F32))), Fraction(float(np.uint32(hi).view(F32)))
  if a - vlo < vhi - a or (a - vlo == vhi - a and lo % 2 == 0):
    pick = lo
  else:
    pick = hi
  return F32(sign * float(np.uint32(pick).view(F32)))


def _fma_exact(a, b, c):
  q = Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c))
  if q == 0:
    p = float(a) * float(b)
    # an exact zero sum: -0 only when both addends are -0 (round to nearest)
    neg = np.signbit(p) and np.signbit(c) and (p == 0)
    return F32(-0.0) if neg else F32(0.0)
  return _round_f32(q)


def _check_fma(a, b, c):
  got = sr.fma32(a, b, c)
  for i in range(len(a)):
    want = _fma_exact(a[i], b[i], c[i])
    assert got[i].view(np.uint32) == want.view(np.uint32), (a[i], b[i], c[i], got[i], want)


def test_fma32_random_triples():
  rng = np.random.default_rng(0)
  n = 100000
  a = (rng.standard_normal(n) * 10.0 ** rng.integers(-6, 6, n)).astype(F32)
  b = (rng.standard_normal(n) * 10.0 ** rng.integers(-6, 6, n)).astype(F32)
  c = (-(a.astype(np.float64) * b) * (1 + rng.standard_normal(n) * 10.0 ** rng.integers(-9, 1, n))).astype(F32)
  got = sr.fma32(a, b, c)
  up = np.nextafter(got, F32(np.inf))
  down = np.nextafter(got, F32(-np.inf))
  for i in range(n):
    # got is the nearest fp32 to the exact value, and on a tie the even one
    q = Fraction(float(a[i])) * Fraction(float(b[i])) + Fraction(float(c[i]))
    d = abs(q - Fraction(float(got[i])))
    for nb in (up[i], down[i]):
      dn = abs(q - Fraction(float(nb)))
      assert d < dn or (d == dn and got[i].view(np.uint32) % 2 == 0), (a[i], b[i], c[i], got[i])
    if i % 997 == 0:
      assert got[i].view(np.uint32) == _fma_exact(a[i], b[i], c[i]).view(np.uint32)


def test_fma32_ties_cancellation_and_subnormals():
  one = F32(1.0)
  ulp = np.spacing(one)                      # 2^-23
  # exact halfway between 1 and 1 + ulp: the tie goes to even (1); a tie above an odd
  # significand goes up; a product a hair off the tie decides it
  a = np.array([one + ulp, one + ulp, one + 2 * ulp, F32(3.0)], F32)
  b = np.array([one + ulp, F32(1.0), F32(1.0), F32(1 / 3)], F32)
  c = np.array([-(one + 2 * ulp), ulp / 2, ulp / 2, F32(-1.0)], F32)
  _check_fma(a, b, c)
  # (1 + 2^-12)^2 = 1 + 2^-11 + 2^-24: a tie in fp32 only through the product
  x = F32(1 + 2.0 ** -12)
  _check_fma(np.array([x, x, -x], F32), np.array([x, x, x], F32), np.array([0.0, ulp / 2, 0.0], F32))
  # products that cancel c exactly: the zero's sign
  v = F32(1.5)
  a = np.array([v, -v, v, F32(0.0), F32(-0.0), F32(0.0)], F32)
  b = np.array([F32(2.0), F32(2.0), F32(-2.0), F32(5.0), F32(5.0), F32(-5.0)], F32)
  c = np.array([F32(-3.0), F32(3.0), F32(3.0), F32(-0.0), F32(-0.0), F32(-0.0)], F32)
  got = sr.fma32(a, b, c)
  assert [bool(np.signbit(g)) for g in got] == [False, False, False, False, True, True]
  _check_fma(a, b, c)
  # subnormal results, and a product below the fp32 range rounded against c
  tiny = F32(2.0 ** -126)
  a = np.array([tiny, tiny, F32(2.0 ** -100), F32(3.0 * 2 ** -75)], F32)
  b = np.array([F32(0.75), F32(-0.5), F32(2.0 ** -45), F32(2.0 ** -75)], F32)
  c = np.array([F32(0.0), tiny, F32(2.0 ** -149), F32(-(2.0 ** -149))], F32)
  _check_fma(a, b, c)
  assert sr.fma32(a, b, c)[0] == F32(0.75) * tiny


def _bar(A, xn, xe, rn, re_):
  """tests/test_algdist_gpu.py's reference bar: |d - d_ref| <= 1e-5 d_ref + 1e-6 sqrt(R)."""
  R = rn.shape[1]
  d, dr = incidence_distances(A, xn, xe), incidence_distances(A, rn, re_)
  assert (np.abs(d - dr) / (1e-5 * dr + 1e-6 * np.sqrt(R))).max() <= 1.0


@pytest.mark.parametrize("name", ["tiny", "rand25", "youtube"])
def test_restatement_computes_the_reference_relaxation_on_the_goldens(name):
  from oracle import port
  g = load_golden("algdist_" + name)
  r = np.searchsorted(g["node_ids"], g["pairs"][:, 0])
  c = np.searchsorted(g["edge_ids"], g["pairs"][:, 1])
  A = csr_from_pairs(np.stack([r, c], 1), shape=(len(g["node_ids"]), len(g["edge_ids"])))
  R, iters = int(g["dim"]), int(g["iters"])
  rng = np.random.default_rng(R)
  xn0 = rng.random((A.shape[0], R)).astype(F32)
  xe0 = rng.random((A.shape[1], R)).astype(F32)
  xn, xe, lohi = sr.relax(sr.Incidence.from_csr(A), xn0, xe0, iters)
  rn, re_ = port.algdist_vectorised(A, A.T.tocsr(), xn0, xe0, iters)
  _bar(A, xn, xe, rn, re_)
  assert lohi.shape == (iters, 2, R) and (lohi[:, 0] < lohi[:, 1]).all()


@pytest.mark.parametrize("edge_path", ["untiled", ("tiled", 700), ("sharded", 3)])
def test_restatement_with_multi_chunk_rows_against_the_port(edge_path):
  """Long rows of 3000 and 2500 incidences on both sides (3 chunks at the defaults, 94 at
  chunk = 32) and signed inputs, on each edge-half path."""
  from oracle import port
  rng = np.random.default_rng(3)
  n, e = 3000, 2500
  rows = np.concatenate([np.arange(n), rng.integers(0, n, 6000), np.zeros(e, int)])
  cols = np.concatenate([np.zeros(n, int), rng.integers(0, e, 6000), np.arange(e)])
  A = csr_from_pairs(np.stack([rows, cols], 1), shape=(n, e))
  inc = sr.Incidence.from_csr(A)
  for R, light, chunk in ((3, 128, 1024), (33, 8, 32)):
    xn0 = (rng.random((n, R)) * 2 - 1).astype(F32)
    xe0 = (rng.random((e, R)) * 2 - 1).astype(F32)
    xn, xe, _ = sr.relax(inc, xn0, xe0, 6, light_max=light, chunk=chunk, edge_path=edge_path)
    rn, re_ = port.algdist_vectorised(A, A.T.tocsr(), xn0, xe0, 6)
    _bar(A, xn, xe, rn, re_)


# ---- the bookkeeping, one row at a time ---------------------------------------------------------

def _seq(vals):
  s = F32(0.0)
  for v in vals:
    s = F32(s + v)
  return s


def _one_row(vals, light_max, chunk, G):
  """row_sums of a single row whose incidences gather the scalar rows `vals` in order."""
  Y = np.asarray(vals, F32)[:, None]
  idx = np.arange(len(vals))
  return sr.row_sums([0], [len(vals)], idx, Y, light_max, chunk, G)[0, 0]


def _order_sensitive(n, rng):
  """Values whose fp32 sum depends on the order: large and tiny magnitudes mixed."""
  return (rng.standard_normal(n) * 10.0 ** rng.integers(-4, 5, n)).astype(F32)


@pytest.mark.parametrize("deg", [3, 4, 7, 8])
def test_light_rows_add_in_csr_order(deg):
  """A light row's sum is its gathered rows added one at a time in CSR order.  The restatement
  has no own slot to model: k_stream_light puts the row itself in slot steps * 4 - 1 and k_sweep
  does not add it, so where that slot falls (degrees 3, 4, 7, 8) only shows on the device --
  tests/test_sweep_exact_gpu.py runs rows of those degrees on both sides."""
  rng = np.random.default_rng(deg)
  for _ in range(50):
    v = _order_sensitive(deg, rng)
    assert _one_row(v, 128, 1024, 4).view(np.uint32) == _seq(v).view(np.uint32)
  # a row whose order shows: 1 + 2^-24 + 2^-24 is 1 in order, 1 + 2^-23 the other way round
  v = np.array([1.0, 2.0 ** -24, 2.0 ** -24], F32)
  assert _one_row(v, 128, 1024, 8) == F32(1.0) and _seq(v[::-1]) == F32(1.0 + 2.0 ** -23)


def test_one_chunk_goes_to_groups_in_quads_and_through_the_butterfly():
  """G = 4: incidence j is summed by group (j // 4) % 4; the chunk's sum is
  ((s0 + s1) + (s2 + s3)), not a sequential sum."""
  rng = np.random.default_rng(1)
  hits = 0
  for _ in range(200):
    v = _order_sensitive(40, rng)
    groups = [_seq([v[j] for j in range(40) if (j // 4) % 4 == g]) for g in range(4)]
    want = F32(F32(groups[0] + groups[1]) + F32(groups[2] + groups[3]))
    got = _one_row(v, 8, 64, 4)
    assert got.view(np.uint32) == want.view(np.uint32)
    hits += got != _seq(v)
  assert hits > 20       # the grouping is visible in the last bits


def test_multi_chunk_row_with_more_chunks_than_groups():
  """chunk = 32, G = 2, 7 chunks: group g Kahan-sums chunks g, g + 2, ... in increasing order,
  then tot - comp, then the butterfly."""
  rng = np.random.default_rng(2)
  G, chunk = 2, 32

  def chunk_sum(c):
    g = [_seq([c[j] for j in range(len(c)) if (j // 4) % G == k]) for k in range(G)]
    return F32(g[0] + g[1])

  for _ in range(100):
    v = _order_sensitive(7 * chunk - 5, rng)
    sums = [chunk_sum(v[k * chunk:(k + 1) * chunk]) for k in range(7)]
    tots = []
    for g in range(G):
      s, c = F32(0.0), F32(0.0)
      for k in range(g, 7, G):
        y = F32(sums[k] - c)
        t = F32(s + y)
        c = F32(F32(t - s) - y)
        s = t
      tots.append(F32(s - c))
    want = F32(tots[0] + tots[1])
    assert _one_row(v, 1, chunk, G).view(np.uint32) == want.view(np.uint32)
  # the compensation matters: chunk sums 1, then 16 of 2^-24 each lost in a plain sum
  sums_row = np.concatenate([[1.0], np.zeros(chunk - 1), np.tile(np.r_[2.0 ** -24, np.zeros(chunk - 1)], 16)])
  got = _one_row(sums_row.astype(F32), 1, chunk, 1)
  assert got == F32(1.0 + 16 * 2.0 ** -24) and _seq(sums_row.astype(F32)) == F32(1.0)


def test_tile_boundary_inside_a_member_list():
  """One edge whose members straddle a tile boundary: the raw sum is the sum of the two
  sub-range sums, each summed on its own, not one sequential sum."""
  N, E = 8, 1
  A = csr_from_pairs(np.array([[n, 0] for n in range(N)]), shape=(N, E))
  inc = sr.Incidence.from_csr(A)
  st = sr.Relaxation(inc, 1, edge_path=("tiled", 3))
  assert st.tile_pos[:, 0].tolist() == [0, 3, 6, 8]
  yn = np.array([1.0, 0.0, 0.0, 2.0 ** -24, 2.0 ** -24, 0.0, 0.5, 2.0 ** -24], F32)[:, None]
  raw = np.zeros((1, 1), F32)
  for t in range(3):
    raw = raw + sr.row_sums(st.tile_pos[t], st.tile_pos[t + 1], inc.e_idx, yn, 128, 1024, 1)
  parts = [_seq(yn[0:3, 0]), _seq(yn[3:6, 0]), _seq(yn[6:8, 0])]
  assert raw[0, 0].view(np.uint32) == F32(F32(parts[0] + parts[1]) + parts[2]).view(np.uint32)
  # 1 + 2^-24 + 2^-24 is 1 in one sequential sum; the second tile adds its 2^-23 at once
  # and the third tile's 0.5 + 2^-24 lands on a tie that rounds up
  assert raw[0, 0] == F32(1.5 + 2.0 ** -22) and _seq(yn[:, 0]) == F32(1.5)


def test_edge_finalize_and_store_follow_the_compiled_contractions():
  """k_edge_finalize at sweep 0 is 0.5 * fma(y, deg, raw * invs) (own never rounded alone),
  later sweeps 0.5 * fma(raw, invs, fma(inv, y * deg, -lo * inv)); k_store_rows with a map is
  fma(y, deg, -lo) / (hi - lo).  Inputs where each contraction shows in the result."""
  rng = np.random.default_rng(4)
  n = 20000
  deg = rng.integers(1, 5000, n)
  y = rng.random((n, 1)).astype(F32) / deg[:, None].astype(F32)
  raw = rng.random((n, 1)).astype(F32)
  invs = rng.random(n).astype(F32)
  x0, _ = sr.edge_finalize(deg, invs, y, raw, None)
  plain = F32(0.5) * (y * deg[:, None].astype(F32) + raw * invs[:, None])
  assert (x0 != plain).any() and (x0 == plain).mean() > 0.5
  lo, hi = np.array([-0.3], F32), np.array([1.7], F32)
  x1, _ = sr.edge_finalize(deg, invs, y, raw, (lo, hi))
  inv = F32(1) / (hi - lo)
  own = sr.fma32(inv, y * deg[:, None].astype(F32), -lo * inv)
  assert np.array_equal(x1, F32(0.5) * sr.fma32(raw, invs[:, None], own))
  inc = sr.Incidence.from_csr(csr_from_pairs(np.array([[0, 0], [1, 0], [1, 1]]), shape=(2, 2)))
  st = sr.Relaxation(inc, 1)
  st.yn = rng.random((2, 1)).astype(F32) / 3
  st.ye = rng.random((2, 1)).astype(F32) / 3
  st.mm = [np.stack([sr.enc(lo), sr.enc(hi)])]
  xn, _ = st.store(1)
  degf = inc.n_deg.astype(F32)[:, None]
  assert np.array_equal(xn, sr.fma32(st.yn, degf, -lo) / (hi - lo))


def test_weight_sums_follow_the_kernel_order():
  """k_row_wsum (8 lanes, xor 4 2 1) and k_row_wsum_long (1000 and 3000 incidences) against a
  direct restatement of the same order, and against fsum to within rounding."""
  import math
  rng = np.random.default_rng(5)
  other = rng.integers(1, 10 ** 6, 5000)
  lens = [1, 7, 8, 9, 512, 513, 1000, 3000]
  ptr = np.concatenate([[0], np.cumsum(lens)])
  idx = rng.integers(0, len(other), ptr[-1])
  got = sr.weight_sums(ptr, idx, other)
  for r, L in enumerate(lens):
    w = 1.0 / other[idx[ptr[r]:ptr[r + 1]]].astype(np.float64)
    assert abs(got[r] - math.fsum(w)) <= 1e-15 * math.fsum(w) * L
    if L <= 512:
      lane = [0.0] * 8
      for p in range(L):
        lane[p % 8] = lane[p % 8] + w[p]
      for off in (4, 2, 1):
        lane = [lane[i] + lane[i ^ off] for i in range(8)]
      assert got[r] == lane[0]
