"""Numpy restatement of the seeded parts of device-resident hypergraph2vec training
(csrc/hge_hg2v_train.cu): the epoch order of hge_shuffle_order and the initial tables of
hge_hg2v_create_seeded.  Both read Philox4x32-10 word streams in the layout of the device sampler
(csrc/hge_philox.cuh, restated in oracle/device_sampler_ref.py): key = the seed, counter =
{block, item lo, item hi, phase}, words read in order, four per counter block.

Test infrastructure only.
"""
import numpy as np

from oracle.device_sampler_ref import MASK, philox4x32_10

# phases of csrc/hge_philox.cuh (HgePhase) beyond the sampler's
PHASE = dict(SHUFFLE=12, INIT_NODES=13, INIT_EDGES=14)


def _key(seed):
  seed = int(seed) & 0xFFFFFFFFFFFFFFFF
  return np.uint64(seed & 0xFFFFFFFF), np.uint64(seed >> 32)


def shuffle_order(seed, epoch, n):
  """hge_shuffle_order: item i's key is (word 2e << 32) | word 2e + 1 of its SHUFFLE stream; the
  order is the stable argsort of the keys."""
  items = np.arange(int(n), dtype=np.uint64)
  w = philox4x32_10((np.uint64(epoch // 2), items & MASK, items >> np.uint64(32), np.uint64(PHASE["SHUFFLE"])),
                    _key(seed))
  j = 2 * (int(epoch) % 2)
  keys = (w[j] << np.uint64(32)) | w[j + 1]
  return np.argsort(keys, kind="stable").astype(np.int32)


def init_table(seed, phase, rows, dim):
  """hge_hg2v_create_seeded's table of `rows` x `dim`: element (r, c) = -0.05 + 0.1 * ((word c of
  row r's stream) >> 8) * 2^-24, every operation in float32."""
  r = np.arange(int(rows), dtype=np.uint64)
  cols = []
  for b in range((int(dim) + 3) // 4):
    cols += philox4x32_10((np.uint64(b), r & MASK, r >> np.uint64(32), np.uint64(phase)), _key(seed))
  w = np.stack(cols[:int(dim)], axis=1) if dim else np.zeros((int(rows), 0), np.uint64)
  u = (w >> np.uint64(8)).astype(np.float32) * np.float32(2.0**-24)
  return np.float32(-0.05) + np.float32(0.1) * u
