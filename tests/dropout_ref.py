"""The dropout mask stream of csrc/dropout.cuh in NumPy (TEST INFRASTRUCTURE); the float64 model that applies the masks
is oracle.model_ref_np (forward / loss_and_grads with ``masks`` and ``rate``).

Mask stream (the data format csrc/dropout.cuh defines; this file is its only other statement):
  u    = word (col & 3) of Philox4x32-10(ctr = (col >> 2, row, block, step lo32), key = (seed lo32, seed hi32))
  keep = u >= t,  t = (uint32) min(floor(rate * 2^32), 2^32 - 1),  scale = (float32)(1 / (1 - rate))
with rate the float32 value the C config holds, widened to double.
"""
from __future__ import annotations

import numpy as np

M32 = 0xFFFFFFFF
PHILOX_M0, PHILOX_M1 = 0xD2511F53, 0xCD9E8D57
PHILOX_W0, PHILOX_W1 = 0x9E3779B9, 0xBB67AE85


def philox4x32_10(ctr, key):
    """Random123 Philox4x32-10, vectorised: ctr a tuple of four uint32 arrays (broadcastable), key a pair of uint32
    scalars.  Returns the four uint32 output words."""
    c0, c1, c2, c3 = (np.asarray(v, dtype=np.uint64) & M32 for v in ctr)
    k0, k1 = int(key[0]) & M32, int(key[1]) & M32
    for r in range(10):
        if r:
            k0, k1 = (k0 + PHILOX_W0) & M32, (k1 + PHILOX_W1) & M32
        p0 = np.uint64(PHILOX_M0) * c0
        p1 = np.uint64(PHILOX_M1) * c2
        hi0, lo0 = p0 >> np.uint64(32), p0 & np.uint64(M32)
        hi1, lo1 = p1 >> np.uint64(32), p1 & np.uint64(M32)
        c0, c1, c2, c3 = hi1 ^ c1 ^ np.uint64(k0), lo1, hi0 ^ c3 ^ np.uint64(k1), lo0
    return tuple(v.astype(np.uint32) for v in (c0, c1, c2, c3))


def threshold(rate):
    r = float(np.float32(rate))
    return int(min(np.floor(r * 2.0 ** 32), 2.0 ** 32 - 1))


def scale(rate):
    return np.float32(1.0 / (1.0 - float(np.float32(rate))))


def keep_mask(seed, step, block, rows, cols, rate):
    """bool [rows, cols]: the keep mask of dense block ``block`` in step ``step``."""
    r = np.arange(rows, dtype=np.uint64)[:, None]
    c = np.arange(cols, dtype=np.uint64)[None, :]
    seed = int(seed) & ((1 << 64) - 1)
    words = philox4x32_10((c >> np.uint64(2), r, np.full_like(r, block), np.full_like(r, int(step) & M32)),
                          (seed & M32, seed >> 32))
    w = np.broadcast_to(c & np.uint64(3), (rows, cols))
    u = np.choose(w.astype(np.int64), [np.broadcast_to(x, (rows, cols)) for x in words])
    return u >= np.uint32(threshold(rate)) if threshold(rate) else np.ones((rows, cols), dtype=bool)


def model_masks(specs, cfg, n_nodes, rows_post, rate, seed, step):
    """One keep mask per dense block, in block order (node-level blocks [n_nodes, m_out], post blocks [rows_post, .])."""
    P, L = cfg.pre_process, cfg.message_passing
    return [keep_mask(seed, step, bi, n_nodes if bi < P + L else rows_post, sp_.m_out, rate) for bi, sp_ in enumerate(specs)]
