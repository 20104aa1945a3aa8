"""Reference restatements of GeneralGNN(dropout=rate) (TEST INFRASTRUCTURE): the mask stream of csrc/dropout.cuh in
NumPy, and the float64 training-mode forward and backward with given masks for every pool, connectivity, aggregation,
edge weights and head, built on the oracle's aggregation and pool functions, which stay as they are.

Mask stream (the data format csrc/dropout.cuh defines; this file is its only other statement):
  u    = word (col & 3) of Philox4x32-10(ctr = (col >> 2, row, block, step lo32), key = (seed lo32, seed hi32))
  keep = u >= t,  t = (uint32) min(floor(rate * 2^32), 2^32 - 1),  scale = (float32)(1 / (1 - rate))
with rate the float32 value the C config holds, widened to double.

Every dense block is Dense -> BatchNormalization -> Dropout -> activation (the last post block too: its dropout acts on
the logits).  With m the keep mask and s the scale, the block output is act(m * s * z), z = bn(h); BatchNorm statistics
are those of h.  Backward: dz = m * s * act'(m * s * z) * da, dalpha = sum da * min(m * s * z, 0).
"""
from __future__ import annotations

import numpy as np

from oracle import model_ref_np as O1

import pool_ref
import sw_ref

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


# ---------------------------------------------------------------- float64 model with given masks
def _block_fwd(blk, x, eps, m, s):
    h = x @ blk.W + blk.b
    mean = h.mean(0)
    var = ((h - mean) ** 2).mean(0)
    rstd = 1.0 / np.sqrt(var + eps)
    inv = blk.gamma * rstd
    z = h * inv + (blk.beta - mean * inv)
    zd = np.where(m, z * s, 0.0)
    a = np.where(zd > 0, zd, blk.alpha * zd) if blk.alpha is not None else zd
    return a, dict(x=x, h=h, mean=mean, var=var, rstd=rstd, z=z, zd=zd, m=m, s=s)


def _block_bwd(blk, c, da, grads, need_dx=True, branch=None):
    sp_ = blk.spec
    zd, m, s = c["zd"], c["m"], c["s"]
    if blk.alpha is not None:
        side = np.sign(zd) if branch is None else np.where(m, branch, 0)
        slope = np.where(side > 0, 1.0, np.where(side < 0, blk.alpha, 0.0))
        dzd = da * slope
        o, n = sp_.alpha
        grads[o:o + n] = (da * np.minimum(zd, 0.0)).sum(0)
    else:
        dzd = da
    dz = np.where(m, dzd * s, 0.0)
    xhat = (c["h"] - c["mean"]) * c["rstd"]
    dgamma = (dz * xhat).sum(0)
    dbeta = dz.sum(0)
    n_rows = dz.shape[0]
    dh = blk.gamma * c["rstd"] * (dz - dbeta / n_rows - xhat * (dgamma / n_rows))
    for rng, v in ((sp_.gamma, dgamma), (sp_.beta, dbeta), (sp_.kernel, (c["x"].T @ dh).reshape(-1)), (sp_.bias, dh.sum(0))):
        grads[rng[0]:rng[0] + rng[1]] = v
    return dh @ blk.W.T if need_dx else None


def forward(cfg, specs, w, s, x, rows, cols, seg, n_graphs, masks, rate, edge_weight=None):
    """Training-mode forward with the keep masks ``masks`` (model_masks): (logits [rows_post, C], ctx)."""
    blocks = [O1.Block(sp_, w, s) for sp_ in specs]
    P, L = cfg.pre_process, cfg.message_passing
    sc = float(scale(rate)) if threshold(rate) else 1.0
    n = x.shape[0]
    ew = None if edge_weight is None else np.asarray(edge_weight, dtype=np.float64)
    caches = []
    out = np.asarray(x, dtype=np.float64)
    for bi in range(P):
        out, c = _block_fwd(blocks[bi], out, cfg.bn_epsilon, masks[bi], sc)
        caches.append(c)
    for bi in range(P, P + L):
        a, c = _block_fwd(blocks[bi], out, cfg.bn_epsilon, masks[bi], sc)
        caches.append(c)
        z, c["agg_ctx"] = O1.aggregate(rows, cols, a, n, cfg.aggregate, ew)
        c["agg_out"] = z
        out = np.concatenate([z, out], axis=1) if cfg.connectivity == "cat" else (z + out if cfg.connectivity == "sum" else z)
    node_out, pool_ctx = out, None
    if cfg.pool == "sum":
        out = O1.segment_sum(out, seg, n_graphs)
    elif cfg.pool == "avg":
        out = pool_ref.segment_mean(out, seg, n_graphs)
    elif cfg.pool == "attn_sum":
        o, k = pool_ref.pool_kernel_range(specs)
        out, pool_ctx = pool_ref.attn_sum_pool(out, w[o:o + k].astype(np.float64), seg, n_graphs)
    for bi in range(P + L, len(blocks)):
        out, c = _block_fwd(blocks[bi], out, cfg.bn_epsilon, masks[bi], sc)
        caches.append(c)
    return out, dict(blocks=blocks, caches=caches, node_out=node_out, pool_ctx=pool_ctx)


def backward(cfg, specs, w, ctx, d, x, rows, cols, seg, n_graphs, prelu_branch=None, edge_weight=None):
    """float64 gradient of the flat trainable buffer from dLoss/dlogits ``d``."""
    blocks, caches = ctx["blocks"], ctx["caches"]
    grads = np.zeros(w.shape[0], dtype=np.float64)
    P, L, H = cfg.pre_process, cfg.message_passing, cfg.hidden
    br = prelu_branch if prelu_branch is not None else [None] * len(blocks)
    ew = None if edge_weight is None else np.asarray(edge_weight, dtype=np.float64)
    for bi in range(len(blocks) - 1, P + L - 1, -1):
        d = _block_bwd(blocks[bi], caches[bi], d, grads, branch=br[bi])
    if cfg.pool is None:
        dout = d
    elif cfg.pool == "attn_sum":
        o, k = pool_ref.pool_kernel_range(specs)
        dout, grads[o:o + k] = pool_ref.attn_sum_pool_bwd(ctx["node_out"], w[o:o + k].astype(np.float64), seg, d,
                                                          ctx["pool_ctx"])
    elif cfg.pool == "avg":
        dout = (d / np.maximum(np.bincount(seg, minlength=n_graphs), 1.0)[:, None])[seg]
    else:
        dout = d[seg]
    for k in range(L - 1, -1, -1):
        bi = P + k
        if cfg.connectivity == "cat":
            dz, dprev = dout[:, :H], dout[:, H:]
        else:
            dz, dprev = dout, (dout if cfg.connectivity == "sum" else 0.0)
        da = O1.aggregate_bwd(rows, cols, dz, x.shape[0], cfg.aggregate, ew, caches[bi]["agg_ctx"], caches[bi]["agg_out"])
        dout = dprev + _block_bwd(blocks[bi], caches[bi], da, grads, branch=br[bi])
    for bi in range(P - 1, -1, -1):
        dout = _block_bwd(blocks[bi], caches[bi], dout, grads, need_dx=bi > 0, branch=br[bi])
    return grads


def head(cfg, loss):
    """The sw_ref head name of a config and a loss name (None: the head's own)."""
    return cfg.activation if cfg.activation in ("softmax", "sigmoid") else (loss or "mse")


def loss_and_grads(cfg, specs, w, s, x, rows, cols, seg, y, n_graphs, masks, rate, loss=None, sw=None, delta=1.0,
                   prelu_branch=None, edge_weight=None):
    """float64 train step with the given masks: dict(loss, metric, logits, grads, new_state)."""
    z, ctx = forward(cfg, specs, w, s, x, rows, cols, seg, n_graphs, masks, rate, edge_weight)
    weights = np.ones(z.shape[0]) if sw is None else sw
    lval, metric, d = sw_ref.weighted_loss(head(cfg, loss), z, y, weights, delta)
    grads = backward(cfg, specs, w, ctx, d, x, rows, cols, seg, n_graphs, prelu_branch, edge_weight)
    new_state = s.astype(np.float64).copy()
    for blk, c in zip(ctx["blocks"], ctx["caches"]):
        o, n = blk.spec.moving_mean
        new_state[o:o + n] = blk.mm - (blk.mm - c["mean"]) * (1.0 - cfg.bn_momentum)
        o, n = blk.spec.moving_variance
        new_state[o:o + n] = blk.mv - (blk.mv - c["var"]) * (1.0 - cfg.bn_momentum)
    return dict(loss=lval, metric=metric, logits=z, grads=grads, new_state=new_state)


def loss_at(cfg, specs, w, s, x, rows, cols, seg, y, n_graphs, masks, rate, loss=None, sw=None, delta=1.0,
            edge_weight=None):
    """The float64 loss of the training-mode forward at parameters w with fixed masks (for finite differences)."""
    z, _ = forward(cfg, specs, w, s, x, rows, cols, seg, n_graphs, masks, rate, edge_weight)
    weights = np.ones(z.shape[0]) if sw is None else sw
    return sw_ref.weighted_loss(head(cfg, loss), z, y, weights, delta)[0]
