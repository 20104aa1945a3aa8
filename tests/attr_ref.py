"""float64 restatement of the attribution backward (gradients with respect to the node features x and the per-entry
edge weights), hand-derived on top of oracle/model_ref_np: the same forward, the same pool and aggregation backward,
and per dense block either the training-mode BatchNorm backward (batch statistics) or the inference-mode one (moving
statistics: dh = gamma * rsqrt(mv + eps) * slope(z) * da).

Edge weights w_e of the stored entries e = (i, j), messages w_e * a[j] (a = the conv block's output activation):
  sum  dw_e = dZ[i] . a[j]        mean  the same / (entries of row i)
  max  sum over the columns where w_e * a[j, c] attains Z[i, c] of dZ[i, c] a[j, c] / ties[i, c]
summed over the L GeneralConv layers.  Output gradients of the model output: softmax p * (d - p . d), sigmoid
d * p (1 - p), linear d (output_grad)."""
from __future__ import annotations

import numpy as np

from oracle import model_ref_np as O1


def output_grad(activation, probs, d):
    """dlogits = J^T d of the head's activation on its output ``probs``."""
    p = np.asarray(probs, dtype=np.float64)
    d = np.asarray(d, dtype=np.float64)
    if activation == "softmax":
        return p * (d - (p * d).sum(1, keepdims=True))
    if activation == "sigmoid":
        return d * p * (1.0 - p)
    return d


def _frozen_bwd(blk, c, da, branch=None):
    """Inference-mode backward of one block to its input: moving statistics, no parameter gradients."""
    zd = c["zd"]
    if blk.alpha is not None:
        side = np.sign(zd) if branch is None else branch
        dz = da * np.where(side > 0, 1.0, np.where(side < 0, blk.alpha, 0.0))
    else:
        dz = da
    return (dz * blk.gamma * c["rstd"]) @ blk.W.T


def _block_dx(blk, c, da, training, branch, scratch):
    if training:                                    # the parameter gradients go to scratch
        return O1._block_bwd(blk, c, da, scratch, branch=branch)
    return _frozen_bwd(blk, c, da, branch)


def _act(blk, c):
    zd = c["zd"]
    return np.where(zd > 0, zd, blk.alpha * zd) if blk.alpha is not None else zd


def _edge_grad(cfg, rows, cols, n, a, dz, ew, c):
    g = (dz[rows] * a[cols])
    if cfg.aggregate == "mean":
        g = g / np.maximum(c["agg_ctx"], 1.0)[rows][:, None]
    elif cfg.aggregate == "max":
        msg, z = c["agg_ctx"], c["agg_out"]
        sel = (msg == z[rows]).astype(np.float64)
        num = np.zeros_like(dz)
        np.add.at(num, rows, sel)
        g = sel * g / np.maximum(num, 1.0)[rows]
    return g.sum(1)


def input_grads(cfg, specs, w, s, x, rows, cols, seg, n_graphs, dlogits, *, training=False, edge_weight=None,
                masks=None, rate=0.0, prelu_branch=None):
    """float64 (dx [N, F], d edge_weight [nnz] or None) of <dlogits, logits> for the forward of ``training`` mode
    (masks / rate: dropout, training mode only).  ``prelu_branch`` pins PReLU's kink side as in
    model_ref_np.loss_and_grads."""
    _, ctx = O1.forward(cfg, specs, w, s, x, rows, cols, seg, n_graphs, training=training, edge_weight=edge_weight,
                        masks=masks, rate=rate)
    return input_grads_from(cfg, specs, w, ctx, np.asarray(x, dtype=np.float64), rows, cols, seg, n_graphs, dlogits,
                            training=training, edge_weight=edge_weight, prelu_branch=prelu_branch)


def input_grads_from(cfg, specs, w, ctx, x, rows, cols, seg, n_graphs, dlogits, *, training, edge_weight=None,
                     prelu_branch=None):
    blocks, caches = ctx["blocks"], ctx["caches"]
    P, L, H = cfg.pre_process, cfg.message_passing, cfg.hidden
    br = prelu_branch if prelu_branch is not None else [None] * len(blocks)
    ew = None if edge_weight is None else np.asarray(edge_weight, dtype=np.float64)
    n = x.shape[0]
    scratch = np.zeros(np.asarray(w).shape[0])
    d = np.asarray(dlogits, dtype=np.float64)
    for bi in range(len(blocks) - 1, P + L - 1, -1):
        d = _block_dx(blocks[bi], caches[bi], d, training, br[bi], scratch)
    if cfg.pool is None:
        dout = d
    elif cfg.pool == "attn_sum":
        o, k = O1.pool_kernel_range(specs)
        dout, _ = O1.attn_sum_pool_bwd(ctx["node_out"], w[o:o + k].astype(np.float64), seg, d, ctx["pool_ctx"])
    elif cfg.pool == "avg":
        dout = (d / np.maximum(np.bincount(seg, minlength=n_graphs), 1.0)[:, None])[seg]
    else:
        dout = d[seg]
    dew = None if ew is None else np.zeros(ew.shape[0])
    for bi in range(P + L - 1, P - 1, -1):
        if cfg.connectivity == "cat":
            dz, dprev = dout[:, :H], dout[:, H:]
        else:
            dz, dprev = dout, (dout if cfg.connectivity == "sum" else 0.0)
        c = caches[bi]
        if dew is not None:
            dew += _edge_grad(cfg, rows, cols, n, _act(blocks[bi], c), dz, ew, c)
        da = O1.aggregate_bwd(rows, cols, dz, n, cfg.aggregate, ew, c["agg_ctx"], c["agg_out"])
        dout = dprev + _block_dx(blocks[bi], c, da, training, br[bi], scratch)
    for bi in range(P - 1, -1, -1):
        dout = _block_dx(blocks[bi], caches[bi], dout, training, br[bi], scratch)
    return dout, dew


def calibrated_state(cfg, specs, w, s, x, rows, cols, seg, n_graphs, edge_weight=None):
    """Moving statistics equal to the batch statistics of a training-mode forward (float32, flat): the inference model
    then sees normalised activations, as a trained model does, instead of the scale of freshly initialised ones."""
    _, ctx = O1.forward(cfg, specs, w, s, x, rows, cols, seg, n_graphs, training=True, edge_weight=edge_weight)
    out = np.asarray(s, dtype=np.float32).copy()
    for blk, c in zip(ctx["blocks"], ctx["caches"]):
        for (o, n), v in ((blk.spec.moving_mean, c["mean"]), (blk.spec.moving_variance, c["var"])):
            out[o:o + n] = v
    return out


def objective(cfg, specs, w, s, x, rows, cols, seg, n_graphs, dlogits, *, training=False, edge_weight=None, masks=None,
              rate=0.0):
    """<dlogits, logits> in float64: the scalar whose gradient input_grads returns (finite differences)."""
    _, ctx = O1.forward(cfg, specs, w, s, x, rows, cols, seg, n_graphs, training=training, edge_weight=edge_weight,
                        masks=masks, rate=rate)
    return float((ctx["logits"] * dlogits).sum())
