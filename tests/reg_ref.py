"""Reference restatements of GeneralGNN(activation=None) trained with the Keras regression losses MeanSquaredError,
MeanAbsoluteError and Huber (TEST INFRASTRUCTURE), for the graph-level pools 'sum' / 'avg' / 'attn_sum' and for
node-level output (pool=None).  Built on pool_ref.forward and node_ref.forward (which return the logits for any
activation but softmax), bce_ref.torch_logits and the oracle's dense-block, aggregation and pool backward.

Keras semantics on the predictions z of a linear head, e = z - y:
  MSE    l = e^2                                                   dl/dz = 2e
  MAE    l = |e|                                                   dl/dz = sign(e), sign(0) = 0
  Huber  l = 0.5 e^2 if |e| <= delta, else delta |e| - 0.5 delta^2   dl/dz = e, or delta sign(e)
  loss = mean_b mean_c l[b, c]     mae = mean_b mean_c |e[b, c]|     dLoss/dz = dl/dz / (rows * C)

``forward`` / ``loss_and_grads``: float64 NumPy with the hand-derived backward; ``torch_loss_and_grads``: float32
PyTorch-CPU autograd with ``mse_loss``, ``l1_loss`` and ``huber_loss(delta=...)``.
"""
from __future__ import annotations

import numpy as np

from oracle import model_ref_np as O1

import bce_ref
import node_ref
import pool_ref

LOSSES = ("mse", "mae", "huber")


def element_loss(kind, e, delta=1.0):
    a = np.abs(e)
    if kind == "mse":
        return e * e
    if kind == "mae":
        return a
    return np.where(a <= delta, 0.5 * e * e, delta * a - 0.5 * delta * delta)


def element_grad(kind, e, delta=1.0):
    if kind == "mse":
        return 2.0 * e
    if kind == "mae":
        return np.sign(e)
    return np.where(np.abs(e) <= delta, e, delta * np.sign(e))


def regression_loss(kind, z, y, delta=1.0):
    """Mean over the columns, then the rows."""
    return float(element_loss(kind, np.asarray(z) - np.asarray(y), delta).mean(axis=-1).mean())


def mae(z, y):
    return float(np.abs(np.asarray(z) - np.asarray(y)).mean(axis=-1).mean())


def forward(cfg, specs, w, s, x, rows, cols, seg, n_graphs, training=False):
    """Output [rows, C] = the logits of the linear head, and the cache of the backward."""
    assert cfg.activation in (None, "linear")
    if cfg.pool is None:
        _, ctx = node_ref.forward(cfg, specs, w, s, x, rows, cols, training)
    else:
        _, ctx = pool_ref.forward(cfg, specs, w, s, x, rows, cols, seg, n_graphs, training)
    return ctx["logits"], ctx


def backward(cfg, specs, w, ctx, d, x, rows, cols, seg, n_graphs, prelu_branch=None):
    """float64 gradient of the flat trainable buffer from dLoss/dlogits ``d``."""
    blocks, caches = ctx["blocks"], ctx["caches"]
    grads = np.zeros(w.shape[0], dtype=np.float64)
    P, L, H = cfg.pre_process, cfg.message_passing, cfg.hidden
    br = prelu_branch if prelu_branch is not None else [None] * len(blocks)
    for bi in range(len(blocks) - 1, P + L - 1, -1):
        d = O1._block_bwd(blocks[bi], caches[bi], d, grads, branch=br[bi])
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
        da = O1.aggregate_bwd(rows, cols, dz, x.shape[0], cfg.aggregate, None, caches[bi]["agg_ctx"], caches[bi]["agg_out"])
        dout = dprev + O1._block_bwd(blocks[bi], caches[bi], da, grads, branch=br[bi])
    for bi in range(P - 1, -1, -1):
        dout = O1._block_bwd(blocks[bi], caches[bi], dout, grads, need_dx=bi > 0, branch=br[bi])
    return grads


def loss_and_grads(cfg, specs, w, s, x, rows, cols, seg, y, n_graphs, kind="mse", delta=1.0, prelu_branch=None,
                   grad_scale=None):
    """float64 train step: dict(loss, mae, pred, grads, new_state, ctx)."""
    y = np.asarray(y, dtype=np.float64)
    z, ctx = forward(cfg, specs, w, s, x, rows, cols, seg, n_graphs, training=True)
    n_rows, C = z.shape
    scale = 1.0 / n_rows if grad_scale is None else grad_scale
    d = element_grad(kind, z - y, delta) * scale / C
    grads = backward(cfg, specs, w, ctx, d, x, rows, cols, seg, n_graphs, prelu_branch)
    new_state = s.astype(np.float64).copy()
    mom = cfg.bn_momentum
    for blk, c in zip(ctx["blocks"], ctx["caches"]):
        o, n = blk.spec.moving_mean
        new_state[o:o + n] = blk.mm - (blk.mm - c["mean"]) * (1.0 - mom)
        o, n = blk.spec.moving_variance
        new_state[o:o + n] = blk.mv - (blk.mv - c["var"]) * (1.0 - mom)
    return dict(loss=regression_loss(kind, z, y, delta), mae=mae(z, y), pred=z, grads=grads, new_state=new_state,
                ctx=ctx)


def torch_loss(kind, z, y, delta=1.0):
    import torch.nn.functional as F
    if kind == "mse":
        return F.mse_loss(z, y)
    if kind == "mae":
        return F.l1_loss(z, y)
    return F.huber_loss(z, y, delta=delta)


def torch_loss_and_grads(cfg, specs, w, s, x, rows, cols, seg, y, n_graphs, kind="mse", delta=1.0):
    """The same train step in float32 autograd (pool.attn_kernel a leaf); the mean over every element equals the mean
    over the columns, then the rows."""
    import torch
    stats = []
    z, params, attn = bce_ref.torch_logits(cfg, specs, w, s, x, rows, cols, seg, n_graphs, True, stats)
    yt = torch.tensor(np.asarray(y, dtype=np.float32))
    loss = torch_loss(kind, z, yt, delta)
    loss.backward()
    grads = np.zeros(w.shape[0], dtype=np.float32)
    for p in params:
        sp_ = p["spec"]
        for key, rng in (("W", sp_.kernel), ("b", sp_.bias), ("gamma", sp_.gamma), ("beta", sp_.beta), ("alpha", sp_.alpha)):
            o, k = rng
            if k:
                grads[o:o + k] = p[key].grad.reshape(-1).numpy()
    if attn is not None:
        ao, an = pool_ref.pool_kernel_range(specs)
        grads[ao:ao + an] = attn.grad.reshape(-1).numpy()
    new_state = np.asarray(s, dtype=np.float32).copy()
    for p, (mean, var) in zip(params, stats):
        for rng, old, batch in ((p["spec"].moving_mean, p["mm"], mean), (p["spec"].moving_variance, p["mv"], var)):
            o, k = rng
            new_state[o:o + k] = (old - (old - batch) * (1.0 - cfg.bn_momentum)).numpy()
    return dict(loss=float(loss.detach()), pred=z.detach().numpy(), grads=grads, new_state=new_state)
