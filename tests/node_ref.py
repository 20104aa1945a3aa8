"""Reference restatements of GeneralGNN with pool=None (TEST INFRASTRUCTURE): the node-level train step, built on the
oracle's dense-block, aggregation and loss functions, which stay as they are.

Without a pool the post-MLP runs on every node row and the loss is the mean categorical cross-entropy over the N node
rows of the batch (Spektral's node-level mode: y [N, C] = np.vstack of the graphs' node labels).

``forward`` / ``loss_and_grads``: float64 NumPy with the hand-derived backward (the counterpart of
oracle.model_ref_np); ``torch_loss_and_grads``: float32 PyTorch-CPU autograd (the counterpart of oracle.model_ref_torch).
"""
from __future__ import annotations

import numpy as np

from oracle import model_ref_np as O1
from oracle import model_ref_torch as O2


def forward(cfg, specs, w, s, x, rows, cols, training=False):
    """Node-level output [N, C] (probabilities with activation='softmax'), and the cache of the backward."""
    assert cfg.pool is None
    blocks = [O1.Block(sp_, w, s) for sp_ in specs]
    P, L = cfg.pre_process, cfg.message_passing
    n = x.shape[0]
    caches = []
    out = x.astype(np.float64)
    for blk in blocks[:P]:
        out, c = O1._block_fwd(blk, out, training, cfg.bn_epsilon)
        caches.append(c)
    for blk in blocks[P:P + L]:
        a, c = O1._block_fwd(blk, out, training, cfg.bn_epsilon)
        caches.append(c)
        z, c["agg_ctx"] = O1.aggregate(rows, cols, a, n, cfg.aggregate)
        c["agg_out"] = z
        out = np.concatenate([z, out], axis=1) if cfg.connectivity == "cat" else (z + out if cfg.connectivity == "sum" else z)
    for blk in blocks[P + L:]:
        out, c = O1._block_fwd(blk, out, training, cfg.bn_epsilon)
        caches.append(c)
    logits = out
    if cfg.activation == "softmax":
        e = np.exp(logits - logits.max(1, keepdims=True))
        out = e / e.sum(1, keepdims=True)
    return out, dict(blocks=blocks, caches=caches, logits=logits)


def loss_and_grads(cfg, specs, w, s, x, rows, cols, y, prelu_branch=None, grad_scale=None):
    """float64 train step: dict(loss, acc, probs, grads, new_state, ctx).  The gradient is that of the mean loss over
    the N rows (``grad_scale`` replaces 1/N, e.g. 1/global_N for one data-parallel shard)."""
    assert cfg.activation == "softmax" and cfg.pool is None
    y = y.astype(np.float64)
    probs, ctx = forward(cfg, specs, w, s, x, rows, cols, training=True)
    blocks, caches, logits = ctx["blocks"], ctx["caches"], ctx["logits"]
    loss, _ = O1.xent_from_logits(logits, y)
    grads = np.zeros(w.shape[0], dtype=np.float64)
    scale = 1.0 / logits.shape[0] if grad_scale is None else grad_scale
    d = (probs * y.sum(1, keepdims=True) - y) * scale
    P, L, H = cfg.pre_process, cfg.message_passing, cfg.hidden
    br = prelu_branch if prelu_branch is not None else [None] * len(blocks)
    flips = 0
    for bi, (blk, c) in enumerate(zip(blocks, caches)):
        if br[bi] is not None and blk.alpha is not None:
            flips += int((np.sign(c["z"]) != br[bi]).sum())
    ctx["prelu_flips"] = flips
    for bi in range(len(blocks) - 1, P + L - 1, -1):
        d = O1._block_bwd(blocks[bi], caches[bi], d, grads, branch=br[bi])
    dout = d                                   # no pool: the post-MLP's input gradient is dLoss/d(node output)
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
    new_state = s.astype(np.float64).copy()
    mom = cfg.bn_momentum
    for blk, c in zip(blocks, caches):
        o, n = blk.spec.moving_mean
        new_state[o:o + n] = blk.mm - (blk.mm - c["mean"]) * (1.0 - mom)
        o, n = blk.spec.moving_variance
        new_state[o:o + n] = blk.mv - (blk.mv - c["var"]) * (1.0 - mom)
    return dict(loss=float(loss), acc=O1.accuracy(probs, y), probs=probs, grads=grads, new_state=new_state, ctx=ctx)


def torch_loss_and_grads(cfg, specs, w, s, x, rows, cols, y):
    """The same train step in float32 PyTorch autograd."""
    import torch
    assert cfg.pool is None
    params = O2.unpack(specs, w, s)
    xt = torch.tensor(np.asarray(x, dtype=np.float32))
    rt, ct = (torch.tensor(np.asarray(v, dtype=np.int64)) for v in (rows, cols))
    yt = torch.tensor(np.asarray(y, dtype=np.float32))
    P, L = cfg.pre_process, cfg.message_passing
    stats = []
    out = xt
    for p in params[:P]:
        out = O2._block(p, out, True, cfg.bn_epsilon, stats)
    n = xt.shape[0]
    for p in params[P:P + L]:
        a = O2._block(p, out, True, cfg.bn_epsilon, stats)
        z = torch.zeros(n, a.shape[1], dtype=a.dtype).index_add_(0, rt, a[ct])
        out = torch.cat([z, out], dim=1) if cfg.connectivity == "cat" else (z + out if cfg.connectivity == "sum" else z)
    for p in params[P + L:]:
        out = O2._block(p, out, True, cfg.bn_epsilon, stats)
    logits = out
    loss = -(yt * torch.log_softmax(logits, dim=1)).sum(1).mean()
    loss.backward()
    grads = np.zeros(w.shape[0], dtype=np.float32)
    for p in params:
        sp_ = p["spec"]
        for key, rng in (("W", sp_.kernel), ("b", sp_.bias), ("gamma", sp_.gamma), ("beta", sp_.beta), ("alpha", sp_.alpha)):
            o, k = rng
            if k:
                grads[o:o + k] = p[key].grad.reshape(-1).numpy()
    probs = torch.softmax(logits.detach(), dim=1).numpy()
    new_state = np.asarray(s, dtype=np.float32).copy()
    for p, (mean, var) in zip(params, stats):
        for rng, old, batch in ((p["spec"].moving_mean, p["mm"], mean), (p["spec"].moving_variance, p["mv"], var)):
            o, k = rng
            new_state[o:o + k] = (old - (old - batch) * (1.0 - cfg.bn_momentum)).numpy()
    return dict(loss=float(loss.detach()), probs=probs, grads=grads, stats=stats, new_state=new_state)
