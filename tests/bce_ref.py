"""Reference restatements of GeneralGNN(activation='sigmoid') trained with BinaryCrossentropy (TEST INFRASTRUCTURE),
for the graph-level pools 'sum' / 'avg' / 'attn_sum' and for node-level output (pool=None).  Built on pool_ref.forward
and node_ref.forward (which return the logits for any activation but softmax) and on the oracle's dense-block,
aggregation and pool backward; those stay as they are.

Keras semantics (tf.keras.losses.BinaryCrossentropy on the logits z of a sigmoid output):
  l[b, c] = max(z, 0) - z*y + log1p(exp(-|z|))        loss = mean_b mean_c l[b, c]
  binary_accuracy = mean_b mean_c (y == (sigmoid(z) > 0.5))
  dLoss/dz = (sigmoid(z) - y) / (rows * C)             (grad_scale replaces 1 / rows)

``forward`` / ``loss_and_grads``: float64 NumPy with the hand-derived backward; ``torch_loss_and_grads``: float32
PyTorch-CPU autograd with ``binary_cross_entropy_with_logits``.
"""
from __future__ import annotations

import numpy as np

from oracle import model_ref_np as O1
from oracle import model_ref_torch as O2

import node_ref
import pool_ref


def sigmoid(z):
    e = np.exp(-np.abs(z))
    return np.where(z >= 0, 1.0 / (1.0 + e), e / (1.0 + e))


def bce_from_logits(z, y):
    """Mean over the columns, then the rows, of TF's sigmoid_cross_entropy_with_logits."""
    return float((np.maximum(z, 0.0) - z * y + np.log1p(np.exp(-np.abs(z)))).mean(axis=-1).mean())


def bce_from_probs(p, y, eps=1e-7):
    """Keras' fallback on probabilities of unknown origin: clip to [eps, 1 - eps], then -(y log(p+eps) + (1-y) log(1-p+eps))."""
    p = np.clip(p, eps, 1.0 - eps)
    return float((-(y * np.log(p + eps) + (1.0 - y) * np.log(1.0 - p + eps))).mean(axis=-1).mean())


def binary_accuracy(y, p, threshold=0.5):
    """Per-row mean over the columns of y == (p > threshold)."""
    return (np.asarray(y) == (np.asarray(p) > threshold).astype(np.asarray(p).dtype)).mean(axis=-1)


def forward(cfg, specs, w, s, x, rows, cols, seg, n_graphs, training=False):
    """Output [rows, C] = sigmoid(logits) and the cache of the backward (logits in cache['logits'])."""
    assert cfg.activation == "sigmoid"
    if cfg.pool is None:
        logits, ctx = node_ref.forward(cfg, specs, w, s, x, rows, cols, training)
    else:
        logits, ctx = pool_ref.forward(cfg, specs, w, s, x, rows, cols, seg, n_graphs, training)
    return sigmoid(ctx["logits"]), ctx


def loss_and_grads(cfg, specs, w, s, x, rows, cols, seg, y, n_graphs, prelu_branch=None, grad_scale=None):
    """float64 train step: dict(loss, acc, probs, grads, new_state, ctx)."""
    y = np.asarray(y, dtype=np.float64)
    probs, ctx = forward(cfg, specs, w, s, x, rows, cols, seg, n_graphs, training=True)
    blocks, caches, logits = ctx["blocks"], ctx["caches"], ctx["logits"]
    n_rows, C = logits.shape
    scale = 1.0 / n_rows if grad_scale is None else grad_scale
    d = (probs - y) * scale / C
    grads = np.zeros(w.shape[0], dtype=np.float64)
    P, L, H = cfg.pre_process, cfg.message_passing, cfg.hidden
    br = prelu_branch if prelu_branch is not None else [None] * len(blocks)
    flips = 0
    for bi, (blk, c) in enumerate(zip(blocks, caches)):
        if br[bi] is not None and blk.alpha is not None:
            flips += int((np.sign(c["z"]) != br[bi]).sum())
    ctx["prelu_flips"] = flips
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
    new_state = s.astype(np.float64).copy()
    mom = cfg.bn_momentum
    for blk, c in zip(blocks, caches):
        o, n = blk.spec.moving_mean
        new_state[o:o + n] = blk.mm - (blk.mm - c["mean"]) * (1.0 - mom)
        o, n = blk.spec.moving_variance
        new_state[o:o + n] = blk.mv - (blk.mv - c["var"]) * (1.0 - mom)
    return dict(loss=bce_from_logits(logits, y), acc=float(binary_accuracy(y, probs).mean()), probs=probs, grads=grads,
                new_state=new_state, ctx=ctx)


def torch_logits(cfg, specs, w, s, x, rows, cols, seg, n_graphs, training, stats=None, requires_grad=True):
    """float32 forward to the logits: (logits, params of O2.unpack, pool.attn_kernel leaf or None)."""
    import torch
    params = O2.unpack(specs, w, s, requires_grad=requires_grad)
    xt = torch.tensor(np.asarray(x, dtype=np.float32))
    rt, ct = (torch.tensor(np.asarray(v, dtype=np.int64)) for v in (rows, cols))
    st = torch.tensor(np.asarray(seg, dtype=np.int64)) if seg is not None else None
    attn = None
    if cfg.pool == "attn_sum":
        ao, an = pool_ref.pool_kernel_range(specs)
        attn = torch.tensor(np.asarray(w[ao:ao + an], dtype=np.float32)).reshape(an, 1).requires_grad_(requires_grad)
    P, L = cfg.pre_process, cfg.message_passing
    out = xt
    for p in params[:P]:
        out = O2._block(p, out, training, cfg.bn_epsilon, stats)
    n = xt.shape[0]
    for p in params[P:P + L]:
        a = O2._block(p, out, training, cfg.bn_epsilon, stats)
        z = torch.zeros(n, a.shape[1], dtype=a.dtype).index_add_(0, rt, a[ct])
        out = torch.cat([z, out], dim=1) if cfg.connectivity == "cat" else (z + out if cfg.connectivity == "sum" else z)
    if cfg.pool in ("sum", "avg"):
        pooled = torch.zeros(n_graphs, out.shape[1], dtype=out.dtype).index_add_(0, st, out)
        if cfg.pool == "avg":
            pooled = pooled / torch.bincount(st, minlength=n_graphs).to(out.dtype).clamp(min=1.0)[:, None]
        out = pooled
    elif cfg.pool == "attn_sum":
        sc = (out @ attn)[:, 0]
        mx = torch.zeros(n_graphs, dtype=out.dtype).scatter_reduce_(0, st, sc.detach(), "amax", include_self=False)
        e = torch.exp(sc - mx[st])
        den = torch.zeros(n_graphs, dtype=out.dtype).index_add_(0, st, e)
        p = e / (den[st] + 1e-9)
        out = torch.zeros(n_graphs, out.shape[1], dtype=out.dtype).index_add_(0, st, p[:, None] * out)
    for p in params[P + L:]:
        out = O2._block(p, out, training, cfg.bn_epsilon, stats)
    return out, params, attn


def torch_loss_and_grads(cfg, specs, w, s, x, rows, cols, seg, y, n_graphs):
    """The same train step in float32 autograd (pool.attn_kernel a leaf)."""
    import torch
    stats = []
    logits, params, attn = torch_logits(cfg, specs, w, s, x, rows, cols, seg, n_graphs, True, stats)
    yt = torch.tensor(np.asarray(y, dtype=np.float32))
    loss = torch.nn.functional.binary_cross_entropy_with_logits(logits, yt)      # mean over every element = mean_b mean_c
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
    probs = torch.sigmoid(logits.detach()).numpy()
    new_state = np.asarray(s, dtype=np.float32).copy()
    for p, (mean, var) in zip(params, stats):
        for rng, old, batch in ((p["spec"].moving_mean, p["mm"], mean), (p["spec"].moving_variance, p["mv"], var)):
            o, k = rng
            new_state[o:o + k] = (old - (old - batch) * (1.0 - cfg.bn_momentum)).numpy()
    return dict(loss=float(loss.detach()), probs=probs, grads=grads, stats=stats, new_state=new_state)
