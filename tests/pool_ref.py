"""Reference restatements of GeneralGNN with pool='avg' | 'attn_sum' (TEST INFRASTRUCTURE), built on the oracle's
dense-block, aggregation and loss functions, which stay as they are:

  pool='avg'       GlobalAvgPool: tf.math.segment_mean(out, i), 0 for an empty graph
  pool='attn_sum'  GlobalAttnSumPool: s = out . attn_kernel, p = unsorted_segment_softmax(s, i)
                   = exp(s - max_g) / (sum_g exp(s - max_g) + 1e-9), pooled[g] = sum_{n in g} p_n out_n
                   (attn_kernel [Wc, 1] follows the last block in the flat trainable buffer)

``forward`` / ``loss_and_grads``: float64 NumPy with the hand-derived backward (the counterpart of
oracle.model_ref_np); ``torch_loss_and_grads``: float32 PyTorch-CPU autograd (the counterpart of oracle.model_ref_torch).
Both also take pool='sum'.
"""
from __future__ import annotations

import numpy as np

from oracle import model_ref_np as O1
from oracle import model_ref_torch as O2


def segment_mean(x, seg, n_seg):
    cnt = np.bincount(seg, minlength=n_seg).astype(x.dtype)
    return O1.segment_sum(x, seg, n_seg) / np.maximum(cnt, 1.0)[:, None]


def pool_kernel_range(specs):
    """(offset, Wc) of pool.attn_kernel: right after the last block; Wc = input width of the first post block."""
    last = specs[-1]
    post0 = next(sp_ for sp_ in specs if sp_.name == "post.0")
    return last.offset + last.n_trainable, post0.k_in


def attn_sum_pool(x, a, seg, n_seg):
    """GlobalAttnSumPool in disjoint mode -> (pooled [B, W], ctx for attn_sum_pool_bwd)."""
    sc = x @ a
    mx = np.full(n_seg, -np.inf)
    np.maximum.at(mx, seg, sc)
    e = np.exp(sc - mx[seg])
    den = np.zeros(n_seg)
    np.add.at(den, seg, e)
    p = e / (den[seg] + 1e-9)
    out = O1.segment_sum(p[:, None] * x, seg, n_seg)
    return out, dict(p=p, out=out, scores=sc)


def attn_sum_pool_bwd(x, a, seg, dout, ctx):
    """-> (dX, d attn_kernel) with u_g = out_g . dOut_g: ds_n = p_n (X_n . dOut_g - u_g), dX_n = p_n dOut_g + ds_n a,
    da = sum_n ds_n X_n."""
    p, out = ctx["p"], ctx["out"]
    dn = dout[seg]
    u = (out * dout).sum(1)
    ds = p * ((x * dn).sum(1) - u[seg])
    return p[:, None] * dn + ds[:, None] * a[None, :], ds @ x


def forward(cfg, specs, w, s, x, rows, cols, seg, n_graphs, training=False):
    """O1.forward with the pool variants.  Returns (output [B, C], cache)."""
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
    node_out, pool_ctx = out, None
    if cfg.pool == "sum":
        out = O1.segment_sum(out, seg, n_graphs)
    elif cfg.pool == "avg":
        out = segment_mean(out, seg, n_graphs)
    elif cfg.pool == "attn_sum":
        o, k = pool_kernel_range(specs)
        out, pool_ctx = attn_sum_pool(out, w[o:o + k].astype(np.float64), seg, n_graphs)
    for blk in blocks[P + L:]:
        out, c = O1._block_fwd(blk, out, training, cfg.bn_epsilon)
        caches.append(c)
    logits = out
    if cfg.activation == "softmax":
        e = np.exp(logits - logits.max(1, keepdims=True))
        out = e / e.sum(1, keepdims=True)
    return out, dict(blocks=blocks, caches=caches, logits=logits, node_out=node_out, pool_ctx=pool_ctx)


def loss_and_grads(cfg, specs, w, s, x, rows, cols, seg, y, n_graphs, prelu_branch=None):
    """O1.loss_and_grads with the pool variants (no edge weights).  Same return dict."""
    assert cfg.activation == "softmax" and cfg.pool in ("sum", "avg", "attn_sum")
    y = y.astype(np.float64)
    probs, ctx = forward(cfg, specs, w, s, x, rows, cols, seg, n_graphs, training=True)
    blocks, caches, logits = ctx["blocks"], ctx["caches"], ctx["logits"]
    loss, _ = O1.xent_from_logits(logits, y)
    grads = np.zeros(w.shape[0], dtype=np.float64)
    d = (probs * y.sum(1, keepdims=True) - y) / logits.shape[0]
    P, L, H = cfg.pre_process, cfg.message_passing, cfg.hidden
    br = prelu_branch if prelu_branch is not None else [None] * len(blocks)
    flips = 0
    for bi, (blk, c) in enumerate(zip(blocks, caches)):
        if br[bi] is not None and blk.alpha is not None:
            flips += int((np.sign(c["z"]) != br[bi]).sum())
    ctx["prelu_flips"] = flips
    for bi in range(len(blocks) - 1, P + L - 1, -1):
        d = O1._block_bwd(blocks[bi], caches[bi], d, grads, branch=br[bi])
    if cfg.pool == "attn_sum":
        o, k = pool_kernel_range(specs)
        dout, grads[o:o + k] = attn_sum_pool_bwd(ctx["node_out"], w[o:o + k].astype(np.float64), seg, d, ctx["pool_ctx"])
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
    return dict(loss=float(loss), acc=O1.accuracy(probs, y), probs=probs, grads=grads, new_state=new_state, ctx=ctx)


def torch_loss_and_grads(cfg, specs, w, s, x, rows, cols, seg, y, n_graphs):
    """O2.loss_and_grads with the pool variants: float32 autograd, attn_kernel a leaf."""
    import torch
    params = O2.unpack(specs, w, s)
    xt = torch.tensor(np.asarray(x, dtype=np.float32))
    rt, ct, st = (torch.tensor(np.asarray(v, dtype=np.int64)) for v in (rows, cols, seg))
    yt = torch.tensor(np.asarray(y, dtype=np.float32))
    attn = None
    if cfg.pool == "attn_sum":
        ao, an = pool_kernel_range(specs)
        attn = torch.tensor(np.asarray(w[ao:ao + an], dtype=np.float32)).reshape(an, 1).requires_grad_(True)
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
    if cfg.pool in ("sum", "avg"):
        pooled = torch.zeros(n_graphs, out.shape[1], dtype=out.dtype).index_add_(0, st, out)
        if cfg.pool == "avg":
            pooled = pooled / torch.bincount(st, minlength=n_graphs).to(out.dtype).clamp(min=1.0)[:, None]
        out = pooled
    else:
        sc = (out @ attn)[:, 0]
        mx = torch.zeros(n_graphs, dtype=out.dtype).scatter_reduce_(0, st, sc.detach(), "amax", include_self=False)
        e = torch.exp(sc - mx[st])
        den = torch.zeros(n_graphs, dtype=out.dtype).index_add_(0, st, e)
        p = e / (den[st] + 1e-9)
        out = torch.zeros(n_graphs, out.shape[1], dtype=out.dtype).index_add_(0, st, p[:, None] * out)
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
    if attn is not None:
        grads[ao:ao + an] = attn.grad.reshape(-1).numpy()
    probs = torch.softmax(logits.detach(), dim=1).numpy()
    new_state = np.asarray(s, dtype=np.float32).copy()
    for p, (mean, var) in zip(params, stats):
        for rng, old, batch in ((p["spec"].moving_mean, p["mm"], mean), (p["spec"].moving_variance, p["mv"], var)):
            o, k = rng
            new_state[o:o + k] = (old - (old - batch) * (1.0 - cfg.bn_momentum)).numpy()
    return dict(loss=float(loss.detach()), probs=probs, grads=grads, stats=stats, new_state=new_state)
