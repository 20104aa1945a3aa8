"""O1 — NumPy float64 restatement of GeneralGNN forward, backward and optimizers
(TEST INFRASTRUCTURE; the numerical truth tolerances are measured against).

Reference call sites: /root/reference/src/scripts/gcn.py:320 (model), :326,:335 (loss),
:321-325,:338 (SGD + PiecewiseConstantDecay), :334,:351 (training / inference calls).
Upstream algorithms restated (SURVEY.md §8 a2-a11; parity unpinned, see oracle/__init__):

  GeneralGNN.call   out = pre(x); for conv: z = conv([out, a]); out = concat([z, out]);
                    out = pool(out, i); out = post(out)
  MLP layer         Dense -> BatchNormalization -> Dropout -> PReLU | final activation
  GeneralConv.call  x.W + b -> BatchNormalization -> Dropout -> PReLU -> propagate:
                    out[t] = sum_{(t,s) in a.indices} x[s]   (values of ``a`` never read)
  BatchNormalization(momentum=.99, eps=1e-3), training: biased two-pass moments,
                    y = h*inv + (beta - mean*inv), inv = gamma*rsqrt(var+eps);
                    moving -= (moving - batch) * (1 - momentum); inference: moving stats
  Dropout           with keep mask m and scale s = (float32)(1 / (1 - rate)): act(m * s * z); the statistics
                    are those of h, and the last post block's dropout acts on the logits
  PReLU             f(z) = relu(z) - alpha*relu(-z), alpha per channel; d/dz at z == 0 is 0
  pool='sum'        segment_sum(out, i)
  pool='avg'        GlobalAvgPool: tf.math.segment_mean(out, i), 0 for an empty graph
  pool='attn_sum'   GlobalAttnSumPool: s = out . attn_kernel, p = unsorted_segment_softmax(s, i)
                    = exp(s - max_g) / (sum_g exp(s - max_g) + 1e-9), pooled[g] = sum_{n in g} p_n out_n
                    (attn_kernel [Wc, 1] follows the last block in the flat trainable buffer)
  pool=None         node-level output: the post-MLP runs on every node row
  CategoricalCrossentropy on softmax output (Keras recovers the logits):
                    loss = mean_b( logsumexp(z_b) * sum(y_b) - y_b . z_b )
  categorical_accuracy   mean(argmax(y) == argmax(p))
  BinaryCrossentropy on sigmoid output: l = max(z, 0) - z*y + log1p(exp(-|z|)), mean over the columns, then
                    the rows; binary_accuracy = mean(y == (sigmoid(z) > 0.5))
  linear head, e = z - y: MSE e^2, MAE |e|, Huber 0.5 e^2 if |e| <= delta else delta |e| - 0.5 delta^2, mean
                    over the columns, then the rows; metric mean |e|
  sample_weight     loss = sum_r w_r l_r / rows, metric = sum_r w_r m_r / sum_r w_r (0 when sum w = 0),
                    dLoss/dz_r = w_r * (the unweighted dLoss/dz_r)
"""
from __future__ import annotations

import numpy as np


class Block:
    """Parameters of one dense block as float64 arrays."""

    def __init__(self, spec, w, s):
        f = np.float64
        self.spec = spec
        o, n = spec.kernel
        self.W = w[o:o + n].astype(f).reshape(spec.k_in, spec.m_out)
        o, n = spec.bias
        self.b = w[o:o + n].astype(f)
        o, n = spec.gamma
        self.gamma = w[o:o + n].astype(f)
        o, n = spec.beta
        self.beta = w[o:o + n].astype(f)
        o, n = spec.alpha
        self.alpha = w[o:o + n].astype(f) if n else None
        o, n = spec.moving_mean
        self.mm = s[o:o + n].astype(f)
        o, n = spec.moving_variance
        self.mv = s[o:o + n].astype(f)


def _block_fwd(blk, x, training, eps, mask=None, scale=1.0):
    """One dense block; ``mask`` (bool [rows, width]) applies dropout with ``scale`` between BatchNorm and PReLU."""
    h = x @ blk.W + blk.b
    if training:
        mean = h.mean(0)
        var = ((h - mean) ** 2).mean(0)
    else:
        mean, var = blk.mm, blk.mv
    rstd = 1.0 / np.sqrt(var + eps)
    inv = blk.gamma * rstd
    z = h * inv + (blk.beta - mean * inv)
    zd = z if mask is None else np.where(mask, z * scale, 0.0)
    a = np.where(zd > 0, zd, blk.alpha * zd) if blk.alpha is not None else zd
    return a, dict(x=x, h=h, mean=mean, var=var, rstd=rstd, z=z, zd=zd, m=mask, s=scale)


def _block_bwd(blk, c, da, grads, need_dx=True, branch=None):
    """Training-mode backward of one block; writes into the flat ``grads``.  ``branch`` (int8 [rows, width]: 1 / -1 / 0)
    overrides the side of PReLU's kink every element is differentiated on - see loss_and_grads."""
    sp_ = blk.spec
    zd, m = c["zd"], c["m"]
    if blk.alpha is not None:
        side = np.sign(zd) if branch is None else (branch if m is None else np.where(m, branch, 0))
        slope = np.where(side > 0, 1.0, np.where(side < 0, blk.alpha, 0.0))
        dz = da * slope
        o, n = sp_.alpha
        grads[o:o + n] = (da * np.minimum(zd, 0.0)).sum(0)
    else:
        dz = da
    if m is not None:
        dz = np.where(m, dz * c["s"], 0.0)
    xhat = (c["h"] - c["mean"]) * c["rstd"]
    dgamma = (dz * xhat).sum(0)
    dbeta = dz.sum(0)
    n_rows = dz.shape[0]
    dh = blk.gamma * c["rstd"] * (dz - dbeta / n_rows - xhat * (dgamma / n_rows))
    for (o, n), v in ((sp_.gamma, dgamma), (sp_.beta, dbeta), (sp_.kernel, (c["x"].T @ dh).reshape(-1)), (sp_.bias, dh.sum(0))):
        grads[o:o + n] = v
    return dh @ blk.W.T if need_dx else None


def spmm_sum(rows, cols, x, n):
    """out[t] = sum over entries (t, s) of x[s] — tf.gather + unsorted_segment_sum."""
    out = np.zeros((n, x.shape[1]), dtype=x.dtype)
    np.add.at(out, rows, x[cols])
    return out


def aggregate(rows, cols, x, n, agg="sum", w=None):
    """spektral.layers.ops scatter_sum / scatter_mean / scatter_max over messages w_ij * x[j] (SURVEY.md §8 f3):
    tf.math.unsorted_segment_{sum,mean,max}(messages, targets, n).  An empty row gives 0 (sum, mean) or the lowest
    float (max).  Returns (out, ctx) with what the gradient needs."""
    msg = x[cols] if w is None else x[cols] * w[:, None]
    if agg == "sum":
        out = np.zeros((n, x.shape[1]), dtype=x.dtype)
        np.add.at(out, rows, msg)
        return out, None
    cnt = np.bincount(rows, minlength=n).astype(x.dtype)
    if agg == "mean":
        out = np.zeros((n, x.shape[1]), dtype=x.dtype)
        np.add.at(out, rows, msg)
        return out / np.maximum(cnt, 1.0)[:, None], cnt
    assert agg == "max"
    out = np.full((n, x.shape[1]), np.finfo(np.float32).min, dtype=x.dtype)
    np.maximum.at(out, rows, msg)
    return out, msg


def aggregate_bwd(rows, cols, dz, n, agg="sum", w=None, ctx=None, z=None):
    """Gradient of ``aggregate`` with respect to x.  max: tf's _UnsortedSegmentMinOrMaxGrad - the entries that attain a
    row's maximum share its gradient equally."""
    g = dz[rows]
    if agg == "mean":
        g = g / np.maximum(ctx, 1.0)[rows][:, None]
    if agg == "max":
        sel = (ctx == z[rows]).astype(dz.dtype)
        num = np.zeros_like(dz)
        np.add.at(num, rows, sel)
        g = sel * g / np.maximum(num, 1.0)[rows]
    if w is not None:
        g = g * w[:, None]
    out = np.zeros((n, dz.shape[1]), dtype=dz.dtype)
    np.add.at(out, cols, g)
    return out


def segment_sum(x, seg, n_seg):
    out = np.zeros((n_seg, x.shape[1]), dtype=x.dtype)
    np.add.at(out, seg, x)
    return out


def segment_mean(x, seg, n_seg):
    cnt = np.bincount(seg, minlength=n_seg).astype(x.dtype)
    return segment_sum(x, seg, n_seg) / np.maximum(cnt, 1.0)[:, None]


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
    out = segment_sum(p[:, None] * x, seg, n_seg)
    return out, dict(p=p, out=out, scores=sc)


def attn_sum_pool_bwd(x, a, seg, dout, ctx):
    """-> (dX, d attn_kernel) with u_g = out_g . dOut_g: ds_n = p_n (X_n . dOut_g - u_g), dX_n = p_n dOut_g + ds_n a,
    da = sum_n ds_n X_n."""
    p, out = ctx["p"], ctx["out"]
    dn = dout[seg]
    u = (out * dout).sum(1)
    ds = p * ((x * dn).sum(1) - u[seg])
    return p[:, None] * dn + ds[:, None] * a[None, :], ds @ x


def dropout_scale(rate):
    """Keras Dropout's 1 / (1 - rate), rounded to float32 from the float32 rate the C config holds."""
    return float(np.float32(1.0 / (1.0 - float(np.float32(rate)))))


def forward(cfg, specs, w, s, x, rows, cols, seg, n_graphs, training=False, edge_weight=None, masks=None, rate=0.0):
    """Returns (output [rows, C] after the head's activation, ctx).  ``edge_weight``: optional per-entry weights (the
    reference's unfinished ``use_edge_data`` switch); GeneralConv itself ignores adjacency values.  ``masks``: one keep
    mask per dense block (dropout at ``rate``), or None.  ctx holds logits, node_out, pool_ctx, blocks and caches."""
    blocks = [Block(sp_, w, s) for sp_ in specs]
    P, L = cfg.pre_process, cfg.message_passing
    n = x.shape[0]
    ew = None if edge_weight is None else np.asarray(edge_weight, dtype=np.float64)
    masks = masks if masks is not None else [None] * len(blocks)
    scale = dropout_scale(rate)
    caches = []

    def block(bi, inp):
        a, c = _block_fwd(blocks[bi], inp, training, cfg.bn_epsilon, masks[bi], scale)
        caches.append(c)
        return a

    out = np.asarray(x, dtype=np.float64)
    for bi in range(P):
        out = block(bi, out)
    for bi in range(P, P + L):
        a = block(bi, out)
        c = caches[-1]
        z, c["agg_ctx"] = aggregate(rows, cols, a, n, cfg.aggregate, ew)
        c["agg_out"] = z
        # Concatenate()([z, out]) | Add()([z, out]) | no skip connection (GeneralGNN.call)
        out = np.concatenate([z, out], axis=1) if cfg.connectivity == "cat" else (z + out if cfg.connectivity == "sum" else z)
    node_out, pool_ctx = out, None
    if cfg.pool == "sum":
        out = segment_sum(out, seg, n_graphs)
    elif cfg.pool == "avg":
        out = segment_mean(out, seg, n_graphs)
    elif cfg.pool == "attn_sum":
        o, k = pool_kernel_range(specs)
        out, pool_ctx = attn_sum_pool(out, w[o:o + k].astype(np.float64), seg, n_graphs)
    for bi in range(P + L, len(blocks)):
        out = block(bi, out)
    logits = out
    if cfg.activation == "softmax":
        e = np.exp(logits - logits.max(1, keepdims=True))
        out = e / e.sum(1, keepdims=True)
    elif cfg.activation == "sigmoid":
        out = sigmoid(logits)
    return out, dict(blocks=blocks, caches=caches, logits=logits, node_out=node_out, pool_ctx=pool_ctx)


def backward(cfg, specs, w, ctx, dlogits, x, rows, cols, seg, n_graphs, prelu_branch=None, edge_weight=None):
    """float64 gradient of the flat trainable buffer from dLoss/dlogits."""
    blocks, caches = ctx["blocks"], ctx["caches"]
    grads = np.zeros(w.shape[0], dtype=np.float64)
    P, L, H = cfg.pre_process, cfg.message_passing, cfg.hidden
    br = prelu_branch if prelu_branch is not None else [None] * len(blocks)
    ew = None if edge_weight is None else np.asarray(edge_weight, dtype=np.float64)
    d = dlogits
    for bi in range(len(blocks) - 1, P + L - 1, -1):
        d = _block_bwd(blocks[bi], caches[bi], d, grads, branch=br[bi])
    if cfg.pool is None:
        dout = d                                        # the post-MLP's input gradient is dLoss/d(node output)
    elif cfg.pool == "attn_sum":
        o, k = pool_kernel_range(specs)
        dout, grads[o:o + k] = attn_sum_pool_bwd(ctx["node_out"], w[o:o + k].astype(np.float64), seg, d, ctx["pool_ctx"])
    elif cfg.pool == "avg":
        dout = (d / np.maximum(np.bincount(seg, minlength=n_graphs), 1.0)[:, None])[seg]
    else:
        dout = d[seg]                                   # grad of segment_sum
    for bi in range(P + L - 1, P - 1, -1):
        if cfg.connectivity == "cat":
            dz, dprev = dout[:, :H], dout[:, H:]
        else:                                           # Add: the gradient reaches both operands; None: only z
            dz, dprev = dout, (dout if cfg.connectivity == "sum" else 0.0)
        da = aggregate_bwd(rows, cols, dz, x.shape[0], cfg.aggregate, ew, caches[bi]["agg_ctx"], caches[bi]["agg_out"])
        dout = dprev + _block_bwd(blocks[bi], caches[bi], da, grads, branch=br[bi])
    for bi in range(P - 1, -1, -1):
        dout = _block_bwd(blocks[bi], caches[bi], dout, grads, need_dx=bi > 0, branch=br[bi])
    return grads


def xent_from_logits(logits, y):
    m = logits.max(1, keepdims=True)
    lse = (m + np.log(np.exp(logits - m).sum(1, keepdims=True)))[:, 0]
    per = lse * y.sum(1) - (y * logits).sum(1)
    return per.mean(), per


def accuracy(probs, y):
    return float((probs.argmax(1) == y.argmax(1)).mean())


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


HEADS = ("softmax", "sigmoid") + LOSSES


def activation(head):
    return head if head in ("softmax", "sigmoid") else None


def head_of(cfg, loss=None):
    """The head a config trains: its activation's, or the loss on a linear head (MSE by default)."""
    return cfg.activation if cfg.activation in ("softmax", "sigmoid") else (loss or "mse")


def row_terms(head, z, y, delta=1.0):
    """float64 (l [rows], m [rows], d [rows, C]): row loss, row metric and the unweighted dl_r/dz (no 1/rows)."""
    z = np.asarray(z, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    C = z.shape[1]
    if head == "softmax":
        e = np.exp(z - z.max(axis=1, keepdims=True))
        p = e / e.sum(axis=1, keepdims=True)
        hit = (y.argmax(axis=1) == z.argmax(axis=1)).astype(np.float64)
        return xent_from_logits(z, y)[1], hit, p * y.sum(axis=1, keepdims=True) - y
    if head == "sigmoid":
        p = sigmoid(z)
        l = (np.maximum(z, 0.0) - z * y + np.log1p(np.exp(-np.abs(z)))).mean(axis=1)
        return l, binary_accuracy(y, p), (p - y) / C
    e = z - y
    return element_loss(head, e, delta).mean(axis=1), np.abs(e).mean(axis=1), element_grad(head, e, delta) / C


def weighted_loss(head, z, y, w=None, delta=1.0, grad_scale=None):
    """float64 (loss, metric, dlogits) of the head on logits z, weighted by ``w`` (None: unweighted); grad_scale
    defaults to 1 / rows."""
    l, m, d = row_terms(head, z, y, delta)
    rows = l.shape[0]
    scale = (1.0 / rows if rows else 0.0) if grad_scale is None else grad_scale
    if w is None:
        return float(l.mean()), float(m.mean()), d * scale
    w = np.asarray(w, dtype=np.float64).reshape(-1)
    loss = float((w * l).sum() / rows) if rows else 0.0
    metric = float((w * m).sum() / w.sum()) if w.sum() != 0 else 0.0
    return loss, metric, d * w[:, None] * scale


def _new_state(cfg, s, ctx):
    """Flat float64 moving statistics after a training-mode forward."""
    new_state = np.asarray(s, dtype=np.float64).copy()
    for blk, c in zip(ctx["blocks"], ctx["caches"]):
        for rng, old, batch in ((blk.spec.moving_mean, blk.mm, c["mean"]), (blk.spec.moving_variance, blk.mv, c["var"])):
            o, n = rng
            new_state[o:o + n] = old - (old - batch) * (1.0 - cfg.bn_momentum)
    return new_state


def loss_and_grads(cfg, specs, w, s, x, rows, cols, seg, y, n_graphs, *, loss=None, delta=1.0, sample_weight=None,
                   grad_scale=None, masks=None, rate=0.0, prelu_branch=None, edge_weight=None):
    """One training-mode forward + backward.  Returns dict(loss, metric (also under acc, the key this function has
    always returned the accuracy under), probs (the output after the head's activation), logits, dlogits, grads (flat
    float64, same layout as w), new_state (flat float64 moving statistics), ctx).  ``loss``: 'mse' | 'mae' | 'huber'
    (with ``delta``) on a linear head; ``grad_scale`` replaces 1/rows, e.g. 1/global_rows for one data-parallel shard;
    ``masks`` / ``rate``: dropout, see forward.

    ``prelu_branch``: optional list (one entry per block, None for blocks without PReLU) of int8 arrays giving the
    branch of PReLU (1: z > 0, -1: z < 0, 0: z == 0) another implementation differentiated each element on.  PReLU's
    derivative jumps at 0, so an input within float32 rounding of 0 may land on either side in a float32
    implementation; with the branches pinned the comparison measures arithmetic error only.  ``ctx['prelu_flips']``
    counts the elements whose pinned branch differs from the float64 sign."""
    probs, ctx = forward(cfg, specs, w, s, x, rows, cols, seg, n_graphs, training=True, edge_weight=edge_weight,
                         masks=masks, rate=rate)
    logits = ctx["logits"]
    lval, metric, d = weighted_loss(head_of(cfg, loss), logits, y, sample_weight, delta, grad_scale)
    br = prelu_branch if prelu_branch is not None else [None] * len(ctx["blocks"])
    ctx["prelu_flips"] = sum(int((np.sign(c["z"]) != b).sum())
                             for blk, c, b in zip(ctx["blocks"], ctx["caches"], br) if b is not None and blk.alpha is not None)
    grads = backward(cfg, specs, w, ctx, d, x, rows, cols, seg, n_graphs, prelu_branch, edge_weight)
    return dict(loss=lval, metric=metric, acc=metric, probs=probs, logits=logits, dlogits=d, grads=grads,
                new_state=_new_state(cfg, s, ctx), ctx=ctx)


def loss_at(cfg, specs, w, s, x, rows, cols, seg, y, n_graphs, *, loss=None, delta=1.0, sample_weight=None, masks=None,
            rate=0.0, edge_weight=None):
    """The float64 loss of the training-mode forward at parameters w (for finite differences)."""
    _, ctx = forward(cfg, specs, w, s, x, rows, cols, seg, n_graphs, training=True, edge_weight=edge_weight, masks=masks,
                     rate=rate)
    return weighted_loss(head_of(cfg, loss), ctx["logits"], y, sample_weight, delta)[0]


def piecewise_constant(step, boundaries, values):
    """tf.keras.optimizers.schedules.PiecewiseConstantDecay: values[0] for step <=
    boundaries[0], values[k] for boundaries[k-1] < step <= boundaries[k], else values[-1]."""
    for b, v in zip(boundaries, values):
        if step <= b:
            return v
    return values[-1]


def sgd_step(w, g, lr):
    """Keras SGD without momentum (gcn.py:325): w <- w - lr * g."""
    return w - lr * g


def adam_step(w, g, m, v, t, lr, beta1=0.9, beta2=0.999, eps=1e-7):
    """Keras Adam (epsilon outside the bias-corrected root), t = 1-based step."""
    m = beta1 * m + (1 - beta1) * g
    v = beta2 * v + (1 - beta2) * g * g
    lr_t = lr * np.sqrt(1 - beta2 ** t) / (1 - beta1 ** t)
    return w - lr_t * m / (np.sqrt(v) + eps), m, v
