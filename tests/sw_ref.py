"""Reference restatements of the sample-weighted losses (TEST INFRASTRUCTURE): Keras' ``loss(y, pred, sample_weight=w)``
with the default "sum_over_batch_size" reduction for every head the library trains, and the weighted train step.

With l_r the row loss of the head (softmax cross-entropy; the mean over the C columns for binary cross-entropy and the
regression losses) and m_r the row metric (categorical accuracy, binary accuracy, mean absolute error):
  loss   = sum_r w_r l_r / rows          metric = sum_r w_r m_r / sum_r w_r (0 when sum w = 0)
  dLoss/dz_r = w_r * (the unweighted dLoss/dz_r)

The model part is that of reg_ref (float64, hand-derived backward) and bce_ref.torch_logits (float32 autograd) on the
linear form of the config: every head has the same parameter layout and the same logits, only the loss differs.
"""
from __future__ import annotations

import dataclasses

import numpy as np

import bce_ref
import pool_ref
import reg_ref

HEADS = ("softmax", "sigmoid", "mse", "mae", "huber")


def activation(head):
    return head if head in ("softmax", "sigmoid") else None


def row_terms(head, z, y, delta=1.0):
    """float64 (l [rows], m [rows], d [rows, C]): row loss, row metric and the unweighted dl_r/dz (no 1/rows)."""
    z = np.asarray(z, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    C = z.shape[1]
    if head == "softmax":
        m = z.max(axis=1, keepdims=True)
        e = np.exp(z - m)
        lse = m[:, 0] + np.log(e.sum(axis=1))
        p = e / e.sum(axis=1, keepdims=True)
        ysum = y.sum(axis=1)
        l = lse * ysum - (y * z).sum(axis=1)
        hit = (y.argmax(axis=1) == z.argmax(axis=1)).astype(np.float64)
        return l, hit, p * ysum[:, None] - y
    if head == "sigmoid":
        p = bce_ref.sigmoid(z)
        l = (np.maximum(z, 0.0) - z * y + np.log1p(np.exp(-np.abs(z)))).mean(axis=1)
        return l, bce_ref.binary_accuracy(y, p), (p - y) / C
    e = z - y
    return (reg_ref.element_loss(head, e, delta).mean(axis=1), np.abs(e).mean(axis=1),
            reg_ref.element_grad(head, e, delta) / C)


def weighted_loss(head, z, y, w, delta=1.0, grad_scale=None):
    """float64 (loss, metric, dlogits) of the weighted head on logits z (grad_scale defaults to 1 / rows)."""
    w = np.asarray(w, dtype=np.float64).reshape(-1)
    l, m, d = row_terms(head, z, y, delta)
    rows = l.shape[0]
    scale = (1.0 / rows if rows else 0.0) if grad_scale is None else grad_scale
    loss = float((w * l).sum() / rows) if rows else 0.0
    metric = float((w * m).sum() / w.sum()) if w.sum() != 0 else 0.0
    return loss, metric, d * w[:, None] * scale


def linear_cfg(cfg):
    return dataclasses.replace(cfg, activation=None)


def loss_and_grads(cfg, specs, w, s, x, rows, cols, seg, y, n_graphs, sw, head, delta=1.0, grad_scale=None,
                   prelu_branch=None):
    """float64 weighted train step: dict(loss, metric, logits, dlogits, grads)."""
    lin = linear_cfg(cfg)
    z, ctx = reg_ref.forward(lin, specs, w, s, x, rows, cols, seg, n_graphs, training=True)
    loss, metric, d = weighted_loss(head, z, y, sw, delta, grad_scale)
    grads = reg_ref.backward(lin, specs, w, ctx, d, x, rows, cols, seg, n_graphs, prelu_branch)
    return dict(loss=loss, metric=metric, logits=z, dlogits=d, grads=grads)


def loss_at(cfg, specs, w, s, x, rows, cols, seg, y, n_graphs, sw, head, delta=1.0):
    """The float64 weighted loss of a training-mode forward at parameters w (for finite differences)."""
    z, _ = reg_ref.forward(linear_cfg(cfg), specs, w, s, x, rows, cols, seg, n_graphs, training=True)
    return weighted_loss(head, z, y, sw, delta)[0]


def torch_loss_and_grads(cfg, specs, w, s, x, rows, cols, seg, y, n_graphs, sw, head, delta=1.0):
    """The same step in float32 autograd: dict(loss, grads)."""
    import torch
    import torch.nn.functional as F
    z, params, attn = bce_ref.torch_logits(linear_cfg(cfg), specs, w, s, x, rows, cols, seg, n_graphs, True, [])
    yt = torch.tensor(np.asarray(y, dtype=np.float32))
    wt = torch.tensor(np.asarray(sw, dtype=np.float32).reshape(-1))
    if head == "softmax":
        l = torch.logsumexp(z, dim=1) * yt.sum(dim=1) - (yt * z).sum(dim=1)
    elif head == "sigmoid":
        l = F.binary_cross_entropy_with_logits(z, yt, reduction="none").mean(dim=1)
    elif head == "mse":
        l = F.mse_loss(z, yt, reduction="none").mean(dim=1)
    elif head == "mae":
        l = F.l1_loss(z, yt, reduction="none").mean(dim=1)
    else:
        l = F.huber_loss(z, yt, reduction="none", delta=delta).mean(dim=1)
    loss = (wt * l).sum() / z.shape[0]
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
    return dict(loss=float(loss.detach()), grads=grads)


def roc_curve(y, score, sw):
    """scikit-learn's roc_curve(y, score, sample_weight=sw, drop_intermediate=False) in NumPy float64: zero weights
    dropped, weighted cumulative true / false positives at each distinct threshold."""
    y, score, sw = (np.asarray(a, dtype=np.float64).reshape(-1) for a in (y, score, sw))
    keep = sw != 0
    y, score, sw = y[keep], score[keep], sw[keep]
    order = np.argsort(-score, kind="stable")
    y, score, sw = y[order], score[order], sw[order]
    idx = np.r_[np.nonzero(np.diff(score))[0], y.size - 1]
    tps = np.cumsum(y * sw)[idx]
    fps = np.cumsum((1 - y) * sw)[idx]
    tps, fps = np.r_[0.0, tps], np.r_[0.0, fps]
    return fps / fps[-1], tps / tps[-1], np.r_[np.inf, score[idx]]
