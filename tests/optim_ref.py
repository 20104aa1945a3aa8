"""Reference restatements of the optimizer options (TEST INFRASTRUCTURE): Keras OptimizerV2 SGD with momentum and
Nesterov, Adam with amsgrad, and the clipping keywords clipvalue / clipnorm / global_clipnorm, in float64 NumPy.

Semantics [upstream, from memory], Keras OptimizerV2 of the TF 2.6-2.7 era:
- SGD with momentum (ResourceApplyKerasMomentum), slot `momentum`, initialised to zeros:
  accum = momentum*accum - lr*g; then w += accum, or with nesterov=True w += momentum*accum - lr*g.
  With momentum == 0, Keras runs plain gradient descent whatever nesterov says.  momentum must lie in [0, 1].
- Adam with amsgrad, extra slot vhat: m, v and lr_t as without it, then vhat = max(vhat, v) and
  w -= lr_t*m/(sqrt(vhat) + eps).  The eps stays outside the root.
- Clipping, applied after any aggregation and in this order: clipvalue, then clipnorm or global_clipnorm, on g*grad_scale.
  - clipvalue=v: clamp each element to [-v, v]; a NaN stays NaN.
  - clipnorm=c: per variable (each trainable tensor); the factor is c/||g_t|| when ||g_t|| > c and exactly 1 otherwise.
    TF writes g*c/max(||g||, c), which differs from this by at most one rounding.  An inf element gives c/inf = 0 for
    the tensor's finite entries and NaN for the inf entry.
  - global_clipnorm=c: one factor from sqrt(sum_t ||g_t||^2) by the same rule; a non-finite global norm makes the
    factor NaN, so every parameter becomes NaN (tf.clip_by_global_norm).
  - each value must be >= 0; clipnorm together with global_clipnorm is a ValueError.
"""
from __future__ import annotations

import numpy as np


def clip_value(g, v):
    g = np.asarray(g, dtype=np.float64)
    return np.where(g > v, v, np.where(g < -v, -v, g))


def clip_factor(norm, c, is_global=False):
    if is_global and not np.isfinite(norm):
        return np.nan
    return 1.0 if norm <= c else c / norm


def clip(grads, clipvalue=None, clipnorm=None, global_clipnorm=None):
    """Clipped copies of the per-tensor gradients ``grads`` (already multiplied by grad_scale) and the factor each
    tensor was scaled by (1.0 where no norm clip fired)."""
    out = [np.asarray(g, dtype=np.float64) for g in grads]
    if clipvalue is not None:
        out = [clip_value(g, clipvalue) for g in out]
    factors = [1.0] * len(out)
    if clipnorm is not None:
        factors = [clip_factor(np.sqrt(np.sum(g * g)), clipnorm) for g in out]
    elif global_clipnorm is not None:
        f = clip_factor(np.sqrt(sum(np.sum(g * g) for g in out)), global_clipnorm, is_global=True)
        factors = [f] * len(out)
    with np.errstate(invalid="ignore"):                  # inf * 0 and NaN factors are part of the semantics
        return [g * f for g, f in zip(out, factors)], factors


def clip_flat(g, sizes, **kw):
    """``clip`` over a flat buffer holding tensors of ``sizes`` back to back."""
    parts = np.split(np.asarray(g, dtype=np.float64), np.cumsum(sizes)[:-1])
    out, factors = clip(parts, **kw)
    return np.concatenate(out), factors


def sgd(w, g, accum, lr, momentum=0.0, nesterov=False):
    """One Keras SGD step; returns (w, accum).  accum is unused (returned as given) for momentum == 0."""
    if momentum == 0.0:
        return w - lr * g, accum
    accum = momentum * accum - lr * g
    if nesterov:
        return w + momentum * accum - lr * g, accum
    return w + accum, accum


def adam(w, g, m, v, vhat, t, lr, beta1=0.9, beta2=0.999, eps=1e-7, amsgrad=False):
    """One Keras Adam step (t 1-based); returns (w, m, v, vhat)."""
    m = beta1 * m + (1 - beta1) * g
    v = beta2 * v + (1 - beta2) * g * g
    lr_t = lr * np.sqrt(1 - beta2 ** t) / (1 - beta1 ** t)
    if amsgrad:
        vhat = np.maximum(vhat, v)
        return w - lr_t * m / (np.sqrt(vhat) + eps), m, v, vhat
    return w - lr_t * m / (np.sqrt(v) + eps), m, v, vhat
