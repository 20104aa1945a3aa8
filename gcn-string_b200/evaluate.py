"""Evaluation step and metrics (SURVEY.md §8 f2) - the reference's ``evaluate(loader)``
(src/scripts/gcn.py:342-362) and its ROC post-processing (:389-398), with everything up to the
final curve kept on the device.

``evaluate`` runs ``model(inputs, training=False)`` (BatchNorm on moving statistics, folded into
scale/shift; gcs_model_forward) over one pass of the loader, evaluates loss and accuracy with the
fused softmax/cross-entropy kernel (gcs_softmax_xent; sigmoid/binary cross-entropy, gcs_sigmoid_bce, for a model
built with activation='sigmoid') and returns the batch-size-weighted averages
plus the per-batch predictions, like the reference.  ``roc_curve`` / ``auc`` follow scikit-learn's
definitions (the reference calls ``sklearn.metrics.roc_curve(labels, probas)`` and ``auc``); they
are sort + prefix sums and run on whatever device the scores live on.
"""
from __future__ import annotations

import numpy as np

from . import _lib
from .losses import (BinaryCrossentropy, CategoricalCrossentropy, Huber, MeanAbsoluteError, MeanSquaredError,
                     binary_accuracy, categorical_accuracy, mean_absolute_error)


def evaluate(model, loader, loss_fn=None, metric=None):
    """One pass over ``loader`` -> (np.array([loss, acc]) weighted by batch size, [pred per batch]).
    Mirrors gcn.py:342-362; the only host transfers are the two scalars per batch.  The loss and accuracy default to
    BinaryCrossentropy / binary_accuracy for a model built with activation='sigmoid', to CategoricalCrossentropy /
    categorical_accuracy otherwise.  ``metric(y_true, y_pred)`` -> per-row values replaces the accuracy; with a
    regression ``loss_fn`` (MeanSquaredError, MeanAbsoluteError, Huber) it defaults to mean_absolute_error.
    A loader that yields ``(inputs, y, w)`` (DisjointLoader(sample_weights=...)) gives the weighted figures: the loss
    is the sum over the pass of w * l over the total number of rows, the metric sum w * m / sum w (0 when sum w = 0)."""
    torch = _lib.require_cuda()
    sigmoid = getattr(model, "config", {}).get("activation") == "sigmoid"
    if metric is None and isinstance(loss_fn, (MeanSquaredError, MeanAbsoluteError, Huber)):
        metric = mean_absolute_error
    loss_fn = loss_fn or (BinaryCrossentropy() if sigmoid else CategoricalCrossentropy())
    metric = metric or (binary_accuracy if sigmoid else categorical_accuracy)
    stats, preds = [], []
    weighted = False
    step = 0
    while step < loader.steps_per_epoch:
        step += 1
        inputs, target, *w = next(loader)
        pred = model(inputs, training=False)
        preds.append(pred)
        rows = torch.tensor(float(target.shape[0]), device=pred.device)
        if w:
            weighted = True
            w = w[0].reshape(-1).to(torch.float32)
            loss = loss_fn(target, pred, sample_weight=w)
            m = metric(target, pred).reshape(-1)
            stats.append(torch.stack([loss.reshape(()), (w * m).sum(), w.sum(), rows]))
        else:
            stats.append(torch.stack([loss_fn(target, pred).reshape(()), metric(target, pred).mean().reshape(()), rows,
                                      rows]))
    out = torch.stack(stats).cpu().numpy().astype(np.float64)
    if not weighted:
        return np.average(out[:, [0, 1]], 0, weights=out[:, -1]), preds
    loss = np.average(out[:, 0], weights=out[:, -1])
    wsum = out[:, 2].sum()
    return np.array([loss, out[:, 1].sum() / wsum if wsum != 0 else 0.0]), preds


def positive_scores(preds, column: int = 1):
    """gcn.py:390-391: stack the per-batch softmax outputs and keep the positive-class column (``column=0`` for the
    one-column output of a sigmoid head)."""
    torch = _lib.require_cuda()
    return torch.cat([p[:, column] for p in preds])


def _as_torch(a, like=None):
    import torch
    if isinstance(a, torch.Tensor):
        return a
    t = torch.as_tensor(np.asarray(a))
    return t.to(like.device) if like is not None else t


def roc_curve(y_true, y_score, drop_intermediate: bool = True, sample_weight=None):
    """``sklearn.metrics.roc_curve`` for binary labels in {0, 1} (positive = 1): returns
    (fpr, tpr, thresholds) as NumPy arrays.  Sort and prefix sums run on the scores' device.  ``sample_weight`` (one
    per sample) as in scikit-learn: samples of weight 0 are left out, and the true and false positives are the
    cumulative weights of the positive and negative samples."""
    import torch
    s = _as_torch(y_score).reshape(-1).to(torch.float64)
    y = _as_torch(y_true, like=s).reshape(-1).to(s.device).to(torch.float64)
    if y.shape[0] != s.shape[0]:
        raise ValueError(f"y_true has {y.shape[0]} entries, y_score {s.shape[0]}")
    w = None
    if sample_weight is not None:
        w = _as_torch(sample_weight, like=s).reshape(-1).to(s.device).to(torch.float64)
        if w.shape[0] != s.shape[0]:
            raise ValueError(f"sample_weight has {w.shape[0]} entries, y_score {s.shape[0]}")
        keep = w != 0
        s, y, w = s[keep], y[keep], w[keep]
    if y.shape[0] == 0:
        raise ValueError("roc_curve needs at least one sample")
    order = torch.argsort(s, descending=True, stable=True)
    s, y = s[order], y[order]
    n = s.shape[0]
    distinct = torch.nonzero(s[1:] != s[:-1]).reshape(-1)
    idx = torch.cat([distinct, torch.tensor([n - 1], device=s.device)])
    if w is None:
        tps = torch.cumsum(y, 0)[idx]
        fps = (1 + idx).to(torch.float64) - tps
    else:
        w = w[order]
        tps = torch.cumsum(y * w, 0)[idx]
        fps = torch.cumsum((1 - y) * w, 0)[idx]
    thr = s[idx]
    if drop_intermediate and idx.shape[0] > 2:
        d2f, d2t = torch.diff(fps, n=2), torch.diff(tps, n=2)
        keep = torch.cat([torch.tensor([True], device=s.device), (d2f != 0) | (d2t != 0),
                          torch.tensor([True], device=s.device)])
        fps, tps, thr = fps[keep], tps[keep], thr[keep]
    zero = torch.zeros(1, dtype=torch.float64, device=s.device)
    tps, fps = torch.cat([zero, tps]), torch.cat([zero, fps])
    thr = torch.cat([torch.full((1,), float("inf"), dtype=torch.float64, device=s.device), thr])
    fpr = fps / fps[-1] if float(fps[-1]) > 0 else torch.full_like(fps, float("nan"))
    tpr = tps / tps[-1] if float(tps[-1]) > 0 else torch.full_like(tps, float("nan"))
    return fpr.cpu().numpy(), tpr.cpu().numpy(), thr.cpu().numpy()


def auc(x, y) -> float:
    """``sklearn.metrics.auc``: trapezoidal area of y over a monotonic x (sign follows the direction)."""
    x = np.asarray(x, dtype=np.float64).reshape(-1)
    y = np.asarray(y, dtype=np.float64).reshape(-1)
    if x.shape[0] != y.shape[0]:
        raise ValueError("x and y must have the same length")
    if x.shape[0] < 2:
        raise ValueError(f"At least 2 points are needed to compute area under curve, but x.shape = {x.shape[0]}")
    dx = np.diff(x)
    direction = 1.0
    if np.any(dx < 0):
        if np.all(dx <= 0):
            direction = -1.0
        else:
            raise ValueError("x is neither increasing nor decreasing : {}.".format(x))
    return float(direction * np.trapezoid(y, x))


def roc_auc(y_true, y_score) -> float:
    """Area under the ROC curve (fpr on the x axis)."""
    fpr, tpr, _ = roc_curve(y_true, y_score, drop_intermediate=False)
    return auc(fpr, tpr)
