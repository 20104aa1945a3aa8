"""The weighted ROC curve in NumPy float64 (TEST INFRASTRUCTURE); the weighted losses and the weighted train step are
oracle.model_ref_np (weighted_loss, loss_and_grads with ``sample_weight``)."""
from __future__ import annotations

import numpy as np


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
