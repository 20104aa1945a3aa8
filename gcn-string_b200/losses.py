"""``CategoricalCrossentropy`` and ``categorical_accuracy`` as the reference uses them
(src/scripts/gcn.py:6-7 imports, :326 ``loss_fn = CategoricalCrossentropy()``, :335,:353
calls, :339,:355 accuracy).  Keras evaluates the loss on the LOGITS of a softmax output
(it recovers them from the activation); the model attaches them to its output the same way
(``_gcs_logits``), and the native kernel computes loss, accuracy and dLoss/dlogits in one
launch (csrc/loss.cu).  Reduction is the Keras default: mean over the batch.

``BinaryCrossentropy`` and ``binary_accuracy`` are the Keras pair for a sigmoid head (binary and multi-label targets):
on the logits of a ``GeneralGNN(activation='sigmoid')`` output, or with ``from_logits=True``, they run the fused kernel
of csrc/loss.cu.

``MeanSquaredError``, ``MeanAbsoluteError`` and ``Huber`` are the Keras regression losses for the linear head of a
default ``GeneralGNN(C)`` (activation=None); with ``mean_squared_error`` / ``mean_absolute_error`` they run the fused
kernel of csrc/loss.cu.

Every loss takes Keras' ``sample_weight``: one weight per row (``[rows]`` or ``[rows, 1]``), with the default
"sum_over_batch_size" reduction, so the loss is sum_r w_r l_r / rows (the number of rows, not sum w).  The fused paths
run the weighted kernel (gcs_weighted_loss); the host fallbacks weight the same way in torch."""
from __future__ import annotations

from . import _lib, ops


def _weighted_mean(per_row, sample_weight):
    """Keras' "sum_over_batch_size" reduction of the per-row losses: sum(w * l) / rows (plain mean without weights)."""
    if sample_weight is None:
        return per_row.mean()
    import torch
    w = sample_weight if isinstance(sample_weight, torch.Tensor) else torch.as_tensor(sample_weight)
    ops.check_sample_weight_shape(w.shape, per_row.shape[0])
    w = w.to(device=per_row.device, dtype=per_row.dtype).reshape(-1)
    return (w * per_row).sum() / per_row.shape[0]


def categorical_crossentropy_from_probs(y, p, sample_weight=None):
    """Keras' loss on probabilities of unknown origin: normalise, clip to [1e-7, 1 - 1e-7], -sum y log p per row, then
    the (weighted) mean over the rows.  Runs on the tensors' device."""
    p = p / p.sum(dim=-1, keepdim=True)
    p = p.clamp(1e-7, 1.0 - 1e-7)
    return _weighted_mean(-(y * p.log()).sum(dim=-1), sample_weight)


def binary_crossentropy_from_probs(y, p, sample_weight=None):
    """Keras' binary cross-entropy on probabilities: clip, -(y log(p + eps) + (1 - y) log(1 - p + eps)), the mean over
    the last axis, then the (weighted) mean over the rows.  Runs on the tensors' device."""
    eps = 1e-7
    p = p.clamp(eps, 1.0 - eps)
    bce = y * (p + eps).log() + (1.0 - y) * (1.0 - p + eps).log()
    return _weighted_mean((-bce).mean(dim=-1), sample_weight)


class CategoricalCrossentropy:
    def __init__(self, from_logits=False, reduction="sum_over_batch_size", name="categorical_crossentropy"):
        if reduction not in ("sum_over_batch_size", "auto"):
            raise NotImplementedError("only the default mean-over-batch reduction is built")
        self.from_logits = from_logits
        self.name = name

    def __call__(self, y_true, y_pred, sample_weight=None):
        torch = _lib.require_cuda()
        y = _lib.as_tensor(y_true).to(device="cuda", dtype=torch.float32)
        logits = y_pred if self.from_logits else getattr(y_pred, "_gcs_logits", None)
        if logits is None:
            # probabilities of unknown origin: Keras' fallback (normalise, clip, -sum y log p)
            return categorical_crossentropy_from_probs(y, y_pred, sample_weight)
        tape = getattr(y_pred, "_gcs_tape", None)
        _, loss_acc, dlogits = ops.softmax_xent(logits, y, want_grad=tape is not None, sample_weight=sample_weight)
        loss = loss_acc[0]
        if tape is not None:
            tape.loss_record = dict(dlogits=dlogits, loss_acc=loss_acc)
        return loss


def categorical_accuracy(y_true, y_pred):
    """Per-sample 0/1 accuracy, like tf.keras.metrics.categorical_accuracy."""
    torch = _lib.require_cuda()
    y = _lib.as_tensor(y_true).to(device="cuda")
    return (y.argmax(dim=-1) == y_pred.argmax(dim=-1)).to(torch.float32)


class BinaryCrossentropy:
    """tf.keras.losses.BinaryCrossentropy: per element ``max(z, 0) - z*y + log1p(exp(-|z|))`` on the logits z, the mean
    over the last axis, then over the rows.  Labels may be multi-hot or soft, in [0, 1]."""

    def __init__(self, from_logits=False, label_smoothing=0.0, axis=-1, reduction="sum_over_batch_size",
                 name="binary_crossentropy"):
        if label_smoothing != 0.0:
            raise NotImplementedError("label_smoothing is not built")
        if axis != -1:
            raise NotImplementedError("only axis=-1 is built")
        if reduction not in ("sum_over_batch_size", "auto"):
            raise NotImplementedError("only the default mean-over-batch reduction is built")
        self.from_logits = from_logits
        self.name = name

    def __call__(self, y_true, y_pred, sample_weight=None):
        torch = _lib.require_cuda()
        y = _lib.as_tensor(y_true).to(device="cuda", dtype=torch.float32)
        if self.from_logits:
            logits = y_pred
        elif getattr(y_pred, "_gcs_activation", None) == "sigmoid":
            logits = y_pred._gcs_logits
        else:
            # probabilities of unknown origin: Keras' fallback (clip, then -(y log(p + eps) + (1 - y) log(1 - p + eps)))
            return binary_crossentropy_from_probs(y, y_pred, sample_weight)
        tape = getattr(y_pred, "_gcs_tape", None)
        _, loss_acc, dlogits = ops.sigmoid_bce(logits, y, want_grad=tape is not None, sample_weight=sample_weight)
        if tape is not None:
            tape.loss_record = dict(dlogits=dlogits, loss_acc=loss_acc)
        return loss_acc[0]


def binary_accuracy(y_true, y_pred, threshold=0.5):
    """Per-row mean over the columns of ``y_true == (y_pred > threshold)``, like tf.keras.metrics.binary_accuracy (the
    comparison is on the float32 probabilities)."""
    torch = _lib.require_cuda()
    y = _lib.as_tensor(y_true).to(device="cuda", dtype=torch.float32)
    pred = (_lib.as_tensor(y_pred) > threshold).to(torch.float32)
    return (y == pred).to(torch.float32).mean(dim=-1)


class _RegressionLoss:
    """Shared body of the Keras regression losses: the mean over the last axis, then over the rows, of the element loss
    of e = y_pred - y_true, on the predictions of a linear head (the logits the model attached to its output) or on
    ``y_pred`` itself.  Under an active ``GradientTape`` it records dLoss/dlogits for the model's backward."""
    kind = ""         # ops.regression_loss name
    code = 0          # gcs_model_config.loss

    def __init__(self, reduction, name, delta=1.0):
        if reduction not in ("sum_over_batch_size", "auto"):
            raise NotImplementedError("only the default mean-over-batch reduction is built")
        self.name = name
        self.delta = float(delta)

    def __call__(self, y_true, y_pred, sample_weight=None):
        torch = _lib.require_cuda()
        y = _lib.as_tensor(y_true).to(device="cuda", dtype=torch.float32)
        linear = getattr(y_pred, "_gcs_activation", None) in (None, "linear")
        pred = y_pred._gcs_logits if linear and hasattr(y_pred, "_gcs_logits") else y_pred
        tape = getattr(y_pred, "_gcs_tape", None)
        if tape is not None and not linear:
            raise NotImplementedError(f"{type(self).__name__} is built for a linear head (activation=None); the model's "
                                      f"output has activation={y_pred._gcs_activation!r}")
        loss_acc, dlogits = ops.regression_loss(pred, y, self.kind, self.delta, want_grad=tape is not None,
                                                sample_weight=sample_weight)
        if tape is not None:
            tape.loss_record = dict(dlogits=dlogits, loss_acc=loss_acc)
        return loss_acc[0]


class MeanSquaredError(_RegressionLoss):
    """tf.keras.losses.MeanSquaredError: mean of (y_pred - y_true)^2."""
    kind, code = "mse", 1

    def __init__(self, reduction="sum_over_batch_size", name="mean_squared_error"):
        super().__init__(reduction, name)


class MeanAbsoluteError(_RegressionLoss):
    """tf.keras.losses.MeanAbsoluteError: mean of |y_pred - y_true|; its gradient at an exact tie is 0, as in TF."""
    kind, code = "mae", 2

    def __init__(self, reduction="sum_over_batch_size", name="mean_absolute_error"):
        super().__init__(reduction, name)


class Huber(_RegressionLoss):
    """tf.keras.losses.Huber: 0.5 e^2 where |e| <= delta, delta |e| - 0.5 delta^2 elsewhere."""
    kind, code = "huber", 3

    def __init__(self, delta=1.0, reduction="sum_over_batch_size", name="huber_loss"):
        delta = float(delta)
        if not (0.0 < delta < float("inf")):
            raise ValueError(f"Huber: delta must be finite and > 0, got {delta}")
        super().__init__(reduction, name, delta)


def mean_squared_error(y_true, y_pred):
    """Per-row mean over the columns of (y_pred - y_true)^2, like tf.keras.metrics.mean_squared_error."""
    torch = _lib.require_cuda()
    y = _lib.as_tensor(y_true).to(device="cuda", dtype=torch.float32)
    return (_lib.as_tensor(y_pred) - y).square().mean(dim=-1)


def mean_absolute_error(y_true, y_pred):
    """Per-row mean over the columns of |y_pred - y_true|, like tf.keras.metrics.mean_absolute_error."""
    torch = _lib.require_cuda()
    y = _lib.as_tensor(y_true).to(device="cuda", dtype=torch.float32)
    return (_lib.as_tensor(y_pred) - y).abs().mean(dim=-1)


def fused_loss_fields(loss, activation):
    """(gcs_model_config.loss, .huber_delta) for the fused train step of a head with ``activation``: ``None`` gives
    (0, 1.0), the head's own loss; a regression loss needs a linear head."""
    if loss is None:
        return 0, 1.0
    if not isinstance(loss, _RegressionLoss):
        raise NotImplementedError(f"the fused train step takes loss=None (the head's own loss) or MeanSquaredError, "
                                  f"MeanAbsoluteError or Huber, not {type(loss).__name__}")
    if activation not in (None, "linear"):
        raise NotImplementedError(f"{type(loss).__name__} is built for a linear head (activation=None), not "
                                  f"activation={activation!r}")
    return loss.code, loss.delta
