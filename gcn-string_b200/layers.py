"""Layer-level call surface: ``GeneralConv``, ``GlobalSumPool``, ``GlobalAvgPool``, ``GlobalAttnSumPool``, ``MLP``.

Signatures follow Spektral (SURVEY.md §8b): ``GeneralConv(channels=256, batch_norm=True,
dropout=0.0, aggregate='sum', activation='prelu', use_bias=True)([x, a]) -> [N, channels]``,
``GlobalSumPool()([x, i]) -> [B, W]`` (likewise ``GlobalAvgPool()`` and
``GlobalAttnSumPool()``; ``[x]`` alone pools over all nodes, keepdims), ``MLP(output, hidden=256, layers=2, batch_norm=True,
dropout=0.0, activation='prelu', final_activation=None)(x)``.  They are inference/forward
building blocks over the same kernels GeneralGNN uses (the reference only ever reaches them
through GeneralGNN, src/scripts/gcn.py:320); training goes through the model entry points.  ``dropout`` is Keras'
rate: the identity in inference, as in Keras; a training-mode call with ``dropout > 0`` raises (GeneralGNN trains it).
"""
from __future__ import annotations

import numpy as np

from . import _lib, ops
from .data import SparseAdjacency
from .params import check_dropout_rate


def _check_training_dropout(layer, rate, training):
    if training and rate > 0.0:
        raise NotImplementedError(f"{layer}(dropout={rate}) is forward-only in training mode: train dropout through "
                                  "GeneralGNN(dropout=...), whose fused train step applies and differentiates the masks")


def _param(arr):
    torch = _lib.require_cuda()
    return torch.from_numpy(np.ascontiguousarray(arr, dtype=np.float32)).cuda()


class _DenseBlock:
    """kernel/bias + BatchNormalization + PReLU parameters of one block."""

    def __init__(self, k_in, m_out, has_alpha, rng, use_bias=True, batch_norm=True):
        lim = np.sqrt(6.0 / (k_in + m_out))
        self.kernel = _param(rng.uniform(-lim, lim, size=(k_in, m_out)))
        self.bias = _param(np.zeros(m_out)) if use_bias else None
        self.batch_norm = batch_norm
        self.gamma = _param(np.ones(m_out))
        self.beta = _param(np.zeros(m_out))
        self.moving_mean = _param(np.zeros(m_out))
        self.moving_variance = _param(np.ones(m_out))
        self.alpha = _param(np.zeros(m_out)) if has_alpha else None
        self.epsilon, self.momentum = 1e-3, 0.99

    def linear(self, x):
        return ops.linear_fwd(x, self.kernel, self.bias)

    def fold(self, h, training):
        torch = _lib.require_cuda()
        if not self.batch_norm:
            one = torch.ones_like(self.gamma)
            return one, torch.zeros_like(one)
        if training:
            mean, var = ops.bn_stats(h)
            return ops.bn_fold(mean, var, self.gamma, self.beta, self.epsilon, self.momentum,
                               self.moving_mean, self.moving_variance)
        return ops.bn_fold(self.moving_mean, self.moving_variance, self.gamma, self.beta, self.epsilon, self.momentum)


def _as_adjacency(a, n):
    if isinstance(a, SparseAdjacency):
        return a
    if not (hasattr(a, "indices") and hasattr(a, "dense_shape")):
        raise AssertionError("A must be a SparseTensor")
    return SparseAdjacency.from_indices(a.indices, a.dense_shape)


class GeneralConv:
    def __init__(self, channels=256, batch_norm=True, dropout=0.0, aggregate="sum", activation="prelu",
                 use_bias=True, seed=0, **kwargs):
        if aggregate not in ops.AGGREGATE:
            raise NotImplementedError("native path implements aggregate in {'sum', 'mean', 'max'}")
        check_dropout_rate(dropout)
        if activation not in ("prelu", None, "linear"):
            raise NotImplementedError("native path implements activation in {'prelu', None}")
        self.aggregate, self.dropout = aggregate, dropout
        self.channels, self.use_batch_norm, self.activation, self.use_bias = channels, batch_norm, activation, use_bias
        self.seed = seed
        self.block = None

    def __call__(self, inputs, training=False):
        _check_training_dropout("GeneralConv", self.dropout, training)
        torch = _lib.require_cuda()
        x, a = inputs[0], inputs[1]
        x = _lib.as_tensor(x)
        if self.block is None:
            self.block = _DenseBlock(x.shape[1], self.channels, self.activation == "prelu",
                                     np.random.default_rng(self.seed), self.use_bias, self.use_batch_norm)
        a = _as_adjacency(a, x.shape[0])
        h = self.block.linear(x)
        scale, shift = self.block.fold(h, training)
        alpha = self.block.alpha if self.block.alpha is not None else torch.ones_like(scale)
        if self.aggregate == "sum":
            return ops.spmm_sum(a.rowptr, a.colidx, h, scale, shift, alpha, rb4=a.rb4)
        return ops.spmm_aggregate(a.rowptr, a.colidx, h, scale, shift, alpha, aggregate=self.aggregate)


def _pool_inputs(inputs):
    """[x, i] -> (x, graph_ptr of the sorted batch index i); [x] or x -> (x, one graph of all nodes: single mode)."""
    torch = _lib.require_cuda()
    if isinstance(inputs, (list, tuple)) and len(inputs) == 2:
        x, i = inputs
        i = _lib.as_tensor(i)
        if i.dim() == 2:
            i = i[:, 0]
        i = i.to(device="cuda", dtype=torch.int64).contiguous()
        n_graphs = int(i[-1].item()) + 1 if i.numel() else 0
        return _lib.as_tensor(x), ops.segment_ptr(i, n_graphs)
    x = _lib.as_tensor(inputs[0] if isinstance(inputs, (list, tuple)) else inputs)
    return x, torch.tensor([0, x.shape[0]], dtype=torch.int32, device="cuda")


class GlobalSumPool:
    def __call__(self, inputs):
        return ops.segment_sum_fwd(*_pool_inputs(inputs))


class GlobalAvgPool:
    """tf.math.segment_mean over the graphs (0 for an empty graph)."""

    def __call__(self, inputs):
        return ops.segment_mean_fwd(*_pool_inputs(inputs))


class GlobalAttnSumPool:
    """Attention-weighted sum: ``softmax_g(x . attn_kernel)`` per graph weights the rows of x.  ``attn_kernel`` [W, 1]
    is created on the first call, glorot-uniform from ``seed``."""

    def __init__(self, seed=0):
        self.seed = seed
        self.attn_kernel = None

    def __call__(self, inputs):
        x, gp = _pool_inputs(inputs)
        if self.attn_kernel is None:
            w = x.shape[1]
            lim = np.sqrt(6.0 / (w + 1))
            self.attn_kernel = _param(np.random.default_rng(self.seed).uniform(-lim, lim, size=(w, 1)))
        out, _, _ = ops.attn_sum_pool_fwd(x, self.attn_kernel, gp)
        return out


class MLP:
    def __init__(self, output, hidden=256, layers=2, batch_norm=True, dropout=0.0, activation="prelu",
                 final_activation=None, seed=0):
        check_dropout_rate(dropout)
        if activation != "prelu":
            raise NotImplementedError("native path implements activation='prelu' only")
        if final_activation not in (None, "linear", "softmax", "sigmoid", "prelu"):
            raise NotImplementedError("final_activation must be None, 'prelu', 'softmax' or 'sigmoid'")
        self.output, self.hidden, self.layers, self.batch_norm = output, hidden, layers, batch_norm
        self.final_activation, self.dropout = final_activation, dropout
        self.seed = seed
        self.blocks = None

    def __call__(self, x, training=False):
        _check_training_dropout("MLP", self.dropout, training)
        x = _lib.as_tensor(x)
        if self.blocks is None:
            rng = np.random.default_rng(self.seed)
            k = x.shape[1]
            self.blocks = []
            for j in range(self.layers):
                last = j == self.layers - 1
                m = self.output if last else self.hidden
                self.blocks.append(_DenseBlock(k, m, (not last) or self.final_activation == "prelu", rng,
                                               True, self.batch_norm))
                k = m
        out = x
        for blk in self.blocks:
            h = blk.linear(out)
            scale, shift = blk.fold(h, training)
            out = ops.bn_prelu_fwd(h, scale, shift, blk.alpha)
        if self.final_activation == "softmax":
            out, _, _ = ops.softmax_xent(out)
        elif self.final_activation == "sigmoid":
            out, _, _ = ops.sigmoid_bce(out)
        return out
