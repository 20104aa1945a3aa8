"""``GeneralGNN`` with the Spektral/Keras call surface the reference script uses.

Reference call sites (src/scripts/gcn.py): :320 ``GeneralGNN(dataset.n_labels,
activation="softmax")``; :334,:351 ``model(inputs, training=...)`` with ``inputs = (x, a,
i)``; :335 ``model.losses``; :337-338 ``model.trainable_variables``; :383
``model.get_weights()``.  Constructor keywords and defaults are those of
``spektral.models.GeneralGNN`` (SURVEY.md §8 a2/b).  All arithmetic happens in the C-ABI
library (csrc/model.cu); this class owns the flat parameter / gradient / state tensors and
the workspace, nothing else.
"""
from __future__ import annotations

import threading
from typing import List, Optional

import numpy as np

from . import _lib, ops
from ._lib import check, ptr, stream_ptr
from .data import SparseAdjacency
from .losses import fused_loss_fields
from .params import (GNNConfig, block_specs, check_dropout_rate, dropout_seed, init_params, n_state, n_trainable,
                     named_slices)

_tape_stack = threading.local()


def _active_tape():
    st = getattr(_tape_stack, "stack", None)
    return st[-1] if st else None


class GradientTape:
    """Minimal stand-in for ``tf.GradientTape`` for the pattern of gcn.py:333-337:

        with GradientTape() as tape:
            predictions = model(inputs, training=True)
            loss = loss_fn(target, predictions) + sum(model.losses)
        gradients = tape.gradient(loss, model.trainable_variables)

    The tape records the training-mode forward (whose activations stay in the model's
    workspace), the dropout of that call (its step, so that the backward regenerates the forward's masks) and the
    loss; ``gradient`` runs the native backward."""

    def __init__(self, persistent=False):
        self.model = None
        self.ctx = None
        self.loss_record = None

    def __enter__(self):
        if not hasattr(_tape_stack, "stack"):
            _tape_stack.stack = []
        _tape_stack.stack.append(self)
        return self

    def __exit__(self, *exc):
        _tape_stack.stack.pop()
        return False

    def gradient(self, loss, variables):
        if self.model is None or self.loss_record is None:
            raise RuntimeError("GradientTape.gradient: no training-mode model call and loss were recorded")
        self.model._backward(self.ctx, self.loss_record["dlogits"])
        by_name = {v.name: v for v in self.model.trainable_variables}
        out = []
        for v in variables:
            if getattr(v, "name", None) not in by_name:
                raise ValueError("GradientTape.gradient: variable does not belong to the recorded model")
            out.append(by_name[v.name].grad_view)
        return out


class Variable:
    """A named view into the model's flat parameter buffer (and the matching gradient)."""

    def __init__(self, name, value, grad_view, trainable):
        self.name, self.value, self.grad_view, self.trainable = name, value, grad_view, trainable

    @property
    def shape(self):
        return tuple(self.value.shape)

    def numpy(self):
        return self.value.detach().cpu().numpy()

    def assign(self, new):
        torch = _lib.require_cuda()
        self.value.copy_(torch.as_tensor(np.asarray(new), dtype=torch.float32).reshape(self.value.shape))

    def __repr__(self):
        return f"<Variable {self.name} shape={self.shape} trainable={self.trainable}>"


class GeneralGNN:
    def __init__(self, output, activation=None, hidden=256, message_passing=4, pre_process=2, post_process=2,
                 connectivity="cat", batch_norm=True, dropout=0.0, aggregate="sum", hidden_activation="prelu",
                 pool="sum", seed: Optional[int] = None, use_edge_weights: bool = False):
        # the layout keywords (params.GNNConfig); Keras' dropout rate changes no layout and is kept apart
        self.config = dict(output=output, activation=activation, hidden=hidden, message_passing=message_passing,
                           pre_process=pre_process, post_process=post_process, connectivity=connectivity,
                           batch_norm=batch_norm, aggregate=aggregate, hidden_activation=hidden_activation, pool=pool)
        check_dropout_rate(dropout)
        self.dropout = float(dropout)
        # validate everything that does not depend on the input width now (no silent fallback)
        GNNConfig(in_features=1, **self.config).validate()
        self.seed = seed
        # dropout: every training-mode call (train_step_grads, model(inputs, training=True)) consumes one step of the
        # mask stream; the stream's key comes from the model's seed and, under DataParallelTrainer, the rank
        self.dropout_step = 0
        self.dropout_rank = 0
        # GeneralConv ignores adjacency values (SURVEY.md 8 a5); the reference's `use_edge_data` switch (gcn.py:73-80)
        # wanted them: with use_edge_weights=True the aggregation weights every message by a.edge_weight[entry]
        self.use_edge_weights = bool(use_edge_weights)
        self.built = False
        self.losses: List = []          # no regularisers (gcn.py:335 adds sum(model.losses) == 0)
        self.cfg: Optional[GNNConfig] = None
        self._ws = None
        self.use_rb4 = True      # row-block (RB4) aggregation format, built once per batch

    # ------------------------------------------------------------------ build / parameters
    def build(self, in_features: int):
        torch = _lib.require_cuda()
        lib = _lib.load()
        self.cfg = GNNConfig(in_features=int(in_features), **self.config)
        self._c = _lib.model_config(self.cfg)
        nw, ns = n_trainable(self.cfg), n_state(self.cfg)
        if lib.gcs_model_num_params(self._c) != nw or lib.gcs_model_num_state(self._c) != ns:
            raise RuntimeError("parameter layout mismatch between params.py and csrc/model.cu")
        seed = self.seed if self.seed is not None else int(np.random.randint(0, 2**31 - 1))
        self._seed = seed
        w, s = init_params(self.cfg, seed)
        self.params = torch.from_numpy(w).cuda()
        self.state = torch.from_numpy(s).cuda()
        self.grads = torch.zeros_like(self.params)
        self._variables = []
        for name, shape, off, buf in named_slices(self.cfg):
            n = int(np.prod(shape))
            if buf == "trainable":
                self._variables.append(Variable(name, self.params[off:off + n].view(shape),
                                                self.grads[off:off + n].view(shape), True))
            else:
                self._variables.append(Variable(name, self.state[off:off + n].view(shape), None, False))
        self.built = True

    @property
    def variables(self):
        return list(self._variables)

    @property
    def trainable_variables(self):
        return [v for v in self._variables if v.trainable]

    @property
    def non_trainable_variables(self):
        return [v for v in self._variables if not v.trainable]

    def get_weights(self):
        """NumPy copies in ``named_slices`` order (per block: kernel, bias, gamma, beta,
        [alpha], moving_mean, moving_variance); names via ``get_named_weights``."""
        return [v.numpy() for v in self._variables]

    def get_named_weights(self):
        return {v.name: v.numpy() for v in self._variables}

    def set_weights(self, weights):
        if isinstance(weights, dict):
            for v in self._variables:
                if v.name in weights:
                    v.assign(weights[v.name])
            return
        if len(weights) != len(self._variables):
            raise ValueError(f"expected {len(self._variables)} arrays, got {len(weights)}")
        for v, w in zip(self._variables, weights):
            v.assign(w)

    def load_flat(self, w, s):
        """Load flat numpy buffers in the params.py layout (parity tests)."""
        torch = _lib.require_cuda()
        self.params.copy_(torch.from_numpy(np.asarray(w, dtype=np.float32)))
        self.state.copy_(torch.from_numpy(np.asarray(s, dtype=np.float32)))

    # ------------------------------------------------------------------ inputs
    def _prepare(self, inputs, need_transpose):
        torch = _lib.require_cuda()
        if not isinstance(inputs, (list, tuple)) or len(inputs) not in (2, 3):
            raise ValueError("inputs must be [x, a] or [x, a, i]")
        x, a = inputs[0], inputs[1]
        i = inputs[2] if len(inputs) == 3 else None
        x = _lib.as_tensor(x)
        if not x.is_cuda:
            x = x.cuda()
        if x.dim() != 2:
            raise ValueError("x must be rank 2 [n_nodes, n_features]")
        if x.dtype == torch.float64:
            x = ops.cast_f64_f32(x)                      # Keras autocast (SURVEY.md §8 a1)
        elif x.dtype != torch.float32:
            raise ValueError(f"x must be float32 or float64, got {x.dtype}")
        if x.stride(1) != 1:
            x = x.contiguous()
        if not self.built:
            self.build(x.shape[1])
        if x.shape[1] != self.cfg.in_features:
            raise ValueError(f"x has {x.shape[1]} features, the model was built for {self.cfg.in_features}")
        if not isinstance(a, SparseAdjacency):
            if not (hasattr(a, "indices") and hasattr(a, "dense_shape")):
                raise AssertionError("A must be a SparseTensor")     # upstream GeneralConv assert
            a = SparseAdjacency.from_indices(a.indices, a.dense_shape)
        if a.n_rows != x.shape[0]:
            raise ValueError(f"a is {a.dense_shape} but x has {x.shape[0]} rows")
        graph_ptr, n_graphs, seg = None, 0, None
        if self.cfg.pool is not None:
            if i is None:
                # upstream: no batch index -> single-graph mode, pool over all nodes
                graph_ptr = torch.tensor([0, x.shape[0]], dtype=torch.int32, device="cuda")
                n_graphs = 1
                seg = torch.zeros(x.shape[0], dtype=torch.int64, device="cuda")
            else:
                i = _lib.as_tensor(i)
                if i.dim() == 2:
                    i = i[:, 0]
                seg = i.to(device="cuda", dtype=torch.int64).contiguous()
                if a.graph_ptr is not None:
                    graph_ptr, n_graphs = a.graph_ptr, a.graph_ptr.shape[0] - 1
                else:
                    n_graphs = int(seg[-1].item()) + 1 if seg.numel() else 0
                    graph_ptr = ops.segment_ptr(seg, n_graphs)
            if seg.shape[0] != x.shape[0]:
                raise ValueError(f"i has {seg.shape[0]} entries but x has {x.shape[0]} rows")
        elif a.graph_ptr is not None:
            graph_ptr, n_graphs = a.graph_ptr, a.graph_ptr.shape[0] - 1
        rp_t, ci_t = a.transposed() if need_transpose else (None, None)
        use_rb4 = self.use_rb4 and x.shape[0] < (1 << 24) and self.cfg.hidden % 4 == 0
        height = a.rb_height() if use_rb4 else 0
        rb4 = a.rb(height) if use_rb4 else (None, None)
        rb4_t = a.rb_t(height) if (use_rb4 and need_transpose) else (None, None)   # the same arrays when the pattern is symmetric
        max_nodes = a.max_graph_nodes if a.graph_ptr is not None else (x.shape[0] if n_graphs == 1 else 0)
        ew, ew_t = None, None
        if self.use_edge_weights:
            if getattr(a, "edge_weight", None) is None:
                raise ValueError("use_edge_weights=True but the adjacency carries no edge_weight")
            a.edge_weight = a.edge_weight.to(device="cuda", dtype=torch.float32).contiguous()
            if a.edge_weight.shape[0] != a.nnz:
                raise ValueError("edge_weight must hold one value per stored entry (CSR order)")
            ew, ew_t = a.edge_weight, (a.edge_weight_t() if need_transpose else None)
        batch = _lib.Batch(x.shape[0], a.nnz, n_graphs, height, ptr(a.rowptr), ptr(a.colidx), ptr(rp_t), ptr(ci_t),
                           ptr(graph_ptr), ptr(x), x.stride(0) if x.shape[0] > 1 else x.shape[1], None,
                           ptr(seg), ptr(rb4[0]), ptr(rb4[1]), ptr(rb4_t[0]), ptr(rb4_t[1]), int(max_nodes), 0, ptr(ew), ptr(ew_t))
        keep = (x, a, graph_ptr, rp_t, ci_t, rb4, rb4_t, seg, ew, ew_t)   # keep device buffers alive
        return batch, keep

    def _workspace(self, batch, training):
        torch = _lib.require_cuda()
        lib = _lib.load()
        flags = _lib.WORKSPACE_SAMPLE_WEIGHTS if batch.sample_weight else 0
        need = lib.gcs_model_workspace_bytes_ex(self._c, batch.n_nodes, batch.nnz, batch.n_graphs, int(training), flags)
        if need < 0:
            raise RuntimeError("gcs_model_workspace_bytes failed: " + lib.gcs_last_error().decode())
        if self._ws is None or self._ws.numel() < need:
            self._ws = None
            self._ws = torch.empty(int(need * 1.08) + 256, dtype=torch.uint8, device="cuda")
        return self._ws

    def _call_dropout(self, training):
        """The gcs_dropout of one call: a training-mode call consumes the next step of the mask stream, keyed by the
        model's seed and rank (host values only: no device synchronisation); inference draws nothing (None)."""
        if not training:
            return None
        d = _lib.Dropout(self.dropout, 0, dropout_seed(self._seed, self.dropout_rank), self.dropout_step)
        self.dropout_step += 1
        return d

    def _rows_out(self, batch):
        return batch.n_graphs if self.cfg.pool is not None else batch.n_nodes

    # ------------------------------------------------------------------ forward / backward
    def __call__(self, inputs, training=False):
        torch = _lib.require_cuda()
        lib = _lib.load()
        tape = _active_tape() if training else None
        batch, keep = self._prepare(inputs, need_transpose=tape is not None)
        ws = self._workspace(batch, training)
        drop = self._call_dropout(training)
        out = torch.empty(self._rows_out(batch), self.cfg.output, dtype=torch.float32, device="cuda")
        check(lib.gcs_model_forward_ex(self._c, ptr(self.params), ptr(self.state), batch, int(training), ptr(out),
                                       ptr(ws), ws.numel(), stream_ptr(), drop), "gcs_model_forward")
        off = lib.gcs_model_logits_offset(self._c, batch.n_nodes, batch.n_graphs, int(training))
        logits = ws[off:off + out.numel() * 4].view(torch.float32).view(out.shape)
        out._gcs_logits = logits       # like Keras' `_keras_logits`: lets the loss use the logits
        out._gcs_activation = self.cfg.activation
        if tape is not None:
            tape.model = self
            tape.ctx = dict(batch=batch, keep=keep, ws=ws, out=out, dropout=drop)
            out._gcs_tape = tape
        return out

    call = __call__

    def _backward(self, ctx, dlogits):
        lib = _lib.load()
        check(lib.gcs_model_backward_ex(self._c, ptr(self.params), ctx["batch"], ptr(dlogits), ptr(self.grads),
                                        ptr(ctx["ws"]), ctx["ws"].numel(), stream_ptr(), ctx["dropout"]),
              "gcs_model_backward")

    def train_step_grads(self, inputs, target, grad_scale: Optional[float] = None, comm=None, sync_bn: bool = False,
                         loss=None, sample_weight=None):
        """Fused training-mode forward + loss + backward (one C call): categorical cross-entropy with
        activation='softmax', binary cross-entropy (mean over the C columns, then the rows) with activation='sigmoid',
        and with the linear head (activation=None) the regression loss ``loss`` - ``MeanSquaredError()`` (the default),
        ``MeanAbsoluteError()`` or ``Huber(delta)``.
        Leaves the gradients in ``self.grads``; returns (loss_acc [2] device tensor = {loss,
        accuracy} - {loss, mean absolute error} for a regression loss -, probs [B, C] - the predictions of a linear
        head).  ``grad_scale`` defaults to 1/B (mean loss, gcn.py:335).
        ``comm`` (distributed.NativeComm): the data-parallel form - the gradients are SUM all-reduced over the
        communicator, bucket by bucket on its own stream while the backward is still running
        (gcs_model_train_step_dp); the current stream waits for the reductions.
        ``sample_weight`` ([rows] or [rows, 1], one weight per graph - per node without pooling): Keras' per-row loss
        weights; the loss is sum w l / rows, the metric the weighted mean, and each row's gradient is scaled by its
        weight."""
        torch = _lib.require_cuda()
        lib = _lib.load()
        code, delta = fused_loss_fields(loss, self.config["activation"])
        batch, keep = self._prepare(inputs, need_transpose=True)
        c = self._c
        if code:                                         # for this call only: the layout never depends on the loss
            c = _lib.ModelConfig.from_buffer_copy(self._c)
            c.loss, c.huber_delta = code, delta
        drop = self._call_dropout(True)
        y = _lib.as_tensor(target)
        y = y.to(device="cuda", dtype=torch.float32).contiguous()
        rows = self._rows_out(batch)
        if tuple(y.shape) != (rows, self.cfg.output):
            raise ValueError(f"target must be [{rows}, {self.cfg.output}], got {tuple(y.shape)}")
        batch.y = ptr(y)
        w = ops.sample_weight_vector(sample_weight, rows) if sample_weight is not None else None
        batch.sample_weight = ptr(w)
        ws = self._workspace(batch, True)
        probs = torch.empty(rows, self.cfg.output, dtype=torch.float32, device="cuda")
        loss_acc = torch.empty(2, dtype=torch.float32, device="cuda")
        gs = 1.0 / rows if grad_scale is None else float(grad_scale)
        if comm is not None:
            check(lib.gcs_model_train_step_dp_ex(c, ptr(self.params), ptr(self.state), batch, gs, ptr(self.grads),
                                                 ptr(probs), ptr(loss_acc), ptr(ws), ws.numel(), stream_ptr(),
                                                 comm.handle, comm.stream.cuda_stream, int(bool(sync_bn)), drop),
                  "gcs_model_train_step_dp")
        else:
            check(lib.gcs_model_train_step_ex(c, ptr(self.params), ptr(self.state), batch, gs, ptr(self.grads),
                                              ptr(probs), ptr(loss_acc), ptr(ws), ws.numel(), stream_ptr(), drop),
                  "gcs_model_train_step")
        self._keep = (keep, y, w)
        return loss_acc, probs
