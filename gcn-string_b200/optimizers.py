"""``SGD`` / ``Adam`` and ``schedules.PiecewiseConstantDecay`` with Keras semantics
(reference: src/scripts/gcn.py:321-325 schedule + SGD, :338 ``apply_gradients``; SURVEY.md §8
a11).  ``apply_gradients`` over a model's full variable list is ONE fused kernel over the
flat parameter buffer (csrc/optim.cu); partial lists fall back to one launch per tensor.

Keras' options are built into the same kernels: ``SGD(momentum, nesterov)``, ``Adam(amsgrad)`` and the clipping
keywords of every Keras optimizer, ``clipvalue``, ``clipnorm`` (per variable) and ``global_clipnorm``.  A norm-clipped
step is two launches (norm pass, update) over a chunk table that is built and uploaded once per variable layout."""
from __future__ import annotations

import numpy as np

from . import _lib, ops

# Elements per chunk of the clipping norm pass (one thread block each).  The cfg3 layout (1 064 454 parameters in 39
# tensors) gives 548 chunks, over three blocks per SM of a B200; tensors smaller than a chunk are one chunk each.
CHUNK = 2048


def chunk_table(sizes, chunk: int = CHUNK):
    """int64 [n_chunks, 3] rows (begin, end, tensor) over a flat buffer that holds tensors of ``sizes`` elements back to
    back: each tensor is cut into pieces of ``chunk`` elements from its own start (the last one shorter), so no chunk
    crosses a tensor and a tensor's chunks do not depend on where it sits in the buffer."""
    rows, off = [], 0
    for t, n in enumerate(sizes):
        n = int(n)
        rows.extend((off + b, off + min(b + chunk, n), t) for b in range(0, n, chunk))
        off += n
    return np.asarray(rows, dtype=np.int64).reshape(-1, 3)


def device_rows(table, relative: bool = False):
    """The device form of a chunk table (gcs_grad_clip.chunks): int64 [n_chunks, 4] = (begin, end, lo, hi) with
    [lo, hi) the rows of the chunk's tensor.  ``relative=True``: begin / end from the start of each tensor (one launch
    per tensor)."""
    t = table[:, 2]
    first = np.searchsorted(t, t, side="left")
    last = np.searchsorted(t, t, side="right")
    begin, end = table[:, 0], table[:, 1]
    if relative:
        begin, end = begin - begin[first], end - begin[first]
    return np.ascontiguousarray(np.stack([begin, end, first, last], axis=1).astype(np.int64))


class PiecewiseConstantDecay:
    """values[0] for step <= boundaries[0]; values[k] for boundaries[k-1] < step <=
    boundaries[k]; values[-1] afterwards (tf.keras.optimizers.schedules)."""

    def __init__(self, boundaries, values, name=None):
        if len(values) != len(boundaries) + 1:
            raise ValueError("The length of boundaries should be 1 less than the length of values")
        self.boundaries, self.values = list(boundaries), list(values)

    def __call__(self, step):
        for b, v in zip(self.boundaries, self.values):
            if step <= b:
                return v
        return self.values[-1]


class schedules:  # namespace, like tf.keras.optimizers.schedules
    PiecewiseConstantDecay = PiecewiseConstantDecay


class _Optimizer:
    def __init__(self, learning_rate, clipnorm=None, clipvalue=None, global_clipnorm=None, **kwargs):
        if "decay" in kwargs:
            raise NotImplementedError("the legacy `decay` keyword is not built; pass a learning-rate schedule")
        for k in kwargs:
            raise TypeError(f"Unexpected keyword argument passed to optimizer: {k}")
        if clipnorm is not None and global_clipnorm is not None:
            raise ValueError(f"Cannot accept both `clipnorm` and `global_clipnorm`, passed `clipnorm` {clipnorm}, "
                             f"`global_clipnorm` {global_clipnorm}")
        for k, val in (("clipnorm", clipnorm), ("clipvalue", clipvalue), ("global_clipnorm", global_clipnorm)):
            if val is not None and not val >= 0:
                raise ValueError(f"Expected {k} >= 0, received: {val}")
        self.learning_rate = learning_rate
        self.iterations = 0
        self.clipnorm, self.clipvalue, self.global_clipnorm = clipnorm, clipvalue, global_clipnorm
        self._slots = {}
        self._clips = {}          # variable layout -> device chunk table, partials and descriptors, built once

    def _lr(self):
        lr = self.learning_rate
        return float(lr(self.iterations)) if callable(lr) else float(lr)

    def _slot(self, key, w, count):
        """The ``count`` zero-initialised slot tensors of ``key``, allocated on first use."""
        if key not in self._slots:
            torch = _lib.require_cuda()
            self._slots[key] = tuple(torch.zeros_like(w) for _ in range(count))
        return self._slots[key]

    # ------------------------------------------------------------------ clipping descriptors
    @property
    def _norm_clip(self):
        return self.clipnorm is not None or self.global_clipnorm is not None

    def _clip_struct(self):
        c = _lib.GradClip()
        if self.clipvalue is not None:
            c.mode |= _lib.CLIP_VALUE
            c.clipvalue = float(self.clipvalue)
        if self._norm_clip:
            c.mode |= _lib.CLIP_NORM if self.clipnorm is not None else _lib.CLIP_GLOBAL_NORM
            c.clipnorm = float(self.clipnorm if self.clipnorm is not None else self.global_clipnorm)
        return c

    def _layout(self, key, sizes, relative):
        """Chunk table (uploaded once) and fp64 partials of a variable layout, with one descriptor for the whole
        buffer (``relative=False``) or one per tensor (``relative=True``)."""
        ck = (key, sizes)
        if ck not in self._clips:
            torch = _lib.require_cuda()
            table = chunk_table(sizes)
            rows = torch.from_numpy(device_rows(table, relative)).cuda()
            partials = torch.zeros(table.shape[0], dtype=torch.float64, device="cuda")
            n = table.shape[0]
            if not relative:
                c = self._clip_struct()
                c.chunks, c.partials, c.n_chunks, c.chunk_base, c.n_partials = rows.data_ptr(), partials.data_ptr(), n, 0, n
                clips = c
            else:
                clips, lo = [], 0
                for size in sizes:
                    hi = lo + (int(size) + CHUNK - 1) // CHUNK
                    c = self._clip_struct()
                    c.mode |= _lib.CLIP_PARTIALS_READY
                    c.chunks, c.partials = rows.data_ptr() + 32 * lo, partials.data_ptr()
                    c.n_chunks, c.chunk_base, c.n_partials = hi - lo, lo, n
                    clips.append(c)
                    lo = hi
            self._clips[ck] = (rows, partials, clips)
        return self._clips[ck][2]

    def _flat_clip(self, sizes):
        """Descriptor of a fused step over the flat buffer holding tensors of ``sizes`` (None: no clipping)."""
        if self._norm_clip:
            return self._layout("flat", tuple(int(n) for n in sizes), False)
        if self.clipvalue is not None:
            if "value" not in self._clips:
                self._clips["value"] = self._clip_struct()
            return self._clips["value"]
        return None

    # ------------------------------------------------------------------ steps
    @staticmethod
    def _flat(grads_and_vars):
        """If the list covers exactly one model's trainable variables in order, return the
        flat (params, grads) pair so that a single fused launch can be used."""
        gv = list(grads_and_vars)
        if not gv:
            return gv, None
        first = gv[0][1]
        base_w = getattr(first.value, "_base", None)
        base_w = first.value._base if first.value._base is not None else None
        if base_w is None:
            return gv, None
        total = 0
        expect = base_w.data_ptr()
        gbase = gv[0][0]._base if gv[0][0]._base is not None else None
        if gbase is None:
            return gv, None
        gexpect = gbase.data_ptr()
        for g, v in gv:
            if v.value._base is not base_w or v.value.data_ptr() != expect + 4 * total:
                return gv, None
            if g._base is not gbase or g.data_ptr() != gexpect + 4 * total:
                return gv, None
            total += v.value.numel()
        if total != base_w.numel() or gbase.numel() != total:
            return gv, None
        return gv, (base_w, gbase)

    def apply_gradients(self, grads_and_vars, grad_scale: float = 1.0):
        gv, flat = self._flat(grads_and_vars)
        if flat is not None:
            self._step(flat[0], flat[1], "flat", grad_scale, self._flat_clip([v.value.numel() for _, v in gv]))
        elif self._norm_clip:
            # per tensor: every tensor's norm pass first, then the updates, which read all partials
            gv = [(g, v) for g, v in gv if v.value.numel()]
            clips = self._layout("tensors", tuple(v.value.numel() for _, v in gv), True)
            for (g, _), clip in zip(gv, clips):
                ops.grad_clip_partials(g.reshape(-1), clip, grad_scale)
            for (g, v), clip in zip(gv, clips):
                self._step(v.value.view(-1), g.reshape(-1), v.name, grad_scale, clip)
        else:
            clip = self._flat_clip(())
            for g, v in gv:
                self._step(v.value.view(-1), g.reshape(-1), v.name, grad_scale, clip)
        self.iterations += 1

    def apply_flat(self, params, grads, grad_scale: float = 1.0, variables=None):
        """Fused step over explicit flat buffers (the data-parallel trainer's path).  ``variables``: the trainable
        variables that lie back to back in ``params`` (``model.trainable_variables``); ``clipnorm`` needs them for
        the tensor boundaries, ``global_clipnorm`` without them takes the norm of the whole buffer."""
        clip = None
        if self._norm_clip or self.clipvalue is not None:
            if variables is None:
                if self.clipnorm is not None:
                    raise ValueError("clipnorm is per variable: apply_flat needs variables=model.trainable_variables")
                sizes = (params.numel(),)
            else:
                sizes, off, base = [], 0, params.data_ptr()
                for v in variables:
                    if v.value.data_ptr() != base + 4 * off:
                        raise ValueError(f"variable {v.name} does not lie at its offset in params")
                    sizes.append(v.value.numel())
                    off += sizes[-1]
                if off != params.numel():
                    raise ValueError(f"the variables hold {off} elements, params {params.numel()}")
            clip = self._flat_clip(sizes)
        self._step(params, grads, "flat", grad_scale, clip)
        self.iterations += 1


class SGD(_Optimizer):
    def __init__(self, learning_rate=0.01, momentum=0.0, nesterov=False, name="SGD", **kwargs):
        if callable(momentum):
            raise NotImplementedError("a callable momentum is not built")
        if momentum < 0 or momentum > 1:
            raise ValueError("`momentum` must be between [0, 1].")
        super().__init__(learning_rate, **kwargs)
        self.momentum, self.nesterov = float(momentum), bool(nesterov)

    def _step(self, w, g, key, grad_scale, clip=None):
        if clip is None and self.momentum == 0.0:        # plain Keras SGD: today's kernel
            ops.sgd_step(w, g, self._lr(), grad_scale)
            return
        accum = self._slot(key, w, 1)[0] if self.momentum != 0.0 else None
        ops.sgd_step_ex(w, g, accum, self._lr(), self.momentum, self.nesterov, grad_scale, clip)


class Adam(_Optimizer):
    def __init__(self, learning_rate=0.001, beta_1=0.9, beta_2=0.999, epsilon=1e-7, amsgrad=False, name="Adam",
                 **kwargs):
        super().__init__(learning_rate, **kwargs)
        self.beta_1, self.beta_2, self.epsilon = beta_1, beta_2, epsilon
        self.amsgrad = bool(amsgrad)

    def _step(self, w, g, key, grad_scale, clip=None):
        slots = self._slot(key, w, 3 if self.amsgrad else 2)
        m, v = slots[0], slots[1]
        if clip is None and not self.amsgrad:
            ops.adam_step(w, g, m, v, self.iterations + 1, self._lr(), self.beta_1, self.beta_2, self.epsilon, grad_scale)
            return
        ops.adam_step_ex(w, g, m, v, slots[2] if self.amsgrad else None, self.iterations + 1, self._lr(), self.beta_1,
                         self.beta_2, self.epsilon, grad_scale, clip)
