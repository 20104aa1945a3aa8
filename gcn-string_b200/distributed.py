"""Data-parallel training: graphs shard across GPUs, one gradient all-reduce per step.

The reference is single-process, single-device (SURVEY.md §2: no tf.distribute, no NCCL);
this is the sharding BASELINE.json's north_star asks for.  A disjoint batch is block-diagonal:
no edge crosses graphs, pooling is per graph, the loss is a mean over graphs (SURVEY.md §8e) —
so each rank batches ITS graphs on its GPU and runs forward/backward locally, and the only
collective is one ``all_reduce(SUM)`` over the flat fp32 gradient buffer (4.26 MB at hidden
256) through torch.distributed (NCCL over NVLink; gloo on CPU in the tests).

Scaling of the mean loss: every rank back-propagates with grad_scale = 1 / global_batch
(graphs over ALL ranks; nodes over all ranks for a node-level model, pool=None), so the summed gradient is the
gradient of the mean loss over the global batch, also when shards are unequal (short last batch).

BatchNorm statistics stay replica-local (the all-reduce is the only collective): a G-GPU
step equals G reference steps on the shards with count-weighted gradient averaging, not one
reference step on the union.  Moving statistics are rank-local; rank 0's are the ones
``get_weights`` reports after ``sync_state``.
"""
from __future__ import annotations

from typing import Optional


def world():
    """(rank, world_size) from torch.distributed if initialised, else (0, 1)."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_bounds(start: int, stop: int, rank: int, world_size: int):
    """Contiguous part of the global batch slice [start, stop) owned by ``rank`` (same rule as
    data.DisjointLoader): sizes differ by at most one graph, lower ranks take the remainder."""
    n = stop - start
    base, rem = divmod(n, world_size)
    lo = start + rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def balanced_shard(ids, cost, rank: int, world_size: int):
    """The part of a global batch owned by ``rank`` when shards are balanced by WORK instead of graph
    count (SURVEY.md §8e: step time ~ nodes*H^2 + nnz*H, protein lengths are log-normal).  ``ids`` are the
    graph ids of the batch, ``cost`` their work estimates (same length).  Deterministic and identical on
    every rank: longest-processing-time greedy - graphs in descending cost (ties by position) go to the
    least-loaded rank that still has room (ties to the lowest rank).  Shard sizes are those of
    ``shard_bounds`` (they differ by at most one graph, which keeps the 1/global_batch scaling and the
    per-rank BatchNorm sample sizes as in the contiguous split); order inside a shard follows the batch."""
    import heapq
    import numpy as np
    ids = np.asarray(ids)
    cost = np.asarray(cost)
    n = ids.shape[0]
    if world_size == 1:
        return ids
    room = [shard_bounds(0, n, r, world_size)[1] - shard_bounds(0, n, r, world_size)[0] for r in range(world_size)]
    heap = [(0, r) for r in range(world_size) if room[r] > 0]
    heapq.heapify(heap)
    mine = []
    for k in np.argsort(-cost, kind="stable").tolist():
        load, r = heapq.heappop(heap)
        if r == rank:
            mine.append(k)
        room[r] -= 1
        if room[r] > 0:
            heapq.heappush(heap, (load + int(cost[k]), r))
    mine.sort()
    return ids[np.asarray(mine, dtype=np.int64)]


def allreduce_gradients(flat_grads, group=None):
    """In-place SUM all-reduce of the flat gradient bucket (no-op for a single process)."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(flat_grads, op=dist.ReduceOp.SUM, group=group)
    return flat_grads


def broadcast_parameters(model, src: int = 0, group=None):
    """Make every replica start from rank ``src``'s parameters and BatchNorm state."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.broadcast(model.params, src=src, group=group)
        dist.broadcast(model.state, src=src, group=group)


def sync_batchnorm_hook(model, group=None):
    """The all-reduce callback of synchronised BatchNorm for ``model``: sums the per-column fp64 statistics the
    native BatchNorm kernels leave in the model's workspace over all ranks (torch.distributed, on the stream the
    step runs on).  Returns ``fn(device_ptr, n_doubles, stream)`` for ``_lib.set_allreduce_hook``."""
    import torch
    import torch.distributed as dist

    def fn(ptr, n, stream):
        ws = model._ws
        off = ptr - ws.data_ptr() if ws is not None else -1
        if off < 0 or off + 8 * n > ws.numel():
            raise RuntimeError("sync-BatchNorm buffer is not inside the model workspace")
        dist.all_reduce(ws[off:off + 8 * n].view(torch.float64), op=dist.ReduceOp.SUM, group=group)
    return fn


class NativeComm:
    """The library's own NCCL communicator (gcs_comm_init): rank 0 draws the 128-byte unique id and torch.distributed
    (any backend) only carries it to the other ranks - the collectives themselves go through the C ABI
    (gcs_allreduce_grads / gcs_model_train_step_dp), as a host without torch would issue them."""

    def __init__(self, group=None):
        import ctypes
        import torch
        import torch.distributed as dist
        from . import _lib
        lib = _lib.load()
        rank, ws = world()
        ident = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            buf = (ctypes.c_char * 128)()
            _lib.check(lib.gcs_comm_unique_id(buf), "gcs_comm_unique_id")
            ident = torch.frombuffer(bytearray(buf.raw), dtype=torch.uint8).clone()
        if ws > 1:
            dev = ident.cuda() if dist.get_backend(group) == "nccl" else ident
            dist.broadcast(dev, src=0, group=group)
            ident = dev.cpu()
        handle = ctypes.c_void_p()
        raw = (ctypes.c_char * 128).from_buffer_copy(bytes(ident.numpy().tobytes()))
        _lib.check(lib.gcs_comm_init(raw, rank, ws, ctypes.byref(handle)), "gcs_comm_init")
        self.handle, self.rank, self.world_size = handle, rank, ws
        self.stream = torch.cuda.Stream()                 # the collective's own stream (overlaps the backward)
        self._lib = lib

    def allreduce_grads(self, flat):
        from . import _lib
        _lib.check(self._lib.gcs_allreduce_grads(self.handle, flat.data_ptr(), flat.numel(), _lib.stream_ptr()), "gcs_allreduce_grads")
        return flat

    def close(self):
        if self.handle:
            self._lib.gcs_comm_destroy(self.handle)
            self.handle = None


class DataParallelTrainer:
    """train_step = local fused forward/backward (grad_scale = 1/global_batch) -> one flat
    all-reduce -> fused optimizer step, identical on every rank.

    ``sync_bn=True`` additionally all-reduces the BatchNorm statistics (2H+1 doubles per layer in the forward,
    3H+1 in the backward): the step then equals ONE single-device step on the union of the shards - same loss
    gradient, same BatchNorm state on every rank - instead of a count-weighted average of per-shard steps."""

    def __init__(self, model, optimizer, group=None, sync_bn: bool = False, native_comm: bool = False, loss=None):
        """``native_comm=True``: the gradient all-reduce goes through the library's own NCCL communicator and is
        started bucket by bucket during the backward (gcs_model_train_step_dp) instead of one torch.distributed
        all-reduce after it.  ``loss``: what ``GeneralGNN.train_step_grads`` runs (None = the head's own loss;
        ``MeanSquaredError()``, ``MeanAbsoluteError()`` or ``Huber(delta)`` for a linear head)."""
        self.model, self.optimizer, self.group, self.loss = model, optimizer, group, loss
        self.sync_bn = bool(sync_bn)
        self._synced = False
        self.comm = NativeComm(group) if native_comm and world()[1] > 1 else None

    def _hooked(self, fn):
        """Run ``fn`` with the sync-BatchNorm hook installed (no-op for one process or sync_bn=False)."""
        from . import _lib
        _, ws = world()
        if not self.sync_bn or ws == 1:
            return fn()
        _lib.set_allreduce_hook(sync_batchnorm_hook(self.model, self.group), ws)
        try:
            return fn()
        finally:
            _lib.set_allreduce_hook(None)

    def train_step(self, inputs, target, global_batch: Optional[int] = None, sample_weight=None):
        """One step; ``sample_weight`` ([rows] or [rows, 1]): this rank's per-row loss weights.  With the 1/global_batch
        scaling the summed gradient is that of sum w l / global_batch, Keras' weighted mean over the global batch."""
        rank, ws = world()
        self.model.dropout_rank = rank            # per-rank dropout masks (params.dropout_seed); the all-reduce keeps
                                                  # the parameters identical
        if not self.model.built:                  # build before the first step: a dry run would move the BatchNorm statistics
            from . import _lib
            self.model.build(int(_lib.as_tensor(inputs[0]).shape[1]))
        if not self._synced:
            broadcast_parameters(self.model, 0, self.group)
            self._synced = True
        a = inputs[1]
        if global_batch is None:
            # the mean loss is over graphs, or over nodes when the model has no pool (node-level output)
            key = "global_batch_nodes" if self.model.config["pool"] is None else "global_batch_graphs"
            global_batch = getattr(a, key, None) or target.shape[0] * ws
        if self.comm is not None:                 # the library's own communicator: collectives (and synchronised BatchNorm) per call
            loss_acc, probs = self.model.train_step_grads(inputs, target, grad_scale=1.0 / float(global_batch), comm=self.comm,
                                                          sync_bn=self.sync_bn, loss=self.loss, sample_weight=sample_weight)
        else:
            step = lambda: self.model.train_step_grads(inputs, target, grad_scale=1.0 / float(global_batch),   # noqa: E731
                                                       loss=self.loss, sample_weight=sample_weight)
            loss_acc, probs = self._hooked(step)
        if self.comm is None:
            allreduce_gradients(self.model.grads, self.group)
        self.optimizer.apply_flat(self.model.params, self.model.grads, variables=self.model.trainable_variables)
        return loss_acc, probs
