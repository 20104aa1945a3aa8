"""Data side of the drop-in surface: ``Graph``, ``Dataset``, ``DisjointLoader``.

Mirrors the parts of ``spektral.data`` the reference uses (src/scripts/gcn.py:9 import,
:66-197 ``MyDataset(Dataset)``, :293-294 ``dataset[idx_array]``, :316-317 loaders, :328
``tf_signature()``, :348,372 ``steps_per_epoch``, :350,367 iteration).  Upstream's collate
(np.vstack / sp.block_diag / sp.find / tf.sparse.reorder / np.repeat on the host, every
step; SURVEY.md §8 a1) is replaced by ONE upload of the packed dataset into HBM and a
device batching kernel per step (csrc/batching.cu); the host only slices the epoch
permutation and sums per-graph sizes.
"""
from __future__ import annotations

from typing import List, Optional, Sequence

import numpy as np

from . import _lib, ops
from ._lib import check, ptr, stream_ptr
from .synthetic import PackedGraphs, pack_graphs


class Graph:
    """``spektral.data.Graph``: container for x [n,F], a [n,n] (scipy sparse / ndarray), e, y."""

    def __init__(self, x=None, a=None, e=None, y=None, **kwargs):
        self.x, self.a, self.e, self.y = x, a, e, y
        for k, v in kwargs.items():
            setattr(self, k, v)

    @property
    def n_nodes(self):
        return self.x.shape[0] if self.x is not None else self.a.shape[0]

    @property
    def n_node_features(self):
        return self.x.shape[-1] if self.x is not None else None

    @property
    def n_labels(self):
        if self.y is None:
            return None
        shp = np.shape(self.y)
        return 1 if len(shp) == 0 else shp[-1]

    def numpy(self):
        return tuple(v for v in (self.x, self.a, self.e, self.y) if v is not None)

    def __repr__(self):
        return f"Graph(n_nodes={self.n_nodes}, n_node_features={self.n_node_features}, n_labels={self.n_labels})"


class Dataset:
    """``spektral.data.Dataset``: subclass and implement ``read()`` returning a list of Graph
    (the reference's MyDataset, gcn.py:66-102).  Supports ``len``, iteration, and indexing by
    int / slice / integer or boolean array (gcn.py:293-294)."""

    def __init__(self, transforms=None, **kwargs):
        for k, v in kwargs.items():
            setattr(self, k, v)
        self.graphs = self.read()
        if len(self.graphs) == 0:
            raise ValueError("Datasets cannot be empty")
        if transforms is not None:
            for t in (transforms if isinstance(transforms, (list, tuple)) else [transforms]):
                self.graphs = [t(g) for g in self.graphs]

    def read(self) -> List[Graph]:
        raise NotImplementedError

    @classmethod
    def from_graphs(cls, graphs: Sequence[Graph]) -> "Dataset":
        ds = cls.__new__(cls)
        ds.graphs = list(graphs)
        return ds

    def __len__(self):
        return len(self.graphs)

    def __iter__(self):
        return iter(self.graphs)

    def __getitem__(self, key):
        if isinstance(key, (int, np.integer)):
            return self.graphs[int(key)]
        if isinstance(key, slice):
            return Dataset.from_graphs(self.graphs[key])
        key = np.asarray(key)
        if key.dtype == bool:
            key = np.nonzero(key)[0]
        return Dataset.from_graphs([self.graphs[int(k)] for k in key])

    def __setitem__(self, key, value):
        self.graphs[key] = value

    @property
    def n_graphs(self):
        return len(self)

    @property
    def n_node_features(self):
        return self.graphs[0].n_node_features

    @property
    def n_labels(self):
        return self.graphs[0].n_labels


class SparseAdjacency:
    """What the loader yields as ``a``: a SparseTensor-like view (``indices`` [nnz,2] int64
    row-major, ``values``, ``dense_shape``) over a device CSR.  The CSR (+ its transpose,
    aliased when the pattern is symmetric) is what the kernels consume; ``indices`` is only
    materialised on request.  ``values`` exist for API compatibility and are never read:
    GeneralConv ignores adjacency values (SURVEY.md §8 a5)."""

    def __init__(self, rowptr, colidx, n_rows, graph_ptr=None, max_graph_nodes=0, indices=None,
                 symmetric: Optional[bool] = None):
        self.rowptr, self.colidx = rowptr, colidx
        self.n_rows = int(n_rows)
        self.graph_ptr = graph_ptr
        self.max_graph_nodes = int(max_graph_nodes)
        self._indices = indices
        self._symmetric = symmetric
        self._t = None
        self._rb = {}
        self._rb_t = {}
        self.edge_weight = None        # optional float32 [nnz] in CSR order; read only by GeneralGNN(use_edge_weights=True)
        self._edge_weight_t = None

    @classmethod
    def from_indices(cls, indices, dense_shape, values=None):
        """From a canonical (row-major sorted) SparseTensor triple."""
        n = int(dense_shape[0])
        if int(dense_shape[1]) != n:
            raise ValueError("A must be square")
        torch = _lib.require_cuda()
        idx = _lib.as_tensor(indices)
        if not idx.is_cuda:
            idx = idx.cuda()
        rowptr, colidx = ops.coo_to_csr(idx.to(torch.int64), n)
        return cls(rowptr, colidx, n, indices=idx)

    @property
    def nnz(self):
        return int(self.colidx.shape[0])

    @property
    def dense_shape(self):
        return (self.n_rows, self.n_rows)

    shape = dense_shape

    @property
    def indices(self):
        if self._indices is None:
            torch = _lib.require_cuda()
            counts = (self.rowptr[1:] - self.rowptr[:-1]).to(torch.int64)
            rows = torch.repeat_interleave(torch.arange(self.n_rows, device="cuda"), counts)
            self._indices = torch.stack([rows, self.colidx.to(torch.int64)], dim=1)
        return self._indices

    @property
    def values(self):
        torch = _lib.require_cuda()
        return torch.ones(self.nnz, dtype=torch.int64, device="cuda")

    @property
    def symmetric(self) -> bool:
        if self._symmetric is None:
            self._symmetric = ops.csr_is_symmetric(self.rowptr, self.colidx)
        return self._symmetric

    def rb(self, height: int = 4):
        """(blk_ptr, ent): row-block form (2 or 4 rows per block) of the pattern for the aggregation kernels."""
        if height not in self._rb:
            self._rb[height] = ops.build_rb(self.rowptr, self.colidx, height)
        return self._rb[height]

    def rb_t(self, height: int = 4):
        """Row-block form of the transposed pattern (the same arrays when symmetric)."""
        if height not in self._rb_t:
            self._rb_t[height] = self.rb(height) if self.symmetric else ops.build_rb(*self.transposed(), height)
        return self._rb_t[height]

    @property
    def rb4(self):
        return self.rb(4)

    @property
    def rb4_t(self):
        return self.rb_t(4)

    def slab_ok(self) -> bool:
        """Whether the per-graph shared-memory aggregation kernel takes this batch (the rule of csrc/spmm_slab.cu)."""
        if self.graph_ptr is None or self.max_graph_nodes <= 0:
            return False
        b = int(self.graph_ptr.shape[0]) - 1
        cap = int(_lib.load().gcs_spmm_slab_stage_bytes())
        return b > 0 and (self.max_graph_nodes + 32) * 16 <= cap and (self.n_rows // b + 32) * 64 <= cap

    def rb_height(self) -> int:
        """Block height the model entry points are given: 4 rows per block is the faster format at every width and
        degree of the cfg4 sweep (profiles/r02_cfg4_spmm_sweep.jsonl; 2 rows per block only ties at degree 4)."""
        return 4

    def edge_weight_t(self):
        """The edge weights in the entry order of the transposed pattern (columns ascending, then rows).  Cached per
        tensor and per in-place version of it: ``a.edge_weight.copy_(w)`` between two steps is seen by the backward."""
        if self.edge_weight is None:
            return None
        w = self.edge_weight
        if self._edge_weight_t is None or self._edge_weight_t[0] is not w or self._edge_weight_t[1] != w._version:
            torch = _lib.require_cuda()
            counts = (self.rowptr[1:] - self.rowptr[:-1]).to(torch.int64)
            rows = torch.repeat_interleave(torch.arange(self.n_rows, device="cuda"), counts)
            key = self.colidx.to(torch.int64) * self.n_rows + rows
            self._edge_weight_t = (w, w._version, w[torch.argsort(key)].contiguous())
        return self._edge_weight_t[2]

    def transposed(self):
        """(rowptr_t, colidx_t) of pattern(A)^T; the same arrays when symmetric."""
        if self._t is None:
            self._t = (self.rowptr, self.colidx) if self.symmetric else ops.csr_transpose(self.rowptr, self.colidx)
        return self._t


class _PinnedRing:
    """Small host -> device uploads of the steady-state loop (graph ids of a batch, the epoch's permutation, gather
    offsets) staged through a ring of PERSISTENT pinned buffers.  ``tensor.pin_memory()`` per step looks harmless - the
    host allocator caches its blocks - but every miss is a ``cudaHostAlloc``, which takes the driver's lock and was
    measured to stall the launching thread for 30-190 ms now and then (one such step at every epoch boundary of
    bench.py in about one run out of five).  A slot is reused only after the copy out of it has run (its event)."""

    def __init__(self, depth=4):
        self.bufs, self.events, self.k = [None] * depth, [None] * depth, 0

    def stage(self, arr):
        """A pinned tensor holding a copy of the NumPy array ``arr``; pass the returned slot to ``uploaded``."""
        torch = _lib.require_cuda()
        arr = np.ascontiguousarray(arr)
        k = self.k
        self.k = (k + 1) % len(self.bufs)
        if self.events[k] is not None:
            self.events[k].synchronize()                       # long since complete in a running loop
            self.events[k] = None
        nbytes = max(int(arr.nbytes), 8)
        if self.bufs[k] is None or self.bufs[k].numel() < nbytes:
            # set-up / growth only, and for ALL slots at once: the first use pays every cudaHostAlloc of the ring
            for e in self.events:
                if e is not None:
                    e.synchronize()
            self.events = [None] * len(self.bufs)
            self.bufs = [torch.empty(2 * nbytes, dtype=torch.uint8).pin_memory() for _ in self.bufs]
        t = self.bufs[k][:arr.nbytes].view(getattr(torch, str(arr.dtype))).view(arr.shape)
        t.numpy()[...] = arr
        return t, k

    def uploaded(self, k):
        """Call after enqueueing the copy out of slot k on the current stream."""
        torch = _lib.require_cuda()
        ev = torch.cuda.Event()
        ev.record()
        self.events[k] = ev

    def upload(self, arr):
        """Stage + asynchronous copy to a fresh device tensor on the current stream."""
        t, k = self.stage(arr)
        dev = t.cuda(non_blocking=True)
        self.uploaded(k)
        return dev


class DeviceGraphStore:
    """The packed dataset resident in HBM + the host-side per-graph sizes."""

    def __init__(self, packed: PackedGraphs, symmetric: Optional[bool] = None):
        torch = _lib.require_cuda()
        _lib.load()
        self.n_graphs = packed.n_graphs
        self.n_feat = int(packed.x.shape[1])
        self.n_classes = int(packed.y.shape[1]) if packed.y.ndim == 2 else 0
        self.h_n_nodes = packed.n_nodes.astype(np.int64)
        self.h_n_edges = packed.n_edges.astype(np.int64)
        self.node_off = torch.from_numpy(packed.node_off).cuda()
        self.rowptr = torch.from_numpy(packed.rowptr).cuda()
        self.col = torch.from_numpy(packed.col).cuda()
        self.x = torch.from_numpy(np.ascontiguousarray(packed.x, dtype=np.float32)).cuda()
        self.y = torch.from_numpy(np.ascontiguousarray(packed.y, dtype=np.float32)).cuda() if self.n_classes else None
        self.node_level = bool(packed.node_level)
        self.symmetric = symmetric

    def batch(self, graph_ids_dev, graph_ids_host, want_coo=False, want_labels=True):
        """Run K0 for the graphs ``graph_ids`` (device int64 tensor + the same ids on host); node labels are then
        gathered by gcs_gather_node_rows at the graph offsets K0 wrote."""
        torch = _lib.require_cuda()
        lib = _lib.load()
        b = int(graph_ids_host.shape[0])
        n = int(self.h_n_nodes[graph_ids_host].sum())
        nnz = int(self.h_n_edges[graph_ids_host].sum())
        max_nodes = int(self.h_n_nodes[graph_ids_host].max()) if b else 0
        i32 = dict(dtype=torch.int32, device="cuda")
        graph_ptr = torch.empty(b + 1, **i32)
        edge_ptr = torch.empty(b + 1, **i32)
        rowptr = ops.empty_bucketed(n + 1, dtype=torch.int32)          # bucketed sizes: no cudaMalloc inside a running loop
        colidx = ops.empty_bucketed(nnz, dtype=torch.int32)
        x = ops.empty_bucketed(n, self.n_feat, dtype=torch.float32)
        seg = ops.empty_bucketed(n, dtype=torch.int64)
        y = None
        if want_labels and self.y is not None:
            y = (ops.empty_bucketed(n, self.n_classes, dtype=torch.float32) if self.node_level
                 else torch.empty(b, self.n_classes, dtype=torch.float32, device="cuda"))
        coo = ops.empty_bucketed(nnz, 2, dtype=torch.int64) if want_coo else None
        flag = torch.zeros(1, **i32)
        graph_y = None if self.node_level else self.y
        check(lib.gcs_batch_disjoint(ptr(self.node_off), ptr(self.rowptr), ptr(self.col), ptr(self.x), ptr(graph_y),
                                     self.n_feat, max(self.n_classes, 1), ptr(graph_ids_dev), b, n, nnz,
                                     ptr(graph_ptr), ptr(edge_ptr), ptr(rowptr), ptr(colidx), ptr(x), ptr(seg),
                                     None if self.node_level else ptr(y), ptr(coo), ptr(flag), stream_ptr()),
              "gcs_batch_disjoint")
        if self.node_level and y is not None:
            check(lib.gcs_gather_node_rows(ptr(graph_ids_dev), b, ptr(self.node_off), ptr(self.y), self.n_classes,
                                           ptr(graph_ptr), ptr(y), stream_ptr()), "gcs_gather_node_rows")
        a = SparseAdjacency(rowptr, colidx, n, graph_ptr=graph_ptr, max_graph_nodes=max_nodes, indices=coo,
                            symmetric=self.symmetric)
        a.edge_ptr = edge_ptr
        a.status = flag
        return x, a, seg, y


class HostGraphStore:
    """Streaming variant: the packed dataset stays in PINNED host memory and every step moves only the graphs of its
    batch to the device, inside the step.
    ``zero_copy=False`` (default): consecutive graph ids (shuffle=False) are uploaded as slices with cudaMemcpyAsync; a
    shuffled batch is first gathered into a pinned staging buffer on the host, then uploaded; the batching kernel runs
    on the copies.
    ``zero_copy=True``: the batching kernel itself reads the batch's graphs out of the pinned host arrays (they are
    device-addressable under unified virtual addressing) - no CPU-side packing, no staging buffer.  Measured on B200
    (cfg3 step, 94 MB per batch): the kernel's row-granular reads reach only 4-6 GB/s over the host link, 18.8-27 ms
    per step against 17.6 ms for the sliced upload, so it is an option for shuffled epochs, not the default."""

    def __init__(self, packed: PackedGraphs, symmetric: Optional[bool] = None, zero_copy: bool = False,
                 device_gather: bool = False):
        self.zero_copy = bool(zero_copy)
        # device_gather=True: a non-consecutive (shuffled) batch is gathered by gcs_gather_graphs - a kernel that copies
        # each selected graph's slices out of the pinned arrays in coalesced runs - instead of a Python loop on the host
        self.device_gather = bool(device_gather)
        torch = _lib.require_cuda()
        _lib.load()
        self.n_graphs = packed.n_graphs
        self.n_feat = int(packed.x.shape[1])
        self.n_classes = int(packed.y.shape[1]) if packed.y.ndim == 2 else 0
        self.h_n_nodes = packed.n_nodes.astype(np.int64)
        self.h_n_edges = packed.n_edges.astype(np.int64)
        self.h_node_off = packed.node_off
        self.h_rowptr = packed.rowptr
        pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()   # noqa: E731
        self.node_off, self.rowptr, self.col = pin(packed.node_off), pin(packed.rowptr), pin(packed.col)
        self.x = pin(packed.x.astype(np.float32, copy=False))
        self.y = pin(packed.y.astype(np.float32, copy=False)) if self.n_classes else None
        self.node_level = bool(packed.node_level)
        self.symmetric = symmetric
        self.h2d_bytes_last = 0
        self._ring = _PinnedRing(depth=6)

    def _gather(self, ids):
        """Pack the graphs ``ids`` (any order) into a fresh pinned mini-dataset."""
        torch = _lib.require_cuda()
        sub = PackedGraphs(*_take_graphs(self, ids), node_level=self.node_level)
        pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()   # noqa: E731
        return pin(sub.node_off), pin(sub.rowptr), pin(sub.col), pin(sub.x), (pin(sub.y) if self.n_classes else None)

    def batch(self, graph_ids_dev, graph_ids_host, want_coo=False, want_labels=True):
        torch = _lib.require_cuda()
        lib = _lib.load()
        ids = np.asarray(graph_ids_host, dtype=np.int64)
        b = int(ids.shape[0])
        consecutive = b > 0 and np.array_equal(ids, np.arange(ids[0], ids[0] + b))
        if self.zero_copy:
            parts = (self.node_off, self.rowptr, self.col, self.x, self.y)           # the pinned dataset itself
            g0 = n0 = e0 = 0
            ids_local = torch.from_numpy(ids)
        elif consecutive:
            g0, g1 = int(ids[0]), int(ids[0]) + b
            n0, n1 = int(self.h_node_off[g0]), int(self.h_node_off[g1])
            e0, e1 = int(self.h_rowptr[n0]), int(self.h_rowptr[n1])
            y_rows = (n0, n1) if self.node_level else (g0, g1)        # node labels: one contiguous node range
            parts = (self.node_off[g0:g1 + 1], self.rowptr[n0:n1 + 1], self.col[e0:e1], self.x[n0:n1],
                     self.y[y_rows[0]:y_rows[1]] if self.y is not None else None)
            ids_local = torch.arange(g0, g1, dtype=torch.int64)
        elif self.device_gather:
            parts = None
            g0 = n0 = e0 = 0
            ids_local = torch.arange(0, b, dtype=torch.int64)
        else:
            parts = self._gather(ids)
            g0 = n0 = e0 = 0
            ids_local = torch.arange(0, b, dtype=torch.int64)
        n = int(self.h_n_nodes[ids].sum())
        nnz = int(self.h_n_edges[ids].sum())
        if self.zero_copy:
            dev = list(parts)
            # uploaded on THIS stream: with prefetch the kernel runs on a side stream, which is not ordered after the
            # loader's asynchronous upload of the epoch order (graph_ids_dev)
            ids_dev = self._ring.upload(ids_local.numpy())
            # bytes the kernel pulls over the host link: per graph its node offsets, row pointers, columns, features, label
            self.h2d_bytes_last = (16 * b + 8 * (n + b) + 4 * nnz + 4 * self.n_feat * n
                                   + 4 * self.n_classes * (n if self.node_level else b) + 8 * b)
        elif parts is None:
            # the selected graphs' offsets in the mini-dataset (host knows the sizes), then one gather kernel
            off = np.zeros((3, b + 1), dtype=np.int64)
            np.cumsum(self.h_n_nodes[ids], out=off[0, 1:])
            np.cumsum(self.h_n_edges[ids], out=off[1, 1:])
            off[2, :b] = ids
            off_dev = self._ring.upload(off)
            d_node_off = off_dev[0]
            d_rowptr = ops.empty_bucketed(n + 1, dtype=torch.int64)
            d_col = ops.empty_bucketed(max(nnz, 1), dtype=torch.int32)
            d_x = ops.empty_bucketed(max(n, 1), self.n_feat, dtype=torch.float32)
            # node labels are gathered straight into the batch after K0 (gcs_gather_node_rows), not into the mini-dataset
            graph_y = None if self.node_level else self.y
            d_y = torch.empty(b, self.n_classes, dtype=torch.float32, device="cuda") if graph_y is not None else None
            check(lib.gcs_gather_graphs(ptr(off_dev[2]), b, ptr(self.node_off), ptr(self.rowptr), ptr(self.col), ptr(self.x),
                                        ptr(graph_y), self.n_feat, self.n_classes, ptr(off_dev[0]), ptr(off_dev[1]),
                                        ptr(d_rowptr), ptr(d_col), ptr(d_x), ptr(d_y), stream_ptr()), "gcs_gather_graphs")
            dev = [d_node_off, d_rowptr, d_col, d_x, d_y]
            ids_dev = self._ring.upload(ids_local.numpy())
            self.h2d_bytes_last = (16 * b + 8 * (n + b) + 4 * nnz + 4 * self.n_feat * n
                                   + 4 * self.n_classes * (n if self.node_level else b) + 24 * (b + 1))
        else:
            dev = []
            for t in parts:                              # pinned slices -> bucketed device buffers
                if t is None:
                    dev.append(None)
                    continue
                d = ops.empty_bucketed(t.shape[0], *t.shape[1:], dtype=t.dtype)
                d.copy_(t, non_blocking=True)
                dev.append(d)
            ids_dev = self._ring.upload(ids_local.numpy())
            self.h2d_bytes_last = sum(t.numel() * t.element_size() for t in parts if t is not None) + ids_local.numel() * 8
        d_node_off, d_rowptr, d_col, d_x, d_y = dev
        max_nodes = int(self.h_n_nodes[ids].max()) if b else 0
        i32 = dict(dtype=torch.int32, device="cuda")
        graph_ptr, edge_ptr = torch.empty(b + 1, **i32), torch.empty(b + 1, **i32)
        rowptr, colidx = ops.empty_bucketed(n + 1, dtype=torch.int32), ops.empty_bucketed(nnz, dtype=torch.int32)
        x = ops.empty_bucketed(n, self.n_feat, dtype=torch.float32)
        seg = ops.empty_bucketed(n, dtype=torch.int64)
        coo = ops.empty_bucketed(nnz, 2, dtype=torch.int64) if want_coo else None
        flag = torch.zeros(1, **i32)
        if self.node_level:
            y, graph_y = None, None
            if want_labels and self.y is not None:
                if parts is not None and not self.zero_copy:
                    y = d_y                      # the copied slice / staged rows are already the batch's rows, in order
                else:
                    y = ops.empty_bucketed(n, self.n_classes, dtype=torch.float32)
        else:
            y = torch.empty(b, self.n_classes, dtype=torch.float32, device="cuda") if (want_labels and d_y is not None) else None
            graph_y = (ptr(d_y) - 4 * self.n_classes * g0) if d_y is not None else None
        # the uploaded slices are addressed with DATASET-global ids: rebase the pointers instead
        # of the index arrays (the kernel only touches [g0, g1], [n0, n1], [e0, e1))
        check(lib.gcs_batch_disjoint(ptr(d_node_off) - 8 * g0, ptr(d_rowptr) - 8 * n0, ptr(d_col) - 4 * e0,
                                     ptr(d_x) - 4 * self.n_feat * n0, graph_y,
                                     self.n_feat, max(self.n_classes, 1), ptr(ids_dev), b, n, nnz, ptr(graph_ptr),
                                     ptr(edge_ptr), ptr(rowptr), ptr(colidx), ptr(x), ptr(seg),
                                     None if self.node_level else ptr(y), ptr(coo), ptr(flag), stream_ptr()),
              "gcs_batch_disjoint")
        if self.node_level and y is not None and y is not d_y:
            # zero_copy: the batch's graph ids index the pinned dataset; device_gather: the same ids (off_dev[2])
            gids = ids_dev if self.zero_copy else off_dev[2]
            check(lib.gcs_gather_node_rows(ptr(gids), b, ptr(self.node_off), ptr(self.y), self.n_classes, ptr(graph_ptr),
                                           ptr(y), stream_ptr()), "gcs_gather_node_rows")
        a = SparseAdjacency(rowptr, colidx, n, graph_ptr=graph_ptr, max_graph_nodes=max_nodes, indices=coo,
                            symmetric=self.symmetric)
        a.edge_ptr, a.status = edge_ptr, flag
        a._keep = (dev, ids_dev)
        return x, a, seg, y


def _take_graphs(store, ids):
    """Host gather of whole graphs into a packed mini-dataset (node_off, rowptr, col, x, y)."""
    node_off = np.zeros(len(ids) + 1, dtype=np.int64)
    np.cumsum(store.h_n_nodes[ids], out=node_off[1:])
    hn, hr = store.h_node_off, store.h_rowptr
    col_np, x_np = store.col.numpy(), store.x.numpy()
    rp_np = store.rowptr.numpy()
    rps, cols, xs, ys = [], [], [], []
    e_off = 0
    y_np = store.y.numpy() if store.y is not None else None
    for g in ids:
        n0, n1 = int(hn[g]), int(hn[g + 1])
        e0, e1 = int(hr[n0]), int(hr[n1])
        rps.append(rp_np[n0:n1] - e0 + e_off)
        cols.append(col_np[e0:e1])
        xs.append(x_np[n0:n1])
        if store.node_level and y_np is not None:
            ys.append(y_np[n0:n1])
        e_off += e1 - e0
    rowptr = np.concatenate(rps + [np.array([e_off], dtype=np.int64)])
    if y_np is None:
        y = np.zeros((len(ids), 0), np.float32)
    else:
        y = np.concatenate(ys) if store.node_level else y_np[ids]
    return node_off, rowptr, np.concatenate(cols), np.concatenate(xs), y


class _Spec:
    """Stand-in for tf.TensorSpec / tf.SparseTensorSpec in ``tf_signature()``."""

    def __init__(self, shape, dtype, sparse=False):
        self.shape, self.dtype, self.sparse = shape, dtype, sparse

    def __repr__(self):
        return f"{'Sparse' if self.sparse else ''}TensorSpec(shape={self.shape}, dtype={self.dtype})"


class DisjointLoader:
    """``spektral.data.DisjointLoader(dataset, node_level=False, batch_size=1, epochs=None,
    shuffle=True)``.  Iterating yields ``((x, a, i), y)`` with everything on the device: y [B, C] graph labels, or
    with ``node_level=True`` y [N, C], the graphs' node labels stacked in batch order (Spektral's np.vstack).

    Batch order follows upstream's ``batch_generator``: per epoch an in-place
    ``np.random.shuffle`` (cumulative across epochs, global NumPy RNG), then consecutive
    slices of ``batch_size``; the last batch may be short; ``steps_per_epoch =
    ceil(len / batch_size)``.  With ``device_resident=False`` the dataset stays in pinned host
    memory and each step uploads its own graphs.  ``dataset`` may be a ``Dataset``, a list of ``Graph`` or an
    already packed ``PackedGraphs``.  ``rank`` / ``world_size`` shard every global batch by
    graph across data-parallel ranks (rank r takes the r-th contiguous part of the slice); the adjacency carries the
    global slice's graph and node counts (``a.global_batch_graphs`` / ``a.global_batch_nodes``), the denominators of
    the graph- and node-level mean loss.

    ``sample_weights`` (the name of Spektral's ``SingleLoader`` argument): a host array with one loss weight per graph,
    or with ``node_level=True`` one per node in dataset order ([n] or [n, 1]).  Iterating then yields
    ``((x, a, i), y, w)``, w [B] or [N] float32 on the device in batch order, for ``loss_fn(y, pred, sample_weight=w)``
    or ``train_step_grads(..., sample_weight=w)``.  The weights are kept in HBM in every store mode (4 bytes per row) and
    gathered per batch by the batch's graph ids: ``index_select`` per graph, ``gcs_gather_node_rows`` at width 1 per
    node, into buffers of bucketed size.
    """

    def __init__(self, dataset, node_level=False, batch_size=1, epochs=None, shuffle=True, rank=0, world_size=1,
                 want_coo=False, symmetric=None, device_resident=True, prefetch=None, balance=None, zero_copy=False,
                 device_gather=False, sample_weights=None):
        node_level = bool(node_level)
        packed = dataset if isinstance(dataset, PackedGraphs) else pack_graphs(list(dataset), node_level=node_level)
        if packed.n_graphs == 0:
            raise ValueError("Datasets cannot be empty")
        if bool(packed.node_level) != node_level:
            raise ValueError(f"DisjointLoader(node_level={node_level}) got a dataset with "
                             f"{'node' if packed.node_level else 'graph'} labels")
        if symmetric is None:
            symmetric = getattr(packed, "symmetric", None)      # recorded by the shard writer (shards.py)
        self.dataset = dataset
        # device_resident=False keeps the dataset in pinned host memory and uploads per batch
        self.store = (DeviceGraphStore(packed, symmetric=symmetric) if device_resident
                      else HostGraphStore(packed, symmetric=symmetric, zero_copy=zero_copy, device_gather=device_gather))
        self.node_level = node_level
        self.batch_size = int(batch_size)
        self.epochs = epochs
        self.shuffle = shuffle
        self.rank, self.world_size = int(rank), int(world_size)
        if balance not in (None, "count", "nnz"):
            raise ValueError("balance must be None, 'count' or 'nnz'")
        # 'nnz': shards of a global batch are balanced by stored entries + nodes (distributed.balanced_shard) instead
        # of being contiguous runs of equal graph count
        self.balance = None if balance == "count" else balance
        self.want_coo = want_coo
        # one batch ahead on a side stream: the H2D upload (host-resident store) and the batching
        # kernels of step t+1 overlap the training step t
        self.prefetch = (not device_resident) if prefetch is None else bool(prefetch)
        self._n = packed.n_graphs
        self._order = np.arange(self._n, dtype=np.int64)
        self._order_dev = None
        self._order_epoch = -1
        self._ring = _PinnedRing(depth=4)
        self._w, self._w_node_off = None, None
        if sample_weights is not None:
            torch = _lib.require_cuda()
            rows = int(packed.node_off[-1]) if node_level else packed.n_graphs
            w = np.asarray(sample_weights, dtype=np.float32)
            ops.check_sample_weight_shape(w.shape, rows)
            self._w = torch.from_numpy(np.ascontiguousarray(w.reshape(rows))).cuda()
            if node_level:
                self._w_node_off = (self.store.node_off if device_resident
                                    else torch.from_numpy(np.ascontiguousarray(packed.node_off)).cuda())
        self._generator = self._generate()

    @property
    def steps_per_epoch(self) -> int:
        """ceil(len / batch_size) as upstream; under data parallelism a short last batch with fewer graphs than ranks is
        dropped on EVERY rank (each rank decides from the global slice, so no rank enters the gradient all-reduce
        alone)."""
        full, tail = divmod(self._n, self.batch_size)
        return full + (1 if tail >= max(self.world_size, 1) else 0)

    def __len__(self):
        return self.steps_per_epoch

    def __iter__(self):
        return self

    def __next__(self):
        return next(self._generator)

    def load(self):
        return self

    def tf_signature(self):
        """Shape/dtype contract of one batch (gcn.py:328): dynamic N, nnz, B."""
        f, c = self.store.n_feat, self.store.n_classes
        spec = ((_Spec((None, f), "float32"), _Spec((None, None), "int64", sparse=True), _Spec((None,), "int64")),
                _Spec((None, c), "float32"))
        return spec + ((_Spec((None,), "float32"),) if self._w is not None else ())

    def _slices_of_rank(self, start, stop):
        """This rank's contiguous part of the global slice [start, stop)."""
        if self.world_size == 1:
            return start, stop
        n = stop - start
        base, rem = divmod(n, self.world_size)
        lo = start + self.rank * base + min(self.rank, rem)
        return lo, lo + base + (1 if self.rank < rem else 0)

    def _slices(self):
        """(epoch, lo, hi, host ids, (global batch graphs, global batch nodes)) of every step, epoch after epoch.  Nothing is uploaded here:
        the device copies of the ids are made by _launch on the stream the batching kernels run on."""
        epochs = np.inf if self.epochs is None or self.epochs == -1 else self.epochs
        epoch = 0
        while epoch < epochs:
            epoch += 1
            if self.shuffle:
                np.random.shuffle(self._order)
            order_host = self._order.copy()
            for b in range(int(np.ceil(self._n / self.batch_size))):
                start = b * self.batch_size
                stop = min(start + self.batch_size, self._n)
                if stop - start < self.world_size:
                    continue                       # a tail shorter than the number of ranks: dropped by every rank alike
                lo, hi = self._slices_of_rank(start, stop)
                nodes = int(self.store.h_n_nodes[order_host[start:stop]].sum())
                if self.balance == "nnz" and self.world_size > 1:
                    from .distributed import balanced_shard
                    ids = order_host[start:stop]
                    cost = self.store.h_n_edges[ids] + 4 * self.store.h_n_nodes[ids]
                    mine = np.ascontiguousarray(balanced_shard(ids, cost, self.rank, self.world_size))
                    yield epoch, None, None, mine, (stop - start, nodes), order_host
                else:
                    yield epoch, lo, hi, order_host[lo:hi], (stop - start, nodes), order_host

    def _launch(self, item, stream):
        """Enqueue upload + batching kernels for one step on `stream`.  The graph ids go to the device on the SAME
        stream (pinned staging, asynchronous copy): the batching kernels that read them are ordered behind the copy by
        the stream itself, whichever stream the training step runs on."""
        torch = _lib.require_cuda()
        epoch, lo, hi, ids_host, (global_count, global_nodes), order_host = item
        with torch.cuda.stream(stream):
            # persistent pinned staging (see _PinnedRing: no pinned allocation inside the loop)
            if lo is None:                                     # work-balanced shard: its own id list
                ids_dev = self._ring.upload(ids_host)
            else:
                if self._order_epoch != epoch:                 # one upload of the epoch's permutation, then slices of it
                    self._order_dev = self._ring.upload(order_host)
                    self._order_epoch = epoch
                ids_dev = self._order_dev[lo:hi]
            staged = None
            x, a, i, y = self.store.batch(ids_dev, ids_host, want_coo=self.want_coo)
            w = self._batch_weights(ids_dev, a) if self._w is not None else None
            a.global_batch_graphs = global_count
            a.global_batch_nodes = global_nodes
            a._ids_keepalive = (ids_dev, staged)
            event = torch.cuda.Event()
            event.record(stream)
        return (x, a, i, y, w), event

    def _batch_weights(self, ids_dev, a):
        """The batch's sample weights in batch order: the weights of its graphs, or of its nodes graph after graph at
        the offsets the batching kernel wrote (a.graph_ptr)."""
        torch = _lib.require_cuda()
        b = int(ids_dev.shape[0])
        if not self.node_level:
            w = torch.empty(b, dtype=torch.float32, device="cuda")
            return torch.index_select(self._w, 0, ids_dev, out=w)
        w = ops.empty_bucketed(a.n_rows, dtype=torch.float32)
        check(_lib.load().gcs_gather_node_rows(ptr(ids_dev), b, ptr(self._w_node_off), ptr(self._w), 1, ptr(a.graph_ptr),
                                               ptr(w), stream_ptr()), "gcs_gather_node_rows")
        return w

    def _generate(self):
        torch = _lib.require_cuda()
        it = self._slices()
        if not self.prefetch:
            for item in it:
                (x, a, i, y, w), _ = self._launch(item, torch.cuda.current_stream())
                yield ((x, a, i), y, w) if w is not None else ((x, a, i), y)
            return
        side = torch.cuda.Stream()
        first = next(it, None)
        pending = self._launch(first, side) if first is not None else None
        while pending is not None:
            (x, a, i, y, w), event = pending
            nxt = next(it, None)
            pending = self._launch(nxt, side) if nxt is not None else None      # step t+1 in flight
            main = torch.cuda.current_stream()
            main.wait_event(event)
            for t in (x, i, y, w, a.rowptr, a.colidx, a.graph_ptr, a.edge_ptr, a.status, a._indices):
                if t is not None:
                    t.record_stream(main)       # allocated on the side stream, consumed on the main one
            yield ((x, a, i), y, w) if w is not None else ((x, a, i), y)
