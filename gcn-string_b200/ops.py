"""Thin functional wrappers: one Python function per C-ABI entry point.

They take torch CUDA tensors (or DLPack objects), validate dtype / device / row-major
layout, allocate the outputs and workspaces with torch's caching allocator, and enqueue on
torch's current stream.  No arithmetic happens in Python.
"""
from __future__ import annotations

import numpy as np

from typing import Optional, Tuple

from . import _lib
from ._lib import as_tensor, check, ptr, stream_ptr


def _t():
    return _lib.require_cuda()


def _mat(t, name, dtype=None):
    """Validate a row-major 2-D view; returns (tensor, leading dimension)."""
    torch = _t()
    t = as_tensor(t)
    dtype = dtype or torch.float32
    if not t.is_cuda:
        raise ValueError(f"{name} must be a CUDA tensor")
    if t.dtype != dtype:
        raise ValueError(f"{name} must be {dtype}, got {t.dtype}")
    if t.dim() != 2:
        raise ValueError(f"{name} must be rank 2, got shape {tuple(t.shape)}")
    if t.shape[1] > 1 and t.stride(1) != 1:
        raise ValueError(f"{name} must be row-major (unit stride along the last axis)")
    ld = t.stride(0) if t.shape[0] > 1 else max(t.shape[1], t.stride(0))
    if ld < t.shape[1]:
        raise ValueError(f"{name}: overlapping rows are not supported")
    return t, ld


def _vec(t, name, dtype=None, n=None):
    torch = _t()
    t = as_tensor(t)
    dtype = dtype or torch.float32
    if not t.is_cuda or t.dtype != dtype or t.dim() != 1 or not t.is_contiguous():
        raise ValueError(f"{name} must be a contiguous 1-D CUDA {dtype} tensor")
    if n is not None and t.shape[0] != n:
        raise ValueError(f"{name} must have {n} elements, got {t.shape[0]}")
    return t


def bucket_rows(n: int) -> int:
    """Leading dimension actually allocated for ``n`` rows: ``n`` itself below 4096, otherwise ``n`` rounded up to a
    multiple of 2**(bit_length(n) - 4), i.e. to 1/16 .. 1/8 of itself (at most 12.5 % more than asked for)."""
    n = int(n)
    if n < 4096:
        return n
    g = 1 << (n.bit_length() - 4)
    return (n + g - 1) // g * g


def empty_bucketed(n, *rest, dtype=None, zero=False):
    """``torch.empty((n, *rest))`` on the device, carved out of an allocation whose leading dimension is rounded up to
    1/16 .. 1/8 of its size.  The per-batch tensors of a training loop (rows, entries, features of a disjoint batch)
    change size by a per cent or two from step to step; with exact sizes the caching allocator keeps meeting requests
    it has no block for and falls through to ``cudaMalloc`` in the middle of the loop - measured: 5 ms on the launching
    thread at the least, 25-75 ms now and then, with the GPU idle behind it.  Bucketed, every step after the first few
    is served from the cache."""
    torch = _t()
    n = int(n)
    pad = bucket_rows(n)
    dtype = dtype or torch.float32
    _reserve_spares(torch, pad * int(np.prod(rest, dtype=np.int64)) * dtype.itemsize)
    make = torch.zeros if zero else torch.empty
    return make((pad, *rest), dtype=dtype, device="cuda")[:n]


_SPARES_SEEN = set()


def _reserve_spares(torch, nbytes):
    """The first time a block size is asked for, three more blocks of that size are allocated and released, and the pool
    of small blocks (< 1 MB: row-block pointers, graph pointers, labels) is grown by a few segments once: how many
    batch tensors of a size are alive at the same moment changes over the first steps (prefetch, an epoch boundary, a
    batch the caller still holds), and the caching allocator answers 'one more block of this size' with a cudaMalloc -
    5 ms on the launching thread when all goes well, 30-300 ms now and then on this pool's hosts (measured: one such
    step in every third 10-step region of bench.py, always the first step of the second epoch, a 2 MB segment for the
    small pool).  Afterwards the loop allocates nothing from the driver."""
    dev = torch.cuda.current_device()
    if (dev, 0) not in _SPARES_SEEN:
        _SPARES_SEEN.add((dev, 0))
        warm = [torch.empty(900_000, dtype=torch.uint8, device="cuda") for _ in range(16)]
        del warm
    key = (dev, int(nbytes))
    if (1 << 20) <= key[1] <= (1 << 28) and key not in _SPARES_SEEN:      # 1 MB .. 256 MB: the per-batch tensors
        _SPARES_SEEN.add(key)
        spare = [torch.empty(key[1], dtype=torch.uint8, device="cuda") for _ in range(3)]
        del spare


def _ws(nbytes):
    torch = _t()
    return empty_bucketed(max(int(nbytes), 256), dtype=torch.uint8)


def check_status_flag(flag, what):
    """Host read of a device status word (synchronises)."""
    if int(flag.item()) != 0:
        raise ValueError(what)


# ------------------------------------------------------------------ structure (K0)
def coo_to_csr(indices, n_rows: int, validate: bool = True):
    """Row-major sorted int64 COO [nnz, 2] -> (rowptr int32 [n_rows+1], colidx int32 [nnz])."""
    torch = _t()
    lib = _lib.load()
    indices = as_tensor(indices)
    if indices.dtype != torch.int64 or indices.dim() != 2 or indices.shape[1] != 2:
        raise ValueError("A.indices must be int64 of shape [nnz, 2] (a rank-2 SparseTensor)")
    indices = indices.contiguous()
    nnz = indices.shape[0]
    rowptr = torch.empty(n_rows + 1, dtype=torch.int32, device="cuda")
    colidx = torch.empty(nnz, dtype=torch.int32, device="cuda")
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    check(lib.gcs_coo_to_csr(ptr(indices), nnz, n_rows, ptr(rowptr), ptr(colidx), ptr(flag), stream_ptr()),
          "gcs_coo_to_csr")
    if validate:
        check_status_flag(flag, "A.indices must be in canonical row-major order with in-range entries "
                                "(tf.sparse.reorder); got unsorted, duplicate or out-of-range indices")
    return rowptr, colidx


def segment_ptr(seg_ids, n_graphs: int, validate: bool = True):
    torch = _t()
    lib = _lib.load()
    seg_ids = _vec(seg_ids, "i", torch.int64)
    gp = torch.empty(n_graphs + 1, dtype=torch.int32, device="cuda")
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    check(lib.gcs_segment_ptr(ptr(seg_ids), seg_ids.shape[0], n_graphs, ptr(gp), ptr(flag), stream_ptr()),
          "gcs_segment_ptr")
    if validate:
        check_status_flag(flag, "the batch index i must be sorted and within [0, n_graphs)")
    return gp


def csr_is_symmetric(rowptr, colidx) -> bool:
    torch = _t()
    lib = _lib.load()
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    check(lib.gcs_csr_is_symmetric(ptr(rowptr), ptr(colidx), rowptr.shape[0] - 1, ptr(flag), stream_ptr()),
          "gcs_csr_is_symmetric")
    return bool(flag.item())


def csr_transpose(rowptr, colidx):
    torch = _t()
    lib = _lib.load()
    n = rowptr.shape[0] - 1
    nnz = colidx.shape[0]
    rp_t = empty_bucketed(n + 1, dtype=torch.int32)
    ci_t = empty_bucketed(nnz, dtype=torch.int32)
    ws = empty_bucketed(n + 1, dtype=torch.int32)
    check(lib.gcs_csr_transpose(ptr(rowptr), ptr(colidx), n, nnz, ptr(rp_t), ptr(ci_t), ptr(ws), stream_ptr()),
          "gcs_csr_transpose")
    return rp_t, ci_t


def cast_f64_f32(x):
    torch = _t()
    lib = _lib.load()
    x = as_tensor(x).contiguous()
    out = torch.empty(x.shape, dtype=torch.float32, device="cuda")
    check(lib.gcs_cast_f64_f32(ptr(x), ptr(out), x.numel(), stream_ptr()), "gcs_cast_f64_f32")
    return out


# ------------------------------------------------------------------ dense (K1/K9)
def linear_fwd(a, w, bias=None, out=None):
    torch = _t()
    lib = _lib.load()
    a, lda = _mat(a, "A")
    w, ldw = _mat(w, "W")
    if ldw != w.shape[1]:
        raise ValueError("W must be contiguous")
    m, k = a.shape
    if w.shape[0] != k:
        raise ValueError(f"shape mismatch: A is [{m},{k}], W is {tuple(w.shape)}")
    n = w.shape[1]
    if bias is not None:
        bias = _vec(bias, "bias", n=n)
    if out is None:
        out = torch.empty(m, n, dtype=torch.float32, device="cuda")
    out, ldc = _mat(out, "C")
    ws = _ws(lib.gcs_linear_workspace_bytes(m, k, n))
    check(lib.gcs_linear_fwd(ptr(a), lda, ptr(w), ptr(bias), ptr(out), ldc, m, k, n, ptr(ws), ws.numel(), stream_ptr()),
          "gcs_linear_fwd")
    return out


def linear_bwd_weight(a, dh, want_db=True):
    torch = _t()
    lib = _lib.load()
    a, lda = _mat(a, "A")
    dh, ldh = _mat(dh, "dH")
    m, k = a.shape
    n = dh.shape[1]
    if dh.shape[0] != m:
        raise ValueError("A and dH must have the same number of rows")
    dw = torch.empty(k, n, dtype=torch.float32, device="cuda")
    db = torch.empty(n, dtype=torch.float32, device="cuda") if want_db else None
    nb = lib.gcs_linear_bwd_weight_workspace_bytes(m, k, n)
    ws = _ws(nb)
    check(lib.gcs_linear_bwd_weight(ptr(a), lda, ptr(dh), ldh, ptr(dw), ptr(db), m, k, n, ptr(ws), ws.numel(),
                                    stream_ptr()), "gcs_linear_bwd_weight")
    return dw, db


def linear_bwd_input(dh, w, out=None, accumulate=False):
    torch = _t()
    lib = _lib.load()
    dh, ldh = _mat(dh, "dH")
    w, _ = _mat(w, "W")
    w = w.contiguous()
    m, n = dh.shape
    k = w.shape[0]
    if w.shape[1] != n:
        raise ValueError("dH and W disagree on the output width")
    if out is None:
        if accumulate:
            raise ValueError("accumulate=True needs an existing output")
        out = torch.empty(m, k, dtype=torch.float32, device="cuda")
    out, lda = _mat(out, "dA")
    ws = _ws(lib.gcs_linear_workspace_bytes(m, n, k))
    check(lib.gcs_linear_bwd_input(ptr(dh), ldh, ptr(w), ptr(out), lda, m, k, n, int(accumulate), ptr(ws), ws.numel(),
                                   stream_ptr()), "gcs_linear_bwd_input")
    return out


# ------------------------------------------------------------------ BatchNorm + PReLU (K2/K8)
def bn_stats(h):
    torch = _t()
    lib = _lib.load()
    h, ldh = _mat(h, "h")
    m, c = h.shape
    mean = torch.empty(c, dtype=torch.float32, device="cuda")
    var = torch.empty(c, dtype=torch.float32, device="cuda")
    ws = _ws(lib.gcs_bn_workspace_bytes(m, c))
    check(lib.gcs_bn_stats(ptr(h), ldh, m, c, ptr(mean), ptr(var), ptr(ws), ws.numel(), stream_ptr()), "gcs_bn_stats")
    return mean, var


def bn_fold(mean, var, gamma, beta, eps=1e-3, momentum=0.99, moving_mean=None, moving_var=None):
    torch = _t()
    lib = _lib.load()
    c = mean.shape[0]
    scale = torch.empty(c, dtype=torch.float32, device="cuda")
    shift = torch.empty(c, dtype=torch.float32, device="cuda")
    check(lib.gcs_bn_fold(ptr(mean), ptr(var), ptr(gamma), ptr(beta), eps, momentum, ptr(moving_mean),
                          ptr(moving_var), ptr(scale), ptr(shift), c, stream_ptr()), "gcs_bn_fold")
    return scale, shift


def bn_prelu_fwd(h, scale, shift, alpha=None, out=None):
    torch = _t()
    lib = _lib.load()
    h, ldh = _mat(h, "h")
    m, c = h.shape
    if out is None:
        out = torch.empty(m, c, dtype=torch.float32, device="cuda")
    out, ldo = _mat(out, "out")
    check(lib.gcs_bn_prelu_fwd(ptr(h), ldh, ptr(scale), ptr(shift), ptr(alpha), ptr(out), ldo, m, c, stream_ptr()),
          "gcs_bn_prelu_fwd")
    return out


def bn_prelu_bwd(da, h, mean, var, gamma, beta, alpha=None, eps=1e-3, want_dbias=False):
    """-> (dh, dgamma, dbeta, dalpha[, dbias]); dbias = column sums of dh (bias gradient of the dense layer in front)."""
    torch = _t()
    lib = _lib.load()
    da, ldda = _mat(da, "da")
    h, ldh = _mat(h, "h")
    m, c = h.shape
    dh = torch.empty(m, c, dtype=torch.float32, device="cuda")
    dgamma = torch.empty(c, dtype=torch.float32, device="cuda")
    dbeta = torch.empty(c, dtype=torch.float32, device="cuda")
    dalpha = torch.empty(c, dtype=torch.float32, device="cuda") if alpha is not None else None
    dbias = torch.empty(c, dtype=torch.float32, device="cuda") if want_dbias else None
    ws = _ws(lib.gcs_bn_workspace_bytes(m, c))
    check(lib.gcs_bn_prelu_bwd(ptr(da), ldda, ptr(h), ldh, ptr(mean), ptr(var), ptr(gamma), ptr(beta), ptr(alpha),
                               eps, ptr(dh), c, ptr(dgamma), ptr(dbeta), ptr(dalpha), ptr(dbias), m, c, ptr(ws),
                               ws.numel(), stream_ptr()), "gcs_bn_prelu_bwd")
    return (dh, dgamma, dbeta, dalpha, dbias) if want_dbias else (dh, dgamma, dbeta, dalpha)


# ------------------------------------------------------------------ aggregation (K3/K7)
def build_rb(rowptr, colidx, height: int = 4):
    """Row-block format of a CSR pattern (block height 2 or 4) -> (blk_ptr int32 [ceil(n/height)+1],
    ent uint32-as-int32 [nnz])."""
    torch = _t()
    lib = _lib.load()
    if height not in (2, 4):
        raise ValueError("row-block height must be 2 or 4")
    n = rowptr.shape[0] - 1
    nnz = colidx.shape[0]
    n_blk = (n + height - 1) // height
    blk_ptr = empty_bucketed(n_blk + 4, dtype=torch.int32, zero=True)[:n_blk + 1]    # 3 words of slack: read in 16-byte units
    ent = empty_bucketed(max(nnz + 3 * ((n + height - 1) // height), 4), dtype=torch.int32)   # blocks are padded to 4 entries
    ws = _ws(lib.gcs_spmm_rb_workspace_bytes(n, height))
    check(lib.gcs_spmm_build_rb(ptr(rowptr), ptr(colidx), n, nnz, height, ptr(blk_ptr), ptr(ent), ptr(ws), ws.numel(),
                                stream_ptr()), "gcs_spmm_build_rb")
    return blk_ptr, ent


def build_rb4(rowptr, colidx):
    return build_rb(rowptr, colidx, 4)


def spmm_sum_graphs(graph_ptr, max_graph_nodes, rowptr, colidx, x, scale=None, shift=None, alpha=None, residual=None,
                    out=None, rb=None, rb_height=0):
    """The aggregation of a disjoint batch (gcs_spmm_sum_graphs): graph g owns rows / columns
    [graph_ptr[g], graph_ptr[g+1]); each graph's slice of x is staged in shared memory.  ``rb`` = (blk_ptr, ent) from
    ``build_rb(..., rb_height)`` or None (gathers walk the CSR).  Same results as ``spmm_sum``."""
    torch = _t()
    lib = _lib.load()
    x, ldx = _mat(x, "x")
    n, hdim = x.shape
    if rowptr.shape[0] != n + 1:
        raise ValueError(f"A has {rowptr.shape[0] - 1} rows but x has {n}")
    ldr = 0
    if residual is not None:
        residual, ldr = _mat(residual, "residual")
        if tuple(residual.shape) != (n, hdim):
            raise ValueError("residual must have the shape of the output")
    if out is None:
        out = torch.empty(n, hdim, dtype=torch.float32, device="cuda")
    out, ldy = _mat(out, "y")
    bp, en = rb if rb is not None else (None, None)
    n_graphs = graph_ptr.shape[0] - 1 if graph_ptr is not None else 0
    check(lib.gcs_spmm_sum_graphs(ptr(graph_ptr), n_graphs, int(max_graph_nodes), ptr(rowptr), ptr(colidx), ptr(bp), ptr(en),
                                  int(rb_height), n, ptr(x), ldx, ptr(scale), ptr(shift), ptr(alpha), ptr(residual), ldr,
                                  ptr(out), ldy, hdim, stream_ptr()), "gcs_spmm_sum_graphs")
    return out


def spmm_sum(rowptr, colidx, x, scale=None, shift=None, alpha=None, out=None, rb4=None):
    """Y = pattern(A) . prelu(x*scale + shift, alpha)  (identity prologue when scale is None).
    ``rb4`` = (blk_ptr, ent) from ``build_rb4`` selects the row-block kernel (same results)."""
    torch = _t()
    lib = _lib.load()
    x, ldx = _mat(x, "x")
    n, hdim = x.shape
    if rowptr.shape[0] != n + 1:
        raise ValueError(f"A has {rowptr.shape[0] - 1} rows but x has {n}")
    if out is None:
        out = torch.empty(n, hdim, dtype=torch.float32, device="cuda")
    out, ldy = _mat(out, "y")
    bp, en = rb4 if rb4 is not None else (None, None)
    check(lib.gcs_spmm_sum(ptr(rowptr), ptr(colidx), ptr(bp), ptr(en), n, ptr(x), ldx, ptr(scale), ptr(shift),
                           ptr(alpha), ptr(out), ldy, hdim, stream_ptr()), "gcs_spmm_sum")
    return out


AGGREGATE = {"sum": 0, "mean": 1, "max": 2}


def spmm_aggregate(rowptr, colidx, x, scale=None, shift=None, alpha=None, values=None, residual=None,
                   aggregate="sum", out=None, rb4=None):
    """Y = agg_j(values_ij * prelu(x[j]*scale + shift, alpha)) + residual  (gcs_spmm_aggregate).
    ``values``: float32 per stored entry in CSR order or None; ``aggregate`` in {'sum', 'mean', 'max'}
    (Spektral's scatter_sum / scatter_mean / scatter_max); ``residual``: [n, H] or None."""
    torch = _t()
    lib = _lib.load()
    if aggregate not in AGGREGATE:
        raise ValueError(f"aggregate must be one of {sorted(AGGREGATE)}")
    x, ldx = _mat(x, "x")
    n, hdim = x.shape
    if rowptr.shape[0] != n + 1:
        raise ValueError(f"A has {rowptr.shape[0] - 1} rows but x has {n}")
    if values is not None:
        if values.shape[0] != colidx.shape[0]:
            raise ValueError("values must hold one weight per stored entry")
        values = values.to(device="cuda", dtype=torch.float32).contiguous()
    ldr = 0
    if residual is not None:
        residual, ldr = _mat(residual, "residual")
        if tuple(residual.shape) != (n, hdim):
            raise ValueError("residual must have the shape of the output")
    if out is None:
        out = torch.empty(n, hdim, dtype=torch.float32, device="cuda")
    out, ldy = _mat(out, "y")
    bp, en = rb4 if rb4 is not None else (None, None)
    check(lib.gcs_spmm_aggregate(ptr(rowptr), ptr(colidx), ptr(values), ptr(bp), ptr(en), n, ptr(x), ldx, ptr(scale),
                                 ptr(shift), ptr(alpha), ptr(residual), ldr, ptr(out), ldy, hdim, AGGREGATE[aggregate],
                                 stream_ptr()), "gcs_spmm_aggregate")
    return out


def spmm_aggregate_bwd(rowptr_t, colidx_t, rowptr, colidx, dz, aggregate="sum", values_t=None, values=None, x=None,
                       scale=None, shift=None, alpha=None, z=None, out=None, ties=None):
    """Gradient of ``spmm_aggregate`` with respect to f(x) (gcs_spmm_aggregate_bwd) -> dA [n, H].
    ``(rowptr_t, colidx_t)``: the transposed pattern, ``values_t`` the weights in its entry order (with ``values``, the
    same weights in CSR order); ``dz``: dLoss/dY.  max also takes the forward's ``x`` with its prologue
    (``scale`` / ``shift`` / ``alpha``) and its output ``z``, and counts the entries that attain each maximum into
    ``ties`` [n, H] (allocated when not given)."""
    torch = _t()
    lib = _lib.load()
    if aggregate not in AGGREGATE:
        raise ValueError(f"aggregate must be one of {sorted(AGGREGATE)}")
    dz, lddz = _mat(dz, "dz")
    n, hdim = dz.shape
    if rowptr.shape[0] != n + 1 or rowptr_t.shape[0] != n + 1:
        raise ValueError(f"A and A^T must have {n} rows, like dz")
    if colidx_t.shape[0] != colidx.shape[0]:
        raise ValueError("A and A^T must have the same number of entries")
    if (values is None) != (values_t is None):
        raise ValueError("values and values_t go together (the same weights in CSR and transposed order)")
    if values is not None:
        if values.shape[0] != colidx.shape[0] or values_t.shape[0] != colidx.shape[0]:
            raise ValueError("values and values_t must hold one weight per stored entry")
        values = values.to(device="cuda", dtype=torch.float32).contiguous()
        values_t = values_t.to(device="cuda", dtype=torch.float32).contiguous()
    if (scale is None) != (shift is None) or (scale is None) != (alpha is None):
        raise ValueError("scale, shift and alpha must be all None or all set")
    if scale is not None:
        scale, shift, alpha = _vec(scale, "scale", n=hdim), _vec(shift, "shift", n=hdim), _vec(alpha, "alpha", n=hdim)
    ldx = ldz = ldt = 0
    if aggregate == "max":
        if x is None or z is None:
            raise ValueError("aggregate='max' needs the forward input x and output z")
        x, ldx = _mat(x, "x")
        z, ldz = _mat(z, "z")
        if tuple(x.shape) != (n, hdim) or tuple(z.shape) != (n, hdim):
            raise ValueError(f"x and z must be [{n}, {hdim}] like dz")
        if ties is None:
            ties = torch.empty(n, hdim, dtype=torch.float32, device="cuda")
    else:
        x = z = None                                      # read by max only
    if ties is not None:
        ties, ldt = _mat(ties, "ties")
        if tuple(ties.shape) != (n, hdim):
            raise ValueError(f"ties must be [{n}, {hdim}]")
    if out is None:
        out = torch.empty(n, hdim, dtype=torch.float32, device="cuda")
    out, ldda = _mat(out, "dA")
    if tuple(out.shape) != (n, hdim):
        raise ValueError(f"dA must be [{n}, {hdim}]")
    check(lib.gcs_spmm_aggregate_bwd(ptr(rowptr_t), ptr(colidx_t), ptr(values_t), ptr(rowptr), ptr(colidx), ptr(values), n,
                                     ptr(dz), lddz, AGGREGATE[aggregate], ptr(x), ldx, ptr(scale), ptr(shift), ptr(alpha),
                                     ptr(z), ldz, ptr(ties), ldt, ptr(out), ldda, hdim, stream_ptr()),
          "gcs_spmm_aggregate_bwd")
    return out


# ------------------------------------------------------------------ pooling (K4/K6)
def _segment_fwd(fn, x, graph_ptr, out):
    torch = _t()
    lib = _lib.load()
    x, ldx = _mat(x, "x")
    b = graph_ptr.shape[0] - 1
    w = x.shape[1]
    if out is None:
        out = torch.empty(b, w, dtype=torch.float32, device="cuda")
    out, ldo = _mat(out, "out")
    check(getattr(lib, fn)(ptr(x), ldx, ptr(graph_ptr), b, w, ptr(out), ldo, stream_ptr()), fn)
    return out


def _segment_bwd(fn, dout, graph_ptr, n_nodes, out):
    torch = _t()
    lib = _lib.load()
    dout, ldo = _mat(dout, "dout")
    b, w = dout.shape
    if out is None:
        out = torch.empty(n_nodes, w, dtype=torch.float32, device="cuda")
    out, ldx = _mat(out, "dx")
    check(getattr(lib, fn)(ptr(dout), ldo, ptr(graph_ptr), b, w, ptr(out), ldx, stream_ptr()), fn)
    return out


def segment_sum_fwd(x, graph_ptr, out=None):
    return _segment_fwd("gcs_segment_sum_fwd", x, graph_ptr, out)


def segment_sum_bwd(dout, graph_ptr, n_nodes: int, out=None):
    return _segment_bwd("gcs_segment_sum_bwd", dout, graph_ptr, n_nodes, out)


def segment_mean_fwd(x, graph_ptr, out=None):
    """tf.math.segment_mean over the graphs of graph_ptr (0 for an empty graph)."""
    return _segment_fwd("gcs_segment_mean_fwd", x, graph_ptr, out)


def segment_mean_bwd(dout, graph_ptr, n_nodes: int, out=None):
    return _segment_bwd("gcs_segment_mean_bwd", dout, graph_ptr, n_nodes, out)


def attn_sum_pool_fwd(x, kernel, graph_ptr, out=None):
    """GlobalAttnSumPool: out[g] = sum_{n in g} softmax_g(x . kernel)_n x_n.  ``kernel``: [W] or [W, 1].
    Returns (out [B, W], scores [N], gstats [B, 2] = {max_g, softmax denominator}); the last two feed the backward."""
    torch = _t()
    lib = _lib.load()
    x, ldx = _mat(x, "x")
    n, w = x.shape
    kernel = _vec(as_tensor(kernel).reshape(-1), "kernel", n=w)
    b = graph_ptr.shape[0] - 1
    if out is None:
        out = torch.empty(b, w, dtype=torch.float32, device="cuda")
    out, ldo = _mat(out, "out")
    scores = torch.empty(n, dtype=torch.float32, device="cuda")
    gstats = torch.empty(b, 2, dtype=torch.float32, device="cuda")
    ws = _ws(lib.gcs_attn_pool_workspace_bytes(n, b, w))
    check(lib.gcs_attn_sum_pool_fwd(ptr(x), ldx, n, ptr(kernel), ptr(graph_ptr), b, w, ptr(out), ldo, ptr(scores),
                                    ptr(gstats), ptr(ws), ws.numel(), stream_ptr()), "gcs_attn_sum_pool_fwd")
    return out, scores, gstats


def attn_sum_pool_bwd(dout, x, kernel, graph_ptr, out, scores, gstats, dx=None):
    """Gradient of ``attn_sum_pool_fwd`` given dout [B, W] and what the forward returned -> (dx [N, W], dkernel [W])."""
    torch = _t()
    lib = _lib.load()
    dout, lddo = _mat(dout, "dout")
    x, ldx = _mat(x, "x")
    out, ldo = _mat(out, "out")
    n, w = x.shape
    b = graph_ptr.shape[0] - 1
    kernel = _vec(as_tensor(kernel).reshape(-1), "kernel", n=w)
    scores = _vec(scores, "scores", n=n)
    gstats = _vec(as_tensor(gstats).reshape(-1), "gstats", n=2 * b)
    if tuple(dout.shape) != (b, w) or tuple(out.shape) != (b, w):
        raise ValueError(f"dout and out must be [{b}, {w}]")
    if dx is None:
        dx = torch.empty(n, w, dtype=torch.float32, device="cuda")
    dx, lddx = _mat(dx, "dx")
    dkernel = torch.empty(w, dtype=torch.float32, device="cuda")
    ws = _ws(lib.gcs_attn_pool_workspace_bytes(n, b, w))
    check(lib.gcs_attn_sum_pool_bwd(ptr(dout), lddo, ptr(x), ldx, n, ptr(kernel), ptr(graph_ptr), b, w, ptr(out), ldo,
                                    ptr(scores), ptr(gstats), ptr(dx), lddx, ptr(dkernel), ptr(ws), ws.numel(),
                                    stream_ptr()), "gcs_attn_sum_pool_bwd")
    return dx, dkernel


# ------------------------------------------------------------------ loss (K5) / optimizers (K10)
def softmax_xent(logits, y=None, grad_scale: Optional[float] = None, want_grad=False):
    """Returns (probs, loss_acc[2] or None, dlogits or None)."""
    torch = _t()
    lib = _lib.load()
    logits, _ = _mat(logits, "logits")
    logits = logits.contiguous()
    b, c = logits.shape
    probs = torch.empty_like(logits)
    loss_acc = torch.empty(2, dtype=torch.float32, device="cuda") if y is not None else None
    dlogits = torch.empty_like(logits) if (want_grad and y is not None) else None
    if y is not None:
        y, _ = _mat(y, "y")
        y = y.contiguous()
    gs = (1.0 / b if b else 0.0) if grad_scale is None else grad_scale
    check(lib.gcs_softmax_xent(ptr(logits), ptr(y), b, c, ptr(probs), ptr(loss_acc), ptr(dlogits), gs, stream_ptr()),
          "gcs_softmax_xent")
    return probs, loss_acc, dlogits


def sgd_step(w, g, lr: float, grad_scale: float = 1.0):
    lib = _lib.load()
    check(lib.gcs_sgd_step(ptr(w), ptr(g), w.numel(), lr, grad_scale, stream_ptr()), "gcs_sgd_step")


def adam_step(w, g, m, v, step: int, lr: float, beta1=0.9, beta2=0.999, eps=1e-7, grad_scale: float = 1.0):
    lib = _lib.load()
    check(lib.gcs_adam_step(ptr(w), ptr(g), ptr(m), ptr(v), w.numel(), lr, beta1, beta2, eps, step, grad_scale,
                            stream_ptr()), "gcs_adam_step")
