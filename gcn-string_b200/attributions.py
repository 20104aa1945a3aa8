"""Residue and contact attributions of a trained ``GeneralGNN``: which residues (nodes) and which contacts (stored
adjacency entries) drive the prediction of one class.

    res = attribute(model, (x, a, i), class_index=1)
    res[g]["residues"]            # [n_g] score per residue of graph g
    rows, cols, scores = res[g]["contacts"]   # graph-local (row, col) of every stored entry of graph g and its score

The gradient is that of ``model(inputs, training=...)[:, class_index]`` (summed over the output rows), taken with the
native input-gradient backward (``GradientTape.watch`` on x and the adjacency).  ``method``:
  'saliency'      residue: sum_f |d pred / d x[n, f]|;       contact: |d pred / d w_e|
  'grad_x_input'  residue: sum_f x[n, f] * d pred / d x[n, f]; contact: w_e * d pred / d w_e
``training=False`` (the default) attributes the inference model (BatchNorm on moving statistics): each graph's scores
depend on that graph alone.  With training=True the batch statistics couple the graphs of the batch.

Contact scores need a model built with ``use_edge_weights=True``: only then does the aggregation read the edge
weights, and all-ones weights reproduce the unweighted model.  Without it ``contacts`` is None.
"""
from __future__ import annotations

import numpy as np

from . import _lib
from .models import GradientTape

METHODS = ("saliency", "grad_x_input")


def attribute(model, inputs, class_index, method="saliency", training=False):
    """Per-graph residue scores and per-contact (row, col, score) in graph-local indices; see the module docstring.
    Returns a list with one dict(residues=[n_g], contacts=(rows, cols, scores) or None) per graph (one entry for a
    single graph without batch index)."""
    torch = _lib.require_cuda()
    if method not in METHODS:
        raise ValueError(f"method must be one of {METHODS}, got {method!r}")
    x, a = inputs[0], inputs[1]
    i = inputs[2] if len(inputs) > 2 else None
    contacts = bool(model.use_edge_weights)
    with GradientTape() as tape:
        tape.watch(x)
        if contacts:
            tape.watch(a)
        pred = model(inputs, training=training)
    C = pred.shape[1]
    if not 0 <= int(class_index) < C:
        raise ValueError(f"class_index must be in [0, {C}), got {class_index}")
    og = torch.zeros_like(pred)
    og[:, int(class_index)] = 1.0
    sources = [x, a] if contacts else [x]
    grads = tape.gradient(pred, sources, output_gradients=og)
    xt = _lib.as_tensor(x).to(device="cuda", dtype=torch.float64)
    dx = grads[0].to(torch.float64)
    node = (dx.abs() if method == "saliency" else dx * xt).sum(dim=1).cpu().numpy()
    edge = None
    if contacts:
        dw = grads[1].to(torch.float64)
        w = a.edge_weight.to(dtype=torch.float64)
        edge = (dw.abs() if method == "saliency" else dw * w).cpu().numpy()
    rowptr = a.rowptr.cpu().numpy().astype(np.int64)
    colidx = a.colidx.cpu().numpy().astype(np.int64)
    return split_by_graph(graph_offsets(a, i, x.shape[0]), rowptr, colidx, node, edge)


def graph_offsets(a, i, n_nodes):
    """Node offsets [B + 1] of the graphs of a disjoint batch: the adjacency's graph_ptr, else from the sorted batch
    index i, else one graph."""
    if getattr(a, "graph_ptr", None) is not None:
        return a.graph_ptr.cpu().numpy().astype(np.int64)
    if i is None:
        return np.array([0, n_nodes], dtype=np.int64)
    seg = _lib.as_tensor(i).cpu().numpy().reshape(-1).astype(np.int64)
    n_graphs = int(seg[-1]) + 1 if seg.size else 0
    return np.concatenate([[0], np.cumsum(np.bincount(seg, minlength=n_graphs))]).astype(np.int64)


def split_by_graph(graph_ptr, rowptr, colidx, node_scores, edge_scores=None):
    """Split batch-level node scores [N] and entry scores [nnz] (CSR order) into per-graph dicts with graph-local
    indices.  The entries of graph g are those of its rows, rowptr[graph_ptr[g]] .. rowptr[graph_ptr[g + 1]]."""
    out = []
    for g in range(len(graph_ptr) - 1):
        n0, n1 = int(graph_ptr[g]), int(graph_ptr[g + 1])
        item = dict(residues=np.asarray(node_scores[n0:n1]), contacts=None)
        if edge_scores is not None:
            e0, e1 = int(rowptr[n0]), int(rowptr[n1])
            rows = np.repeat(np.arange(n0, n1), np.diff(rowptr[n0:n1 + 1])) - n0
            item["contacts"] = (rows, colidx[e0:e1] - n0, np.asarray(edge_scores[e0:e1]))
        out.append(item)
    return out
