"""Synthetic "E. coli inter-protein shape" graphs (SURVEY.md §8d) as a packed store.

What the reference's offline generator emits per protein pair, restated as a sampler
(reference: src/utilities/gcn_utills.py):
  * two proteins, one residue per node, node order = protein a then protein b
    (``nx.union`` with a-/b- prefixes, gcn_utills.py:345; relabelled to ints at
    src/scripts/gcn.py:189);
  * per protein a symmetric CA-CA contact graph WITH self-loops (10 A threshold on a
    distance matrix whose diagonal is 0, gcn_utills.py:225-227,256-257) - here a band
    |i-j| <= w plus long-range contacts with P(d) ~ 1/d;
  * 20 symmetric inter-protein DCA "bridge" edges (gcn_utills.py:87,345-351);
  * adjacency values are all 1 (src/scripts/gcn.py:187-197 pops ``weight``);
  * node features: 16 NetSurfP columns in the real data (gcn_utills.py:293-311),
    mostly probabilities -> U[0,1); width F is a parameter (BASELINE.json uses 32);
  * labels one-hot [0,1] positive / [1,0] negative, balanced (src/scripts/gcn.py:259,262);
    ``node_level=True`` instead labels every residue (a per-residue task such as interface residues): one-hot of the
    argmax of a fixed random projection of the summed neighbour features, which a GeneralGNN can learn;
    ``task='regression'`` gives continuous targets instead: tanh of that projection per residue, or its mean over
    each graph (a continuous score per protein pair).

Everything is NumPy with ``default_rng(seed + graph_id)`` so any graph can be
regenerated alone.  The output is the packed layout the device batching kernel consumes
(``PackedGraphs``): per-graph CSR with LOCAL column indices, concatenated.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List

import numpy as np


@dataclass
class PackedGraphs:
    """Concatenated per-graph CSR + features + labels (host, NumPy).

    node_off[G+1]  int64  node offset of each graph in ``x`` / ``rowptr``
    rowptr[sumN+1] int64  start of each node's neighbour list in ``col`` (dataset-global)
    col[sumNNZ]    int32  neighbour index LOCAL to the graph, ascending within a row
    x[sumN, F]     float32
    y[G, C]        float32 one-hot graph labels, or y[sumN, C] node labels (rows in node order) when node_level
    """
    node_off: np.ndarray
    rowptr: np.ndarray
    col: np.ndarray
    x: np.ndarray
    y: np.ndarray
    node_level: bool = False

    @property
    def n_graphs(self) -> int:
        return int(self.node_off.shape[0] - 1)

    @property
    def n_nodes(self) -> np.ndarray:
        return np.diff(self.node_off)

    @property
    def n_edges(self) -> np.ndarray:
        return self.rowptr[self.node_off[1:]] - self.rowptr[self.node_off[:-1]]

    def graph(self, g: int):
        """(x[n,F], scipy CSR int64 ones [n,n], y[C]) for graph g — the per-graph objects
        the reference's MyDataset hands to Spektral (src/scripts/gcn.py:161-181)."""
        import scipy.sparse as sp
        n0, n1 = int(self.node_off[g]), int(self.node_off[g + 1])
        e0, e1 = int(self.rowptr[n0]), int(self.rowptr[n1])
        n = n1 - n0
        a = sp.csr_matrix((np.ones(e1 - e0, dtype=np.int64), self.col[e0:e1].astype(np.int32),
                           (self.rowptr[n0:n1 + 1] - e0).astype(np.int32)), shape=(n, n))
        return self.x[n0:n1], a, (self.y[n0:n1] if self.node_level else self.y[g])


def _protein_pairs(rng, n, deg):
    """Undirected contact keys i*n+j (i<j) of one protein: band + 1/d long-range."""
    lr_per_node = 3 if deg >= 8 else 1
    w = max(1, (deg - 1 - lr_per_node) // 2)
    w = min(w, max(1, n - 1))
    i = np.repeat(np.arange(n, dtype=np.int64), w)
    d = np.tile(np.arange(1, w + 1, dtype=np.int64), n)
    keep = i + d < n
    bi, bj = i[keep], (i + d)[keep]
    band_nnz = n + 2 * bi.size
    m = max(0, int(round((deg * n - band_nnz) / 2.0)))
    if m > 0 and n > w + 2:
        u = rng.random(m)
        dd = np.floor((w + 1) * np.exp(u * np.log(n / (w + 1.0)))).astype(np.int64)
        dd = np.clip(dd, w + 1, n - 1)
        li = np.floor(rng.random(m) * (n - dd)).astype(np.int64)
        lj = li + dd
        bi = np.concatenate([bi, li])
        bj = np.concatenate([bj, lj])
    return bi, bj


def make_graph(seed: int, graph_id: int, n_mean: int = 500, deg: int = 12, n_feat: int = 32,
               n_bridges: int = 20):
    """One graph -> (rowptr_local int64 [n+1], col_local int32 [nnz], x f32 [n,F])."""
    rng = np.random.default_rng(seed + graph_id)
    half = n_mean / 2.0
    sigma = 0.35
    mu = np.log(half) - 0.5 * sigma * sigma
    lens = np.clip(np.rint(rng.lognormal(mu, sigma, size=2)), 15, 2 * n_mean).astype(np.int64)
    n1, n2 = int(lens[0]), int(lens[1])
    n = n1 + n2
    ai, aj = _protein_pairs(rng, n1, deg)
    bi, bj = _protein_pairs(rng, n2, deg)
    br_i = rng.integers(0, n1, size=n_bridges)
    br_j = rng.integers(0, n2, size=n_bridges) + n1
    ui = np.concatenate([ai, bi + n1, br_i])
    uj = np.concatenate([aj, bj + n1, br_j])
    diag = np.arange(n, dtype=np.int64)
    rows = np.concatenate([ui, uj, diag])
    cols = np.concatenate([uj, ui, diag])
    keys = np.unique(rows * n + cols)          # sorted row-major, duplicates merged
    r = keys // n
    c = (keys - r * n).astype(np.int32)
    rowptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(r, minlength=n), out=rowptr[1:])
    x = rng.random((n, n_feat), dtype=np.float32)
    return rowptr, c, x


def neighbour_scores(packed: PackedGraphs, n_out: int, seed: int) -> np.ndarray:
    """float64 [sum N, n_out] score of every node of a packed dataset: (sum over the stored neighbours j of n of
    (x_j - 1/2)) . V, with V [F, n_out] standard normal from ``default_rng(seed)`` - a function of the graph that one
    aggregation step can express."""
    import scipy.sparse as sp
    n = int(packed.node_off[-1])
    rows = np.repeat(np.arange(n, dtype=np.int64), np.diff(packed.rowptr))
    cols = packed.col.astype(np.int64) + np.repeat(packed.node_off[:-1], packed.n_nodes)[rows]
    a = sp.csr_matrix((np.ones(rows.shape[0]), (rows, cols)), shape=(n, n))
    v = np.random.default_rng(seed).standard_normal((packed.x.shape[1], n_out))
    return (a @ (np.asarray(packed.x, dtype=np.float64) - 0.5)) @ v


def node_labels(packed: PackedGraphs, n_classes: int, seed: int) -> np.ndarray:
    """One-hot [sum N, C] node labels of a packed dataset: row n is one-hot at argmax_c of its ``neighbour_scores``."""
    score = neighbour_scores(packed, n_classes, seed)
    n = score.shape[0]
    y = np.zeros((n, n_classes), dtype=np.float32)
    y[np.arange(n), np.argmax(score, axis=1)] = 1.0
    return y


def regression_targets(packed: PackedGraphs, n_out: int, seed: int, node_level: bool) -> np.ndarray:
    """Continuous float32 targets in (-1, 1): tanh of the ``neighbour_scores``, per node [sum N, n_out] with
    ``node_level``, else their mean over each graph's nodes [G, n_out] (what a sum or average pool can express)."""
    t = np.tanh(neighbour_scores(packed, n_out, seed))
    if node_level:
        return t.astype(np.float32)
    counts = packed.n_nodes
    seg = np.repeat(np.arange(packed.n_graphs, dtype=np.int64), counts)
    sums = np.stack([np.bincount(seg, weights=t[:, k], minlength=packed.n_graphs) for k in range(n_out)], axis=1)
    return (sums / np.maximum(counts, 1)[:, None]).astype(np.float32)


def _with_node_labels(p: PackedGraphs, n_classes: int, seed: int) -> PackedGraphs:
    return PackedGraphs(p.node_off, p.rowptr, p.col, p.x, node_labels(p, n_classes, seed + 0x5EED), node_level=True)


def _with_regression_targets(p: PackedGraphs, n_out: int, seed: int, node_level: bool) -> PackedGraphs:
    return PackedGraphs(p.node_off, p.rowptr, p.col, p.x, regression_targets(p, n_out, seed + 0x5EED, node_level),
                        node_level=node_level)


TASKS = ("classification", "regression")


def make_dataset(n_graphs: int, seed: int = 0, n_mean: int = 500, deg: int = 12,
                 n_feat: int = 32, n_classes: int = 2, node_level: bool = False,
                 task: str = "classification") -> PackedGraphs:
    """G(seed, n_mean, deg, F) of SURVEY.md §8d, packed.  ``node_level=True``: per-node labels (``node_labels``, one
    projection for the whole dataset) instead of the balanced graph labels; the graphs themselves are the same.
    ``task='regression'``: ``n_classes`` continuous targets per graph or per node (``regression_targets``) instead of
    one-hot labels."""
    if task not in TASKS:
        raise ValueError(f"task must be one of {TASKS}, got {task!r}")
    rps: List[np.ndarray] = []
    cols: List[np.ndarray] = []
    xs: List[np.ndarray] = []
    node_off = np.zeros(n_graphs + 1, dtype=np.int64)
    e_off = 0
    for g in range(n_graphs):
        rp, c, x = make_graph(seed, g, n_mean, deg, n_feat)
        node_off[g + 1] = node_off[g] + x.shape[0]
        rps.append(rp[:-1] + e_off)
        e_off += int(rp[-1])
        cols.append(c)
        xs.append(x)
    rowptr = np.concatenate(rps + [np.array([e_off], dtype=np.int64)]) if n_graphs else np.zeros(1, np.int64)
    col = np.concatenate(cols) if n_graphs else np.zeros(0, np.int32)
    x = np.concatenate(xs) if n_graphs else np.zeros((0, n_feat), np.float32)
    if task == "regression":
        return _with_regression_targets(PackedGraphs(node_off, rowptr, col, x, np.zeros((0, n_classes), np.float32)),
                                        n_classes, seed, node_level)
    if node_level:
        return _with_node_labels(PackedGraphs(node_off, rowptr, col, x, np.zeros((0, n_classes), np.float32)), n_classes,
                                 seed)
    y = np.zeros((n_graphs, n_classes), dtype=np.float32)
    lab = np.arange(n_graphs) % n_classes          # balanced (gcn.py:265-266)
    y[np.arange(n_graphs), lab] = 1.0
    return PackedGraphs(node_off, rowptr, col, x, y)


def concat_packed(parts: List[PackedGraphs]) -> PackedGraphs:
    """Concatenate packed datasets (graph order = order of the parts).  Graph- and node-labelled parts do not mix."""
    kinds = {bool(p.node_level) for p in parts}
    if len(kinds) > 1:
        raise ValueError("cannot concatenate graph-labelled and node-labelled datasets")
    if len(parts) == 1:
        return parts[0]
    node_off = [np.zeros(1, dtype=np.int64)]
    rowptr = []
    n0, e0 = 0, 0
    for p in parts:
        node_off.append(p.node_off[1:] + n0)
        rowptr.append(p.rowptr[:-1] + e0)
        n0 += int(p.node_off[-1])
        e0 += int(p.rowptr[-1])
    rowptr.append(np.array([e0], dtype=np.int64))
    return PackedGraphs(np.concatenate(node_off), np.concatenate(rowptr), np.concatenate([p.col for p in parts]),
                        np.concatenate([p.x for p in parts]), np.concatenate([p.y for p in parts]), kinds.pop())


def _make_range(args):
    seed, g0, g1, n_mean, deg, n_feat, n_classes = args
    rps, cols, xs = [], [], []
    node_off = np.zeros(g1 - g0 + 1, dtype=np.int64)
    e_off = 0
    for k, gid in enumerate(range(g0, g1)):
        rp, c, x = make_graph(seed, gid, n_mean, deg, n_feat)
        node_off[k + 1] = node_off[k] + x.shape[0]
        rps.append(rp[:-1] + e_off)
        e_off += int(rp[-1])
        cols.append(c)
        xs.append(x)
    y = np.zeros((g1 - g0, n_classes), dtype=np.float32)
    y[np.arange(g1 - g0), np.arange(g0, g1) % n_classes] = 1.0
    return PackedGraphs(node_off, np.concatenate(rps + [np.array([e_off], dtype=np.int64)]), np.concatenate(cols),
                        np.concatenate(xs), y)


def make_dataset_parallel(n_graphs: int, seed: int = 0, n_mean: int = 500, deg: int = 12, n_feat: int = 32,
                          n_classes: int = 2, workers: int = 0, node_level: bool = False) -> PackedGraphs:
    """make_dataset over a process pool (the same graphs: every graph is seeded by its id).  workers = 0: the cores this
    process may run on."""
    import multiprocessing as mp
    import os
    workers = workers or len(os.sched_getaffinity(0))
    if workers <= 1 or n_graphs < 4 * workers:
        return make_dataset(n_graphs, seed, n_mean, deg, n_feat, n_classes, node_level=node_level)
    chunk = -(-n_graphs // (4 * workers))
    jobs = [(seed, g0, min(g0 + chunk, n_graphs), n_mean, deg, n_feat, n_classes) for g0 in range(0, n_graphs, chunk)]
    with mp.get_context("fork").Pool(workers) as pool:
        parts = pool.map(_make_range, jobs)
    out = concat_packed(parts)
    return _with_node_labels(out, n_classes, seed) if node_level else out


def tile_dataset(packed: PackedGraphs, n_graphs: int) -> PackedGraphs:
    """The first n_graphs graphs of `packed` repeated end to end (a large epoch out of a smaller set of unique
    synthetic graphs; labels and features repeat with them)."""
    g = packed.n_graphs
    reps = -(-n_graphs // g)
    out = concat_packed([packed] * reps)
    if out.n_graphs == n_graphs:
        return out
    n1 = int(out.node_off[n_graphs])
    e1 = int(out.rowptr[n1])
    return PackedGraphs(out.node_off[:n_graphs + 1], out.rowptr[:n1 + 1], out.col[:e1], out.x[:n1],
                        out.y[:n1] if out.node_level else out.y[:n_graphs], out.node_level)


def pack_graphs(graphs, node_level: bool = False) -> PackedGraphs:
    """Pack a list of per-graph objects exposing ``.x [n,F]``, ``.a`` (scipy sparse / dense
    [n,n]) and ``.y`` — what the reference's MyDataset.read returns (gcn.py:84-102) — into
    the device-ready layout.  Explicit zeros are dropped and duplicates merged, exactly as
    ``sp.find`` does in Spektral's collate (SURVEY.md §8 a1); values are otherwise ignored
    (a5: GeneralConv never reads them).  ``node_level=True``: every ``.y`` is [n_nodes, C] (one label row per node,
    all with the same C) and the rows are stacked in node order."""
    import scipy.sparse as sp
    node_off = np.zeros(len(graphs) + 1, dtype=np.int64)
    rps, cols, xs, ys = [], [], [], []
    e_off = 0
    for g, gr in enumerate(graphs):
        a = sp.csr_matrix(gr.a, copy=True)     # never mutate the caller's matrix
        a.sum_duplicates()
        a.eliminate_zeros()
        a.sort_indices()
        n = a.shape[0]
        x = np.asarray(gr.x)
        if x.shape[0] != n:
            raise ValueError(f"graph {g}: x has {x.shape[0]} rows but a is {a.shape}")
        node_off[g + 1] = node_off[g] + n
        rps.append(a.indptr[:-1].astype(np.int64) + e_off)
        e_off += int(a.indptr[-1])
        cols.append(a.indices.astype(np.int32))
        xs.append(x.astype(np.float32))
        if node_level:
            yg = np.asarray(gr.y, dtype=np.float32) if gr.y is not None else None
            if yg is None or yg.ndim != 2 or yg.shape[0] != n or (ys and yg.shape[1] != ys[0].shape[1]):
                want = f"[{n}, {ys[0].shape[1]}]" if ys else f"[{n}, C]"
                raise ValueError(f"graph {g}: node-level labels must be {want}, got "
                                 f"{None if yg is None else tuple(yg.shape)}")
            ys.append(yg)
        else:
            ys.append(np.asarray(gr.y, dtype=np.float32).reshape(-1))
    rowptr = np.concatenate(rps + [np.array([e_off], dtype=np.int64)]) if graphs else np.zeros(1, np.int64)
    col = np.concatenate(cols) if graphs else np.zeros(0, np.int32)
    x = np.concatenate(xs) if graphs else np.zeros((0, 0), np.float32)
    if node_level:
        return PackedGraphs(node_off, rowptr, col, x, np.concatenate(ys) if graphs else np.zeros((0, 0), np.float32), True)
    y = np.stack(ys) if graphs else np.zeros((0, 0), np.float32)
    return PackedGraphs(node_off, rowptr, col, x, y)
