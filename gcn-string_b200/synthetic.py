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

import dataclasses
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np


@dataclass
class PackedGraphs:
    """Concatenated per-graph CSR + features + labels (host, NumPy).

    node_off[G+1]  int64  node offset of each graph in ``x`` / ``rowptr``
    rowptr[sumN+1] int64  start of each node's neighbour list in ``col`` (dataset-global)
    col[sumNNZ]    int32  neighbour index LOCAL to the graph, ascending within a row
    x[sumN, F]     float32
    y[G, C]        float32 one-hot graph labels, or y[sumN, C] node labels (rows in node order) when node_level
    symmetric      True when every graph's pattern equals its transpose (a shard header records it), False when some
                   graph's does not, None when unknown: the loader then checks each batch's pattern on the device
    """
    node_off: np.ndarray
    rowptr: np.ndarray
    col: np.ndarray
    x: np.ndarray
    y: np.ndarray
    node_level: bool = False
    symmetric: Optional[bool] = None

    @classmethod
    def from_graphs(cls, rowptrs, cols, xs, ys, node_level: bool = False, n_feat: int = 0, n_classes: int = 0,
                    symmetric: Optional[bool] = None) -> "PackedGraphs":
        """Pack per-graph pieces, in order: local ``rowptr [n+1]``, ``col [nnz]`` int32, ``x [n, F]`` float32, and a label
        row ``y [C]`` per graph or, with ``node_level``, ``y [n, C]``, all float32.  ``n_feat`` / ``n_classes`` are the
        widths of ``x`` / ``y`` when there are no graphs."""
        node_off = np.zeros(len(xs) + 1, dtype=np.int64)
        np.cumsum([x.shape[0] for x in xs], out=node_off[1:])
        e_off = np.zeros(len(rowptrs) + 1, dtype=np.int64)
        np.cumsum([rp[-1] for rp in rowptrs], out=e_off[1:])
        rowptr = np.concatenate([np.asarray(rp[:-1], dtype=np.int64) + e for rp, e in zip(rowptrs, e_off)] + [e_off[-1:]])
        col = np.concatenate(cols) if cols else np.zeros(0, np.int32)
        x = np.concatenate(xs) if xs else np.zeros((0, n_feat), np.float32)
        if not ys:
            y = np.zeros((0, n_classes), np.float32)
        else:
            y = np.concatenate(ys) if node_level else np.stack(ys)
        return cls(node_off, rowptr, col, x, y, node_level, symmetric)

    @property
    def n_graphs(self) -> int:
        return int(self.node_off.shape[0] - 1)

    @property
    def n_nodes(self) -> np.ndarray:
        return np.diff(self.node_off)

    @property
    def n_edges(self) -> np.ndarray:
        return self.rowptr[self.node_off[1:]] - self.rowptr[self.node_off[:-1]]

    def span(self, g0: int, g1: int):
        """(n0, n1, e0, e1): the graphs [g0, g1) hold the nodes [n0, n1) of ``x`` / ``rowptr`` and the entries [e0, e1) of
        ``col``."""
        n0, n1 = int(self.node_off[g0]), int(self.node_off[g1])
        return n0, n1, int(self.rowptr[n0]), int(self.rowptr[n1])

    def graph(self, g: int):
        """(x[n,F], scipy CSR int64 ones [n,n], y[C]) for graph g — the per-graph objects
        the reference's MyDataset hands to Spektral (src/scripts/gcn.py:161-181)."""
        import scipy.sparse as sp
        n0, n1, e0, e1 = self.span(g, g + 1)
        n = n1 - n0
        a = sp.csr_matrix((np.ones(e1 - e0, dtype=np.int64), self.col[e0:e1].astype(np.int32),
                           (self.rowptr[n0:n1 + 1] - e0).astype(np.int32)), shape=(n, n))
        return self.x[n0:n1], a, (self.y[n0:n1] if self.node_level else self.y[g])

    def take(self, ids) -> "PackedGraphs":
        """A new pack of the graphs ``ids``, in that order (a graph may repeat)."""
        spans = [self.span(g, g + 1) for g in ids]
        return PackedGraphs.from_graphs(
            [self.rowptr[n0:n1 + 1] - e0 for n0, n1, e0, _ in spans], [self.col[e0:e1] for _, _, e0, e1 in spans],
            [self.x[n0:n1] for n0, n1, _, _ in spans],
            [self.y[n0:n1] for n0, n1, _, _ in spans] if self.node_level else [self.y[g] for g in ids],
            self.node_level, self.x.shape[1], self.y.shape[1], self.symmetric)


def concat_packed(parts: Sequence[PackedGraphs]) -> PackedGraphs:
    """Concatenate packed datasets (graph order = order of the parts, offsets rebased).  Graph- and node-labelled parts
    do not mix.  Parts without graphs are skipped, and a single remaining part is returned itself, not a copy.  The
    result is symmetric when every part is, not symmetric when any part is not, and unknown otherwise."""
    if len({bool(p.node_level) for p in parts}) > 1:
        raise ValueError("cannot concatenate graph-labelled and node-labelled datasets")
    if not parts:
        raise ValueError("nothing to concatenate")
    parts = [p for p in parts if p.n_graphs] or list(parts[:1])
    if len(parts) == 1:
        return parts[0]
    node_off, rowptr = [np.zeros(1, np.int64)], []
    n0 = e0 = 0
    for p in parts:
        node_off.append(p.node_off[1:] + n0)
        rowptr.append(p.rowptr[:-1] - p.rowptr[0] + e0)
        n0 += int(p.node_off[-1])
        e0 += int(p.rowptr[-1] - p.rowptr[0])
    rowptr.append(np.array([e0], dtype=np.int64))
    sym = [p.symmetric for p in parts]
    symmetric = False if any(s is False for s in sym) else (True if all(sym) else None)
    return PackedGraphs(np.concatenate(node_off), np.concatenate(rowptr), np.concatenate([p.col for p in parts]),
                        np.concatenate([p.x for p in parts]), np.concatenate([p.y for p in parts]), parts[0].node_level,
                        symmetric)


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


def _labelled(p: PackedGraphs, n_classes: int, seed: int, node_level: bool, task: str) -> PackedGraphs:
    """``p`` (graphs with their balanced graph labels) with the labels ``make_dataset`` gives for ``task`` /
    ``node_level``."""
    if task == "regression":
        return dataclasses.replace(p, y=regression_targets(p, n_classes, seed + 0x5EED, node_level), node_level=node_level)
    if node_level:
        return dataclasses.replace(p, y=node_labels(p, n_classes, seed + 0x5EED), node_level=True)
    return p


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
    return _labelled(_make_range((seed, 0, n_graphs, n_mean, deg, n_feat, n_classes)), n_classes, seed, node_level, task)


def _make_range(args):
    """Graphs [g0, g1) with their balanced graph labels (gcn.py:265-266: graph g is of class g % n_classes)."""
    seed, g0, g1, n_mean, deg, n_feat, n_classes = args
    graphs = [make_graph(seed, g, n_mean, deg, n_feat) for g in range(g0, g1)]
    eye = np.eye(n_classes, dtype=np.float32)
    return PackedGraphs.from_graphs([rp for rp, _, _ in graphs], [c for _, c, _ in graphs], [x for _, _, x in graphs],
                                    [eye[g % n_classes] for g in range(g0, g1)], n_feat=n_feat, n_classes=n_classes)


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
    return _labelled(concat_packed(parts), n_classes, seed, node_level, "classification")


def tile_dataset(packed: PackedGraphs, n_graphs: int) -> PackedGraphs:
    """The first n_graphs graphs of `packed` repeated end to end (a large epoch out of a smaller set of unique
    synthetic graphs; labels and features repeat with them)."""
    g = packed.n_graphs
    reps = -(-n_graphs // g)
    out = concat_packed([packed] * reps)
    if out.n_graphs == n_graphs:
        return out
    _, n1, _, e1 = out.span(0, n_graphs)
    return PackedGraphs(out.node_off[:n_graphs + 1], out.rowptr[:n1 + 1], out.col[:e1], out.x[:n1],
                        out.y[:n1] if out.node_level else out.y[:n_graphs], out.node_level, out.symmetric)


def pack_graphs(graphs, node_level: bool = False) -> PackedGraphs:
    """Pack a list of per-graph objects exposing ``.x [n,F]``, ``.a`` (scipy sparse / dense
    [n,n]) and ``.y`` — what the reference's MyDataset.read returns (gcn.py:84-102) — into
    the device-ready layout.  Explicit zeros are dropped and duplicates merged, exactly as
    ``sp.find`` does in Spektral's collate (SURVEY.md §8 a1); values are otherwise ignored
    (a5: GeneralConv never reads them).  ``node_level=True``: every ``.y`` is [n_nodes, C] (one label row per node,
    all with the same C) and the rows are stacked in node order."""
    import scipy.sparse as sp
    rps, cols, xs, ys = [], [], [], []
    for g, gr in enumerate(graphs):
        a = sp.csr_matrix(gr.a, copy=True)     # never mutate the caller's matrix
        a.sum_duplicates()
        a.eliminate_zeros()
        a.sort_indices()
        n = a.shape[0]
        x = np.asarray(gr.x, dtype=np.float32)
        if x.shape[0] != n:
            raise ValueError(f"graph {g}: x has {x.shape[0]} rows but a is {a.shape}")
        rps.append(a.indptr)
        cols.append(a.indices.astype(np.int32))
        xs.append(x)
        if node_level:
            yg = np.asarray(gr.y, dtype=np.float32) if gr.y is not None else None
            if yg is None or yg.ndim != 2 or yg.shape[0] != n or (ys and yg.shape[1] != ys[0].shape[1]):
                want = f"[{n}, {ys[0].shape[1]}]" if ys else f"[{n}, C]"
                raise ValueError(f"graph {g}: node-level labels must be {want}, got "
                                 f"{None if yg is None else tuple(yg.shape)}")
            ys.append(yg)
        else:
            ys.append(np.asarray(gr.y, dtype=np.float32).reshape(-1))
    return PackedGraphs.from_graphs(rps, cols, xs, ys, node_level)
