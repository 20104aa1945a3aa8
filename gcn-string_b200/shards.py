"""Packed graph shards: the device-ready ingest format (SURVEY.md §8 f1).

The reference reads one ``.gpickle`` per protein pair through networkx on every run
(src/scripts/gcn.py:84-102 ``MyDataset.read``, :161-197 ``generate_spektral_graph`` /
``read_graph`` / ``format_graph``; the loop the author notes "takes a very long time") and
re-collates on the host every step.  Here a dataset is converted ONCE into shard files
that hold exactly what the device batching kernel consumes (``PackedGraphs``): per-graph
CSR with local int32 columns, float32 node features, one-hot float32 labels.  A shard is
read with ``np.memmap`` (no parsing, no per-graph Python objects) and goes to pinned host
memory or straight to HBM.

File layout (little endian, every section 64-byte aligned):

    0    8  magic  b"GCSSHRD1"
    8    4  uint32 version (1: graph labels; 2: node labels)
    12   4  uint32 n_feat
    16   4  uint32 n_classes
    20   4  uint32 flags           bit 0: every graph's pattern is symmetric
                                   bit 1: node labels (set exactly when version is 2)
    24   8  uint64 n_graphs
    32   8  uint64 n_nodes
    40   8  uint64 nnz
    48   8  uint64 payload checksum (sum of the payload's uint32 words mod 2^64)
    56   8  reserved (0)
    64      node_off int64 [n_graphs+1] | rowptr int64 [n_nodes+1] | col int32 [nnz]
            | x float32 [n_nodes, n_feat] | y float32 [n_graphs, n_classes]  (version 1)
                                           | y float32 [n_nodes, n_classes]   (version 2, node labels)

A node-labelled shard carries version 2 so that a reader that knows only version 1 refuses it instead of misreading
its y section.  Graph-labelled shards are written as version 1, byte for byte as before.
"""
from __future__ import annotations

import json
import os
import struct
from typing import Iterable, List, Optional, Sequence

import numpy as np

from .synthetic import PackedGraphs, pack_graphs

MAGIC = b"GCSSHRD1"
VERSION = 1                  # graph labels
VERSION_NODE_LEVEL = 2       # node labels
_HEADER = struct.Struct("<8sIIIIQQQQQ")          # 64 bytes
_ALIGN = 64
FLAG_SYMMETRIC = 1
FLAG_NODE_LEVEL = 2


def _pad(n: int) -> int:
    return (-n) % _ALIGN


def _sections(n_graphs: int, n_nodes: int, nnz: int, n_feat: int, n_classes: int, node_level: bool = False):
    """[(name, dtype, shape, offset)] of the payload, offsets from the start of the file."""
    spec = [("node_off", np.dtype("<i8"), (n_graphs + 1,)), ("rowptr", np.dtype("<i8"), (n_nodes + 1,)),
            ("col", np.dtype("<i4"), (nnz,)), ("x", np.dtype("<f4"), (n_nodes, n_feat)),
            ("y", np.dtype("<f4"), (n_nodes if node_level else n_graphs, n_classes))]
    out, off = [], _HEADER.size
    for name, dt, shape in spec:
        nbytes = int(np.prod(shape, dtype=np.int64)) * dt.itemsize
        out.append((name, dt, shape, off))
        off += nbytes + _pad(nbytes)
    return out, off


def _checksum(arrays) -> int:
    total = 0
    for a in arrays:
        b = np.ascontiguousarray(a).view(np.uint8).reshape(-1)
        n4 = b.size // 4 * 4
        total += int(b[:n4].view("<u4").sum(dtype=np.uint64))
        total += int(b[n4:].sum(dtype=np.uint64))
    return total & 0xFFFFFFFFFFFFFFFF


def pattern_is_symmetric(p: PackedGraphs) -> bool:
    """True when every graph's stored pattern equals its transpose (undirected contact graphs)."""
    import scipy.sparse as sp
    n = int(p.node_off[-1])
    if n == 0:
        return True
    rows = np.repeat(np.arange(n, dtype=np.int64), np.diff(p.rowptr))
    base = np.repeat(p.node_off[:-1], p.n_nodes)               # first node of the graph each row belongs to
    cols = p.col.astype(np.int64) + base[rows]
    a = sp.csr_matrix((np.ones(cols.shape[0], np.int8), (rows, cols)), shape=(n, n))
    return (a != a.T).nnz == 0


def write_shard(path: str, packed: PackedGraphs, symmetric: Optional[bool] = None) -> str:
    """Write one shard.  ``symmetric=None`` checks the pattern (recorded in the header so that the
    loader can alias the transposed CSR without a device-side check)."""
    g, n, nnz = packed.n_graphs, int(packed.node_off[-1]), int(packed.col.shape[0])
    if packed.rowptr.shape[0] != n + 1 or int(packed.rowptr[-1]) != nnz:
        raise ValueError("inconsistent PackedGraphs: rowptr does not match node_off / col")
    x = np.ascontiguousarray(packed.x, dtype="<f4").reshape(n, -1) if n else np.zeros((0, packed.x.shape[-1]), "<f4")
    node_level = bool(getattr(packed, "node_level", False))
    y = np.ascontiguousarray(packed.y, dtype="<f4").reshape(n if node_level else g, -1)
    if nnz and (packed.col.min() < 0 or (packed.col >= np.repeat(packed.n_nodes, packed.n_edges)).any()):
        raise ValueError("column index outside its graph")
    arrays = [np.ascontiguousarray(packed.node_off, dtype="<i8"), np.ascontiguousarray(packed.rowptr, dtype="<i8"),
              np.ascontiguousarray(packed.col, dtype="<i4"), x, y]
    if symmetric is None:
        symmetric = pattern_is_symmetric(packed)
    flags = (FLAG_SYMMETRIC if symmetric else 0) | (FLAG_NODE_LEVEL if node_level else 0)
    version = VERSION_NODE_LEVEL if node_level else VERSION
    header = _HEADER.pack(MAGIC, version, x.shape[1], y.shape[1], flags, g, n, nnz, _checksum(arrays), 0)
    tmp = path + ".tmp"
    with open(tmp, "wb") as f:
        f.write(header)
        for a in arrays:
            b = a.tobytes()
            f.write(b)
            f.write(b"\0" * _pad(len(b)))
    os.replace(tmp, path)
    return path


class ShardHeader:
    def __init__(self, raw: bytes, path: str):
        if len(raw) < _HEADER.size:
            raise ValueError(f"{path}: truncated shard header")
        magic, ver, self.n_feat, self.n_classes, self.flags, self.n_graphs, self.n_nodes, self.nnz, self.checksum, _ = \
            _HEADER.unpack(raw[:_HEADER.size])
        if magic != MAGIC:
            raise ValueError(f"{path}: not a gcn_string_b200 shard (bad magic {magic!r})")
        if ver not in (VERSION, VERSION_NODE_LEVEL):
            raise ValueError(f"{path}: shard version {ver}, this reader understands {VERSION} and {VERSION_NODE_LEVEL}")
        if bool(self.flags & FLAG_NODE_LEVEL) != (ver == VERSION_NODE_LEVEL):
            raise ValueError(f"{path}: shard version {ver} disagrees with its node-label flag (flags {self.flags:#x})")
        self.version = ver

    @property
    def symmetric(self) -> bool:
        return bool(self.flags & FLAG_SYMMETRIC)

    @property
    def node_level(self) -> bool:
        return bool(self.flags & FLAG_NODE_LEVEL)


def read_header(path: str) -> ShardHeader:
    with open(path, "rb") as f:
        return ShardHeader(f.read(_HEADER.size), path)


def read_shard(path: str, mmap: bool = True, verify: bool = False) -> PackedGraphs:
    """Open a shard as ``PackedGraphs``.  With ``mmap`` the arrays are read-only views of the file
    (nothing is parsed or copied until the loader uploads it); ``verify`` recomputes the checksum."""
    h = read_header(path)
    secs, end = _sections(h.n_graphs, h.n_nodes, h.nnz, h.n_feat, h.n_classes, h.node_level)
    size = os.path.getsize(path)
    if size < end:
        raise ValueError(f"{path}: truncated shard ({size} bytes, header implies {end})")
    if mmap:
        buf = np.memmap(path, dtype=np.uint8, mode="r")
    else:
        buf = np.fromfile(path, dtype=np.uint8)
    arrs = {}
    for name, dt, shape, off in secs:
        nbytes = int(np.prod(shape, dtype=np.int64)) * dt.itemsize
        arrs[name] = buf[off:off + nbytes].view(dt).reshape(shape)
    if verify and _checksum([arrs[k] for k in ("node_off", "rowptr", "col", "x", "y")]) != h.checksum:
        raise ValueError(f"{path}: payload checksum mismatch")
    p = PackedGraphs(arrs["node_off"], arrs["rowptr"], arrs["col"], arrs["x"], arrs["y"], h.node_level)
    if h.n_graphs and (int(p.node_off[-1]) != h.n_nodes or int(p.rowptr[-1]) != h.nnz or int(p.node_off[0]) != 0):
        raise ValueError(f"{path}: offsets disagree with the header")
    p.symmetric = h.symmetric
    return p


def concat_packed(parts: Sequence[PackedGraphs]) -> PackedGraphs:
    """Concatenate packed datasets (graph order preserved, offsets rebased).  Graph- and node-labelled parts do not
    mix."""
    if len({bool(getattr(p, "node_level", False)) for p in parts}) > 1:
        raise ValueError("cannot concatenate graph-labelled and node-labelled shards")
    parts = [p for p in parts if p.n_graphs]
    if not parts:
        raise ValueError("nothing to concatenate")
    if len(parts) == 1:
        return parts[0]
    node_off, rowptr = [np.zeros(1, np.int64)], [np.zeros(1, np.int64)]
    n0 = e0 = 0
    for p in parts:
        node_off.append(np.asarray(p.node_off[1:], dtype=np.int64) + n0)
        rowptr.append(np.asarray(p.rowptr[1:], dtype=np.int64) + e0)
        n0 += int(p.node_off[-1])
        e0 += int(p.rowptr[-1])
    out = PackedGraphs(np.concatenate(node_off), np.concatenate(rowptr), np.concatenate([p.col for p in parts]),
                       np.concatenate([p.x for p in parts]), np.concatenate([p.y for p in parts]), parts[0].node_level)
    out.symmetric = all(getattr(p, "symmetric", False) for p in parts)
    return out


def write_dataset(graphs: Iterable, out_dir: str, graphs_per_shard: int = 4096, prefix: str = "shard",
                  node_level: bool = False) -> List[str]:
    """Convert a dataset (anything iterable over objects with ``.x``, ``.a``, ``.y`` - what
    ``MyDataset.read`` returns, gcn.py:84-102) into shard files + an ``index.json``; returns the paths.
    ``node_level=True``: every ``.y`` is [n_nodes, C] (version-2 shards; ``index.json`` says ``"labels": "node"``)."""
    os.makedirs(out_dir, exist_ok=True)
    paths, chunk, counts = [], [], []

    def flush():
        if chunk:
            path = os.path.join(out_dir, f"{prefix}-{len(paths):05d}.gcss")
            write_shard(path, pack_graphs(chunk, node_level=node_level))
            paths.append(path)
            counts.append(len(chunk))
            chunk.clear()

    for g in graphs:
        chunk.append(g)
        if len(chunk) == graphs_per_shard:
            flush()
    flush()
    if not paths:
        raise ValueError("Datasets cannot be empty")
    with open(os.path.join(out_dir, "index.json"), "w") as f:
        json.dump({"format": MAGIC.decode(), "version": VERSION_NODE_LEVEL if node_level else VERSION,
                   "labels": "node" if node_level else "graph",
                   "shards": [{"file": os.path.basename(p), "n_graphs": c} for p, c in zip(paths, counts)]}, f, indent=1)
    return paths


def load_dataset(out_dir_or_paths, mmap: bool = True, verify: bool = False) -> PackedGraphs:
    """Open every shard of a directory written by ``write_dataset`` (or an explicit list of shard
    paths) as one ``PackedGraphs`` - pass it to ``DisjointLoader`` like a ``Dataset``."""
    if isinstance(out_dir_or_paths, (str, os.PathLike)):
        d = os.fspath(out_dir_or_paths)
        with open(os.path.join(d, "index.json")) as f:
            idx = json.load(f)
        if idx.get("format") != MAGIC.decode():
            raise ValueError(f"{d}/index.json: unknown format {idx.get('format')!r}")
        paths = [os.path.join(d, s["file"]) for s in idx["shards"]]
    else:
        paths = list(out_dir_or_paths)
    return concat_packed([read_shard(p, mmap=mmap, verify=verify) for p in paths])


def graph_from_networkx(G, label, feature_name: str = "x"):
    """One networkx graph -> ``Graph`` the way the reference does it: integer node labels in
    iteration order (``format_graph``, gcn.py:184-197), adjacency of the stored edges with the
    ``weight`` attribute dropped - i.e. the 0/1 pattern, both directions, self-loops kept
    (``get_adjacency``, :104-117), node features stacked from attribute ``x`` (:119-130), label as
    given (:175).  Duck-typed: needs ``G.nodes(data=...)`` and ``G.edges()`` only."""
    import scipy.sparse as sp
    from .data import Graph
    nodes = list(G.nodes())
    pos = {n: k for k, n in enumerate(nodes)}
    x = np.vstack([np.asarray(v, dtype=np.float64) for _, v in G.nodes(data=feature_name)])
    e = np.array([(pos[u], pos[v]) for u, v in G.edges()], dtype=np.int64).reshape(-1, 2)
    directed = bool(getattr(G, "is_directed", lambda: False)())
    r, c = e[:, 0], e[:, 1]
    if not directed:
        off = r != c
        r, c = np.concatenate([r, c[off]]), np.concatenate([c, e[:, 0][off]])
    a = sp.csr_matrix((np.ones(r.shape[0], np.int64), (r, c)), shape=(len(nodes), len(nodes)))
    a.sum_duplicates()
    a.data[:] = 1
    return Graph(x=x, a=a, y=np.array(label))
