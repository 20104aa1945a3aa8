"""Digest of every batch DisjointLoader yields, for comparing two trees of the package.

    python scripts/loader_ab.py [--root TREE] --out FILE.jsonl

Imports gcn_string_b200 from TREE (default: this repository) and runs every graph store mode - device-resident,
host slices (unshuffled), host-staged, device_gather and zero_copy - graph- and node-level, with and without sample
weights, prefetch on and off, two shuffled epochs; then each mode as rank 0 and rank 1 of a 2-rank balance='nnz'
shard, and three modes over a memory-mapped shard.  One JSON line per run: per batch a SHA-256 over every yielded
tensor (x, indices, rowptr, colidx, graph_ptr, edge_ptr, i, y, w: dtype, shape, bytes) and the batch's symmetric
flag, node and graph counts, the gcs_debug_launch_count delta of the step and h2d_bytes_last of a host store; the
number of copies torch.profiler saw in the run, and a SHA-256 over its count of every CUDA kernel, copy and memset by
name.  Two trees that batch alike write identical files.
"""
from __future__ import annotations

import argparse
import collections
import hashlib
import json
import os
import sys
import tempfile

import numpy as np

MODES = {"device": (dict(device_resident=True), True), "host_slices": (dict(device_resident=False), False),
         "host_staged": (dict(device_resident=False), True),
         "device_gather": (dict(device_resident=False, device_gather=True), True),
         "zero_copy": (dict(device_resident=False, zero_copy=True), True)}


def batch_digest(item):
    (x, a, i), y = item[:2]
    w = item[2] if len(item) > 2 else None
    h = hashlib.sha256(repr((a._symmetric, a.max_graph_nodes, a.global_batch_graphs, a.global_batch_nodes)).encode())
    for t in (x, a.indices, a.rowptr, a.colidx, a.graph_ptr, a.edge_ptr, i, y, w):
        t = None if t is None else t.detach().cpu().contiguous()
        h.update(b"-" if t is None else f"{t.dtype}{tuple(t.shape)}".encode() + t.numpy().tobytes())
    return h.hexdigest()[:12]


def run(g, lib, tag, data, weights, out, **kw):
    import torch
    np.random.seed(1234)
    loader = g.DisjointLoader(data, batch_size=5, epochs=2, want_coo=True, sample_weights=weights, **kw)
    batches, launches, h2d = [], [], []
    acts = [torch.profiler.ProfilerActivity.CPU, torch.profiler.ProfilerActivity.CUDA]
    with torch.profiler.profile(activities=acts) as prof:
        while True:
            n0 = lib.gcs_debug_launch_count()
            item = next(loader, None)
            if item is None:
                break
            launches.append(lib.gcs_debug_launch_count() - n0)
            h2d.append(getattr(loader.store, "h2d_bytes_last", None))
            batches.append(item)
        torch.cuda.synchronize()
    cuda = sorted(collections.Counter(e.name for e in prof.events() if str(e.device_type).endswith("CUDA")).items())
    out.write(json.dumps(dict(run=tag, launches=launches, h2d=h2d, digests=[batch_digest(b) for b in batches],
                              copies=sum(c for name, c in cuda if name.startswith("Memcpy")),
                              cuda=hashlib.sha256(repr(cuda).encode()).hexdigest()[:12])) + "\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    sys.path.insert(0, os.path.abspath(args.root))
    import gcn_string_b200 as g
    from gcn_string_b200 import _lib, shards, synthetic
    assert os.path.abspath(g.__file__).startswith(os.path.abspath(args.root)), g.__file__
    lib = _lib.load()
    rng = np.random.default_rng(5)
    sets = {}
    for node_level in (False, True):
        ds = synthetic.make_dataset(23, seed=11, n_mean=40, deg=8, n_feat=6, n_classes=3, node_level=node_level)
        sets[node_level] = (ds, rng.uniform(0.25, 2.0, int(ds.node_off[-1]) if node_level else 23).astype(np.float32))
    with open(args.out, "w") as out, tempfile.TemporaryDirectory() as tmp:
        for mode, (kw, shuffle) in MODES.items():
            for node_level, (ds, sw) in sets.items():
                for weights in (None, sw):
                    for prefetch in (False, True):
                        run(g, lib, f"{mode} node_level={node_level} weights={weights is not None} prefetch={prefetch}",
                            ds, weights, out, node_level=node_level, shuffle=shuffle, prefetch=prefetch, **kw)
                for rank in (0, 1):
                    run(g, lib, f"{mode} node_level={node_level} rank={rank}/2 balance=nnz", ds, sw, out,
                        node_level=node_level, shuffle=True, rank=rank, world_size=2, balance="nnz", **kw)
        ds = sets[False][0]
        shards.write_dataset([g.Graph(*ds.graph(k)[:2], y=ds.graph(k)[2]) for k in range(ds.n_graphs)], tmp,
                             graphs_per_shard=64)
        packed = shards.load_dataset(tmp)                  # one shard: memory-mapped, symmetric from its header
        for mode in ("device", "host_slices", "host_staged"):
            kw, shuffle = MODES[mode]
            run(g, lib, f"{mode} shard", packed, None, out, shuffle=shuffle, **kw)


if __name__ == "__main__":
    main()
