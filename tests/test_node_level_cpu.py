"""Node-level labels on the CPU: packing, shards (version 2 / flag bit 1 for node labels, graph-level shards unchanged),
the loader's kind check, and the two restatements of the node-level train step (float64 hand-derived backward, float32
autograd) against each other and against finite differences."""
import json
import os
import struct

import numpy as np
import pytest
import scipy.sparse as sp

import gcn_string_b200 as g
from gcn_string_b200 import shards, synthetic
from gcn_string_b200.data import Graph
from gcn_string_b200.params import GNNConfig, block_specs
from oracle import model_ref_np as O1, model_ref_torch as O2

from conftest import rel_err


def _graphs(sizes, c=3, seed=0):
    rng = np.random.default_rng(seed)
    out = []
    for n in sizes:
        a = sp.random(n, n, density=0.3, random_state=int(rng.integers(1 << 30)), format="csr") if n else sp.csr_matrix((0, 0))
        a = ((a + a.T + sp.eye(n)) > 0).astype(np.float64)
        out.append(Graph(x=rng.random((n, 5)), a=a, y=rng.random((n, c)).astype(np.float32)))
    return out


def test_pack_graphs_stacks_node_labels_in_node_order():
    gr = _graphs([4, 0, 1, 7])
    p = synthetic.pack_graphs(gr, node_level=True)
    assert p.node_level and p.y.shape == (12, 3) and p.y.dtype == np.float32
    assert np.array_equal(p.y, np.vstack([x.y for x in gr]))
    for k, x in enumerate(gr):
        assert np.array_equal(p.graph(k)[2], x.y)
    q = synthetic.pack_graphs([Graph(x=x.x, a=x.a, y=np.array([0.0, 1.0])) for x in gr])
    assert not q.node_level and q.y.shape == (4, 2)


@pytest.mark.parametrize("bad", ["vector", "rows", "width", "none"])
def test_pack_graphs_rejects_labels_of_the_wrong_shape(bad):
    gr = _graphs([3, 5, 2])
    n = gr[1].x.shape[0]
    gr[1].y = {"vector": np.zeros(3, np.float32), "rows": np.zeros((n + 1, 3), np.float32),
               "width": np.zeros((n, 4), np.float32), "none": None}[bad]
    with pytest.raises(ValueError, match="graph 1"):
        synthetic.pack_graphs(gr, node_level=True)


def test_make_dataset_node_level_keeps_the_graphs_and_labels_every_node():
    ref = synthetic.make_dataset(6, seed=4, n_mean=40, deg=8, n_feat=9)
    nl = synthetic.make_dataset(6, seed=4, n_mean=40, deg=8, n_feat=9, node_level=True)
    assert not ref.node_level and ref.y.shape == (6, 2)
    assert np.array_equal(ref.y, np.eye(2, dtype=np.float32)[np.arange(6) % 2])
    for name in ("node_off", "rowptr", "col", "x"):
        assert np.array_equal(getattr(ref, name), getattr(nl, name))
    assert nl.node_level and nl.y.shape == (int(nl.node_off[-1]), 2)
    assert np.array_equal(nl.y.sum(1), np.ones(nl.y.shape[0], np.float32))
    frac = nl.y[:, 1].mean()
    assert 0.2 < frac < 0.8                                  # both classes, roughly balanced
    again = synthetic.make_dataset(6, seed=4, n_mean=40, deg=8, n_feat=9, node_level=True)
    assert np.array_equal(again.y, nl.y)


def test_concat_and_tile_carry_node_labels_and_refuse_to_mix():
    a = synthetic.make_dataset(3, seed=1, n_mean=30, deg=6, n_feat=4, node_level=True)
    b = synthetic.make_dataset(2, seed=9, n_mean=30, deg=6, n_feat=4, node_level=True)
    c = synthetic.concat_packed([a, b])
    assert c.node_level and np.array_equal(c.y, np.vstack([a.y, b.y]))
    t = synthetic.tile_dataset(a, 5)
    assert t.node_level and t.n_graphs == 5 and t.y.shape[0] == int(t.node_off[-1])
    assert np.array_equal(t.y, np.vstack([a.y, a.y[:int(a.node_off[2])]]))
    gl = synthetic.make_dataset(2, seed=1, n_mean=30, deg=6, n_feat=4)
    with pytest.raises(ValueError):
        synthetic.concat_packed([a, gl])
    with pytest.raises(ValueError):
        synthetic.concat_packed([gl, a])


def _v1_bytes(p, symmetric):
    """The graph-level shard exactly as the version-1 format defines it (header + 64-byte aligned sections)."""
    n, g_, nnz = int(p.node_off[-1]), p.n_graphs, int(p.col.shape[0])
    arrays = [np.ascontiguousarray(p.node_off, "<i8"), np.ascontiguousarray(p.rowptr, "<i8"),
              np.ascontiguousarray(p.col, "<i4"), np.ascontiguousarray(p.x, "<f4"), np.ascontiguousarray(p.y, "<f4")]
    total = 0
    for a in arrays:
        b = a.view(np.uint8).reshape(-1)
        total += int(b[:b.size // 4 * 4].view("<u4").sum(dtype=np.uint64))
    out = struct.pack("<8sIIIIQQQQQ", b"GCSSHRD1", 1, p.x.shape[1], p.y.shape[1], int(symmetric), g_, n, nnz,
                      total & 0xFFFFFFFFFFFFFFFF, 0)
    for a in arrays:
        raw = a.tobytes()
        out += raw + b"\0" * ((-len(raw)) % 64)
    return out


def test_graph_level_shards_stay_version_1_byte_for_byte(tmp_path):
    p = synthetic.make_dataset(5, seed=2, n_mean=30, deg=6, n_feat=7)
    path = shards.write_shard(str(tmp_path / "g.gcss"), p)
    raw = open(path, "rb").read()
    assert raw == _v1_bytes(p, True)
    h = shards.read_header(path)
    assert h.version == 1 and h.flags == 1 and not h.node_level
    q = shards.read_shard(path, verify=True)
    assert not q.node_level and np.array_equal(q.y, p.y)


def test_node_level_shard_round_trip_is_version_2(tmp_path):
    p = synthetic.make_dataset(5, seed=2, n_mean=30, deg=6, n_feat=7, node_level=True)
    path = shards.write_shard(str(tmp_path / "n.gcss"), p)
    magic, ver, nf, nc, flags = struct.unpack("<8sIIII", open(path, "rb").read(24))
    assert (ver, flags, nf, nc) == (2, 3, 7, 2)
    for mmap in (True, False):
        q = shards.read_shard(path, mmap=mmap, verify=True)
        assert q.node_level and q.symmetric
        for name in ("node_off", "rowptr", "col", "x", "y"):
            assert np.array_equal(getattr(q, name), getattr(p, name)), name
    # a version-1 reader refuses it: its check is `version != 1`
    assert ver != 1


@pytest.mark.parametrize("ver,flags", [(1, 2), (1, 3), (2, 1), (2, 0), (3, 2)])
def test_shard_version_and_node_flag_must_agree(tmp_path, ver, flags):
    p = synthetic.make_dataset(2, seed=2, n_mean=20, deg=4, n_feat=3, node_level=flags & 2 == 2)
    path = shards.write_shard(str(tmp_path / "s.gcss"), p)
    raw = bytearray(open(path, "rb").read())
    raw[8:12] = struct.pack("<I", ver)
    raw[20:24] = struct.pack("<I", flags)
    open(path, "wb").write(bytes(raw))
    with pytest.raises(ValueError):
        shards.read_shard(path)


def test_write_and_load_dataset_of_node_labels(tmp_path):
    gr = _graphs([3, 0, 1, 6, 4], c=2, seed=5)
    d = str(tmp_path / "nl")
    paths = shards.write_dataset(gr, d, graphs_per_shard=2, node_level=True)
    assert len(paths) == 3
    idx = json.load(open(os.path.join(d, "index.json")))
    assert idx["labels"] == "node" and idx["version"] == 2
    p = shards.load_dataset(d, verify=True)
    assert p.node_level and np.array_equal(p.y, np.vstack([x.y for x in gr]))
    dg = str(tmp_path / "gl")
    shards.write_dataset([Graph(x=x.x, a=x.a, y=np.array([1.0, 0.0])) for x in gr], dg, graphs_per_shard=2)
    idx = json.load(open(os.path.join(dg, "index.json")))
    assert idx["labels"] == "graph" and idx["version"] == 1
    mixed = [os.path.join(d, idx["shards"][0]["file"]), os.path.join(dg, idx["shards"][0]["file"])]
    with pytest.raises(ValueError):
        shards.load_dataset(mixed)


def test_loader_refuses_a_dataset_of_the_other_kind():
    nl = synthetic.make_dataset(3, seed=1, n_mean=20, deg=4, n_feat=3, node_level=True)
    gl = synthetic.make_dataset(3, seed=1, n_mean=20, deg=4, n_feat=3)
    with pytest.raises(ValueError, match="node"):
        g.DisjointLoader(nl, batch_size=2)
    with pytest.raises(ValueError, match="graph"):
        g.DisjointLoader(gl, batch_size=2, node_level=True)
    with pytest.raises(ValueError):                      # graph labels in Graph objects, node_level=True
        g.DisjointLoader([Graph(x=np.ones((2, 3)), a=sp.eye(2), y=np.array([0.0, 1.0]))], node_level=True)


def _case(small_case, connectivity, seed=41, soft=False):
    c = small_case
    cfg = GNNConfig(in_features=12, output=3, activation="softmax", hidden=16, message_passing=3,
                    connectivity=connectivity, pool=None)
    specs = block_specs(cfg)
    w, s = g.init_params(cfg, seed=seed, perturb=True)
    n = c["x"].shape[0]
    rng = np.random.default_rng(seed)
    y = np.eye(3, dtype=np.float32)[rng.integers(0, 3, n)]
    if soft:
        y[::5] = rng.random((y[::5].shape[0], 3)).astype(np.float32)        # soft rows, sum != 1
        y[3::7] = 0.0                                                       # rows without a label
    return cfg, specs, w, s, (cfg, specs, w, s, c["x"], c["idx"][:, 0], c["idx"][:, 1], None, y, None)


@pytest.mark.parametrize("connectivity", ["cat", "sum", None])
def test_float64_and_autograd_restatements_agree(small_case, connectivity):
    cfg, specs, w, s, args = _case(small_case, connectivity)
    r1, r2 = O1.loss_and_grads(*args), O2.loss_and_grads(*args)
    assert r1["probs"].shape == (small_case["x"].shape[0], 3)
    assert abs(r1["loss"] - r2["loss"]) < 1e-5 * abs(r1["loss"])
    assert rel_err(r2["probs"], r1["probs"]) < 1e-5
    assert rel_err(r2["grads"], r1["grads"]) < 2e-5
    assert rel_err(r2["new_state"], r1["new_state"]) < 1e-5


@pytest.mark.parametrize("connectivity", ["cat", "sum", None])
def test_manual_backward_matches_finite_differences(small_case, connectivity):
    c = small_case
    cfg, specs, w, s, args = _case(small_case, connectivity, seed=43, soft=True)
    y = args[8].astype(np.float64)
    rows, cols = c["idx"][:, 0], c["idx"][:, 1]
    r = O1.loss_and_grads(*args)

    def loss_at(wv):
        return O1.loss_at(cfg, specs, wv, s, c["x"], rows, cols, None, y, None)

    rng = np.random.default_rng(11)
    scale = np.abs(r["grads"]).max()
    for j in rng.integers(0, w.shape[0], 14):
        wp = w.astype(np.float64).copy()
        wm = wp.copy()
        wp[j] += 1e-6
        wm[j] -= 1e-6
        assert abs((loss_at(wp) - loss_at(wm)) / 2e-6 - r["grads"][j]) < 2e-6 * scale + 1e-9, j


def test_library_exports_the_node_level_entry_points():
    from gcn_string_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = _lib.load()
    for name in ("gcs_gather_node_rows", "gcs_softmax_xent_workspace_bytes", "gcs_softmax_xent_ws"):
        assert hasattr(lib, name) and name in _lib.PROTOTYPES
    # the single-block kernel up to 65 536 rows (no workspace), the grid above
    assert lib.gcs_softmax_xent_workspace_bytes(0, 2) == 0
    assert lib.gcs_softmax_xent_workspace_bytes(65536, 2) == 0
    assert lib.gcs_softmax_xent_workspace_bytes(65537, 2) > 0
    assert lib.gcs_softmax_xent_workspace_bytes(2_000_000, 64) > 0
    # the model reserves it only above the threshold: graph-level plans keep their size
    cfg = _lib.model_config(GNNConfig(in_features=32, output=2, activation="softmax", pool=None))
    per_node = lib.gcs_model_workspace_bytes(cfg, 2, 10, 1, 1) - lib.gcs_model_workspace_bytes(cfg, 1, 10, 1, 1)
    small = lib.gcs_model_workspace_bytes(cfg, 65536, 10, 1, 1) - lib.gcs_model_workspace_bytes(cfg, 65535, 10, 1, 1)
    big = lib.gcs_model_workspace_bytes(cfg, 65537, 10, 1, 1) - lib.gcs_model_workspace_bytes(cfg, 65536, 10, 1, 1)
    assert big > small and per_node > 0
