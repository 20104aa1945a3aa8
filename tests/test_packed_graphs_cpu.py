"""The packed layout on the CPU: the parallel generator against the serial one, PackedGraphs.take against packing the
same graphs, and concat_packed's rebasing and its rule for the symmetric flag."""
import numpy as np
import pytest

from gcn_string_b200 import synthetic
from gcn_string_b200.data import Graph
from gcn_string_b200.synthetic import PackedGraphs, concat_packed

FIELDS = ("node_off", "rowptr", "col", "x", "y")


def _same(p, q):
    assert p.node_level == q.node_level
    for name in FIELDS:
        a, b = getattr(p, name), getattr(q, name)
        assert a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a, b), name


@pytest.mark.parametrize("node_level", [False, True])
def test_make_dataset_parallel_equals_make_dataset(node_level):
    kw = dict(seed=3, n_mean=40, deg=8, n_feat=5, n_classes=3, node_level=node_level)
    _same(synthetic.make_dataset_parallel(16, workers=2, **kw), synthetic.make_dataset(16, **kw))


@pytest.mark.parametrize("node_level", [False, True])
def test_take_equals_pack_graphs_of_the_same_graphs(node_level):
    p = synthetic.make_dataset(9, seed=6, n_mean=30, deg=6, n_feat=4, node_level=node_level)
    ids = np.random.default_rng(2).permutation(9)[:6]
    graphs = [Graph(x, a, y=y) for x, a, y in (p.graph(int(k)) for k in ids)]
    _same(p.take(ids), synthetic.pack_graphs(graphs, node_level=node_level))


def test_span_covers_the_graphs_nodes_and_entries():
    p = synthetic.make_dataset(5, seed=1, n_mean=30, deg=6, n_feat=3)
    n0, n1, e0, e1 = p.span(1, 4)
    assert (n1 - n0, e1 - e0) == (int(p.n_nodes[1:4].sum()), int(p.n_edges[1:4].sum()))
    assert p.span(0, p.n_graphs) == (0, p.x.shape[0], 0, p.col.shape[0])


def test_concat_rebases_each_part_on_its_own_first_entry():
    p = synthetic.make_dataset(5, seed=4, n_mean=30, deg=6, n_feat=3)
    n0, n1, e0, e1 = p.span(2, 4)
    mid = PackedGraphs(p.node_off[2:5] - n0, p.rowptr[n0:n1 + 1], p.col[e0:e1], p.x[n0:n1], p.y[2:4])
    assert mid.rowptr[0] > 0                                 # rows still point into the whole pack's entries
    _same(concat_packed([mid, p]), p.take([2, 3, 0, 1, 2, 3, 4]))


def test_concat_symmetric_rule_and_single_part():
    p = synthetic.make_dataset(3, seed=2, n_mean=20, deg=4, n_feat=3)
    q = synthetic.make_dataset(2, seed=5, n_mean=20, deg=4, n_feat=3)
    assert p.symmetric is None and concat_packed([p, q]).symmetric is None      # synthetic packs stay unknown
    assert synthetic.tile_dataset(p, 5).symmetric is None
    with_flag = lambda pack, s: PackedGraphs(pack.node_off, pack.rowptr, pack.col, pack.x, pack.y, symmetric=s)  # noqa: E731
    for flags, want in [((True, True), True), ((True, False), False), ((None, False), False), ((True, None), None)]:
        assert concat_packed([with_flag(p, flags[0]), with_flag(q, flags[1])]).symmetric is want, flags
    assert concat_packed([p]) is p
    empty = p.take([])
    assert empty.n_graphs == 0 and concat_packed([empty, q, empty]) is q
