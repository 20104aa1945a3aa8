"""CPU tests of the attribution backward's float64 restatement (tests/attr_ref.py) - against central finite
differences of oracle/model_ref_np's forward and against float32 autograd of oracle/model_ref_torch - and of the
Python surface that needs no device: GradientTape.watch / gradient routing and errors, the new prototypes against the
header, and the per-graph split of gcn_string_b200.attributions."""
import os
import re

import numpy as np
import pytest

import gcn_string_b200 as g
from gcn_string_b200 import _lib, attributions, synthetic
from gcn_string_b200.models import GradientTape, _WatchedInputs
from gcn_string_b200.params import GNNConfig, block_specs

from oracle import batching_ref
from oracle import model_ref_np as O1

import attr_ref as A
import dropout_ref as D

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


NG = 5                   # graphs per batch: training-mode BatchNorm over the pooled rows needs more than two


def _batch(n_graphs=NG, seed=4, n_feat=5):
    ds = synthetic.make_dataset(n_graphs, seed=seed, n_mean=9, deg=3, n_feat=n_feat)
    (x, (idx, _, _), seg), _ = batching_ref.collate([ds.graph(k) for k in range(n_graphs)])
    return np.asarray(x, dtype=np.float64), idx[:, 0], idx[:, 1], seg


def _setup(cfg, weighted, seed=1):
    x, rows, cols, seg = _batch(n_feat=cfg.in_features)
    specs = block_specs(cfg)
    w, s = g.init_params(cfg, seed=seed, perturb=True)
    rng = np.random.default_rng(seed)
    ew = rng.uniform(0.3, 1.5, rows.shape[0]) if weighted else None
    r_out = x.shape[0] if cfg.pool is None else NG
    d = rng.standard_normal((r_out, cfg.output))
    return x, rows, cols, seg, specs, w, s, ew, d


def _fd(f, v, idx, eps=1e-6):
    out = []
    for k in idx:
        vp, vm = v.copy(), v.copy()
        vp.flat[k] += eps
        vm.flat[k] -= eps
        out.append((f(vp) - f(vm)) / (2 * eps))
    return np.array(out)


def _check_fd(cfg, weighted, training, rate=0.0, tol=1e-5):
    x, rows, cols, seg, specs, w, s, ew, d = _setup(cfg, weighted)
    n = x.shape[0]
    masks = None
    if rate:
        r_out = n if cfg.pool is None else NG
        masks = D.model_masks(specs, cfg, n, r_out, rate, 11, 2)
    kw = dict(training=training, masks=masks, rate=rate)
    dx, dew = A.input_grads(cfg, specs, w, s, x, rows, cols, seg, NG, d, edge_weight=ew, **kw)
    assert dx.shape == x.shape and (dew is None) == (ew is None)
    rng = np.random.default_rng(0)
    ix = rng.choice(x.size, 24, replace=False)
    fx = _fd(lambda v: A.objective(cfg, specs, w, s, v, rows, cols, seg, NG, d, edge_weight=ew, **kw), x, ix)
    # floor: under training-mode BatchNorm the gradient can be tiny, and the central difference carries ~1e-10 noise
    assert np.abs(dx.flat[ix] - fx).max() / max(np.abs(dx).max(), 1e-4) < tol
    if ew is not None:
        ie = rng.choice(ew.size, min(24, ew.size), replace=False)
        fe = _fd(lambda v: A.objective(cfg, specs, w, s, x, rows, cols, seg, NG, d, edge_weight=v, **kw), ew, ie)
        assert np.abs(dew[ie] - fe).max() / max(np.abs(dew).max(), 1e-4) < tol


@pytest.mark.parametrize("training", [False, True])
@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("pool", ["sum", "avg", "attn_sum", None])
@pytest.mark.parametrize("connectivity", ["cat", "sum", None])
def test_input_grads_match_finite_differences_pools(training, weighted, pool, connectivity):
    cfg = GNNConfig(in_features=5, output=3, activation="softmax", hidden=6, message_passing=2,
                    connectivity=connectivity, pool=pool)
    _check_fd(cfg, weighted, training)


@pytest.mark.parametrize("training", [False, True])
@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("aggregate,connectivity", [("mean", "cat"), ("mean", "sum"), ("max", "cat"), ("max", None)])
def test_input_grads_match_finite_differences_aggregations(training, weighted, aggregate, connectivity):
    cfg = GNNConfig(in_features=5, output=2, activation="softmax", hidden=6, message_passing=2,
                    connectivity=connectivity, aggregate=aggregate)
    _check_fd(cfg, weighted, training)


def test_input_grads_match_finite_differences_with_dropout():
    cfg = GNNConfig(in_features=5, output=2, activation="softmax", hidden=6, message_passing=2, aggregate="mean")
    _check_fd(cfg, True, True, rate=0.3)


@pytest.mark.parametrize("training", [False, True])
@pytest.mark.parametrize("activation", ["softmax", "sigmoid", None])
def test_output_gradients_through_every_head(training, activation):
    """d<dprobs, probs>/dx through the head's Jacobian (output_grad) against finite differences of the probabilities."""
    cfg = GNNConfig(in_features=5, output=3, activation=activation, hidden=6, message_passing=2, pool="avg")
    x, rows, cols, seg, specs, w, s, ew, d = _setup(cfg, True)
    probs, _ = O1.forward(cfg, specs, w, s, x, rows, cols, seg, NG, training=training, edge_weight=ew)
    dl = A.output_grad(activation, probs, d)
    dx, dew = A.input_grads(cfg, specs, w, s, x, rows, cols, seg, NG, dl, training=training, edge_weight=ew)

    def f(xv, ev):
        p, _ = O1.forward(cfg, specs, w, s, xv, rows, cols, seg, NG, training=training, edge_weight=ev)
        return float((p * d).sum())
    ix = np.arange(0, x.size, 3)
    fx = _fd(lambda v: f(v, ew), x, ix)
    assert np.abs(dx.flat[ix] - fx).max() / np.abs(dx).max() < 1e-5
    ie = np.arange(0, ew.size, 3)
    fe = _fd(lambda v: f(x, v), ew, ie)
    assert np.abs(dew[ie] - fe).max() / np.abs(dew).max() < 1e-5


@pytest.mark.parametrize("training", [False, True])
@pytest.mark.parametrize("pool", ["sum", "attn_sum", None])
def test_input_grads_match_float32_autograd(training, pool):
    """The hand-derived float64 dx against torch autograd of the float32 restatement (sum aggregation, no weights)."""
    torch = pytest.importorskip("torch")
    from oracle import model_ref_torch as O2
    cfg = GNNConfig(in_features=5, output=3, activation="softmax", hidden=6, message_passing=2, pool=pool)
    x, rows, cols, seg, specs, w, s, _, d = _setup(cfg, False)
    dx, _ = A.input_grads(cfg, specs, w, s, x, rows, cols, seg, NG, d, training=training)
    params = O2.unpack(specs, w, s, requires_grad=False)
    xt, rt, ct, st = O2.tensors(x, rows, cols, seg if pool else None)
    xt.requires_grad_(True)
    logits = O2.forward(cfg, params, xt, rt, ct, st, NG, training, attn=O2.attn_leaf(cfg, specs, w, False))
    (logits * torch.tensor(d, dtype=torch.float32)).sum().backward()
    got = xt.grad.numpy().astype(np.float64)
    assert np.abs(got - dx).max() / np.abs(dx).max() < 1e-4


def test_inference_mode_is_batch_independent():
    """Moving statistics: a graph's input gradient alone equals its rows inside the batch."""
    cfg = GNNConfig(in_features=5, output=2, activation="softmax", hidden=6, message_passing=2, aggregate="mean")
    x, rows, cols, seg, specs, w, s, ew, d = _setup(cfg, True)
    dx, dew = A.input_grads(cfg, specs, w, s, x, rows, cols, seg, NG, d, edge_weight=ew)
    n0 = int((seg == 0).sum())
    m = rows < n0
    dx0, dew0 = A.input_grads(cfg, specs, w, s, x[:n0], rows[m], cols[m], seg[:n0], 1, d[:1], edge_weight=ew[m])
    assert np.abs(dx0 - dx[:n0]).max() < 1e-12 and np.abs(dew0 - dew[m]).max() < 1e-12


# ---------------------------------------------------------------------------------------------- Python surface


class _Obj:
    pass


def test_watched_inputs_routing():
    x, a, other = _Obj(), _Obj(), _Obj()
    a.edge_weight = _Obj()
    w = _WatchedInputs(x, None, a, None, True)
    assert w.kind(x) == "x" and w.kind(a) == "ew" and w.kind(other) is None and w.kind(None) is None
    w = _WatchedInputs(None, None, None, a.edge_weight, False)
    assert w.kind(a.edge_weight) == "unconnected" and w.kind(x) is None      # the model ignores edge weights


def test_tape_watch_is_idempotent_and_tracks_identity():
    t = GradientTape()
    x = _Obj()
    t.watch(x)
    t.watch([x])
    assert t._is_watched(x) and not t._is_watched(_Obj()) and len(t._watched) == 1


def test_parameter_gradients_of_an_inference_call_raise():
    t = GradientTape()
    t.model = object()
    t.loss_record = dict(dlogits=None)
    t.ctx = dict(mode="inference", inputs=_WatchedInputs(_Obj(), None, None, None, False))
    with pytest.raises(NotImplementedError, match="training=False"):
        t.gradient(object(), [_Obj()])


def test_new_prototypes_match_the_header():
    text = open(os.path.join(ROOT, "include", "gcnstring_b200.h")).read()
    for name, n_args in (("gcs_spmm_edge_grad", 20), ("gcs_model_forward_attr", 8), ("gcs_model_input_grad", 13),
                         ("gcs_output_grad", 7)):
        m = re.search(rf"\bint\s+{name}\s*\(([^)]*)\)", text)
        assert m, name
        assert len(m.group(1).split(",")) == n_args == len(_lib.PROTOTYPES[name][1]), name


def test_split_by_graph_on_a_two_graph_batch():
    # graph 0: nodes 0-2, entries (0,1) (1,0) (1,2) (2,1); graph 1: nodes 3-4, entries (3,4) (4,3) (4,4)
    rowptr = np.array([0, 1, 3, 4, 5, 7])
    colidx = np.array([1, 0, 2, 1, 4, 3, 4])
    node = np.arange(5, dtype=np.float64)
    edge = np.arange(7, dtype=np.float64) * 10
    out = attributions.split_by_graph(np.array([0, 3, 5]), rowptr, colidx, node, edge)
    assert len(out) == 2
    assert np.array_equal(out[0]["residues"], [0, 1, 2]) and np.array_equal(out[1]["residues"], [3, 4])
    r, c, sc = out[0]["contacts"]
    assert np.array_equal(r, [0, 1, 1, 2]) and np.array_equal(c, [1, 0, 2, 1]) and np.array_equal(sc, [0, 10, 20, 30])
    r, c, sc = out[1]["contacts"]
    assert np.array_equal(r, [0, 1, 1]) and np.array_equal(c, [1, 0, 1]) and np.array_equal(sc, [40, 50, 60])
    assert attributions.split_by_graph(np.array([0, 3, 5]), rowptr, colidx, node)[1]["contacts"] is None


def test_graph_offsets_from_the_batch_index():
    import torch

    class _A:
        graph_ptr = None
    assert np.array_equal(attributions.graph_offsets(_A(), torch.tensor([0, 0, 1, 1, 1]), 5), [0, 2, 5])
    assert np.array_equal(attributions.graph_offsets(_A(), None, 4), [0, 4])
