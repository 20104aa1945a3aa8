"""GPU tests of the attribution backward: dx and d(edge weights) through GradientTape.watch against the float64
restatement (tests/attr_ref.py) in inference and training mode over pools, connectivities, aggregations, heads, widths
(FFMA and tensor-core paths), both aggregation paths and dropout; gcs_spmm_edge_grad alone against NumPy; the
attribution forward against the plain inference forward; bit identity (repeated calls, parameter gradients with and
without a watched x); batch independence in inference mode; an allocation-free loop; and the attribute() helper."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

import gcn_string_b200 as g
from gcn_string_b200 import _lib, attributions, synthetic
from gcn_string_b200.params import GNNConfig, block_specs, dropout_seed

from oracle import batching_ref
from oracle import model_ref_np as O1

import attr_ref as A
import dropout_ref as D

from conftest import rel_err
from test_model_gpu import TOL, gpu_prelu_branches, host

pytestmark = pytest.mark.gpu


def _model(cfg, w, s, rate=0.0, weighted=False):
    m = g.GeneralGNN(cfg.output, activation=cfg.activation, hidden=cfg.hidden, message_passing=cfg.message_passing,
                     pre_process=cfg.pre_process, post_process=cfg.post_process, pool=cfg.pool,
                     connectivity=cfg.connectivity, aggregate=cfg.aggregate, dropout=rate, seed=3,
                     use_edge_weights=weighted)
    m.build(cfg.in_features)
    m.load_flat(w, s)
    return m


def _data(ds, B, weighted):
    (xr, (idx, _, _), seg), _ = batching_ref.collate([ds.graph(k) for k in range(B)])
    (x, a, i), _ = next(g.DisjointLoader(ds, batch_size=B, epochs=1, shuffle=False))
    assert np.array_equal(host(a.indices), idx)
    ew = None
    if weighted:
        ew = np.random.default_rng(7).uniform(0.3, 1.5, idx.shape[0]).astype(np.float32)
        a.edge_weight = torch.from_numpy(ew).cuda()
    return (x, a, i), xr, idx[:, 0], idx[:, 1], seg, ew


def attr_vs_ref(cfg, ds, B, training, weighted=True, rate=0.0, max_graph_nodes=None, tol=TOL, x64=False):
    inputs, xr, rows, cols, seg, ew = _data(ds, B, weighted)
    x, a, i = inputs
    if max_graph_nodes is not None:
        a.max_graph_nodes = max_graph_nodes
    if x64:
        x = x.double()
        inputs = (x, a, i)
    specs = block_specs(cfg)
    w, s = g.init_params(cfg, seed=21, perturb=True)
    s = A.calibrated_state(cfg, specs, w, s, xr, rows, cols, seg, B, ew)
    model = _model(cfg, w, s, rate, weighted)
    n = xr.shape[0]
    r_out = n if cfg.pool is None else B
    d = np.random.default_rng(n).standard_normal((r_out, cfg.output)).astype(np.float32)
    step = model.dropout_step
    with g.GradientTape() as tape:
        tape.watch(x)
        tape.watch(a)
        pred = model(inputs, training=training)
    dx, dew = tape.gradient(pred, [x, a], output_gradients=torch.from_numpy(d).cuda())
    assert dx.shape == (n, cfg.in_features) and dx.dtype == (torch.float64 if x64 else torch.float32)
    masks, branches = None, None
    if training:
        masks = D.model_masks(specs, cfg, n, r_out, rate, dropout_seed(3, 0), step) if rate else None
        branches = gpu_prelu_branches(model, cfg, n, B)
    probs, _ = O1.forward(cfg, specs, w, s, xr, rows, cols, seg, B, training=training, edge_weight=ew, masks=masks,
                          rate=rate)
    assert rel_err(host(pred), probs) < tol
    dl = A.output_grad(cfg.activation, host(pred), d)
    rx, re_ = A.input_grads(cfg, specs, w, s, xr, rows, cols, seg, B, dl, training=training, edge_weight=ew,
                            masks=masks, rate=rate, prelu_branch=branches)
    assert rel_err(host(dx), rx) < tol, ("dx", rel_err(host(dx), rx))
    if weighted:
        assert dew.shape == (rows.shape[0],)
        assert rel_err(host(dew), re_) < tol, ("dew", rel_err(host(dew), re_))
    else:
        assert dew is None                                # the aggregation never read the edge weights
    return model, inputs, dx, dew


@pytest.fixture(scope="module")
def small_ds():
    return synthetic.make_dataset(8, seed=3, n_mean=60, deg=8, n_feat=12)


@pytest.mark.parametrize("training", [False, True])
@pytest.mark.parametrize("pool", ["sum", "avg", "attn_sum", None])
@pytest.mark.parametrize("connectivity", ["cat", "sum", None])
def test_pools_and_connectivity(small_ds, training, pool, connectivity):
    cfg = GNNConfig(in_features=12, output=2, activation="softmax", hidden=16, message_passing=3,
                    connectivity=connectivity, pool=pool)
    attr_vs_ref(cfg, small_ds, 8, training)


@pytest.mark.parametrize("training", [False, True])
@pytest.mark.parametrize("aggregate,connectivity", [("sum", "cat"), ("mean", "cat"), ("mean", "sum"), ("max", "cat"),
                                                    ("max", None)])
@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("hidden", [16, 128, 256])
def test_aggregations_and_widths(small_ds, training, aggregate, connectivity, weighted, hidden):
    cfg = GNNConfig(in_features=12, output=2, activation="softmax", hidden=hidden, message_passing=3,
                    connectivity=connectivity, aggregate=aggregate)
    # max: the selection is not pinned to the GPU's here, so a float32 near-tie may pick the other maximum (seen once
    # at 1.2e-4, H = 256); the exact tie-sharing rule is checked bit for bit by test_spmm_edge_grad_against_numpy
    attr_vs_ref(cfg, small_ds, 8, training, weighted=weighted, tol=1e-3 if aggregate == "max" else 2 * TOL)


@pytest.mark.parametrize("training", [False, True])
@pytest.mark.parametrize("activation", ["softmax", "sigmoid", None])
@pytest.mark.parametrize("pool", ["sum", None])
def test_heads_with_output_gradients(small_ds, training, activation, pool):
    cfg = GNNConfig(in_features=12, output=3, activation=activation, hidden=16, message_passing=2, pool=pool)
    attr_vs_ref(cfg, small_ds, 8, training)


@pytest.mark.parametrize("aggregate", ["sum", "mean", "max"])
@pytest.mark.parametrize("hidden", [16, 128])
def test_training_mode_with_dropout(small_ds, aggregate, hidden):
    cfg = GNNConfig(in_features=12, output=2, activation="softmax", hidden=hidden, message_passing=3,
                    aggregate=aggregate)
    attr_vs_ref(cfg, small_ds, 8, True, rate=0.3, tol=2 * TOL)


@pytest.mark.parametrize("training", [False, True])
def test_global_memory_path_and_float64_x(training):
    """No slab (max_graph_nodes = 0): the row-block / row kernels; float64 x returns a float64 gradient."""
    ds = synthetic.make_dataset(6, seed=5, n_mean=300, deg=12, n_feat=16)
    cfg = GNNConfig(in_features=16, output=2, activation="softmax", hidden=128, message_passing=2)
    attr_vs_ref(cfg, ds, 6, training, weighted=False, max_graph_nodes=0)
    attr_vs_ref(cfg, ds, 6, training, weighted=True, x64=True)


def test_attribution_forward_equals_inference_forward(small_ds):
    cfg = GNNConfig(in_features=12, output=2, activation="softmax", hidden=128, message_passing=3)
    inputs, *_ = _data(small_ds, 8, False)
    w, s = g.init_params(cfg, seed=21, perturb=True)
    model = _model(cfg, w, s)
    plain = host(model(inputs, training=False))
    state = host(model.state).copy()
    with g.GradientTape() as tape:
        tape.watch(inputs[0])
        attr = host(model(inputs, training=False))
    assert rel_err(attr, plain) < TOL
    assert np.array_equal(host(model.state), state)            # no moving-statistics update


def test_edge_weights_unconnected_and_parameter_errors(small_ds):
    cfg = GNNConfig(in_features=12, output=2, activation="softmax", hidden=16, message_passing=2)
    inputs, *_ = _data(small_ds, 8, False)
    x, a, _ = inputs
    model = _model(cfg, *g.init_params(cfg, seed=1))
    other = torch.zeros(3, device="cuda")
    with g.GradientTape() as tape:
        tape.watch(x)
        tape.watch(a)
        pred = model(inputs, training=False)
    dx, da, do = tape.gradient(pred, [x, a, other])
    assert dx is not None and da is None and do is None
    with pytest.raises(NotImplementedError, match="training=False"):
        tape.gradient(pred, [x, model.trainable_variables[0]])
    with g.GradientTape() as tape:                               # nothing watched: the plain inference path, no record
        pred = model(inputs, training=False)
    assert not hasattr(pred, "_gcs_tape") and tape.model is None


def test_parameter_gradients_bit_identical_with_and_without_watched_x(small_ds):
    cfg = GNNConfig(in_features=12, output=2, activation="softmax", hidden=128, message_passing=3)
    inputs, xr, rows, cols, seg, _ = _data(small_ds, 8, True)
    x, a, i = inputs
    y = torch.from_numpy(np.eye(2, dtype=np.float32)[np.arange(8) % 2]).cuda()
    w, s = g.init_params(cfg, seed=21, perturb=True)
    model = _model(cfg, w, s, weighted=True)
    loss_fn = g.CategoricalCrossentropy()
    with g.GradientTape() as tape:
        loss = loss_fn(y, model(inputs, training=True))
    ref = [host(t).copy() for t in tape.gradient(loss, model.trainable_variables)]
    model.load_flat(w, s)
    with g.GradientTape() as tape:
        tape.watch(x)
        tape.watch(a)
        loss = loss_fn(y, model(inputs, training=True))
    got = tape.gradient(loss, [x, a] + model.trainable_variables)
    assert got[0] is not None and got[1] is not None
    for r, t in zip(ref, got[2:]):
        assert np.array_equal(r, host(t))


def test_repeated_calls_bit_identical_and_allocation_free(small_ds):
    cfg = GNNConfig(in_features=12, output=2, activation="softmax", hidden=128, message_passing=3, aggregate="max")
    inputs, *_ = _data(small_ds, 8, True)
    model = _model(cfg, *g.init_params(cfg, seed=2, perturb=True), weighted=True)
    x, a, _ = inputs
    og = torch.ones(8, 2, device="cuda")

    def run():
        with g.GradientTape() as tape:
            tape.watch(x)
            tape.watch(a)
            pred = model(inputs, training=False)
        return tape.gradient(pred, [x, a], output_gradients=og)
    first = [host(t).copy() for t in run()]
    for _ in range(3):
        run()
    torch.cuda.synchronize()
    before = torch.cuda.memory_stats().get("num_device_alloc", 0)
    for _ in range(8):
        got = run()
        assert all(np.array_equal(f, host(t)) for f, t in zip(first, got))
    torch.cuda.synchronize()
    assert torch.cuda.memory_stats().get("num_device_alloc", 0) == before


def test_inference_attributions_are_batch_independent():
    ds = synthetic.make_dataset(32, seed=9, n_mean=50, deg=8, n_feat=16)
    model = g.GeneralGNN(2, activation="softmax", hidden=128, message_passing=3, seed=0, use_edge_weights=True,
                         aggregate="mean")
    (x, a, i), _ = next(g.DisjointLoader(ds, batch_size=32, epochs=1, shuffle=False))
    a.edge_weight = torch.rand(a.nnz, device="cuda") + 0.5
    batch = attributions.attribute(model, (x, a, i), 1)
    (x1, a1, i1), _ = next(g.DisjointLoader(ds, batch_size=1, epochs=1, shuffle=False))
    a1.edge_weight = a.edge_weight[:a1.nnz].clone()
    alone = attributions.attribute(model, (x1, a1, i1), 1)
    assert len(batch) == 32 and len(alone) == 1
    assert rel_err(alone[0]["residues"], batch[0]["residues"]) < TOL
    for u, v in zip(alone[0]["contacts"], batch[0]["contacts"]):
        assert rel_err(u, v) < TOL
    gx = attributions.attribute(model, (x, a, i), 0, method="grad_x_input")
    assert gx[5]["residues"].shape == (int(host(a.graph_ptr)[6] - host(a.graph_ptr)[5]),)


# ---------------------------------------------------------------------------------------------- gcs_spmm_edge_grad


def _edge_grad_case(H, agg, weighted, transform, rng):
    n = 23
    rows, cols = [], []
    for r in range(n):
        if r in (4, 11):                                          # empty rows
            continue
        k = rng.integers(1, 6)
        for c in sorted(rng.choice(n, k, replace=False)):
            rows.append(r)
            cols.append(c)
    rows, cols = np.array(rows), np.array(cols)
    rowptr = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=n))]).astype(np.int32)
    X = rng.integers(-3, 4, (n, H)).astype(np.float32)            # small integers: exact ties under max
    vals = rng.choice([0.5, 1.0, 2.0], rows.shape[0]).astype(np.float32) if weighted else None
    sc = rng.uniform(0.5, 1.5, H).astype(np.float32) if transform else None
    sh = rng.uniform(-0.5, 0.5, H).astype(np.float32) if transform else None
    al = rng.uniform(0.1, 0.3, H).astype(np.float32) if transform else None
    dZ = rng.standard_normal((n, H)).astype(np.float32)
    cuda = lambda v: None if v is None else torch.from_numpy(np.ascontiguousarray(v)).cuda()
    dev = dict(rp=cuda(rowptr), ci=cuda(cols.astype(np.int32)), v=cuda(vals), X=cuda(X), sc=cuda(sc), sh=cuda(sh),
               al=cuda(al), dZ=cuda(dZ))
    return n, rows, cols, rowptr, X, vals, sc, sh, al, dZ, dev


@pytest.mark.parametrize("agg", [0, 1, 2])
@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("H", [1, 7, 33, 130, 256])
def test_spmm_edge_grad_against_numpy(agg, weighted, H):
    lib = _lib.load()
    rng = np.random.default_rng(H * 10 + agg)
    transform = H % 2 == 1
    n, rows, cols, rowptr, X, vals, sc, sh, al, dZ, dev = _edge_grad_case(H, agg, weighted, transform, rng)
    p = _lib.ptr
    Z = torch.empty(n, H, device="cuda")
    _lib.check(lib.gcs_spmm_aggregate(p(dev["rp"]), p(dev["ci"]), p(dev["v"]), None, None, n, p(dev["X"]), H,
                                      p(dev["sc"]), p(dev["sh"]), p(dev["al"]), None, 0, p(Z), H, H, agg,
                                      _lib.stream_ptr()))
    ties = torch.empty(n, H, device="cuda")
    dA = torch.empty(n, H, device="cuda")
    # the transposed pattern for gcs_spmm_aggregate_bwd, which leaves the tie counts of max in `ties`
    order = np.lexsort((rows, cols))
    rp_t = np.concatenate([[0], np.cumsum(np.bincount(cols, minlength=n))]).astype(np.int32)
    ci_t = torch.from_numpy(rows[order].astype(np.int32)).cuda()
    v_t = torch.from_numpy(vals[order]).cuda() if weighted else None
    rp_t = torch.from_numpy(rp_t).cuda()
    _lib.check(lib.gcs_spmm_aggregate_bwd(p(rp_t), p(ci_t), p(v_t), p(dev["rp"]), p(dev["ci"]), p(dev["v"]), n,
                                          p(dev["dZ"]), H, agg, p(dev["X"]), H, p(dev["sc"]), p(dev["sh"]),
                                          p(dev["al"]), p(Z), H, p(ties), H, p(dA), H, H, _lib.stream_ptr()))
    dw = torch.full((rows.shape[0],), 5.0, device="cuda")
    for acc in (0, 1):
        _lib.check(lib.gcs_spmm_edge_grad(p(dev["rp"]), p(dev["ci"]), p(dev["v"]), n, p(dev["dZ"]), H, agg,
                                          p(dev["X"]), H, p(dev["sc"]), p(dev["sh"]), p(dev["al"]), p(Z), H, p(ties),
                                          H, H, p(dw), acc, _lib.stream_ptr()))
        if acc == 0:
            once = host(dw).copy()
    a = X.astype(np.float32)
    if transform:                                               # fmaf: one rounding (exact in double, then float)
        z = (a.astype(np.float64) * sc + sh).astype(np.float32)
        a = np.where(z > 0, z, al * z).astype(np.float32)
    zh = host(Z)
    w = vals if weighted else np.ones(rows.shape[0], np.float32)
    g = dZ[rows].astype(np.float64) * a[cols]
    if agg == 1:
        g /= np.bincount(rows, minlength=n)[rows][:, None]
    if agg == 2:
        sel = (a[cols] * w[:, None] if weighted else a[cols]) == zh[rows]
        cnt = np.zeros((n, H))
        np.add.at(cnt, rows, sel)
        g = np.where(sel, g / np.maximum(cnt, 1)[rows], 0.0)
    ref = g.sum(1)
    assert rel_err(once, ref) < 1e-5
    assert rel_err(host(dw), 2 * ref) < 1e-5
