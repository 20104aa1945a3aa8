"""GPU tests of sample weights: the weighted loss kernel of every head against float64 (one block and the full grid,
unaligned inputs, C not a multiple of 4, zero weights, rows = 0, determinism), all-ones weights against the unweighted
kernels bit for bit, the weighted fused train step against the float64 restatement for every head, pool and
connectivity (node level with a 50 % mask), the GradientTape and DataParallelTrainer routes, the undersized workspace,
the loader's weights in every store mode, a masked training loop, and evaluate() with weights."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

import gcn_string_b200 as g
from gcn_string_b200 import _lib, ops, synthetic
from gcn_string_b200.evaluate import evaluate
from gcn_string_b200.params import GNNConfig, block_specs

import sw_ref as S

from conftest import rel_err
from test_model_gpu import TOL, gpu_prelu_branches, grad_errors, host, make_model
from test_regression_head_gpu import _targets_off_the_kinks

pytestmark = pytest.mark.gpu
HEAD = {"softmax": (1, 0), "sigmoid": (2, 0), "mse": (0, 1), "mae": (0, 2), "huber": (0, 3)}
LOSS = {"softmax": lambda: g.CategoricalCrossentropy(), "sigmoid": lambda: g.BinaryCrossentropy(),
        "mse": lambda: g.MeanSquaredError(), "mae": lambda: g.MeanAbsoluteError(), "huber": lambda: g.Huber(0.7)}
DELTA = 0.7


def _case(head, rows, c, seed, zero=False):
    rng = np.random.default_rng(seed)
    z = (2 * rng.standard_normal((rows, c))).astype(np.float32)
    if head == "softmax":
        y = np.eye(c, dtype=np.float32)[rng.integers(0, c, rows)]
    elif head == "sigmoid":
        y = (rng.random((rows, c)) > 0.5).astype(np.float32)
    else:
        y = rng.standard_normal((rows, c)).astype(np.float32)
    w = np.zeros(rows, np.float32) if zero else np.where(rng.random(rows) < 0.3, 0.0, rng.uniform(0.1, 3.0, rows))
    return z, y, w.astype(np.float32)


def _buf(a, offset):
    t = torch.empty(a.size + offset, device="cuda")
    t[offset:] = torch.from_numpy(np.ascontiguousarray(a).reshape(-1)).cuda()
    return t[offset:]


def _run(head, z, y, w, offset=0, weighted=True):
    """gcs_weighted_loss (or, weighted=False, the head's unweighted entry point) on copies `offset` floats into fresh
    buffers; returns host (probs or None, loss_acc, dlogits)."""
    lib = _lib.load()
    rows, c = z.shape
    code, kind = HEAD[head]
    zt, yt, wt = _buf(z, offset), _buf(y, offset), _buf(w, offset)
    probs = None if code == 0 else _buf(np.zeros_like(z), offset)
    dl = _buf(np.zeros_like(z), offset)
    la = torch.empty(2, device="cuda")
    st = _lib.stream_ptr()
    p = lambda t: t.data_ptr() if t is not None else None          # noqa: E731
    if weighted:
        need = lib.gcs_weighted_loss_workspace_bytes(code, rows, c)
        ws = torch.empty(max(need, 8), dtype=torch.uint8, device="cuda")
        _lib.check(lib.gcs_weighted_loss(code, kind, DELTA, p(zt), p(yt), p(wt), rows, c, p(probs), p(la), p(dl),
                                         1.0 / max(rows, 1), p(ws), need, st))
    elif code == 1:
        need = lib.gcs_softmax_xent_workspace_bytes(rows, c)
        ws = torch.empty(max(need, 8), dtype=torch.uint8, device="cuda")
        _lib.check(lib.gcs_softmax_xent_ws(p(zt), p(yt), rows, c, p(probs), p(la), p(dl), 1.0 / max(rows, 1), p(ws),
                                           need, st))
    elif code == 2:
        need = lib.gcs_sigmoid_bce_workspace_bytes(rows, c)
        ws = torch.empty(max(need, 8), dtype=torch.uint8, device="cuda")
        _lib.check(lib.gcs_sigmoid_bce(p(zt), p(yt), rows, c, p(probs), p(la), p(dl), 1.0 / max(rows, 1), p(ws), need, st))
    else:
        need = lib.gcs_regression_loss_workspace_bytes(rows, c)
        ws = torch.empty(max(need, 8), dtype=torch.uint8, device="cuda")
        _lib.check(lib.gcs_regression_loss(kind, DELTA, p(zt), p(yt), rows, c, None, p(la), p(dl), 1.0 / max(rows, 1),
                                           p(ws), need, st))
    return (None if probs is None else host(probs).reshape(z.shape)), host(la), host(dl).reshape(z.shape)


def _gpu_row_metric(head, z, y, probs):
    """The row metric from the kernel's own float32 probabilities (hits exactly as the kernel decides them)."""
    if head == "softmax":
        return (y.argmax(axis=1) == np.asarray(z).argmax(axis=1)).astype(np.float64)
    if head == "sigmoid":
        return (y == (probs > 0.5)).mean(axis=1)
    return np.abs(z.astype(np.float64) - y).mean(axis=1)


@pytest.mark.parametrize("head", list(HEAD))
@pytest.mark.parametrize("rows,c", [(1, 1), (1000, 3), (341, 3), (70_000, 2), (508_428, 1), (508_428, 2),
                                    (508_428, 16)])
def test_weighted_kernel_against_float64(head, rows, c):
    z, y, w = _case(head, rows, c, seed=rows % 997 + c)
    probs, la, dl = _run(head, z, y, w)
    loss, _, dref = S.weighted_loss(head, z, y, w, DELTA)
    assert abs(la[0] - loss) <= 1e-5 * max(abs(loss), 1e-30) + 1e-7, (la[0], loss)
    m = _gpu_row_metric(head, z, y, probs)
    metric = (w * m).sum() / w.sum() if w.sum() else 0.0
    assert abs(la[1] - metric) <= 1e-6 * max(abs(metric), 1.0), (la[1], metric)
    assert rel_err(dl, dref) < 1e-5
    assert not dl[w == 0].any()                                                # masked rows: exactly zero
    if probs is not None:
        assert np.array_equal(probs, _run(head, z, y, w, weighted=False)[0])   # the head's own probabilities
    again = _run(head, z, y, w)
    odd = _run(head, z, y, w, offset=1)                                        # off the 16-byte grid
    for other in (again, odd):
        assert all((a is None and b is None) or np.array_equal(a, b) for a, b in zip(other, (probs, la, dl)))


@pytest.mark.parametrize("head", list(HEAD))
@pytest.mark.parametrize("rows,c", [(1000, 3), (341, 4), (70_000, 2), (508_428, 1), (508_428, 16)])
def test_all_ones_weights_give_the_unweighted_bits(head, rows, c):
    z, y, _ = _case(head, rows, c, seed=7 + c)
    ones = np.ones(rows, np.float32)
    for offset in (0, 1):
        pw, lw, dw = _run(head, z, y, ones, offset=offset)
        pu, lu, du = _run(head, z, y, ones, offset=offset, weighted=False)
        assert lw[0] == lu[0] and np.array_equal(dw, du)
        assert pw is None or np.array_equal(pw, pu)
        assert abs(np.float32(lw[1]) - np.float32(lu[1])) <= np.spacing(np.float32(lu[1]))


@pytest.mark.parametrize("head", list(HEAD))
def test_zero_weights_and_zero_rows(head):
    for rows, c in ((1000, 3), (508_428, 2)):
        z, y, w = _case(head, rows, c, seed=3, zero=True)
        _, la, dl = _run(head, z, y, w)
        assert la.tolist() == [0.0, 0.0] and not dl.any()
    z, y, w = _case(head, 4, 2, seed=1)
    lib = _lib.load()
    code, kind = HEAD[head]
    zt, yt, wt = (torch.from_numpy(a).cuda() for a in (z, y, w))
    la = torch.full((2,), 7.0, device="cuda")
    _lib.check(lib.gcs_weighted_loss(code, kind, DELTA, zt.data_ptr(), yt.data_ptr(), wt.data_ptr(), 0, 2, None,
                                     la.data_ptr(), None, 1.0, None, 0, _lib.stream_ptr()))
    assert host(la).tolist() == [0.0, 0.0]
    # the wrappers: the weights may be [rows] or [rows, 1], anything else is refused before a launch
    fn = {"softmax": ops.softmax_xent, "sigmoid": ops.sigmoid_bce}.get(head)
    if fn is not None:
        a = fn(zt, yt, want_grad=True, sample_weight=wt)
        b = fn(zt, yt, want_grad=True, sample_weight=wt.reshape(4, 1).cpu().numpy())
        assert all(torch.equal(u, v) for u, v in zip(a, b))
        with pytest.raises(ValueError):
            fn(zt, yt, sample_weight=torch.ones(5, device="cuda"))
    else:
        with pytest.raises(ValueError):
            ops.regression_loss(zt, yt, head, DELTA, sample_weight=torch.ones(4, 2, device="cuda"))


# ---------------------------------------------------------------- the weighted train step
def _labels(head, z, seed):
    rng = np.random.default_rng(seed)
    rows, c = z.shape
    if head == "softmax":
        return np.eye(c, dtype=np.float32)[rng.integers(0, c, rows)]
    if head == "sigmoid":
        return (rng.random((rows, c)) > 0.5).astype(np.float32)
    return _targets_off_the_kinks(z, DELTA, seed)


def _weights(rows, node_level, seed):
    rng = np.random.default_rng(seed)
    if node_level:
        return (rng.random(rows) < 0.5).astype(np.float32)                    # a 50 % mask
    return rng.uniform(0.0, 2.5, rows).astype(np.float32)


@pytest.mark.parametrize("head", list(HEAD))
@pytest.mark.parametrize("pool", ["sum", "avg", "attn_sum", None])
@pytest.mark.parametrize("connectivity", ["cat", "sum", None])
def test_weighted_train_step_matches_float64(small_case, head, pool, connectivity):
    c = small_case
    cfg = GNNConfig(in_features=12, output=2, activation=S.activation(head), hidden=16, message_passing=3,
                    connectivity=connectivity, pool=pool)
    specs = block_specs(cfg)
    w, s = g.init_params(cfg, seed=91, perturb=True)
    (x, a, i), _ = next(g.DisjointLoader(c["ds"], batch_size=8, epochs=1, shuffle=False))
    n = c["x"].shape[0]
    base = (cfg, specs, w, s, c["x"], c["idx"][:, 0], c["idx"][:, 1], c["seg"])
    z0 = S.loss_and_grads(*base, np.zeros((n if pool is None else 8, 2)), 8, np.ones(n if pool is None else 8), "mse")["logits"]
    y = _labels(head, z0, seed=n)
    sw = _weights(y.shape[0], pool is None, seed=5)
    model = make_model(cfg, w, s)
    loss = LOSS[head]() if head in ("mse", "mae", "huber") else None
    loss_acc, probs = model.train_step_grads((x, a, i), torch.from_numpy(y).cuda(), loss=loss,
                                             sample_weight=torch.from_numpy(sw).cuda())
    branches = gpu_prelu_branches(model, cfg, n, 8)
    ref = S.loss_and_grads(*base, y, 8, sw, head, DELTA, prelu_branch=branches)
    o2 = S.torch_loss_and_grads(*base, y, 8, sw, head, DELTA)["grads"]
    got = host(loss_acc)
    assert abs(got[0] - ref["loss"]) < TOL * abs(ref["loss"])
    regression = head in ("mse", "mae", "huber")
    pr = host(probs)
    m = _gpu_row_metric(head, ref["logits"] if regression else pr, y, pr)   # hits as the GPU's probabilities decide
    metric = (sw * m).sum() / sw.sum()
    assert abs(got[1] - metric) < (TOL if regression else 1e-6) * max(abs(metric), 1.0)
    e_gpu = grad_errors(host(model.grads), ref["grads"], cfg)
    e_o2 = grad_errors(o2, ref["grads"], cfg)
    bad = {k: (v, e_o2[k]) for k, v in e_gpu.items()
           if v > max(TOL * (2.0 if k == "pool.attn_kernel" else 1.0), 10 * e_o2[k])}
    assert not bad, f"gradient tensors out of tolerance (gpu err, fp32-cpu err): {bad}"


@pytest.mark.parametrize("head", list(HEAD))
@pytest.mark.parametrize("pool", ["sum", None])
def test_tape_and_data_parallel_routes_equal_the_fused_step(head, pool):
    from gcn_string_b200.distributed import DataParallelTrainer
    node_level = pool is None
    task = "regression" if head in ("mse", "mae", "huber") else "classification"
    ds = synthetic.make_dataset(6, seed=11, n_mean=90, deg=10, n_feat=8, n_classes=3, task=task, node_level=node_level)
    (x, a, i), y = next(g.DisjointLoader(ds, node_level=node_level, batch_size=6, epochs=1, shuffle=False))
    if head == "sigmoid":
        y = (y > 0.5).float()
    sw = torch.from_numpy(_weights(y.shape[0], node_level, seed=2)).cuda()
    models = []
    for _ in range(3):
        m = g.GeneralGNN(3, activation=S.activation(head), hidden=64, message_passing=2, seed=0, pool=pool)
        m.build(8)
        wv, sv = g.init_params(m.cfg, seed=5, perturb=True)
        m.load_flat(wv, sv)
        models.append(m)
    fused, taped, dp = models
    reg = LOSS[head]() if head in ("mse", "mae", "huber") else None
    loss_acc, probs = fused.train_step_grads((x, a, i), y, loss=reg, sample_weight=sw)
    with g.GradientTape() as tape:
        pred = taped((x, a, i), training=True)
        loss = LOSS[head]()(y, pred, sample_weight=sw)
    tape.gradient(loss, taped.trainable_variables)
    assert torch.equal(loss_acc[0], loss) and torch.equal(tape.loss_record["loss_acc"], loss_acc)
    assert torch.equal(fused.grads, taped.grads) and torch.equal(fused.state, taped.state)
    opt = g.optimizers.SGD(learning_rate=0.0)
    la_dp, _ = DataParallelTrainer(dp, opt, loss=reg).train_step((x, a, i), y, sample_weight=sw)
    assert torch.equal(la_dp, loss_acc) and torch.equal(dp.grads, fused.grads)


def test_train_step_refuses_the_unweighted_workspace_for_a_weighted_batch():
    ds = synthetic.make_dataset(16, seed=2, n_mean=800, deg=8, n_feat=8, n_classes=3, node_level=True)
    (x, a, i), y = next(g.DisjointLoader(ds, node_level=True, batch_size=16, epochs=1, shuffle=False))
    model = g.GeneralGNN(3, activation="sigmoid", hidden=16, message_passing=2, seed=0, pool=None)
    model.build(8)
    lib = _lib.load()
    batch, keep = model._prepare((x, a, i), need_transpose=True)
    sw = torch.ones(x.shape[0], device="cuda")
    batch.y, batch.sample_weight = y.data_ptr(), sw.data_ptr()
    plain = lib.gcs_model_workspace_bytes(model._c, batch.n_nodes, batch.nnz, batch.n_graphs, 1)
    ex = lib.gcs_model_workspace_bytes_ex(model._c, batch.n_nodes, batch.nnz, batch.n_graphs, 1,
                                          _lib.WORKSPACE_SAMPLE_WEIGHTS)
    assert ex > plain
    ws = torch.empty(ex, dtype=torch.uint8, device="cuda")
    probs, la = torch.empty_like(y), torch.empty(2, device="cuda")
    args = (model._c, model.params.data_ptr(), model.state.data_ptr(), batch, 1.0 / x.shape[0], model.grads.data_ptr(),
            probs.data_ptr(), la.data_ptr(), ws.data_ptr())
    assert lib.gcs_model_train_step(*args, plain, _lib.stream_ptr()) == 3              # GCS_ERR_WORKSPACE
    assert lib.gcs_model_train_step(*args, ex, _lib.stream_ptr()) == 0
    torch.cuda.synchronize()


# ---------------------------------------------------------------- the loader, a training loop and evaluate
def _batches(n_graphs, batch_size, epochs, seed):
    np.random.seed(seed)
    order = np.arange(n_graphs)
    for _ in range(epochs):
        np.random.shuffle(order)
        for b in range(0, n_graphs, batch_size):
            yield order[b:b + batch_size].copy()


@pytest.mark.parametrize("node_level", [False, True])
def test_loader_weights_follow_the_batch_in_every_store_mode(node_level):
    ds = synthetic.make_dataset(11, seed=5, n_mean=50, deg=8, n_feat=7, node_level=node_level)
    rows = int(ds.node_off[-1]) if node_level else ds.n_graphs
    sw = np.random.default_rng(0).uniform(0, 1, rows).astype(np.float32)
    for kw in (dict(device_resident=True), dict(device_resident=False, zero_copy=True), dict(device_resident=False),
               dict(device_resident=False, device_gather=True), dict(device_resident=True, prefetch=True),
               dict(device_resident=False, shuffle=False)):
        shuffle = kw.pop("shuffle", True)
        np.random.seed(77)
        ld = g.DisjointLoader(ds, node_level=node_level, batch_size=4, epochs=2, shuffle=shuffle, sample_weights=sw, **kw)
        assert len(ld.tf_signature()) == 3
        out = list(ld)
        ids = list(_batches(11, 4, 2, 77)) if shuffle else [np.arange(b, min(b + 4, 11)) for b in (0, 4, 8)] * 2
        assert len(out) == len(ids) == 6
        for (inputs, y, w), gids in zip(out, ids):
            ref = (np.concatenate([sw[ds.node_off[k]:ds.node_off[k + 1]] for k in gids]) if node_level else sw[gids])
            assert np.array_equal(host(w), ref) and w.shape[0] == y.shape[0]
    plain = g.DisjointLoader(ds, node_level=node_level, batch_size=4, epochs=1)
    assert len(next(plain)) == 2 and len(plain.tf_signature()) == 2
    with pytest.raises(ValueError):
        g.DisjointLoader(ds, node_level=node_level, batch_size=4, sample_weights=sw[:-1])


def test_masked_node_level_loop_lowers_the_loss_without_driver_allocations():
    ds = synthetic.make_dataset(96, seed=3, n_mean=120, deg=10, n_feat=16, n_classes=2, node_level=True)
    mask = (np.random.default_rng(1).random(int(ds.node_off[-1])) < 0.5).astype(np.float32)
    model = g.GeneralGNN(2, activation="softmax", hidden=64, message_passing=2, seed=0, pool=None)
    model.build(16)
    loader = g.DisjointLoader(ds, node_level=True, batch_size=24, epochs=None, shuffle=True, sample_weights=mask)
    opt = g.optimizers.Adam(learning_rate=1e-2)

    def step():
        (x, a, i), y, w = next(loader)
        la, _ = model.train_step_grads((x, a, i), y, sample_weight=w)
        opt.apply_flat(model.params, model.grads)
        return la
    first = torch.stack([step() for _ in range(4)])
    for _ in range(28):
        step()
    torch.cuda.synchronize()
    before = torch.cuda.memory_stats().get("num_device_alloc", 0)
    last = torch.stack([step() for _ in range(24)])[-4:]
    torch.cuda.synchronize()
    assert torch.cuda.memory_stats().get("num_device_alloc", 0) == before
    f, l_ = host(first).mean(axis=0), host(last).mean(axis=0)
    assert l_[0] < 0.9 * f[0], (f, l_)


def test_evaluate_and_roc_curve_with_weights(small_case):
    from gcn_string_b200.evaluate import positive_scores, roc_curve
    cfg = GNNConfig(in_features=12, output=2, activation="softmax", hidden=16, message_passing=3, pool="avg")
    w, s = g.init_params(cfg, seed=43, perturb=True)
    model = make_model(cfg, w, s)
    sw = np.array([0.0, 1.0, 2.5, 0.5, 0.0, 1.5, 3.0, 1.0], np.float32)
    loader = g.DisjointLoader(small_case["ds"], batch_size=3, epochs=None, shuffle=False, sample_weights=sw)
    (loss, acc), preds = evaluate(model, loader)
    p = host(torch.cat(preds)).astype(np.float64)
    y = small_case["y"].astype(np.float64)
    # the loss is on the logits (no clipping of the probabilities): the same forward again, logits kept per batch
    plain = g.DisjointLoader(small_case["ds"], batch_size=3, epochs=1, shuffle=False)
    z = np.concatenate([host(model(inputs)._gcs_logits) for inputs, _ in plain])
    l_rows = S.row_terms("softmax", z, y)[0]
    assert loss == pytest.approx((sw * l_rows).sum() / 8, rel=1e-5)
    hit = (y.argmax(axis=1) == p.argmax(axis=1)).astype(np.float64)
    assert acc == pytest.approx((sw * hit).sum() / sw.sum(), rel=1e-6)
    fpr, tpr, thr = roc_curve(y[:, 1], positive_scores(preds), drop_intermediate=False, sample_weight=sw)
    rf, rt, rth = S.roc_curve(y[:, 1], p[:, 1].astype(np.float32), sw)
    np.testing.assert_allclose(fpr, rf, rtol=1e-12)
    np.testing.assert_allclose(tpr, rt, rtol=1e-12)
    np.testing.assert_allclose(thr, rth, rtol=1e-7)
