"""GPU tests of the linear head's regression losses: the fused MSE / MAE / Huber kernel against float64 (one block and the
full grid, unaligned inputs, exact ties and |e| == delta, rows = 0, determinism, argument errors), the
GeneralGNN(activation=None) train step against the float64 restatement for every loss, pool and connectivity, the
GradientTape and DataParallelTrainer routes, a training loop on synthetic regression data at graph and node level, and
evaluate() with a regression loss."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

import gcn_string_b200 as g
from gcn_string_b200 import _lib, ops, synthetic
from gcn_string_b200.data import Graph
from gcn_string_b200.params import GNNConfig, block_specs
from oracle import batching_ref, model_ref_np as O1, model_ref_torch as O2

from conftest import rel_err
from test_model_gpu import TOL, gpu_prelu_branches, grad_errors, host, make_model

pytestmark = pytest.mark.gpu
KIND = {"mse": 1, "mae": 2, "huber": 3}
LOSS = {"mse": lambda d: g.MeanSquaredError(), "mae": lambda d: g.MeanAbsoluteError(), "huber": lambda d: g.Huber(d)}


# ---------------------------------------------------------------- the kernel against float64
def _reg_case(rows, c, seed):
    rng = np.random.default_rng(seed)
    z = (2 * rng.standard_normal((rows, c))).astype(np.float32)
    y = rng.standard_normal((rows, c)).astype(np.float32)
    flat_z, flat_y = z.reshape(-1), y.reshape(-1)
    k = min(flat_z.size, 64)
    at = rng.choice(flat_z.size, k, replace=False)
    flat_z[at] = flat_y[at]                                                   # exact ties: e = 0
    return z, y


def _run(kind, z, y, delta=1.0, grad_scale=None, offset=0):
    """gcs_regression_loss with predictions written, on copies placed `offset` floats into fresh buffers."""
    lib = _lib.load()
    rows, c = z.shape
    n = rows * c
    bz = torch.empty(n + offset, device="cuda")
    by = torch.empty(n + offset, device="cuda")
    bz[offset:] = torch.from_numpy(z.reshape(-1)).cuda()
    by[offset:] = torch.from_numpy(y.reshape(-1)).cuda()
    zt, yt = bz[offset:].view(rows, c), by[offset:].view(rows, c)
    probs = torch.empty(n + offset, device="cuda")[offset:].view(rows, c)
    dl = torch.empty(n + offset, device="cuda")[offset:].view(rows, c)
    la = torch.empty(2, device="cuda")
    need = lib.gcs_regression_loss_workspace_bytes(rows, c)
    ws = torch.empty(max(need, 1), dtype=torch.uint8, device="cuda")
    gs = 1.0 / rows if grad_scale is None else grad_scale
    _lib.check(lib.gcs_regression_loss(KIND[kind], delta, zt.data_ptr(), yt.data_ptr(), rows, c, probs.data_ptr(),
                                       la.data_ptr(), dl.data_ptr(), gs, ws.data_ptr(), need, _lib.stream_ptr()))
    return probs, la, dl


def _check_kernel(kind, z, y, probs, la, dl, delta=1.0, grad_scale=None):
    rows, c = z.shape
    e = z.astype(np.float64) - y.astype(np.float64)
    got = host(la)
    loss = O1.regression_loss(kind, z.astype(np.float64), y.astype(np.float64), delta)
    assert abs(got[0] - loss) <= 1e-6 * max(1.0, abs(loss)), (got[0], loss)
    assert abs(got[1] - O1.mae(z, y.astype(np.float64))) <= 1e-6 * max(1.0, abs(got[1]))
    assert np.array_equal(host(probs), z)
    gs = 1.0 / rows if grad_scale is None else grad_scale
    ref = O1.element_grad(kind, e, delta) * gs / c
    assert rel_err(host(dl), ref) < 1e-5
    ties = e == 0
    if kind != "mse":
        assert (host(dl)[ties] == 0).all()                                   # sign(0) = 0, Huber's e = 0


@pytest.mark.parametrize("kind", list(KIND))
@pytest.mark.parametrize("rows,c", [(1, 1), (1000, 1), (1024, 1), (341, 3), (1025, 1), (508_428, 1), (508_428, 2),
                                    (508_428, 16)])
def test_regression_loss_against_float64(kind, rows, c):
    z, y = _reg_case(rows, c, seed=rows % 1000 + c + KIND[kind])
    delta = 0.8
    probs, la, dl = _run(kind, z, y, delta)
    _check_kernel(kind, z, y, probs, la, dl, delta)
    again = _run(kind, z, y, delta)                                           # reruns bit-identical
    assert all(torch.equal(a, b) for a, b in zip(again, (probs, la, dl)))
    odd = _run(kind, z, y, delta, offset=1)                                   # off the 16-byte grid: scalar accesses
    assert all(torch.equal(a, b) for a, b in zip(odd, (probs, la, dl)))
    # the Python wrapper: same sums and gradient, no prediction copy
    la2, dl2 = ops.regression_loss(torch.from_numpy(z).cuda(), torch.from_numpy(y).cuda(), kind, delta, want_grad=True)
    assert torch.equal(la2, la) and torch.equal(dl2, dl)


def test_huber_at_delta_ties_rows_zero_and_argument_errors():
    # |e| == delta exactly: 0.5 e^2 (both branches meet there), dz = e * scale
    z = np.array([[1.25, -0.25, 0.5, 3.0]], np.float32)
    y = np.array([[0.5, 0.5, 0.5, 0.5]], np.float32)
    probs, la, dl = _run("huber", z, y, delta=0.75, grad_scale=1.0)
    assert host(la).tolist() == [(0.28125 + 0.28125 + 0.0 + (0.75 * 2.5 - 0.28125)) / 4, (0.75 + 0.75 + 0.0 + 2.5) / 4]
    assert host(dl).tolist() == [[0.75 / 4, -0.75 / 4, 0.0, 0.75 / 4]]
    _, _, dl_mae = _run("mae", z, y, grad_scale=1.0)
    assert host(dl_mae).tolist() == [[0.25, -0.25, 0.0, 0.25]]
    lib = _lib.load()
    st = _lib.stream_ptr()
    zt, yt = torch.from_numpy(z).cuda(), torch.from_numpy(y).cuda()
    la0 = torch.full((2,), 7.0, device="cuda")
    assert lib.gcs_regression_loss(1, 1.0, zt.data_ptr(), yt.data_ptr(), 0, 4, None, la0.data_ptr(), None, 1.0, None, 0, st) == 0
    assert host(la0).tolist() == [0.0, 0.0]
    # without targets: the predictions are copied, nothing else
    out = torch.zeros_like(zt)
    assert lib.gcs_regression_loss(2, 1.0, zt.data_ptr(), None, 1, 4, out.data_ptr(), None, None, 1.0, None, 0, st) == 0
    assert torch.equal(out, zt)
    assert lib.gcs_regression_loss(2, 1.0, zt.data_ptr(), None, 1, 4, None, la0.data_ptr(), None, 1.0, None, 0, st) == 1
    big_z, big_y = (torch.zeros(5000, 3, device="cuda") for _ in range(2))
    need = lib.gcs_regression_loss_workspace_bytes(5000, 3)
    assert need > 0
    assert lib.gcs_regression_loss(1, 1.0, big_z.data_ptr(), big_y.data_ptr(), 5000, 3, None, la0.data_ptr(), None, 1.0,
                                   None, 0, st) == 3                          # GCS_ERR_WORKSPACE
    assert lib.gcs_regression_loss(3, -1.0, zt.data_ptr(), yt.data_ptr(), 1, 4, None, la0.data_ptr(), None, 1.0, None, 0,
                                   st) == 1
    with pytest.raises(ValueError):
        ops.regression_loss(zt, yt[:, :2])
    with pytest.raises(ValueError):
        ops.regression_loss(zt, yt, loss="hinge")
    torch.cuda.synchronize()


# ---------------------------------------------------------------- whole model against the float64 restatement
def _targets_off_the_kinks(z, delta, seed):
    """y = z -/+ m with m in [0.2, 0.5] or [0.9, 1.5]: every |e| stays at least 0.1 away from 0 and from delta = 0.7 on
    both the GPU and the float64 side, so that MAE and Huber take the same branch everywhere."""
    rng = np.random.default_rng(seed)
    mag = np.where(rng.random(z.shape) < 0.5, rng.uniform(0.2, 0.5, z.shape), rng.uniform(0.9, 1.5, z.shape))
    return (z - np.where(rng.random(z.shape) < 0.5, -1.0, 1.0) * mag).astype(np.float32)


def _node_permuted(args, seed):
    """The same batch with its nodes in another order: parameter gradients are sums over nodes, so this changes only the
    order of the float32 sums of the CPU restatement."""
    cfg, specs, w, s, x, rows, cols, seg, y, n_graphs = args
    perm = np.random.default_rng(seed).permutation(x.shape[0])
    inv = np.empty_like(perm)
    inv[perm] = np.arange(perm.shape[0])
    return (cfg, specs, w, s, x[perm], inv[rows], inv[cols], None if seg is None else seg[perm],
            y[perm] if cfg.pool is None else y, n_graphs)


def _parity(cfg, w, s, inputs, kind, args, n_nodes, n_graphs, delta=0.7, tol=TOL):
    model = make_model(cfg, w, s)
    z0, _ = O1.forward(*args[:8], args[9], training=True)
    y = _targets_off_the_kinks(z0, delta, seed=n_nodes)
    args = args[:8] + (y,) + args[9:]
    yt = torch.from_numpy(y).cuda()
    loss_fn = LOSS[kind](delta)
    loss_acc, probs = model.train_step_grads(inputs, yt, loss=loss_fn)
    branches = gpu_prelu_branches(model, cfg, n_nodes, n_graphs)
    ref = O1.loss_and_grads(*args, loss=kind, delta=delta, prelu_branch=branches)
    o2 = O2.loss_and_grads(*args, loss=kind, delta=delta)["grads"]
    o2p = O2.loss_and_grads(*_node_permuted(args, seed=1), loss=kind, delta=delta)["grads"]
    got = host(loss_acc)
    assert probs.shape == y.shape
    assert abs(got[0] - ref["loss"]) < tol * abs(ref["loss"])
    assert abs(got[1] - ref["metric"]) < tol * abs(ref["metric"])
    assert rel_err(host(probs), ref["logits"]) < tol
    assert rel_err(host(model.state), ref["new_state"]) < tol
    # every tensor to 1e-5 (pool.attn_kernel 2e-5, as for the other heads), or 5x the error of the float32 CPU
    # restatement, the larger of its errors in two node orders.  The gradients of the PReLU slopes, of the attention
    # kernel and of the last post kernel are sums over all rows with cancellation, whose float32 error depends on the
    # order of the sum: the GPU's order is a third sample of it, and it came to 4.0x and 4.1x of that larger error in
    # two of these cases
    e_gpu = grad_errors(host(model.grads), ref["grads"], cfg)
    e_a, e_b = grad_errors(o2, ref["grads"], cfg), grad_errors(o2p, ref["grads"], cfg)
    e_o2 = {k: max(e_a[k], e_b[k]) for k in e_a}
    bad = {k: (v, e_o2[k]) for k, v in e_gpu.items()
           if v > max(tol * (2.0 if k == "pool.attn_kernel" else 1.0), 5 * e_o2[k])}
    assert not bad, f"gradient tensors out of tolerance (gpu err, fp32-cpu err): {bad}"
    g1, p1, la1 = model.grads.clone(), probs.clone(), loss_acc.clone()
    model.load_flat(w, s)
    la2, p2 = model.train_step_grads(inputs, yt, loss=loss_fn)
    assert torch.equal(g1, model.grads) and torch.equal(p1, p2) and torch.equal(la1, la2)
    return model


@pytest.mark.parametrize("kind", list(KIND))
@pytest.mark.parametrize("pool", ["sum", "avg", "attn_sum", None])
@pytest.mark.parametrize("connectivity", ["cat", "sum", None])
def test_train_step_matches_float64(small_case, kind, pool, connectivity):
    c = small_case
    cfg = GNNConfig(in_features=12, output=2, activation=None, hidden=16, message_passing=3,
                    connectivity=connectivity, pool=pool)
    w, s = g.init_params(cfg, seed=81, perturb=True)
    (x, a, i), _ = next(g.DisjointLoader(c["ds"], batch_size=8, epochs=1, shuffle=False))
    args = (cfg, block_specs(cfg), w, s, c["x"], c["idx"][:, 0], c["idx"][:, 1], c["seg"], None, 8)
    _parity(cfg, w, s, (x, a, i), kind, args, c["x"].shape[0], 8)


@pytest.mark.parametrize("kind,pool", [("mse", "sum"), ("huber", None)])
def test_default_architecture_train_step(kind, pool):
    """Hidden 256, 4 GeneralConv layers, F = 32 on 8 E. coli-shaped graphs (the tensor-core GEMMs), C = 1."""
    ds = synthetic.make_dataset(8, seed=0, n_mean=500, deg=12, n_feat=32)
    (xr, (idx, _, _), seg), _ = batching_ref.collate([ds.graph(k) for k in range(8)])
    cfg = GNNConfig(in_features=32, output=1, activation=None, pool=pool)
    w, s = g.init_params(cfg, seed=4, perturb=True)
    args = (cfg, block_specs(cfg), w, s, xr, idx[:, 0], idx[:, 1], seg, None, 8)
    (x, a, i), _ = next(g.DisjointLoader(ds, batch_size=8, epochs=1, shuffle=False))
    _parity(cfg, w, s, (x, a, i), kind, args, xr.shape[0], 8)


def test_default_loss_of_the_linear_head_is_mse(small_case):
    (x, a, i), _ = next(g.DisjointLoader(small_case["ds"], batch_size=8, epochs=1, shuffle=False))
    y = torch.randn(8, 2, device="cuda")
    models = []
    for _ in range(2):
        m = g.GeneralGNN(2, hidden=16, message_passing=2, seed=3)
        m.build(12)
        models.append(m)
    la0, p0 = models[0].train_step_grads((x, a, i), y)
    la1, p1 = models[1].train_step_grads((x, a, i), y, loss=g.MeanSquaredError())
    assert torch.equal(la0, la1) and torch.equal(p0, p1) and torch.equal(models[0].grads, models[1].grads)
    soft = g.GeneralGNN(2, activation="softmax", hidden=16, message_passing=2, seed=3)
    with pytest.raises(NotImplementedError):
        soft.train_step_grads((x, a, i), torch.eye(2, device="cuda")[[0, 1] * 4], loss=g.Huber())


@pytest.mark.parametrize("kind", list(KIND))
@pytest.mark.parametrize("pool", ["sum", None])
def test_gradient_tape_route_equals_fused_step(kind, pool):
    ds = synthetic.make_dataset(6, seed=11, n_mean=90, deg=10, n_feat=8, n_classes=3, task="regression",
                                node_level=pool is None)
    (x, a, i), y = next(g.DisjointLoader(ds, node_level=pool is None, batch_size=6, epochs=1, shuffle=False))
    models = []
    for _ in range(2):
        m = g.GeneralGNN(3, hidden=64, message_passing=2, seed=0, pool=pool)
        m.build(8)
        w, s = g.init_params(m.cfg, seed=5, perturb=True)
        m.load_flat(w, s)
        models.append(m)
    fused, taped = models
    loss_acc, probs = fused.train_step_grads((x, a, i), y, loss=LOSS[kind](0.6))
    with g.GradientTape() as tape:
        pred = taped((x, a, i), training=True)
        loss = LOSS[kind](0.6)(y, pred)
    tape.gradient(loss, taped.trainable_variables)
    assert torch.equal(probs, pred) and torch.equal(loss_acc[0], loss) and torch.equal(tape.loss_record["loss_acc"], loss_acc)
    assert torch.equal(fused.grads, taped.grads) and torch.equal(fused.state, taped.state)
    # the metrics on the same predictions
    assert float((g.mean_absolute_error(y, pred).mean() - loss_acc[1]).abs()) < 1e-6 * float(loss_acc[1])
    if kind == "mse":
        assert float((g.mean_squared_error(y, pred).mean() - loss).abs()) < 1e-6 * float(loss)


def test_data_parallel_trainer_in_one_process_equals_train_step_and_apply_flat():
    from gcn_string_b200.distributed import DataParallelTrainer
    ds = synthetic.make_dataset(12, seed=7, n_mean=100, deg=10, n_feat=16, n_classes=1, task="regression")
    (x, a, i), y = next(g.DisjointLoader(ds, batch_size=12, epochs=1, shuffle=False))
    models = []
    for _ in range(2):
        m = g.GeneralGNN(1, hidden=64, message_passing=2, seed=1)
        m.build(16)
        models.append(m)
    trainer = DataParallelTrainer(models[0], g.optimizers.SGD(learning_rate=0.05), loss=g.Huber(0.3))
    la0, p0 = trainer.train_step((x, a, i), y)
    la1, p1 = models[1].train_step_grads((x, a, i), y, loss=g.Huber(0.3))
    g.optimizers.SGD(learning_rate=0.05).apply_flat(models[1].params, models[1].grads)
    assert torch.equal(la0, la1) and torch.equal(p0, p1)
    assert torch.equal(models[0].params, models[1].params) and torch.equal(models[0].state, models[1].state)


@pytest.mark.parametrize("node_level", [False, True])
def test_training_loop_on_synthetic_regression_data_lowers_the_loss(node_level):
    ds = synthetic.make_dataset(96, seed=3, n_mean=120, deg=10, n_feat=16, n_classes=1, task="regression",
                                node_level=node_level)
    model = g.GeneralGNN(1, hidden=64, message_passing=2, seed=0, pool=None if node_level else "sum")
    model.build(16)
    loader = g.DisjointLoader(ds, node_level=node_level, batch_size=24, epochs=None, shuffle=False)
    opt = g.optimizers.Adam(learning_rate=1e-2)
    loss_fn = g.Huber(0.5)

    def step():
        (x, a, i), y = next(loader)
        la, _ = model.train_step_grads((x, a, i), y, loss=loss_fn)
        opt.apply_flat(model.params, model.grads)
        return la
    first = torch.stack([step() for _ in range(4)])                            # one epoch
    for _ in range(28):
        step()
    torch.cuda.synchronize()
    before = torch.cuda.memory_stats().get("num_device_alloc", 0)
    last = torch.stack([step() for _ in range(24)])[-4:]
    torch.cuda.synchronize()
    assert torch.cuda.memory_stats().get("num_device_alloc", 0) == before
    f, l_ = host(first).mean(axis=0), host(last).mean(axis=0)
    assert l_[0] < 0.8 * f[0] and l_[1] < f[1], (f, l_)


def test_evaluate_returns_batch_weighted_loss_and_mae(small_case):
    from gcn_string_b200.evaluate import evaluate
    rng = np.random.default_rng(4)
    parts = []
    for k in range(8):
        xk, ak, _ = small_case["ds"].graph(k)
        parts.append((xk, ak, rng.standard_normal(2).astype(np.float32)))
    graphs = [Graph(x=xk, a=ak, y=yk) for xk, ak, yk in parts]
    cfg = GNNConfig(in_features=12, output=2, activation=None, hidden=16, message_passing=3, pool="avg")
    specs = block_specs(cfg)
    w, s = g.init_params(cfg, seed=43, perturb=True)
    model = make_model(cfg, w, s)
    loader = g.DisjointLoader(graphs, batch_size=3, epochs=None, shuffle=False)
    (loss, mae), preds = evaluate(model, loader, loss_fn=g.Huber(0.5))
    (mse, mse_metric), _ = evaluate(model, loader, loss_fn=g.MeanSquaredError(), metric=g.mean_squared_error)
    losses, mses, maes, sizes, pred_ref = [], [], [], [], []
    for b0 in range(0, 8, 3):
        ids = list(range(b0, min(b0 + 3, 8)))
        (xr, (idx, _, _), seg), yr = batching_ref.collate([parts[k] for k in ids])
        z, _ = O1.forward(cfg, specs, w, s, xr, idx[:, 0], idx[:, 1], seg, len(ids), training=False)
        pred_ref.append(z)
        yr = yr.astype(np.float64)
        losses.append(O1.regression_loss("huber", z, yr, 0.5))
        mses.append(O1.regression_loss("mse", z, yr))
        maes.append(O1.mae(z, yr))
        sizes.append(len(ids))
    assert abs(loss - np.average(losses, weights=sizes)) < TOL * abs(np.average(losses, weights=sizes))
    assert abs(mae - np.average(maes, weights=sizes)) < TOL * np.average(maes, weights=sizes)
    assert abs(mse - np.average(mses, weights=sizes)) < TOL * np.average(mses, weights=sizes)
    assert abs(mse_metric - mse) < 1e-6 * mse
    assert rel_err(np.concatenate([host(p) for p in preds]), np.concatenate(pred_ref)) < TOL
