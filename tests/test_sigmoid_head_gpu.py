"""GPU tests of the sigmoid head: the fused sigmoid + binary cross-entropy kernel against float64 (rows across its grid
boundaries, any C, multi-hot / soft / all-zero labels, |z| up to 100, determinism, argument errors), the
GeneralGNN(activation='sigmoid') train step against the float64 restatement for every pool and node-level output, the
inference and GradientTape routes, evaluate() with multi-hot node labels, the layers and the data-parallel step."""
import os
import socket

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
ONE_BLOCK = 1024            # rows * C up to which the kernel runs one block (no workspace, one launch)
FULL_GRID = 888 * 1024      # rows * C from which the grid has its maximum block count


# ---------------------------------------------------------------- the kernel against float64
def _bce_case(rows, c, seed):
    rng = np.random.default_rng(seed)
    z = (3 * rng.standard_normal((rows, c))).astype(np.float32)
    flat = z.reshape(-1)
    k = min(flat.size, 64)
    flat[rng.choice(flat.size, k, replace=False)] = rng.choice([100.0, -100.0, 60.0, -60.0, 0.0, 1e-8, -1e-8], k)
    y = (rng.random((rows, c)) < 0.3).astype(np.float32)                    # multi-hot
    soft = rng.random(rows) < 0.1
    y[soft] = rng.random((int(soft.sum()), c)).astype(np.float32)          # soft labels
    y[rng.random(rows) < 0.05] = 0.0                                        # all-zero rows
    return z, y


def _check_kernel(z, y, probs, la, dl, grad_scale=None):
    rows, c = z.shape
    z64, y64 = z.astype(np.float64), y.astype(np.float64)
    p64 = O1.sigmoid(z64)
    loss = O1.bce_from_logits(z64, y64)
    got = host(la)
    assert np.isfinite(got).all()
    assert abs(got[0] - loss) <= 1e-6 * max(1.0, abs(loss)), (got[0], loss)
    p = host(probs)
    assert np.abs(p - p64).max() < 1e-6
    # the accuracy counts y == (p > 0.5) on the kernel's own float32 probabilities
    assert abs(got[1] - O1.binary_accuracy(y, p).mean()) <= 1e-6
    gs = 1.0 / rows if grad_scale is None else grad_scale
    assert rel_err(host(dl), (p64 - y64) * gs / c) < 1e-5


@pytest.mark.parametrize("rows,c", [(1, 1), (1, 300), (1000, 1), (1000, 7), (ONE_BLOCK, 1), (ONE_BLOCK + 1, 1), (341, 3),
                                    (342, 3), (FULL_GRID, 1), (FULL_GRID + 1, 1), (FULL_GRID // 64 + 1, 64),
                                    (508_428, 1), (508_428, 2), (508_428, 64), (3001, 300), (2_100_001, 2)])
def test_sigmoid_bce_against_float64(rows, c):
    z, y = _bce_case(rows, c, seed=rows % 1000 + c)
    zt, yt = torch.from_numpy(z).cuda(), torch.from_numpy(y).cuda()
    probs, la, dl = ops.sigmoid_bce(zt, yt, want_grad=True)
    _check_kernel(z, y, probs, la, dl)
    again = ops.sigmoid_bce(zt, yt, want_grad=True)                        # reruns bit-identical
    assert torch.equal(again[0], probs) and torch.equal(again[1], la) and torch.equal(again[2], dl)
    # the same values at addresses off the 16-byte grid (scalar loads): the same bits, sums included
    buf_z = torch.empty(rows * c + 1, device="cuda")
    buf_y = torch.empty(rows * c + 1, device="cuda")
    buf_z[1:] = zt.reshape(-1)
    buf_y[1:] = yt.reshape(-1)
    odd = ops.sigmoid_bce(buf_z[1:].view(rows, c), buf_y[1:].view(rows, c), want_grad=True)
    assert torch.equal(odd[0], probs) and torch.equal(odd[1], la) and torch.equal(odd[2], dl)
    # probabilities only
    p_only, la_none, dl_none = ops.sigmoid_bce(zt)
    assert la_none is None and dl_none is None and torch.equal(p_only, probs)


def test_sigmoid_bce_grad_scale_rows_zero_and_argument_errors():
    z, y = _bce_case(5000, 3, seed=9)
    zt, yt = torch.from_numpy(z).cuda(), torch.from_numpy(y).cuda()
    probs, la, dl = ops.sigmoid_bce(zt, yt, grad_scale=1.0 / 12345, want_grad=True)
    _check_kernel(z, y, probs, la, dl, grad_scale=1.0 / 12345)
    lib = _lib.load()
    st = _lib.stream_ptr()
    la0 = torch.full((2,), 7.0, device="cuda")
    assert lib.gcs_sigmoid_bce(zt.data_ptr(), yt.data_ptr(), 0, 3, None, la0.data_ptr(), None, 1.0, None, 0, st) == 0
    assert host(la0).tolist() == [0.0, 0.0]
    out = torch.empty_like(zt)
    need = lib.gcs_sigmoid_bce_workspace_bytes(5000, 3)
    assert need > 0
    assert lib.gcs_sigmoid_bce(zt.data_ptr(), yt.data_ptr(), 5000, 3, out.data_ptr(), la.data_ptr(), None, 1.0, None, 0,
                               st) == 3                                   # GCS_ERR_WORKSPACE
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    assert lib.gcs_sigmoid_bce(zt.data_ptr(), yt.data_ptr(), 5000, 3, out.data_ptr(), la.data_ptr(), None, 1.0,
                               ws.data_ptr(), need - 1, st) == 3
    assert lib.gcs_sigmoid_bce(zt.data_ptr(), None, 5000, 3, out.data_ptr(), la.data_ptr(), None, 1.0, ws.data_ptr(), need,
                               st) == 1                                   # loss without labels
    assert lib.gcs_sigmoid_bce(zt.data_ptr(), None, 5000, 3, out.data_ptr(), None, out.data_ptr(), 1.0, None, 0, st) == 1
    assert lib.gcs_sigmoid_bce(zt.data_ptr(), yt.data_ptr(), 5000, 0, out.data_ptr(), None, None, 1.0, None, 0, st) == 1
    assert lib.gcs_sigmoid_bce(None, None, 5, 3, out.data_ptr(), None, None, 1.0, None, 0, st) == 1
    with pytest.raises(ValueError):
        ops.sigmoid_bce(zt, yt[:, :2])
    torch.cuda.synchronize()


# ---------------------------------------------------------------- whole model against the float64 restatement
def _multi_hot(rows, c, seed):
    rng = np.random.default_rng(seed)
    y = (rng.random((rows, c)) < 0.4).astype(np.float32)
    y[::7] = 0.0
    return y


def _parity(cfg, w, s, inputs, y, args, n_nodes, n_graphs, tol=TOL, inference=True):
    model = make_model(cfg, w, s)
    yt = torch.from_numpy(y).cuda()
    loss_acc, probs = model.train_step_grads(inputs, yt)
    branches = gpu_prelu_branches(model, cfg, n_nodes, n_graphs)
    ref = O1.loss_and_grads(*args, prelu_branch=branches)
    o2 = O2.loss_and_grads(*args)["grads"]
    got = host(loss_acc)
    assert probs.shape == y.shape
    assert abs(got[0] - ref["loss"]) < tol * abs(ref["loss"])
    assert abs(got[1] - O1.binary_accuracy(y, host(probs)).mean()) < 1e-6
    assert abs(got[1] - ref["metric"]) <= 2.0 / y.size                       # at most a tie at p = 0.5 apart
    assert rel_err(host(probs), ref["probs"]) < tol
    assert rel_err(host(model.state), ref["new_state"]) < tol
    e_gpu = grad_errors(host(model.grads), ref["grads"], cfg)
    e_o2 = grad_errors(o2, ref["grads"], cfg)
    bad = {k: (v, e_o2[k]) for k, v in e_gpu.items()
           if v > max(tol * (2.0 if k == "pool.attn_kernel" else 1.0), 4 * e_o2[k])}
    assert not bad, f"gradient tensors out of tolerance (gpu err, fp32-cpu err): {bad}"
    g1, p1, la1 = model.grads.clone(), probs.clone(), loss_acc.clone()
    model.load_flat(w, s)
    la2, p2 = model.train_step_grads(inputs, yt)
    assert torch.equal(g1, model.grads) and torch.equal(p1, p2) and torch.equal(la1, la2)
    if inference:
        model.load_flat(w, s)
        p_inf, cache = O1.forward(*args[:8], args[9], training=False)
        out = model(list(inputs), training=False)
        assert out._gcs_activation == "sigmoid"
        z = host(out._gcs_logits).astype(np.float64)
        assert rel_err(z, cache["logits"]) < TOL
        assert np.abs(host(out) - O1.sigmoid(z)).max() < 1e-6             # the kernel's sigmoid of its own logits
        # On the moving statistics of perturbed parameters the logits reach |z| ~ 1 500 (C = 130), where the float32
        # rounding of a logit near 0 alone moves its probability by ~4e-5: the probabilities are held to 1e-5 or 4x the
        # error of the float32 CPU restatement, whose logits carry the same rounding
        with torch.no_grad():
            z32 = O2.forward(cfg, O2.unpack(args[1], w, s, requires_grad=False), *O2.tensors(*args[4:8]), args[9], False,
                             attn=O2.attn_leaf(cfg, args[1], w, requires_grad=False))
        e32 = rel_err(torch.sigmoid(z32).numpy(), p_inf)
        assert rel_err(host(out), p_inf) < max(TOL, 4 * e32), (rel_err(host(out), p_inf), e32)
    return model


@pytest.mark.parametrize("pool", ["sum", "avg", "attn_sum", None])
@pytest.mark.parametrize("connectivity", ["cat", "sum", None])
def test_train_step_and_inference_match_float64(small_case, pool, connectivity):
    c = small_case
    cfg = GNNConfig(in_features=12, output=3, activation="sigmoid", hidden=16, message_passing=3,
                    connectivity=connectivity, pool=pool)
    w, s = g.init_params(cfg, seed=61, perturb=True)
    n = c["x"].shape[0]
    y = _multi_hot(n if pool is None else 8, 3, seed=7)
    (x, a, i), _ = next(g.DisjointLoader(c["ds"], batch_size=8, epochs=1, shuffle=False))
    args = (cfg, block_specs(cfg), w, s, c["x"], c["idx"][:, 0], c["idx"][:, 1], c["seg"], y, 8)
    _parity(cfg, w, s, (x, a, i), y, args, n, 8)


@pytest.mark.parametrize("c_out", [1, 5])
def test_default_architecture_train_step(c_out):
    """Hidden 256, 4 GeneralConv layers, F = 32 on 8 E. coli-shaped graphs: one binary and one multi-label head."""
    ds = synthetic.make_dataset(8, seed=0, n_mean=500, deg=12, n_feat=32)
    (xr, (idx, _, _), seg), _ = batching_ref.collate([ds.graph(k) for k in range(8)])
    cfg = GNNConfig(in_features=32, output=c_out, activation="sigmoid")
    w, s = g.init_params(cfg, seed=4, perturb=True)
    y = _multi_hot(8, c_out, seed=c_out)
    args = (cfg, block_specs(cfg), w, s, xr, idx[:, 0], idx[:, 1], seg, y, 8)
    (x, a, i), _ = next(g.DisjointLoader(ds, batch_size=8, epochs=1, shuffle=False))
    _parity(cfg, w, s, (x, a, i), y, args, xr.shape[0], 8, inference=False)


def test_more_classes_than_the_softmax_cap(small_case):
    c = small_case
    cfg = GNNConfig(in_features=12, output=130, activation="sigmoid", hidden=32, message_passing=2, pool="sum")
    w, s = g.init_params(cfg, seed=62, perturb=True)
    y = _multi_hot(8, 130, seed=3)
    (x, a, i), _ = next(g.DisjointLoader(c["ds"], batch_size=8, epochs=1, shuffle=False))
    args = (cfg, block_specs(cfg), w, s, c["x"], c["idx"][:, 0], c["idx"][:, 1], c["seg"], y, 8)
    _parity(cfg, w, s, (x, a, i), y, args, c["x"].shape[0], 8)


def test_node_level_binary_head_on_a_large_batch():
    ds = synthetic.make_dataset(740, seed=2, n_mean=100, deg=8, n_feat=8, node_level=True)
    (xr, (idx, _, _), _), _ = batching_ref.collate([ds.graph(k) for k in range(740)])
    assert xr.shape[0] >= 72_000
    cfg = GNNConfig(in_features=8, output=1, activation="sigmoid", hidden=32, message_passing=2, pool=None)
    w, s = g.init_params(cfg, seed=6, perturb=True)
    y = _multi_hot(xr.shape[0], 1, seed=5)
    (x, a, i), _ = next(g.DisjointLoader(ds, node_level=True, batch_size=740, epochs=1, shuffle=False))
    args = (cfg, block_specs(cfg), w, s, xr, idx[:, 0], idx[:, 1], None, y, 740)
    _parity(cfg, w, s, (x, a, i), y, args, xr.shape[0], 740, inference=False)


@pytest.mark.parametrize("pool", ["sum", None])
def test_gradient_tape_route_equals_fused_step(pool):
    ds = synthetic.make_dataset(6, seed=11, n_mean=90, deg=10, n_feat=8)
    (x, a, i), _ = next(g.DisjointLoader(ds, batch_size=6, epochs=1, shuffle=False))
    rows = 6 if pool else int(x.shape[0])
    y = torch.from_numpy(_multi_hot(rows, 4, seed=2)).cuda()
    models = []
    for _ in range(2):
        m = g.GeneralGNN(4, activation="sigmoid", hidden=64, message_passing=2, seed=0, pool=pool)
        m.build(8)
        w, s = g.init_params(m.cfg, seed=5, perturb=True)
        m.load_flat(w, s)
        models.append(m)
    fused, taped = models
    loss_acc, probs = fused.train_step_grads((x, a, i), y)
    with g.GradientTape() as tape:
        pred = taped((x, a, i), training=True)
        loss = g.BinaryCrossentropy()(y, pred)
        on_logits = g.BinaryCrossentropy(from_logits=True)(y, pred._gcs_logits)
    tape.gradient(loss, taped.trainable_variables)
    assert torch.equal(probs, pred) and torch.equal(loss_acc[0], loss) and torch.equal(on_logits, loss)
    assert torch.equal(fused.grads, taped.grads) and torch.equal(fused.state, taped.state)
    # an output without sigmoid logits is taken as probabilities (Keras' clip + eps fallback)
    plain = pred.detach().clone()
    ref = O1.bce_from_probs(host(plain).astype(np.float64), host(y).astype(np.float64))
    assert abs(float(g.BinaryCrossentropy()(y, plain)) - ref) < 1e-5 * ref


def test_evaluate_with_multi_hot_node_labels(small_case):
    from gcn_string_b200.evaluate import evaluate, positive_scores
    rng = np.random.default_rng(4)
    parts = []                                                  # (x, a, y [n, 3] multi-hot) per graph
    for k in range(8):
        xk, ak, _ = small_case["ds"].graph(k)
        parts.append((xk, ak, (rng.random((xk.shape[0], 3)) < 0.35).astype(np.float32)))
    graphs = [Graph(x=xk, a=ak, y=yk) for xk, ak, yk in parts]
    # the loader carries multi-hot node labels unchanged
    (_, _, _), yb = next(g.DisjointLoader(graphs, node_level=True, batch_size=8, epochs=1, shuffle=False))
    assert np.array_equal(host(yb), np.vstack([p[2] for p in parts]))
    cfg = GNNConfig(in_features=12, output=3, activation="sigmoid", hidden=16, message_passing=3, pool=None)
    specs = block_specs(cfg)
    w, s = g.init_params(cfg, seed=43, perturb=True)
    model = make_model(cfg, w, s)
    loader = g.DisjointLoader(graphs, node_level=True, batch_size=3, epochs=None, shuffle=False)
    (loss, acc), preds = evaluate(model, loader)
    losses, accs, sizes, probs_ref = [], [], [], []
    for b0 in range(0, 8, 3):
        ids = list(range(b0, min(b0 + 3, 8)))
        (xr, (idx, _, _), _), yr = batching_ref.collate([parts[k] for k in ids])
        yr = yr.astype(np.float64)
        probs, cache = O1.forward(cfg, specs, w, s, xr, idx[:, 0], idx[:, 1], None, len(ids), training=False)
        probs_ref.append(probs)
        losses.append(O1.bce_from_logits(cache["logits"], yr))
        accs.append(O1.binary_accuracy(yr, probs.astype(np.float32)).mean())
        sizes.append(yr.shape[0])
    ref_loss = np.average(losses, weights=sizes)
    assert abs(loss - ref_loss) < TOL * abs(ref_loss)
    assert abs(acc - np.average(accs, weights=sizes)) < 1.5 / (3 * sum(sizes))   # at most one element at p = 0.5 apart
    assert rel_err(np.concatenate([host(p) for p in preds]), np.concatenate(probs_ref)) < TOL
    assert torch.equal(positive_scores(preds, column=0), torch.cat([p[:, 0] for p in preds]))


def test_layers_and_metric(small_case):
    xs = torch.from_numpy(small_case["x"].astype(np.float32)).cuda()
    out = g.MLP(5, hidden=16, final_activation="sigmoid")(xs)
    lin = g.MLP(5, hidden=16)(xs)
    assert torch.equal(out, ops.sigmoid_bce(lin)[0])
    assert float(out.min()) >= 0.0 and float(out.max()) <= 1.0
    y = torch.tensor([[1.0, 0.0, 0.3], [0.0, 0.0, 1.0]], device="cuda")
    p = torch.tensor([[0.5, 0.2, 0.9], [0.6, 0.4, 0.7]], device="cuda")
    assert host(g.binary_accuracy(y, p)).tolist() == pytest.approx([1 / 3, 2 / 3])


# ---------------------------------------------------------------- data parallel
def _dp_child(rank, world, port, queue):
    import torch.distributed as dist
    from gcn_string_b200.distributed import DataParallelTrainer
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
        torch.cuda.set_device(rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
        n_graphs = 12 * world + 1
        ds = synthetic.make_dataset(n_graphs, seed=11, n_mean=200, deg=10, n_feat=16, node_level=True)

        def model():
            m = g.GeneralGNN(2, activation="sigmoid", hidden=64, message_passing=2, seed=0, pool=None)
            m.build(16)
            return m

        m = model()
        w0 = m.params.clone()
        loader = g.DisjointLoader(ds, node_level=True, batch_size=n_graphs, epochs=1, shuffle=False, symmetric=True,
                                  rank=rank, world_size=world, balance="nnz")
        (x, a, i), y = next(loader)
        trainer = DataParallelTrainer(m, g.optimizers.SGD(learning_rate=0.02), native_comm=True, sync_bn=True)
        trainer.train_step((x, a, i), y)
        torch.cuda.synchronize()
        gathered = [torch.empty_like(m.params) for _ in range(world)]
        dist.all_gather(gathered, m.params)
        same = all(torch.equal(gathered[0], t) for t in gathered[1:])
        diff = None
        if rank == 0:
            u = model()
            (xu, au, iu), yu = next(g.DisjointLoader(ds, node_level=True, batch_size=n_graphs, epochs=1, shuffle=False,
                                                     symmetric=True))
            u.train_step_grads((xu, au, iu), yu)
            expect = w0 - 0.02 * u.grads
            diff = float((m.params - expect).abs().max() / (u.grads.abs().max() * 0.02))
        dist.barrier()
        dist.destroy_process_group()
        queue.put((rank, same, diff, None))
    except Exception as e:                                    # reported to the parent
        queue.put((rank, False, None, repr(e)))


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_data_parallel_sigmoid_step_equals_one_step_on_the_union():
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    world = 2
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    queue = ctx.Queue()
    procs = [ctx.Process(target=_dp_child, args=(r, world, port, queue)) for r in range(world)]
    try:
        for p in procs:
            p.start()
        results = sorted(queue.get(timeout=300) for _ in range(world))
    finally:
        for p in procs:
            p.join(timeout=60)
            if p.is_alive():
                p.terminate()
                p.join()
    assert all(r[3] is None for r in results), results
    assert all(r[1] for r in results)
    assert results[0][2] < 1e-5, results[0][2]
