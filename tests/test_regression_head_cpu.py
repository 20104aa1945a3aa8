"""GeneralGNN(activation=None) with MeanSquaredError, MeanAbsoluteError and Huber on the CPU: the parameter and
workspace layout and the C configuration fields, what the library refuses, the float64 and float32 restatements against
each other and against finite differences for every loss and pool, the Keras documentation values, unsupported
arguments, and the synthetic regression targets."""
import os

import numpy as np
import pytest

import gcn_string_b200 as g
from gcn_string_b200 import losses, synthetic
from gcn_string_b200.params import GNNConfig, block_specs, n_state, n_trainable, named_slices

from oracle import model_ref_np as O1, model_ref_torch as O2

from conftest import rel_err

POOLS = ["sum", "avg", "attn_sum", None]


def _lib():
    from gcn_string_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib, _lib.load()


def _with_loss(c, loss, delta=1.0):
    from gcn_string_b200 import _lib
    out = _lib.ModelConfig.from_buffer_copy(c)
    out.loss, out.huber_delta = loss, delta
    return out


def test_linear_layout_does_not_depend_on_the_loss():
    _l, lib = _lib()
    for pool in POOLS:
        for connectivity in ("cat", "sum", None):
            kw = dict(in_features=7, output=3, hidden=12, message_passing=3, connectivity=connectivity, pool=pool)
            lin, soft = GNNConfig(activation=None, **kw), GNNConfig(activation="softmax", **kw)
            assert block_specs(lin) == block_specs(soft) and named_slices(lin) == named_slices(soft)
            w0, s0 = g.init_params(soft, seed=3, perturb=True)
            w1, s1 = g.init_params(lin, seed=3, perturb=True)
            assert np.array_equal(w0, w1) and np.array_equal(s0, s1)
            c = _l.model_config(lin)
            assert (c.loss, c.huber_delta) == (0, 1.0)
            sizes = set()
            for loss, delta in ((0, 1.0), (1, 1.0), (2, 1.0), (3, 0.25), (3, 7.0)):
                cl = _with_loss(c, loss, delta)
                assert lib.gcs_model_num_params(cl) == n_trainable(lin) and lib.gcs_model_num_state(cl) == n_state(lin)
                sizes.add((lib.gcs_model_workspace_bytes(cl, 3000, 30000, 16, 1), lib.gcs_model_workspace_bytes(cl, 3000, 30000, 16, 0),
                           lib.gcs_model_logits_offset(cl, 3000, 16, 1), lib.gcs_model_logits_offset(cl, 3000, 16, 0)))
            assert len(sizes) == 1


def test_zero_filled_config_keeps_every_head_and_softmax_sigmoid_plans_keep_their_size():
    _l, lib = _lib()
    assert [f[0] for f in _l.ModelConfig._fields_[-3:]] == ["aggregate", "loss", "huber_delta"]
    for act in (None, "softmax", "sigmoid"):
        for pool, n, b in (("sum", 5000, 16), (None, 5000, 16), ("attn_sum", 70_000, 700)):
            c = _l.model_config(GNNConfig(in_features=32, output=2, activation=act, pool=pool))
            zero = _with_loss(c, 0, 0.0)                                   # what a zero-filled struct holds
            for training in (0, 1):
                assert lib.gcs_model_workspace_bytes(zero, n, 60000, b, training) == lib.gcs_model_workspace_bytes(c, n, 60000, b, training)
            assert lib.gcs_model_num_params(zero) == lib.gcs_model_num_params(c) > 0
    # the linear plan differs from the softmax plan in its last slot only: the regression partials
    for pool, n, b in (("sum", 5000, 16), ("sum", 100_000, 1024), (None, 5000, 16), (None, 500_000, 1000)):
        kw = dict(in_features=32, output=2, pool=pool)
        soft = _l.model_config(GNNConfig(activation="softmax", **kw))
        lin = _l.model_config(GNNConfig(activation=None, **kw))
        rows = b if pool else n
        for training in (0, 1):
            assert lib.gcs_model_logits_offset(lin, n, b, training) == lib.gcs_model_logits_offset(soft, n, b, training)
        up = lambda v: -(-v // 256) * 256                                  # noqa: E731
        d_soft = up(lib.gcs_softmax_xent_workspace_bytes(rows, 2))
        d_lin = up(lib.gcs_regression_loss_workspace_bytes(rows, 2))
        assert lib.gcs_model_workspace_bytes(lin, n, 60000, b, 1) - lib.gcs_model_workspace_bytes(soft, n, 60000, b, 1) == d_lin - d_soft


def test_library_refuses_regression_losses_on_other_heads_and_bad_deltas():
    _l, lib = _lib()
    for name in ("gcs_regression_loss_workspace_bytes", "gcs_regression_loss"):
        assert hasattr(lib, name) and name in _l.PROTOTYPES
    assert lib.gcs_version() == 100
    for act in ("softmax", "sigmoid"):
        c = _l.model_config(GNNConfig(in_features=8, output=2, activation=act))
        for loss in (1, 2, 3):
            assert lib.gcs_model_num_params(_with_loss(c, loss)) == -1
            assert lib.gcs_model_workspace_bytes(_with_loss(c, loss), 100, 1000, 4, 1) == -1
    lin = _l.model_config(GNNConfig(in_features=8, output=2))
    for delta in (0.0, -1.0, float("inf"), float("nan")):
        assert lib.gcs_model_num_params(_with_loss(lin, 3, delta)) == -1
    for loss in (-1, 4):
        assert lib.gcs_model_num_params(_with_loss(lin, loss)) == -1
    assert lib.gcs_model_num_params(_with_loss(lin, 1, -1.0)) > 0            # delta is read for Huber only
    assert lib.gcs_model_num_params(_with_loss(lin, 3, 1e-3)) > 0
    # the kernel refuses a bad kind or delta before touching a pointer
    assert lib.gcs_regression_loss(0, 1.0, None, None, 0, 1, None, None, None, 1.0, None, 0, None) == 1
    assert lib.gcs_regression_loss(4, 1.0, None, None, 0, 1, None, None, None, 1.0, None, 0, None) == 1
    assert lib.gcs_regression_loss(3, 0.0, None, None, 0, 1, None, None, None, 1.0, None, 0, None) == 1
    assert lib.gcs_regression_loss(3, float("nan"), None, None, 0, 1, None, None, None, 1.0, None, 0, None) == 1
    assert lib.gcs_regression_loss(1, 1.0, None, None, 5, 0, None, None, None, 1.0, None, 0, None) == 1


def test_regression_workspace_is_zero_for_one_block_and_partials_above():
    _l, lib = _lib()
    ws = lib.gcs_regression_loss_workspace_bytes
    assert ws(0, 1) == 0 and ws(1024, 1) == 0 and ws(512, 2) == 0 and ws(1, 1024) == 0
    assert ws(1025, 1) == 2 * 16 and ws(513, 2) == 2 * 16                   # two blocks: {loss, |e|} fp64 each
    assert ws(508_428, 64) == ws(2_100_000, 300) == 888 * 16                 # at most one wave of blocks
    assert ws(-1, 1) == -1 and ws(1, 0) == -1


def _case(small_case, pool, connectivity, c_out=2, seed=71):
    c = small_case
    cfg = GNNConfig(in_features=12, output=c_out, activation=None, hidden=16, message_passing=3,
                    connectivity=connectivity, pool=pool)
    specs = block_specs(cfg)
    w, s = g.init_params(cfg, seed=seed, perturb=True)
    rows = c["x"].shape[0] if pool is None else 8
    y = np.random.default_rng(seed).standard_normal((rows, c_out)).astype(np.float32)
    args = (cfg, specs, w, s, c["x"], c["idx"][:, 0], c["idx"][:, 1], c["seg"], y, 8)
    return cfg, specs, w, s, args


@pytest.mark.parametrize("kind", O1.LOSSES)
@pytest.mark.parametrize("pool", POOLS)
@pytest.mark.parametrize("connectivity", ["cat", "sum", None])
def test_float64_and_autograd_restatements_agree(small_case, kind, pool, connectivity):
    cfg, specs, w, s, args = _case(small_case, pool, connectivity)
    delta = 0.7
    r1 = O1.loss_and_grads(*args, loss=kind, delta=delta)
    r2 = O2.loss_and_grads(*args, loss=kind, delta=delta)
    assert r1["logits"].shape == args[8].shape
    assert abs(r1["loss"] - r2["loss"]) < 1e-5 * abs(r1["loss"])
    assert rel_err(r2["logits"], r1["logits"]) < 1e-5
    assert rel_err(r2["grads"], r1["grads"]) < 2e-5
    assert rel_err(r2["new_state"], r1["new_state"]) < 1e-5


@pytest.mark.parametrize("kind", O1.LOSSES)
@pytest.mark.parametrize("pool", POOLS)
def test_manual_backward_matches_finite_differences(small_case, kind, pool):
    c = small_case
    cfg, specs, w, s, args = _case(small_case, pool, "cat", seed=73)
    rows, cols = c["idx"][:, 0], c["idx"][:, 1]
    delta = 0.7
    # targets that keep every element away from the kinks (MAE at e = 0, Huber at |e| = delta), half of them on each
    # Huber branch, so that finite differences see one smooth piece
    z0, _ = O1.forward(cfg, specs, w, s, c["x"], rows, cols, c["seg"], 8, training=True)
    rng = np.random.default_rng(5)
    mag = np.where(rng.random(z0.shape) < 0.5, rng.uniform(0.2, 0.5, z0.shape), rng.uniform(0.9, 1.5, z0.shape))
    y = z0 - np.where(rng.random(z0.shape) < 0.5, -1.0, 1.0) * mag
    args = args[:8] + (y,) + args[9:]
    r = O1.loss_and_grads(*args, loss=kind, delta=delta)

    def loss_at(wv):
        return O1.loss_at(cfg, specs, wv, s, c["x"], rows, cols, c["seg"], y, 8, loss=kind, delta=delta)

    rng = np.random.default_rng(17)
    picks = list(rng.integers(0, w.shape[0], 10))
    if pool == "attn_sum":
        last = specs[-1]
        picks += list(last.offset + last.n_trainable + rng.integers(0, cfg.cat_width, 4))
    scale = np.abs(r["grads"]).max()
    for j in picks:
        wp = w.astype(np.float64).copy()
        wm = wp.copy()
        wp[j] += 1e-6
        wm[j] -= 1e-6
        assert abs((loss_at(wp) - loss_at(wm)) / 2e-6 - r["grads"][j]) < 2e-6 * scale + 1e-9, j


def test_keras_documentation_values():
    y_true = np.array([[0.0, 1.0], [0.0, 0.0]])
    y_pred = np.array([[1.0, 1.0], [1.0, 0.0]])
    assert O1.regression_loss("mse", y_pred, y_true) == pytest.approx(0.5, abs=1e-15)
    assert O1.regression_loss("mae", y_pred, y_true) == pytest.approx(0.5, abs=1e-15)
    assert O1.regression_loss("huber", np.array([[0.6, 0.4], [0.4, 0.6]]), y_true) == pytest.approx(0.155, abs=1e-12)
    # the branches: |e| == delta is quadratic, above it linear; sign(0) = 0
    e = np.array([-3.0, -1.0, 0.0, 0.5, 1.0, 2.0])
    assert O1.element_loss("huber", e).tolist() == [2.5, 0.5, 0.0, 0.125, 0.5, 1.5]
    assert O1.element_grad("huber", e).tolist() == [-1.0, -1.0, 0.0, 0.5, 1.0, 1.0]
    assert O1.element_grad("mae", e).tolist() == [-1.0, -1.0, 0.0, 1.0, 1.0, 1.0]
    # torch's huber_loss is Keras' form, value and gradient at |e| = delta included
    import torch
    z = torch.tensor([0.0, 2.0, 4.5], requires_grad=True)
    t = torch.tensor([1.5, 0.5, 0.0])
    loss = torch.nn.functional.huber_loss(z, t, delta=1.5, reduction="sum")
    loss.backward()
    ez = (z.detach() - t).numpy().astype(np.float64)
    assert float(loss.detach()) == pytest.approx(O1.element_loss("huber", ez, 1.5).sum())
    assert z.grad.numpy().tolist() == pytest.approx(O1.element_grad("huber", ez, 1.5).tolist())


def test_unsupported_arguments_raise():
    for cls in (g.MeanSquaredError, g.MeanAbsoluteError, g.Huber):
        with pytest.raises(NotImplementedError):
            cls(reduction="sum")
        with pytest.raises(NotImplementedError):
            cls(reduction="none")
        cls(reduction="auto")
    for delta in (0.0, -1.0, float("inf"), float("nan")):
        with pytest.raises(ValueError):
            g.Huber(delta=delta)
    assert g.MeanSquaredError().name == "mean_squared_error" and g.MeanAbsoluteError().name == "mean_absolute_error"
    h = g.Huber(delta=2.5)
    assert h.name == "huber_loss" and h.delta == 2.5
    # the fused step's config fields: for the call only, and only on a linear head
    assert losses.fused_loss_fields(None, None) == (0, 1.0)
    assert losses.fused_loss_fields(g.MeanSquaredError(), None) == (1, 1.0)
    assert losses.fused_loss_fields(g.MeanAbsoluteError(), "linear") == (2, 1.0)
    assert losses.fused_loss_fields(h, None) == (3, 2.5)
    for act in ("softmax", "sigmoid"):
        for loss in (g.MeanSquaredError(), g.MeanAbsoluteError(), g.Huber()):
            with pytest.raises(NotImplementedError):
                losses.fused_loss_fields(loss, act)
    with pytest.raises(NotImplementedError):
        losses.fused_loss_fields(g.CategoricalCrossentropy(), "softmax")
    with pytest.raises(ValueError):
        synthetic.make_dataset(2, n_mean=40, task="ranking")


def test_synthetic_regression_targets():
    kw = dict(seed=5, n_mean=80, deg=8, n_feat=16)
    a = synthetic.make_dataset(12, n_classes=2, task="regression", **kw)
    b = synthetic.make_dataset(12, n_classes=2, task="regression", **kw)
    plain = synthetic.make_dataset(12, n_classes=2, **kw)
    assert np.array_equal(a.y, b.y) and a.y.dtype == np.float32 and a.y.shape == (12, 2) and not a.node_level
    assert np.array_equal(a.x, plain.x) and np.array_equal(a.col, plain.col)    # the same graphs
    assert np.abs(a.y).max() < 1.0 and a.y.std() > 0.05
    nl = synthetic.make_dataset(12, n_classes=2, task="regression", node_level=True, **kw)
    assert nl.node_level and nl.y.shape == (int(nl.node_off[-1]), 2)
    # graph targets are the per-graph means of the node targets; both are tanh of the node_labels score
    for k in range(12):
        n0, n1 = nl.node_off[k], nl.node_off[k + 1]
        assert np.allclose(a.y[k], nl.y[n0:n1].astype(np.float64).mean(axis=0), atol=1e-6)
    score = synthetic.neighbour_scores(nl, 2, 5 + 0x5EED)
    assert np.array_equal(nl.y, np.tanh(score).astype(np.float32))
    cls = synthetic.make_dataset(12, n_classes=2, node_level=True, **kw)
    assert np.array_equal(cls.y.argmax(axis=1), score.argmax(axis=1))
    # node_labels as it was: one-hot at the argmax of the same projection
    y = synthetic.node_labels(nl, 3, 99)
    s3 = synthetic.neighbour_scores(nl, 3, 99)
    assert np.array_equal(y, np.eye(3, dtype=np.float32)[s3.argmax(axis=1)])
    # shards carry continuous labels unchanged
    import tempfile
    from gcn_string_b200 import shards
    with tempfile.TemporaryDirectory() as d:
        for ds in (a, nl):
            path = shards.write_shard(os.path.join(d, "node.gcs" if ds.node_level else "graph.gcs"), ds)
            back = shards.read_shard(path, mmap=False, verify=True)
            assert back.node_level == ds.node_level and np.array_equal(back.y, ds.y)
