"""GeneralGNN(activation='sigmoid') with BinaryCrossentropy on the CPU: configuration and parameter layout, the C
configuration value, the float64 and float32 restatements against each other and against finite differences for every
pool and for node-level output, and hand-computed Keras cases of the loss and the metric."""
import os

import numpy as np
import pytest

import gcn_string_b200 as g
from gcn_string_b200.params import FINAL_ACT, GNNConfig, block_specs, n_state, n_trainable, named_slices

import bce_ref as R

from conftest import rel_err

POOLS = ["sum", "avg", "attn_sum", None]


def test_validate_accepts_sigmoid_and_the_layout_equals_the_softmax_models():
    for pool in POOLS:
        for connectivity in ("cat", "sum", None):
            kw = dict(in_features=7, output=5, hidden=12, message_passing=3, connectivity=connectivity, pool=pool)
            sig, soft = GNNConfig(activation="sigmoid", **kw), GNNConfig(activation="softmax", **kw)
            sig.validate()
            assert block_specs(sig) == block_specs(soft) and named_slices(sig) == named_slices(soft)
            assert n_trainable(sig) == n_trainable(soft) and n_state(sig) == n_state(soft)
            w0, s0 = g.init_params(soft, seed=3, perturb=True)
            w1, s1 = g.init_params(sig, seed=3, perturb=True)
            assert np.array_equal(w0, w1) and np.array_equal(s0, s1)
    # no class cap on the sigmoid head
    GNNConfig(in_features=4, output=300, activation="sigmoid").validate()
    with pytest.raises(NotImplementedError, match="sigmoid"):
        GNNConfig(in_features=4, output=2, activation="tanh").validate()


def test_library_maps_sigmoid_to_2_and_agrees_on_the_layout():
    from gcn_string_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = _lib.load()
    assert FINAL_ACT["sigmoid"] == 2
    for name in ("gcs_sigmoid_bce_workspace_bytes", "gcs_sigmoid_bce"):
        assert hasattr(lib, name) and name in _lib.PROTOTYPES
    for pool in POOLS:
        cfg = GNNConfig(in_features=32, output=130, activation="sigmoid", pool=pool)
        c = _lib.model_config(cfg)
        assert c.final_activation == 2
        assert lib.gcs_model_num_params(c) == n_trainable(cfg) and lib.gcs_model_num_state(c) == n_state(cfg)
        assert lib.gcs_model_workspace_bytes(c, 1000, 12000, 4, 1) > lib.gcs_model_workspace_bytes(c, 1000, 12000, 4, 0) > 0
    # above 64 classes the softmax head is refused, the sigmoid head is not
    assert lib.gcs_model_num_params(_lib.model_config(GNNConfig(in_features=8, output=65, activation="softmax"))) == -1
    # the loss workspace: none for one block (rows * C <= 1024), per-block partials above
    assert lib.gcs_sigmoid_bce_workspace_bytes(0, 1) == 0
    assert lib.gcs_sigmoid_bce_workspace_bytes(1024, 1) == 0 and lib.gcs_sigmoid_bce_workspace_bytes(512, 2) == 0
    assert lib.gcs_sigmoid_bce_workspace_bytes(1025, 1) > 0
    assert lib.gcs_sigmoid_bce_workspace_bytes(508_428, 64) == lib.gcs_sigmoid_bce_workspace_bytes(2_100_000, 300)
    assert lib.gcs_sigmoid_bce_workspace_bytes(-1, 1) == -1 and lib.gcs_sigmoid_bce_workspace_bytes(1, 0) == -1
    # softmax plans keep their size; the sigmoid plan reserves the loss partials last
    for pool, n, b in (("sum", 5000, 16), (None, 5000, 16)):
        kw = dict(in_features=32, output=2, pool=pool)
        soft = lib.gcs_model_workspace_bytes(_lib.model_config(GNNConfig(activation="softmax", **kw)), n, 60000, b, 1)
        sig = lib.gcs_model_workspace_bytes(_lib.model_config(GNNConfig(activation="sigmoid", **kw)), n, 60000, b, 1)
        rows = b if pool else n
        assert sig - soft == -(-lib.gcs_sigmoid_bce_workspace_bytes(rows, 2) // 256) * 256


def _case(small_case, pool, connectivity, c_out=3, seed=51, soft=False):
    c = small_case
    cfg = GNNConfig(in_features=12, output=c_out, activation="sigmoid", hidden=16, message_passing=3,
                    connectivity=connectivity, pool=pool)
    specs = block_specs(cfg)
    w, s = g.init_params(cfg, seed=seed, perturb=True)
    rows = c["x"].shape[0] if pool is None else 8
    rng = np.random.default_rng(seed)
    y = (rng.random((rows, c_out)) < 0.4).astype(np.float32)                 # multi-hot
    y[1] = 0.0                                                               # a row without a positive
    if soft:
        y[::3] = rng.random((y[::3].shape[0], c_out)).astype(np.float32)     # soft labels
    args = (cfg, specs, w, s, c["x"], c["idx"][:, 0], c["idx"][:, 1], c["seg"], y, 8)
    return cfg, specs, w, s, args


@pytest.mark.parametrize("pool", POOLS)
@pytest.mark.parametrize("connectivity", ["cat", "sum", None])
def test_float64_and_autograd_restatements_agree(small_case, pool, connectivity):
    cfg, specs, w, s, args = _case(small_case, pool, connectivity, soft=True)
    r1, r2 = R.loss_and_grads(*args), R.torch_loss_and_grads(*args)
    assert r1["probs"].shape == args[8].shape
    assert abs(r1["loss"] - r2["loss"]) < 1e-5 * abs(r1["loss"])
    assert rel_err(r2["probs"], r1["probs"]) < 1e-5
    assert rel_err(r2["grads"], r1["grads"]) < 2e-5
    assert rel_err(r2["new_state"], r1["new_state"]) < 1e-5


@pytest.mark.parametrize("pool", POOLS)
def test_manual_backward_matches_finite_differences(small_case, pool):
    c = small_case
    cfg, specs, w, s, args = _case(small_case, pool, "cat", seed=53, soft=True)
    y = args[8].astype(np.float64)
    rows, cols = c["idx"][:, 0], c["idx"][:, 1]
    r = R.loss_and_grads(*args)

    def loss_at(wv):
        _, ctx = R.forward(cfg, specs, wv, s, c["x"], rows, cols, c["seg"], 8, training=True)
        return R.bce_from_logits(ctx["logits"], y)

    rng = np.random.default_rng(13)
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


def test_keras_cases_by_hand():
    # two rows, two columns: the mean over the columns, then over the rows
    z = np.array([[0.0, 2.0], [-1.0, 30.0]])
    y = np.array([[1.0, 0.0], [0.0, 1.0]])
    l00 = np.log(2.0)                                     # z = 0
    l01 = 2.0 + np.log1p(np.exp(-2.0))                    # y = 0: softplus(z)
    l10 = np.log1p(np.exp(-1.0))                          # y = 0, z < 0: softplus(-1)
    l11 = np.log1p(np.exp(-30.0))                         # y = 1: softplus(-z)
    assert abs(R.bce_from_logits(z, y) - ((l00 + l01) / 2 + (l10 + l11) / 2) / 2) < 1e-15
    # a row-wise mean differs from a flat mean only through ragged weights: a 1-row case pins the column mean
    assert abs(R.bce_from_logits(z[:1], y[:1]) - (l00 + l01) / 2) < 1e-15
    # Keras' fallback on probabilities: clip to [1e-7, 1 - 1e-7], then log(p + 1e-7) and log(1 - p + 1e-7)
    p = np.array([[1.0, 0.0, 0.25]])
    t = np.array([[1.0, 1.0, 0.5]])
    hi, lo = 1.0 - 1e-7, 1e-7
    ref = -np.mean([np.log(hi + 1e-7), np.log(lo + 1e-7), 0.5 * np.log(0.25 + 1e-7) + 0.5 * np.log(0.75 + 1e-7)])
    assert abs(R.bce_from_probs(p, t) - ref) < 1e-12
    # the sigmoid is stable for both signs, and the loss finite at |z| = 100
    assert R.sigmoid(np.array([-800.0]))[0] == 0.0 and R.sigmoid(np.array([800.0]))[0] == 1.0
    assert abs(R.bce_from_logits(np.array([[100.0, -100.0]]), np.array([[0.0, 1.0]])) - 100.0) < 1e-12
    # binary_accuracy: p == 0.5 predicts 0; soft labels never equal a 0/1 prediction
    assert R.binary_accuracy(np.array([[0.0, 1.0]]), np.array([[0.5, 0.5]], np.float32))[0] == 0.5
    assert R.binary_accuracy(np.array([[0.3, 1.0, 0.0]]), np.array([[0.2, 0.9, 0.1]], np.float32))[0] == pytest.approx(2 / 3)
    assert R.binary_accuracy(np.array([[1.0], [0.0]]), np.array([[0.51], [0.49]], np.float32)).tolist() == [1.0, 1.0]


def test_unsupported_loss_arguments_raise():
    with pytest.raises(NotImplementedError):
        g.BinaryCrossentropy(label_smoothing=0.1)
    with pytest.raises(NotImplementedError):
        g.BinaryCrossentropy(axis=0)
    with pytest.raises(NotImplementedError):
        g.BinaryCrossentropy(reduction="sum")
    loss = g.BinaryCrossentropy(from_logits=True, reduction="auto")
    assert loss.name == "binary_crossentropy" and loss.from_logits
    with pytest.raises(NotImplementedError):
        g.MLP(2, final_activation="tanh")
    g.MLP(2, final_activation="sigmoid")
    g.GeneralGNN(1, activation="sigmoid")                 # validated at construction: accepted
