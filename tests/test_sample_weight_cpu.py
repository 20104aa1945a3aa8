"""Sample weights on the CPU: the Keras documentation values through the float64 reference and the losses' host
fallbacks, the float64 and float32-autograd restatements of the weighted train step against each other and against
finite differences for every head at graph and node level, the C ABI (exports, the gcs_batch tail, workspace sizing,
what the weighted entry point refuses), shape errors, and the weighted ROC curve."""
import os

import numpy as np
import pytest
import torch

import gcn_string_b200 as g
from gcn_string_b200 import losses, ops
from gcn_string_b200.evaluate import roc_curve
from gcn_string_b200.params import GNNConfig, block_specs
from oracle import model_ref_np as O1, model_ref_torch as O2

import sw_ref as S

from conftest import rel_err


def _lib():
    from gcn_string_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib, _lib.load()


def test_keras_documentation_values():
    y2 = np.array([[0.0, 1.0], [0.0, 0.0]])
    cases = [("mse", y2, [[1.0, 1.0], [1.0, 0.0]], [0.7, 0.3], 0.5, 0.25),
             ("mae", y2, [[1.0, 1.0], [1.0, 0.0]], [0.7, 0.3], 0.5, 0.25),
             ("huber", y2, [[0.6, 0.4], [0.4, 0.6]], [1.0, 0.0], 0.155, 0.09),
             ("sigmoid", y2, [[-18.6, 0.51], [2.94, -12.8]], [0.8, 0.2], 0.86546, 0.24364)]
    for head, y, z, w, plain, weighted in cases:
        assert O1.weighted_loss(head, z, y, np.ones(2))[0] == pytest.approx(plain, rel=1e-4), head
        assert O1.weighted_loss(head, z, y, w)[0] == pytest.approx(weighted, rel=1e-4), head
    # the host fallbacks of the losses, on probabilities of unknown origin
    y3 = torch.tensor([[0.0, 1.0, 0.0], [0.0, 0.0, 1.0]], dtype=torch.float64)
    p3 = torch.tensor([[0.05, 0.95, 0.0], [0.1, 0.8, 0.1]], dtype=torch.float64)
    assert float(losses.categorical_crossentropy_from_probs(y3, p3)) == pytest.approx(1.17694, rel=1e-5)
    for w in ([0.3, 0.7], [[0.3], [0.7]], torch.tensor([0.3, 0.7]), np.array([0.3, 0.7], np.float32)):
        assert float(losses.categorical_crossentropy_from_probs(y3, p3, w)) == pytest.approx(0.81360, rel=1e-5)
    p2 = torch.sigmoid(torch.tensor([[-18.6, 0.51], [2.94, -12.8]], dtype=torch.float64))
    yt = torch.tensor(y2)
    assert float(losses.binary_crossentropy_from_probs(yt, p2)) == pytest.approx(0.86546, rel=1e-4)
    assert float(losses.binary_crossentropy_from_probs(yt, p2, [0.8, 0.2])) == pytest.approx(0.24364, rel=1e-4)


def test_weighted_metric_is_the_weighted_mean_and_zero_without_weight():
    rng = np.random.default_rng(0)
    z, y = rng.standard_normal((6, 3)), (rng.random((6, 3)) > 0.5).astype(float)
    for head in O1.HEADS:
        _, m1, _ = O1.weighted_loss(head, z, y, np.ones(6))
        _, mw, d0 = O1.weighted_loss(head, z, y, np.zeros(6))
        assert mw == 0.0 and not d0.any()
        l, m, _ = O1.row_terms(head, z, y)
        assert m1 == pytest.approx(m.mean())


def _case(small_case, pool, head, c_out=3, seed=81):
    c = small_case
    cfg = GNNConfig(in_features=12, output=c_out, activation=O1.activation(head), hidden=16, message_passing=3, pool=pool)
    specs = block_specs(cfg)
    w, s = g.init_params(cfg, seed=seed, perturb=True)
    rows = c["x"].shape[0] if pool is None else 8
    rng = np.random.default_rng(seed)
    if head == "softmax":
        y = np.eye(c_out, dtype=np.float32)[rng.integers(0, c_out, rows)]
    elif head == "sigmoid":
        y = (rng.random((rows, c_out)) > 0.5).astype(np.float32)
    else:
        y = rng.standard_normal((rows, c_out)).astype(np.float32)
    # half the rows masked, the rest with fractional weights
    sw = np.where(rng.random(rows) < 0.5, 0.0, rng.uniform(0.25, 2.0, rows))
    args = (cfg, specs, w, s, c["x"], c["idx"][:, 0], c["idx"][:, 1], c["seg"], y, 8)
    return args, dict(loss=head, sample_weight=sw)


@pytest.mark.parametrize("head", O1.HEADS)
@pytest.mark.parametrize("pool", ["sum", None])
def test_float64_and_autograd_restatements_agree(small_case, head, pool):
    args, kw = _case(small_case, pool, head)
    r1 = O1.loss_and_grads(*args, **kw, delta=0.7)
    r2 = O2.loss_and_grads(*args, **kw, delta=0.7)
    assert abs(r1["loss"] - r2["loss"]) < 1e-5 * abs(r1["loss"])
    assert rel_err(r2["grads"], r1["grads"]) < 2e-5


@pytest.mark.parametrize("head", ["softmax", "sigmoid", "mse"])
@pytest.mark.parametrize("pool", ["avg", None])
def test_manual_backward_matches_finite_differences(small_case, head, pool):
    args, kw = _case(small_case, pool, head, seed=83)
    r = O1.loss_and_grads(*args, **kw)
    w = args[2]
    rng = np.random.default_rng(19)
    scale = np.abs(r["grads"]).max()
    for j in rng.integers(0, w.shape[0], 10):
        wp = w.astype(np.float64).copy()
        wm = wp.copy()
        wp[j] += 1e-6
        wm[j] -= 1e-6
        fd = (O1.loss_at(args[0], args[1], wp, *args[3:], **kw) - O1.loss_at(args[0], args[1], wm, *args[3:], **kw)) / 2e-6
        assert abs(fd - r["grads"][j]) < 2e-6 * scale + 1e-9, j


def test_abi_exports_batch_tail_and_workspace_sizing():
    _l, lib = _lib()
    for name in ("gcs_weighted_loss", "gcs_weighted_loss_workspace_bytes", "gcs_model_workspace_bytes_ex"):
        assert name in _l.PROTOTYPES and hasattr(lib, name)
    assert lib.gcs_version() == 100
    assert _l.Batch._fields_[-1][0] == "sample_weight" and _l.Batch._fields_[-2][0] == "values_t"
    assert _l.Batch().sample_weight is None                       # a zero-filled struct: unweighted
    up = lambda v: -(-v // 256) * 256                              # noqa: E731
    for act, head in ((None, 0), ("softmax", 1), ("sigmoid", 2)):
        for pool, n, b in (("sum", 5000, 16), ("sum", 100_000, 70_000), (None, 5000, 16), (None, 500_000, 1000)):
            c = _l.model_config(GNNConfig(in_features=32, output=2, activation=act, pool=pool))
            rows = b if pool else n
            for training in (0, 1):
                plain = lib.gcs_model_workspace_bytes(c, n, 60000, b, training)
                assert lib.gcs_model_workspace_bytes_ex(c, n, 60000, b, training, 0) == plain
                ex = lib.gcs_model_workspace_bytes_ex(c, n, 60000, b, training, _l.WORKSPACE_SAMPLE_WEIGHTS)
                unweighted = {0: lib.gcs_regression_loss_workspace_bytes, 1: lib.gcs_softmax_xent_workspace_bytes,
                              2: lib.gcs_sigmoid_bce_workspace_bytes}[head](rows, 2)
                weighted = max(lib.gcs_weighted_loss_workspace_bytes(head, rows, 2), unweighted)
                assert ex - plain == up(weighted) - up(unweighted)
                assert lib.gcs_model_workspace_bytes_ex(c, n, 60000, b, training, 2) == -1
            if rows > 65536 or (head != 1 and rows * 2 > 1024):
                assert lib.gcs_weighted_loss_workspace_bytes(head, rows, 2) > 0
    # 24 bytes per block of the grid
    blocks = min(-(-508_428 * 16 // 4 // 256), 6 * 148)
    assert lib.gcs_weighted_loss_workspace_bytes(2, 508_428, 16) == 24 * blocks
    assert lib.gcs_weighted_loss_workspace_bytes(1, 65536, 2) == 0
    assert lib.gcs_weighted_loss_workspace_bytes(3, 10, 2) == -1
    assert lib.gcs_weighted_loss_workspace_bytes(1, -1, 2) == -1


def test_weighted_entry_refuses_null_weights_negative_rows_and_small_workspace():
    _l, lib = _lib()
    fake = 256                                                       # never dereferenced: every call fails first
    st = None
    assert lib.gcs_weighted_loss(2, 0, 1.0, fake, fake, None, 10, 2, None, fake, fake, 0.1, None, 0, st) == 1
    assert lib.gcs_weighted_loss(2, 0, 1.0, fake, fake, fake, -1, 2, None, fake, fake, 0.1, None, 0, st) == 1
    assert lib.gcs_weighted_loss(1, 0, 1.0, fake, fake, fake, 10, 65, None, fake, fake, 0.1, None, 0, st) == 1
    assert lib.gcs_weighted_loss(0, 4, 1.0, fake, fake, fake, 10, 2, None, fake, fake, 0.1, None, 0, st) == 1
    assert lib.gcs_weighted_loss(0, 3, 0.0, fake, fake, fake, 10, 2, None, fake, fake, 0.1, None, 0, st) == 1
    for head in (0, 1, 2):
        rows = 100_000
        need = lib.gcs_weighted_loss_workspace_bytes(head, rows, 2)
        assert lib.gcs_weighted_loss(head, 1, 1.0, fake, fake, fake, rows, 2, None, fake, fake, 0.1, fake, need - 8,
                                     st) == 3
        assert b"workspace" in lib.gcs_last_error()


def test_sample_weight_shapes():
    ops.check_sample_weight_shape((5,), 5)
    ops.check_sample_weight_shape((5, 1), 5)
    for bad in ((4,), (5, 2), (1, 5), (5, 1, 1), ()):
        with pytest.raises(ValueError, match="sample_weight"):
            ops.check_sample_weight_shape(bad, 5)
    y = torch.tensor([[0.0, 1.0], [1.0, 0.0]])
    with pytest.raises(ValueError, match="sample_weight"):
        losses.binary_crossentropy_from_probs(y, torch.full((2, 2), 0.5), [1.0, 2.0, 3.0])
    with pytest.raises(ValueError, match="sample_weight"):
        losses.categorical_crossentropy_from_probs(y, torch.full((2, 2), 0.5), np.ones((2, 2)))


def test_weighted_roc_curve_matches_the_sklearn_formula():
    rng = np.random.default_rng(3)
    y = (rng.random(300) > 0.6).astype(float)
    s = np.round(rng.random(300), 2)                                  # ties
    sw = np.where(rng.random(300) < 0.3, 0.0, rng.uniform(0.1, 3.0, 300))
    fpr, tpr, thr = roc_curve(y, s, drop_intermediate=False, sample_weight=sw)
    rf, rt, rth = S.roc_curve(y, s, sw)
    np.testing.assert_allclose(fpr, rf, rtol=1e-12)
    np.testing.assert_allclose(tpr, rt, rtol=1e-12)
    np.testing.assert_array_equal(thr, rth)
    # unit weights: the unweighted curve; zero weights: those rows leave the curve
    for a, b in zip(roc_curve(y, s, sample_weight=np.ones(300)), roc_curve(y, s)):
        np.testing.assert_allclose(a, b, rtol=1e-12)
    keep = sw != 0
    for a, b in zip(roc_curve(y, s, sample_weight=keep.astype(float)), roc_curve(y[keep], s[keep])):
        np.testing.assert_allclose(a, b, rtol=1e-12)
    with pytest.raises(ValueError):
        roc_curve(y, s, sample_weight=np.ones(299))
