"""GeneralGNN(dropout=rate) on the CPU: the NumPy Philox4x32-10 against Random123's known answers, the threshold and
scale arithmetic, validation, the C configuration fields against the header, the host step counter, per-rank mask
keys, and the float64 restatement with dropout against finite differences."""
import math
import os
import re

import numpy as np
import pytest

import gcn_string_b200 as g
from gcn_string_b200.params import GNNConfig, block_specs, check_dropout_rate, dropout_seed

from oracle import model_ref_np as O1

import dropout_ref as D

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _words(*hexes):
    return tuple(np.uint32(int(h, 16)) for h in hexes)


@pytest.mark.parametrize("ctr,key,expect", [
    (("0", "0", "0", "0"), ("0", "0"), ("6627e8d5", "e169c58d", "bc57ac4c", "9b00dbd8")),
    (("ffffffff",) * 4, ("ffffffff",) * 2, ("408f276d", "41c83b0e", "a20bc7c6", "6d5451fd")),
    (("243f6a88", "85a308d3", "13198a2e", "03707344"), ("a4093822", "299f31d0"),
     ("d16cfe09", "94fdcceb", "5001e420", "24126ea1")),
])
def test_numpy_philox_matches_random123_known_answers(ctr, key, expect):
    got = D.philox4x32_10(tuple(np.array([int(c, 16)], dtype=np.uint64) for c in ctr), [int(k, 16) for k in key])
    assert tuple(int(v[0]) for v in got) == tuple(int(e) for e in _words(*expect))


def test_threshold_and_scale():
    assert D.threshold(0.0) == 0 and D.scale(0.0) == np.float32(1.0)
    assert D.threshold(0.5) == 2 ** 31 and D.scale(0.5) == np.float32(2.0)
    r = float(np.float32(0.1))
    assert D.threshold(0.1) == math.floor(r * 2 ** 32) and D.scale(0.1) == np.float32(1.0 / (1.0 - r))
    assert D.threshold(np.nextafter(np.float32(1.0), np.float32(0.0))) == 2 ** 32 - 2 ** 8
    tiny = 1e-10                                              # below 2^-32: nothing is dropped, and the scale is 1.0f
    assert D.threshold(tiny) == 0 and D.scale(tiny) == np.float32(1.0)
    assert D.keep_mask(1, 2, 3, 5, 7, tiny).all()


def test_mask_is_a_function_of_seed_step_block_row_col():
    m = D.keep_mask(7, 3, 2, 64, 37, 0.3)
    assert np.array_equal(m[10:20, 5:30], D.keep_mask(7, 3, 2, 20, 30, 0.3)[10:20, 5:30])   # no dependence on the shape
    for other in (D.keep_mask(8, 3, 2, 64, 37, 0.3), D.keep_mask(7, 4, 2, 64, 37, 0.3), D.keep_mask(7, 3, 1, 64, 37, 0.3)):
        assert not np.array_equal(m, other)
    frac = 1.0 - D.keep_mask(11, 0, 0, 2000, 64, 0.3).mean()
    assert abs(frac - 0.3) < 6 * math.sqrt(0.3 * 0.7 / (2000 * 64))


@pytest.mark.parametrize("rate", [-0.1, 1.0, 1.5, float("nan"), float("inf"), "0.5", True])
def test_bad_rates_raise_value_error(rate):
    with pytest.raises(ValueError):
        check_dropout_rate(rate)
    with pytest.raises(ValueError):
        g.GeneralGNN(2, activation="softmax", dropout=rate)
    with pytest.raises(ValueError):
        g.layers.GeneralConv(8, dropout=rate)
    with pytest.raises(ValueError):
        g.layers.MLP(2, dropout=rate)


@pytest.mark.parametrize("rate", [0.0, 1e-12, 0.3, 0.5, 0.999])
def test_valid_rates_no_longer_raise(rate):
    """GeneralGNN takes the rate; the layout description GNNConfig stays rate-free (its validate still refuses one)."""
    check_dropout_rate(rate)
    model = g.GeneralGNN(2, activation="softmax", dropout=rate)
    assert model.dropout == rate and "dropout" not in model.config
    g.layers.GeneralConv(8, dropout=rate)
    g.layers.MLP(2, dropout=rate)


def test_forward_only_layers_refuse_training_with_dropout():
    for layer in (g.layers.GeneralConv(8, dropout=0.2), g.layers.MLP(2, dropout=0.2)):
        with pytest.raises(NotImplementedError, match="GeneralGNN"):
            layer(None, training=True)


def _header_struct(text, name):
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), text, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    return re.findall(r"(int32_t|uint32_t|uint64_t|float)\s+(\w+);", body)


def test_dropout_struct_matches_the_header_and_the_model_config_is_unchanged():
    import ctypes
    from gcn_string_b200 import _lib
    text = open(os.path.join(ROOT, "include", "gcnstring_b200.h")).read()
    size = {"int32_t": 4, "uint32_t": 4, "uint64_t": 8, "float": 4}
    for name, struct in (("gcs_dropout", _lib.Dropout), ("gcs_model_config", _lib.ModelConfig)):
        fields = _header_struct(text, name)
        assert [n for _, n in fields] == [f[0] for f in struct._fields_], name
        for (t, n), (_, ct) in zip(fields, struct._fields_):
            assert ctypes.sizeof(ct) == size[t], (name, n)
    assert ctypes.sizeof(_lib.Dropout) == 24 and _lib.Dropout.seed.offset == 8 and _lib.Dropout.step.offset == 16
    assert ctypes.sizeof(_lib.ModelConfig) == 56                  # dropout is a per-call argument, not a config field
    d = _lib.Dropout(0.25, 0, (1 << 64) - 1, 7)
    assert (d.rate, d.seed, d.step) == (0.25, (1 << 64) - 1, 7)


def test_rank_seeds_are_distinct_and_rank_zero_is_the_single_device_stream():
    for seed in (0, 1, 12345, 2 ** 63 + 7):
        keys = [dropout_seed(seed, r) for r in range(64)]
        assert len(set(keys)) == 64 and all(0 <= k < 2 ** 64 for k in keys)
    assert dropout_seed(3) == dropout_seed(3, 0) != dropout_seed(4, 0)


class _Lib:
    """Stands in for the native library: records the dropout of every backward call."""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        def fn(*args):
            d = args[-1]
            self.calls.append((name, None if d is None else (d.rate, d.seed, d.step)))
            return 0
        return fn


def test_step_counter_advances_once_per_training_call(monkeypatch):
    """The host counter: each training-mode call gets its own gcs_dropout carrying the next step, inference draws none,
    and the tape's backward reuses its forward's."""
    from gcn_string_b200 import models
    from gcn_string_b200 import _lib
    fake = _Lib()
    model = g.GeneralGNN(2, activation="softmax", dropout=0.5, seed=9)
    model._c, model._seed, model.built = _lib.model_config(GNNConfig(in_features=4, output=2)), 9, True
    assert model.dropout_step == 0
    assert model._call_dropout(False) is None and model.dropout_step == 0
    d1, d2 = model._call_dropout(True), model._call_dropout(True)
    assert (d1.step, d2.step, model.dropout_step) == (0, 1, 2)
    assert d1.rate == d2.rate == 0.5 and d1.seed == d2.seed == dropout_seed(9, 0)
    model.dropout_rank = 3
    assert model._call_dropout(True).seed == dropout_seed(9, 3)
    monkeypatch.setattr(_lib, "load", lambda: fake)
    monkeypatch.setattr(models, "stream_ptr", lambda: 0)
    model.params = model.grads = None
    model._backward(dict(batch=None, ws=_Ws(), dropout=d1), None)
    assert fake.calls == [("gcs_model_backward_ex", (0.5, dropout_seed(9, 0), 0))]


class _Ws:
    def data_ptr(self):
        return 0

    def numel(self):
        return 0


@pytest.mark.parametrize("pool,connectivity,aggregate,loss", [
    ("sum", "cat", "sum", None), ("avg", "sum", "mean", None), ("attn_sum", None, "max", None), (None, "cat", "sum", "mse"),
    ("sum", "cat", "max", "huber")])
def test_float64_restatement_with_dropout_matches_finite_differences(pool, connectivity, aggregate, loss):
    rng = np.random.default_rng(4)
    n, F, B = 14, 3, 3
    seg = np.sort(rng.integers(0, B, n))
    seg[:B] = np.arange(B)
    seg.sort()
    pairs = [(i, i) for i in range(n)] + [(i, j) for i in range(n) for j in range(n) if i != j and seg[i] == seg[j]
                                          and rng.random() < 0.4]
    rows = np.array([p[0] for p in pairs])
    cols = np.array([p[1] for p in pairs])
    act = None if loss else "softmax"
    cfg = GNNConfig(in_features=F, output=2, activation=act, hidden=6, message_passing=2, pre_process=1, post_process=2,
                    connectivity=connectivity, pool=pool, aggregate=aggregate)
    specs = block_specs(cfg)
    w, s = g.init_params(cfg, seed=2, perturb=True)
    w = w.astype(np.float64)
    x = rng.standard_normal((n, F))
    r_out = n if pool is None else B
    y = np.eye(2)[rng.integers(0, 2, r_out)] if act else rng.standard_normal((r_out, 2))
    ew = rng.uniform(0.5, 1.5, rows.shape[0]) if aggregate == "mean" else None
    masks = D.model_masks(specs, cfg, n, r_out, 0.4, seed=5, step=1)
    args = (cfg, specs, w, s, x, rows, cols, seg, y, B)
    kw = dict(masks=masks, rate=0.4, loss=loss, delta=0.5, edge_weight=ew)
    ref = O1.loss_and_grads(*args, **kw)
    eps = 1e-6
    idx = rng.choice(w.shape[0], 60, replace=False)
    for k in idx:
        wp, wm = w.copy(), w.copy()
        wp[k] += eps
        wm[k] -= eps
        fd = (O1.loss_at(cfg, specs, wp, s, x, rows, cols, seg, y, B, **kw) -
              O1.loss_at(cfg, specs, wm, s, x, rows, cols, seg, y, B, **kw)) / (2 * eps)
        assert abs(fd - ref["grads"][k]) <= 1e-5 * max(1.0, abs(fd)), (k, fd, ref["grads"][k])
    # dropped elements are exactly zero after the activation, and kept ones are scaled by 1 / (1 - rate)
    z, ctx = O1.forward(cfg, specs, w, s, x, rows, cols, seg, B, training=True, edge_weight=ew, masks=masks, rate=0.4)
    c0 = ctx["caches"][0]
    assert not c0["zd"][~masks[0]].any()
    np.testing.assert_allclose(c0["zd"][masks[0]], c0["z"][masks[0]] * float(D.scale(0.4)))
