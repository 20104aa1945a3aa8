"""GeneralGNN(pool='avg' | 'attn_sum') on the CPU: configuration, parameter layout, and the two restatements of the
oracle (float64 hand-derived backward, float32 autograd) against each other and against finite differences."""
import os

import numpy as np
import pytest

import gcn_string_b200 as g
from gcn_string_b200.params import GNNConfig, block_specs, n_trainable, named_slices, pool_kernel_slice
from oracle import model_ref_np as O1, model_ref_torch as O2

from conftest import rel_err

POOLS = ["avg", "attn_sum"]


@pytest.mark.parametrize("pool", POOLS)
def test_validate_accepts_the_new_pools(pool):
    GNNConfig(in_features=4, output=2, pool=pool).validate()
    with pytest.raises(NotImplementedError):
        GNNConfig(in_features=4, output=2, pool="max").validate()
    with pytest.raises(NotImplementedError):
        GNNConfig(in_features=4, output=2, pool="attn").validate()


@pytest.mark.parametrize("connectivity", ["cat", "sum", None])
def test_attn_kernel_is_appended_and_blocks_keep_their_layout_and_values(connectivity):
    kw = dict(in_features=7, output=3, hidden=12, message_passing=3, connectivity=connectivity)
    ref = GNNConfig(pool="sum", **kw)
    for pool in POOLS:
        cfg = GNNConfig(pool=pool, **kw)
        assert block_specs(cfg) == block_specs(ref)
        names = named_slices(cfg)
        extra = cfg.cat_width if pool == "attn_sum" else 0
        assert n_trainable(cfg) == n_trainable(ref) + extra
        if pool == "attn_sum":
            name, shape, off, buf = names[-1]
            assert (name, shape, buf) == ("pool.attn_kernel", (cfg.cat_width, 1), "trainable")
            assert off + cfg.cat_width == n_trainable(cfg) and (off, cfg.cat_width) == pool_kernel_slice(cfg)
        else:
            assert names == named_slices(ref) and pool_kernel_slice(cfg) is None
        for perturb in (False, True):
            w0, s0 = g.init_params(ref, seed=5, perturb=perturb)
            w1, s1 = g.init_params(cfg, seed=5, perturb=perturb)
            assert np.array_equal(w1[:w0.shape[0]], w0) and np.array_equal(s1, s0)
            if pool == "attn_sum":
                lim = np.sqrt(6.0 / (cfg.cat_width + 1))
                k = w1[w0.shape[0]:]
                assert np.abs(k).max() <= lim and np.abs(k).max() > 0.3 * lim


def test_default_parameter_count_with_attention_pooling():
    # the default architecture at F = 32: 1 064 454 trainable floats + attn_kernel [1280, 1]
    cfg = GNNConfig(in_features=32, output=2, activation="softmax", pool="attn_sum")
    assert n_trainable(cfg) == 1_065_734
    assert n_trainable(GNNConfig(in_features=32, output=2, activation="softmax", pool="avg")) == 1_064_454


def test_library_layout_agrees_for_every_pool():
    from gcn_string_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = _lib.load()
    for pool in ("sum", "avg", "attn_sum", None):
        for connectivity in ("cat", "sum", None):
            cfg = GNNConfig(in_features=32, output=2, activation="softmax", pool=pool, connectivity=connectivity)
            c = _lib.model_config(cfg)
            assert lib.gcs_model_num_params(c) == n_trainable(cfg)
            assert lib.gcs_model_workspace_bytes(c, 1000, 12000, 4, 1) > 0
    assert lib.gcs_attn_pool_workspace_bytes(10_000, 4, 96) > 0


def _case(small_case, pool, connectivity, seed=31):
    c = small_case
    cfg = GNNConfig(in_features=12, output=2, activation="softmax", hidden=16, message_passing=3, connectivity=connectivity,
                    pool=pool)
    specs = block_specs(cfg)
    w, s = g.init_params(cfg, seed=seed, perturb=True)
    args = (cfg, specs, w, s, c["x"], c["idx"][:, 0], c["idx"][:, 1], c["seg"], c["y"], 8)
    return cfg, specs, w, s, args


@pytest.mark.parametrize("pool", POOLS)
@pytest.mark.parametrize("connectivity", ["cat", "sum", None])
def test_float64_and_autograd_restatements_agree(small_case, pool, connectivity):
    cfg, specs, w, s, args = _case(small_case, pool, connectivity)
    r1, r2 = O1.loss_and_grads(*args), O2.loss_and_grads(*args)
    assert abs(r1["loss"] - r2["loss"]) < 1e-5 * abs(r1["loss"])
    assert rel_err(r2["probs"], r1["probs"]) < 1e-5
    assert rel_err(r2["grads"], r1["grads"]) < 2e-5
    assert rel_err(r2["new_state"], r1["new_state"]) < 1e-5
    if pool == "attn_sum":
        o, n = pool_kernel_slice(cfg)
        assert rel_err(r2["grads"][o:o + n], r1["grads"][o:o + n]) < 2e-5 and np.abs(r1["grads"][o:o + n]).max() > 0


@pytest.mark.parametrize("pool,connectivity", [("avg", "cat"), ("attn_sum", "cat"), ("attn_sum", "sum"), ("attn_sum", None)])
def test_manual_backward_matches_finite_differences(small_case, pool, connectivity):
    c = small_case
    cfg, specs, w, s, args = _case(small_case, pool, connectivity, seed=33)
    rows, cols = c["idx"][:, 0], c["idx"][:, 1]
    r = O1.loss_and_grads(*args)

    def loss_at(wv):
        return O1.loss_at(cfg, specs, wv, s, c["x"], rows, cols, c["seg"], c["y"], 8)

    rng = np.random.default_rng(9)
    picks = list(rng.integers(0, w.shape[0], 8))
    pk = pool_kernel_slice(cfg)
    if pk:
        picks += list(pk[0] + rng.integers(0, pk[1], 6))
    scale = np.abs(r["grads"]).max()
    for j in picks:
        wp = w.astype(np.float64).copy()
        wm = wp.copy()
        wp[j] += 1e-6
        wm[j] -= 1e-6
        assert abs((loss_at(wp) - loss_at(wm)) / 2e-6 - r["grads"][j]) < 2e-6 * scale + 1e-9, j


def test_empty_graph_and_single_mode_semantics():
    rng = np.random.default_rng(2)
    x = rng.standard_normal((7, 5))
    a = rng.standard_normal(5)
    seg = np.array([0, 0, 0, 2, 2, 3, 3])          # graph 1 has no rows
    mean = O1.segment_mean(x, seg, 4)
    assert np.array_equal(mean[1], np.zeros(5)) and np.allclose(mean[0], x[:3].mean(0))
    out, ctx = O1.attn_sum_pool(x, a, seg, 4)
    assert np.array_equal(out[1], np.zeros(5))
    sc = x[3:5] @ a
    p = np.exp(sc - sc.max()) / np.exp(sc - sc.max()).sum()
    assert np.allclose(out[2], p @ x[3:5], rtol=1e-8, atol=1e-12)
    # the gradient of an empty graph's output reaches no row; da agrees with finite differences
    dout = rng.standard_normal((4, 5))
    dx, da = O1.attn_sum_pool_bwd(x, a, seg, dout, ctx)
    dout_no1 = dout.copy()
    dout_no1[1] = 0.0
    dx2, da2 = O1.attn_sum_pool_bwd(x, a, seg, dout_no1, ctx)
    assert np.array_equal(dx, dx2) and np.array_equal(da, da2)
    for j in range(5):
        ap, am = a.copy(), a.copy()
        ap[j] += 1e-6
        am[j] -= 1e-6
        fd = ((O1.attn_sum_pool(x, ap, seg, 4)[0] * dout).sum() - (O1.attn_sum_pool(x, am, seg, 4)[0] * dout).sum()) / 2e-6
        assert abs(fd - da[j]) < 1e-7
    # single mode (no batch index): one softmax over all nodes, output [1, W]
    one, _ = O1.attn_sum_pool(x, a, np.zeros(7, dtype=np.int64), 1)
    sc = x @ a
    p = np.exp(sc - sc.max()) / np.exp(sc - sc.max()).sum()
    assert one.shape == (1, 5) and np.allclose(one[0], p @ x, rtol=1e-8, atol=1e-12)
    assert np.allclose(O1.segment_mean(x, np.zeros(7, dtype=np.int64), 1)[0], x.mean(0))
