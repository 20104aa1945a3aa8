"""SGD momentum / Nesterov, Adam amsgrad and Keras gradient clipping: the float64 restatements (optim_ref) against
torch.optim and hand cases, the constructor errors, the chunk tables and the exported symbols.  No GPU needed."""
import os
import re

import numpy as np
import pytest

import gcn_string_b200 as g
from gcn_string_b200 import _lib, optimizers

import optim_ref as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("nesterov", [False, True])
def test_momentum_matches_torch_sgd(nesterov):
    """At a constant learning rate Keras' accum = m*accum - lr*g and torch's buf = m*buf + g, w -= lr*buf give the
    same trajectory (torch's buffer is -accum/lr)."""
    import torch
    rng = np.random.default_rng(0)
    w0 = rng.normal(size=7)
    p = torch.tensor(w0, dtype=torch.float64, requires_grad=True)
    opt = torch.optim.SGD([p], lr=0.05, momentum=0.9, nesterov=nesterov)
    w, accum = w0.copy(), np.zeros(7)
    for _ in range(5):
        gr = rng.normal(size=7)
        p.grad = torch.tensor(gr, dtype=torch.float64)
        opt.step()
        w, accum = R.sgd(w, gr, accum, 0.05, 0.9, nesterov)
    assert np.allclose(w, p.detach().numpy(), rtol=1e-12, atol=1e-13)


def test_momentum_zero_is_plain_sgd_whatever_nesterov():
    w, gr = np.array([1.0, -2.0]), np.array([0.5, 0.25])
    for nesterov in (False, True):
        got, _ = R.sgd(w, gr, None, 0.1, 0.0, nesterov)
        assert np.array_equal(got, w - 0.1 * gr)


def test_clip_hand_cases():
    # a zero gradient: norm 0 <= c, factor exactly 1, nothing changes
    out, f = R.clip([np.zeros(3), np.array([3.0, 4.0])], clipnorm=1.0)
    assert f[0] == 1.0 and np.array_equal(out[0], np.zeros(3))
    assert f[1] == pytest.approx(0.2) and np.allclose(out[1], [0.6, 0.8])
    # a norm exactly equal to c does not fire
    out, f = R.clip([np.array([3.0, 4.0])], clipnorm=5.0)
    assert f == [1.0] and np.array_equal(out[0], [3.0, 4.0])
    out, f = R.clip([np.array([3.0]), np.array([4.0])], global_clipnorm=5.0)
    assert f == [1.0, 1.0]
    # global norm: sqrt(3^2 + 4^2) = 5 > 2.5 -> factor 0.5 on both tensors
    out, f = R.clip([np.array([3.0]), np.array([4.0])], global_clipnorm=2.5)
    assert f == [0.5, 0.5] and np.allclose(np.concatenate(out), [1.5, 2.0])
    # clipvalue first, then the norm of the clamped values
    out, f = R.clip([np.array([10.0, -10.0, 0.5])], clipvalue=1.0, clipnorm=1.0)
    assert np.allclose(out[0], np.array([1.0, -1.0, 0.5]) / 1.5)
    # clipvalue keeps NaN
    assert np.isnan(R.clip_value(np.array([np.nan]), 1.0)[0])


def test_clip_inf_in_one_tensor():
    grads = [np.array([1.0, np.inf]), np.array([2.0, 3.0])]
    out, _ = R.clip(grads, global_clipnorm=1.0)
    assert all(np.isnan(t).all() for t in out)          # the global norm is not finite: everything NaN
    out, f = R.clip(grads, clipnorm=1.0)
    assert out[0][0] == 0.0 and np.isnan(out[0][1])     # c / inf = 0 for the finite entry, NaN for the inf one
    assert f[1] == pytest.approx(1.0 / np.sqrt(13.0)) and np.isfinite(out[1]).all()


def test_amsgrad_equals_adam_while_v_does_not_decrease():
    rng = np.random.default_rng(1)
    w = rng.normal(size=5)
    a = [w.copy(), np.zeros(5), np.zeros(5), None]
    b = [w.copy(), np.zeros(5), np.zeros(5), np.zeros(5)]
    mag, sign = rng.uniform(0.5, 1.5, 5), rng.choice([-1.0, 1.0], 5)
    for t in range(1, 6):
        gr = sign * mag * 2.0 ** t                      # |g| doubles every step: v increases every step
        v_before = b[2].copy()
        a = list(R.adam(a[0], gr, a[1], a[2], None, t, 1e-3))
        b = list(R.adam(b[0], gr, b[1], b[2], b[3], t, 1e-3, amsgrad=True))
        assert (b[2] >= v_before).all()
        assert np.array_equal(a[0], b[0]) and np.array_equal(b[3], b[2])
    # once v shrinks, vhat holds the maximum and the steps differ
    a2 = R.adam(a[0], np.zeros(5), a[1], a[2], None, 6, 1e-3)
    b2 = R.adam(b[0], np.zeros(5), b[1], b[2], b[3], 6, 1e-3, amsgrad=True)
    assert (b2[3] > b2[2]).all() and not np.array_equal(a2[0], b2[0])


def test_constructor_errors():
    with pytest.raises(ValueError, match="momentum"):
        optimizers.SGD(momentum=1.5)
    with pytest.raises(ValueError, match="momentum"):
        optimizers.SGD(momentum=-0.1)
    with pytest.raises(NotImplementedError):
        optimizers.SGD(momentum=lambda: 0.9)
    for cls in (optimizers.SGD, optimizers.Adam):
        with pytest.raises(ValueError, match="Cannot accept both `clipnorm` and `global_clipnorm`"):
            cls(clipnorm=1.0, global_clipnorm=1.0)
        for k in ("clipnorm", "clipvalue", "global_clipnorm"):
            with pytest.raises(ValueError, match=f"Expected {k} >= 0"):
                cls(**{k: -1.0})
        with pytest.raises(NotImplementedError, match="decay"):
            cls(decay=1e-4)
        with pytest.raises(TypeError):
            cls(bogus=1)
    # every option accepted, defaults unchanged
    s = optimizers.SGD(0.1, momentum=0.9, nesterov=True, clipvalue=0.5, clipnorm=1.0)
    assert (s.momentum, s.nesterov, s.clipvalue, s.clipnorm, s.global_clipnorm) == (0.9, True, 0.5, 1.0, None)
    a = optimizers.Adam(amsgrad=True, global_clipnorm=2.0)
    assert a.amsgrad and a.global_clipnorm == 2.0 and a.clipnorm is None
    d = optimizers.SGD()
    assert d.momentum == 0.0 and not d.nesterov and d.clipvalue is None and d.clipnorm is None


@pytest.mark.parametrize("kw", [dict(), dict(hidden=512), dict(pool="attn_sum"), dict(pool="avg", connectivity="sum"),
                                dict(hidden=16, message_passing=3, output=3, in_features=12), dict(pool=None)])
def test_chunk_tables(kw):
    cfg = g.GNNConfig(**{**dict(in_features=32, output=2, activation="softmax"), **kw})
    slices = [(off, int(np.prod(shape))) for _, shape, off, buf in g.named_slices(cfg) if buf == "trainable"]
    sizes = [n for _, n in slices]
    t = optimizers.chunk_table(sizes)
    assert t.dtype == np.int64 and t.shape[1] == 3
    assert t[0, 0] == 0 and t[-1, 1] == g.n_trainable(cfg)
    assert np.array_equal(t[1:, 0], t[:-1, 1])                         # no gaps, no overlaps
    assert (t[:, 1] > t[:, 0]).all() and (t[:, 1] - t[:, 0] <= optimizers.CHUNK).all()
    for b, e, k in t:                                                   # inside its own tensor, at the right offsets
        off, n = slices[k]
        assert off <= b and e <= off + n
    assert np.array_equal(np.unique(t[:, 2]), np.arange(len(sizes)))   # every tensor covered
    dev = optimizers.device_rows(t)
    for r, (b, e, lo, hi) in enumerate(dev):
        assert lo <= r < hi and (t[lo:hi, 2] == t[r, 2]).all()
        assert (lo == 0 or t[lo - 1, 2] != t[r, 2]) and (hi == len(t) or t[hi, 2] != t[r, 2])
    rel = optimizers.device_rows(t, relative=True)
    starts = np.cumsum([0] + sizes)[t[:, 2]]
    assert np.array_equal(rel[:, 0], t[:, 0] - starts) and np.array_equal(rel[:, 2:], dev[:, 2:])
    if not kw:                                                          # cfg3: at least two blocks per SM on 148 SMs
        assert g.n_trainable(cfg) == 1_064_454 and len(t) >= 2 * 148


def test_chunk_table_does_not_depend_on_position():
    """A tensor's chunks are cut from its own start, so the per-tensor path (any order) reduces the same pieces."""
    sizes = [5000, 3, 4097, 2048]
    a = optimizers.chunk_table(sizes)
    b = optimizers.chunk_table(sizes[::-1])
    for k, n in enumerate(sizes):
        ra = a[a[:, 2] == k][:, :2] - a[a[:, 2] == k][0, 0]
        rb = b[b[:, 2] == len(sizes) - 1 - k][:, :2] - b[b[:, 2] == len(sizes) - 1 - k][0, 0]
        assert np.array_equal(ra, rb)


def test_reference_clip_flat_matches_per_tensor():
    rng = np.random.default_rng(2)
    sizes = [6, 3, 9]
    flat = rng.normal(size=sum(sizes)) * 3
    out, f = R.clip_flat(flat, sizes, clipvalue=2.0, clipnorm=2.5)
    parts, f2 = R.clip(np.split(flat, np.cumsum(sizes)[:-1]), clipvalue=2.0, clipnorm=2.5)
    assert np.array_equal(out, np.concatenate(parts)) and f == f2


def test_new_symbols_are_exported():
    text = open(os.path.join(ROOT, "include", "gcnstring_b200.h")).read()
    for name in ("gcs_sgd_step_ex", "gcs_adam_step_ex", "gcs_grad_clip_partials"):
        assert name in _lib.PROTOTYPES and re.search(rf"\bint\s+{name}\s*\(", text)
    for name, val in (("GCS_CLIP_VALUE", 1), ("GCS_CLIP_NORM", 2), ("GCS_CLIP_GLOBAL_NORM", 4),
                      ("GCS_CLIP_PARTIALS_READY", 8)):
        assert re.search(rf"\b{name}\s*=\s*{val}\b", text)
    assert (_lib.CLIP_VALUE, _lib.CLIP_NORM, _lib.CLIP_GLOBAL_NORM, _lib.CLIP_PARTIALS_READY) == (1, 2, 4, 8)
    # gcs_grad_clip as the ctypes structure lays it out (LP64): the pointers at 16 and 24, 40 bytes in all
    import ctypes
    assert _lib.GradClip.chunks.offset == 16 and _lib.GradClip.partials.offset == 24
    assert ctypes.sizeof(_lib.GradClip) == 40
    so = _lib.LIB_PATH
    if os.path.exists(so):
        lib = ctypes.CDLL(so)
        for name in ("gcs_sgd_step_ex", "gcs_adam_step_ex", "gcs_grad_clip_partials"):
            assert hasattr(lib, name)
    assert g.optimizers.SGD is optimizers.SGD and hasattr(g.optimizers, "chunk_table")
