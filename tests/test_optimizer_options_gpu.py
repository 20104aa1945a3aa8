"""GPU checks of SGD momentum / Nesterov, Adam amsgrad and Keras gradient clipping on the fused optimizer kernels:
parity with the float64 restatements (optim_ref) over the default model's real layout and chunk table, bit identity of
the option-free and never-firing forms, flat against per-tensor steps, non-finite gradients, and whole training loops
against the oracle."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

import gcn_string_b200 as g
from gcn_string_b200 import ops
from gcn_string_b200.params import named_slices
from oracle import model_ref_np as O1

import optim_ref as R
from conftest import rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-5


def host(t):
    return t.detach().cpu().numpy()


def flat_model(seed=0, **kw):
    """The default GeneralGNN (cfg3 layout, 1 064 454 parameters) built without data: its flat params / grads and
    trainable variables are what the optimizer sees in training."""
    m = g.GeneralGNN(2, activation="softmax", seed=seed, **kw)
    m.build(32)
    return m


def sizes_of(model):
    return [v.value.numel() for v in model.trainable_variables]


def draw_grads(sizes, seed):
    """Per-tensor magnitudes spread over four decades, so that some tensors exceed a clip threshold and others not."""
    rng = np.random.default_rng(seed)
    scale = np.repeat(10.0 ** rng.uniform(-3, 1, len(sizes)), sizes)
    return (rng.standard_normal(sum(sizes)) * scale).astype(np.float32)


OPTS = {
    "sgd": dict(cls="SGD", kw=dict(learning_rate=0.01)),
    "momentum": dict(cls="SGD", kw=dict(learning_rate=0.01, momentum=0.9)),
    "nesterov": dict(cls="SGD", kw=dict(learning_rate=0.01, momentum=0.9, nesterov=True)),
    "adam": dict(cls="Adam", kw=dict(learning_rate=1e-3)),
    "amsgrad": dict(cls="Adam", kw=dict(learning_rate=1e-3, amsgrad=True)),
}
CLIPS = ["none", "clipvalue", "clipnorm", "global_clipnorm", "clipvalue+clipnorm"]


def clip_kwargs(clip, g0, sizes, gs):
    """Thresholds from the first step's scaled gradient: clipvalue at the 99th percentile of |g|, clipnorm at the median
    tensor norm, global_clipnorm at half the global norm."""
    gsc = g0.astype(np.float64) * np.float64(np.float32(gs))
    kw = {}
    if "clipvalue" in clip:
        kw["clipvalue"] = float(np.float32(np.quantile(np.abs(gsc), 0.99)))
    base = R.clip_flat(gsc, sizes, clipvalue=kw.get("clipvalue"))[0] if kw else gsc
    norms = [np.linalg.norm(p) for p in np.split(base, np.cumsum(sizes)[:-1])]
    if "global_clipnorm" in clip:
        kw["global_clipnorm"] = float(np.float32(0.5 * np.sqrt(np.sum(np.square(norms)))))
    elif "clipnorm" in clip:
        kw["clipnorm"] = float(np.float32(np.median(norms)))
    return kw


@pytest.mark.parametrize("gs", [1.0, 0.37])
@pytest.mark.parametrize("clip", CLIPS)
@pytest.mark.parametrize("opt", list(OPTS))
def test_kernel_parity_with_reference(opt, clip, gs):
    model = flat_model()
    sizes = sizes_of(model)
    w0 = host(model.params).astype(np.float64)
    grads = [draw_grads(sizes, s) for s in range(3)]
    ckw = clip_kwargs(clip, grads[0], sizes, gs)
    spec = OPTS[opt]
    o = getattr(g.optimizers, spec["cls"])(**spec["kw"], **ckw)
    n = w0.size
    w, accum, m, v, vhat = w0.copy(), np.zeros(n), np.zeros(n), np.zeros(n), np.zeros(n)
    fired = []
    for t, gr in enumerate(grads, start=1):
        model.grads.copy_(torch.from_numpy(gr))
        o.apply_flat(model.params, model.grads, grad_scale=gs, variables=model.trainable_variables)
        gc, factors = R.clip_flat(gr.astype(np.float64) * np.float64(np.float32(gs)), sizes, **ckw)
        fired.append((factors, np.abs(gr * np.float32(gs)).max()))
        if spec["cls"] == "SGD":
            w, accum = R.sgd(w, gc, accum, 0.01, spec["kw"].get("momentum", 0.0), spec["kw"].get("nesterov", False))
        else:
            w, m, v, vhat = R.adam(w, gc, m, v, vhat, t, 1e-3, amsgrad=spec["kw"].get("amsgrad", False))
    torch.cuda.synchronize()
    assert rel_err(host(model.params), w) < 1e-6
    slots = o._slots.get("flat", ())
    if opt in ("momentum", "nesterov"):
        assert rel_err(host(slots[0]), accum) < 1e-6
    if spec["cls"] == "Adam":
        assert rel_err(host(slots[0]), m) < 1e-6 and rel_err(host(slots[1]), v) < 1e-6
        if opt == "amsgrad":
            assert rel_err(host(slots[2]), vhat) < 1e-6
    if opt == "sgd":
        assert not slots                                  # plain SGD has no slot
    # the clip fired where intended
    factors0, gmax0 = fired[0]
    if "clipvalue" in clip:
        assert ckw["clipvalue"] < gmax0
    if clip.endswith("clipnorm") and clip != "global_clipnorm":
        assert min(factors0) < 1.0 and max(factors0) == 1.0
    if clip == "global_clipnorm":
        assert factors0[0] < 1.0
    if clip == "none":
        assert all(f == 1.0 for f in factors0)


def _pair(fn_a, fn_b, seed=0):
    """Run two update sequences from the same start over the same 3 gradients; return both parameter vectors."""
    out = []
    for fn in (fn_a, fn_b):
        model = flat_model(seed=seed)
        for s in range(3):
            model.grads.copy_(torch.from_numpy(draw_grads(sizes_of(model), s)))
            fn(model)
        out.append(model.params.clone())
    return out


def test_option_free_ex_calls_equal_the_plain_entry_points():
    gs = 0.37
    model = flat_model()
    w = model.params
    gr = torch.from_numpy(draw_grads(sizes_of(model), 0)).cuda()
    ws = [w.clone() for _ in range(4)]
    ops.sgd_step(ws[0], gr, 0.01, gs)
    ops.sgd_step_ex(ws[1], gr, None, 0.01, 0.0, False, gs, None)
    acc = torch.zeros_like(w)
    ops.sgd_step_ex(ws[2], gr, acc, 0.01, 0.0, True, gs, None)          # momentum 0: plain SGD whatever nesterov says
    assert torch.equal(ws[0], ws[1]) and torch.equal(ws[0], ws[2]) and not acc.any()
    slots = [[torch.zeros_like(w) for _ in range(2)] for _ in range(2)]
    wa, wb = w.clone(), w.clone()
    for t in (1, 2):
        ops.adam_step(wa, gr, *slots[0], t, 1e-3, grad_scale=gs)
        ops.adam_step_ex(wb, gr, *slots[1], None, t, 1e-3, grad_scale=gs)
    assert torch.equal(wa, wb) and all(torch.equal(a, b) for a, b in zip(*slots))


@pytest.mark.parametrize("opt", ["momentum", "amsgrad"])
@pytest.mark.parametrize("clip", ["clipnorm", "global_clipnorm", "clipvalue"])
def test_clip_that_never_fires_is_bit_identical(opt, clip):
    spec = OPTS[opt]
    cls = getattr(g.optimizers, spec["cls"])
    big = {"clipnorm": 1e30, "global_clipnorm": 1e30, "clipvalue": 1e6}[clip]   # |g| < 1e3 for every draw
    oa, ob = cls(**spec["kw"]), cls(**spec["kw"], **{clip: big})
    a, b = _pair(lambda m: oa.apply_flat(m.params, m.grads, 0.37, variables=m.trainable_variables),
                 lambda m: ob.apply_flat(m.params, m.grads, 0.37, variables=m.trainable_variables))
    assert torch.equal(a, b)


def test_two_identical_runs_are_equal():
    mk = lambda: g.optimizers.SGD(0.01, momentum=0.9, global_clipnorm=1.0)         # noqa: E731
    oa, ob = mk(), mk()
    a, b = _pair(lambda m: oa.apply_flat(m.params, m.grads, variables=m.trainable_variables),
                 lambda m: ob.apply_flat(m.params, m.grads, variables=m.trainable_variables))
    assert torch.equal(a, b)
    oa, ob = g.optimizers.Adam(amsgrad=True, clipnorm=1.0), g.optimizers.Adam(amsgrad=True, clipnorm=1.0)
    a, b = _pair(lambda m: oa.apply_flat(m.params, m.grads, variables=m.trainable_variables),
                 lambda m: ob.apply_flat(m.params, m.grads, variables=m.trainable_variables))
    assert torch.equal(a, b)


@pytest.mark.parametrize("clip", ["clipnorm", "global_clipnorm"])
@pytest.mark.parametrize("opt", ["nesterov", "amsgrad"])
def test_flat_path_agrees_with_per_tensor_path(opt, clip):
    spec = OPTS[opt]
    cls = getattr(g.optimizers, spec["cls"])
    c = 1.0 if clip == "clipnorm" else 20.0
    oa, ob = cls(**spec["kw"], clipvalue=5.0, **{clip: c}), cls(**spec["kw"], clipvalue=5.0, **{clip: c})
    a, b = _pair(lambda m: oa.apply_gradients(zip([v.grad_view for v in m.trainable_variables], m.trainable_variables)),
                 lambda m: ob.apply_gradients(list(zip([v.grad_view for v in m.trainable_variables],
                                                       m.trainable_variables))[::-1]))
    assert "flat" in oa._slots and "flat" not in ob._slots           # one fused step against one step per tensor
    if clip == "clipnorm":
        assert torch.equal(a, b)
    else:                                                             # only the fp64 summation order differs
        assert rel_err(host(a), host(b)) < 1e-7


@pytest.mark.parametrize("opt", ["momentum", "amsgrad"])
def test_non_finite_gradient(opt):
    spec = OPTS[opt]
    cls = getattr(g.optimizers, spec["cls"])
    for clip in ("global_clipnorm", "clipnorm"):
        model = flat_model()
        w0 = host(model.params)
        gr = draw_grads(sizes_of(model), 0)
        names = [v.name for v in model.trainable_variables]
        k = names.index("gnn.1.kernel")
        off = int(np.sum(sizes_of(model)[:k]))
        gr[off + 5] = np.inf
        model.grads.copy_(torch.from_numpy(gr))
        cls(**spec["kw"], **{clip: 1.0}).apply_flat(model.params, model.grads, variables=model.trainable_variables)
        got = host(model.params)
        if clip == "global_clipnorm":
            assert np.isnan(got).all()
        else:
            n = sizes_of(model)[k]
            bad = got[off:off + n]
            assert np.isnan(bad[5])
            rest = np.concatenate([got[:off], got[off + n:]])
            assert np.isfinite(rest).all() and not np.array_equal(rest, np.concatenate([w0[:off], w0[off + n:]]))
            if opt == "momentum":      # factor c/inf = 0: the finite entries of the tensor do not move
                assert np.array_equal(np.delete(bad, 5), np.delete(w0[off:off + n], 5))


def test_apply_flat_clipnorm_needs_the_variables():
    model = flat_model()
    with pytest.raises(ValueError, match="variables"):
        g.optimizers.SGD(clipnorm=1.0).apply_flat(model.params, model.grads)
    with pytest.raises(ValueError, match="offset"):
        g.optimizers.SGD(clipnorm=1.0).apply_flat(model.params, model.grads,
                                                  variables=model.trainable_variables[::-1])
    g.optimizers.SGD(global_clipnorm=1.0).apply_flat(model.params, model.grads)     # whole-buffer norm: allowed


def test_clipped_step_uploads_nothing_after_the_first():
    """The chunk table and partials are built once per layout: later steps allocate no device memory."""
    model = flat_model()
    o = g.optimizers.SGD(0.01, momentum=0.9, global_clipnorm=1.0)
    for _ in range(2):
        o.apply_flat(model.params, model.grads, variables=model.trainable_variables)
    torch.cuda.synchronize()
    before = torch.cuda.memory_stats().get("allocation.all.allocated", 0)
    for _ in range(5):
        o.apply_flat(model.params, model.grads, variables=model.trainable_variables)
    torch.cuda.synchronize()
    assert torch.cuda.memory_stats().get("allocation.all.allocated", 0) == before
    assert len(o._clips) == 1


def _flat_sizes(cfg):
    return [int(np.prod(shape)) for _, shape, _, buf in named_slices(cfg) if buf == "trainable"]


def test_tape_loop_momentum_nesterov_global_clipnorm_matches_oracle(small_case):
    c = small_case
    cfg, specs = c["cfg"], c["specs"]
    model = g.GeneralGNN(cfg.output, activation=cfg.activation, hidden=cfg.hidden, message_passing=cfg.message_passing)
    model.build(cfg.in_features)
    model.load_flat(c["w"], c["s"])
    rows, cols = c["idx"][:, 0], c["idx"][:, 1]
    r0 = O1.loss_and_grads(cfg, specs, c["w"].astype(np.float64), c["s"].astype(np.float64), c["x"], rows, cols,
                           c["seg"], c["y"], 8)
    clipnorm = float(np.float32(0.5 * np.linalg.norm(r0["grads"])))
    sched = g.optimizers.schedules.PiecewiseConstantDecay([0, 1], [0.02, 0.002, 0.0002])
    optimizer = g.optimizers.SGD(learning_rate=sched, momentum=0.9, nesterov=True, global_clipnorm=clipnorm)
    loss_fn = g.CategoricalCrossentropy()
    sizes = _flat_sizes(cfg)
    w_ref, s_ref = c["w"].astype(np.float64), c["s"].astype(np.float64)
    accum = np.zeros_like(w_ref)
    step, fired = 0, []
    for inputs, target in g.DisjointLoader(c["ds"], batch_size=8, epochs=3, shuffle=False):
        with g.GradientTape() as tape:
            predictions = model(inputs, training=True)
            loss = loss_fn(target, predictions) + sum(model.losses)
        gradients = tape.gradient(loss, model.trainable_variables)
        optimizer.apply_gradients(zip(gradients, model.trainable_variables))
        r = O1.loss_and_grads(cfg, specs, w_ref, s_ref, c["x"], rows, cols, c["seg"], c["y"], 8)
        gc, f = R.clip_flat(r["grads"], sizes, global_clipnorm=clipnorm)
        fired.append(f[0])
        w_ref, accum = R.sgd(w_ref, gc, accum, O1.piecewise_constant(step, [0, 1], [0.02, 0.002, 0.0002]), 0.9, True)
        s_ref = r["new_state"]
        step += 1
    assert step == 3 and fired[0] < 1.0
    assert rel_err(host(model.params), w_ref) < TOL and rel_err(host(model.state), s_ref) < TOL


def test_amsgrad_clipnorm_training_matches_oracle(small_case):
    c = small_case
    cfg, specs = c["cfg"], c["specs"]
    model = g.GeneralGNN(cfg.output, activation=cfg.activation, hidden=cfg.hidden, message_passing=cfg.message_passing)
    model.build(cfg.in_features)
    model.load_flat(c["w"], c["s"])
    sizes = _flat_sizes(cfg)
    (x, a, i), y = next(g.DisjointLoader(c["ds"], batch_size=8, epochs=1, shuffle=False))
    w_ref, s_ref = c["w"].astype(np.float64), c["s"].astype(np.float64)
    rows, cols = c["idx"][:, 0], c["idx"][:, 1]
    r0 = O1.loss_and_grads(cfg, specs, w_ref, s_ref, c["x"], rows, cols, c["seg"], c["y"], 8)
    norms = [np.linalg.norm(p) for p in np.split(r0["grads"], np.cumsum(sizes)[:-1])]
    clipnorm = float(np.float32(np.median(norms)))
    opt = g.optimizers.Adam(learning_rate=1e-3, amsgrad=True, clipnorm=clipnorm)
    m, v, vhat = np.zeros_like(w_ref), np.zeros_like(w_ref), np.zeros_like(w_ref)
    fired = []
    for t in range(1, 4):
        model.train_step_grads([x, a, i], y)
        opt.apply_flat(model.params, model.grads, variables=model.trainable_variables)
        r = O1.loss_and_grads(cfg, specs, w_ref, s_ref, c["x"], rows, cols, c["seg"], c["y"], 8)
        gc, f = R.clip_flat(r["grads"], sizes, clipnorm=clipnorm)
        fired.append(f)
        w_ref, m, v, vhat = R.adam(w_ref, gc, m, v, vhat, t, 1e-3, amsgrad=True)
        s_ref = r["new_state"]
    assert min(fired[0]) < 1.0 and max(fired[0]) == 1.0
    assert rel_err(host(model.state), s_ref) < TOL
    # as test_adam_training_matches_oracle: Adam normalises each gradient by its own running magnitude, so the biases
    # in front of a BatchNorm (true gradient 0, rounding noise in any implementation) move by +-lr at random
    got = host(model.params)
    for name, shape, off, buf in named_slices(cfg):
        if buf == "trainable" and not name.endswith(".bias"):
            n = int(np.prod(shape))
            assert rel_err(got[off:off + n], w_ref[off:off + n]) < 5 * TOL, name


def test_data_parallel_trainer_with_clipped_momentum_equals_train_step_and_apply_gradients(small_case):
    from gcn_string_b200.distributed import DataParallelTrainer
    c = small_case
    cfg = c["cfg"]
    (x, a, i), y = next(g.DisjointLoader(c["ds"], batch_size=8, epochs=1, shuffle=False))
    models = []
    for _ in range(2):
        m = g.GeneralGNN(cfg.output, activation=cfg.activation, hidden=cfg.hidden, message_passing=cfg.message_passing)
        m.build(cfg.in_features)
        m.load_flat(c["w"], c["s"])
        models.append(m)
    mk = lambda: g.optimizers.SGD(0.05, momentum=0.9, clipvalue=0.5, global_clipnorm=0.1)     # noqa: E731
    trainer = DataParallelTrainer(models[0], mk())
    opt = mk()
    for _ in range(3):
        la0, p0 = trainer.train_step((x, a, i), y)
        la1, p1 = models[1].train_step_grads((x, a, i), y)
        opt.apply_gradients(zip([v.grad_view for v in models[1].trainable_variables], models[1].trainable_variables))
        assert torch.equal(la0, la1) and torch.equal(p0, p1)
    assert torch.equal(models[0].params, models[1].params) and torch.equal(models[0].state, models[1].state)
    assert torch.equal(trainer.optimizer._slots["flat"][0], opt._slots["flat"][0])
