"""A/B of the reference models against the per-feature restatements they replaced.

    python scripts/oracle_ab.py [REV]

REV (default HEAD~1) is a revision that still has tests/{pool,node,bce,reg,sw,dropout}_ref.py.  Its reference modules
(those six and oracle/model_ref_{np,torch}.py) are loaded with `git show REV:path` into a temporary directory, and
every old entry point runs next to oracle.model_ref_np (O1) / oracle.model_ref_torch (O2) on the same inputs: the
graphs of the test suite's small_case for pool 'sum' / 'avg' / 'attn_sum' and a node-level batch of them for
pool=None, every connectivity and aggregation, the heads softmax, sigmoid, mse, mae and huber, with and without sample
weights, dropout masks (rate 0.4), edge weights, pinned PReLU branches and grad_scale, wherever the old module took
that option.  float64 results (loss, metric, probs, logits, dlogits, grads, new_state, inference output) must agree to
1e-12 (max-abs relative error); float32 autograd results, computed on one CPU thread, must be bit-identical.  Prints
every failure and exits 1 on any.
"""
from __future__ import annotations

import importlib.util
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

OLD_TESTS = ("pool_ref", "node_ref", "bce_ref", "reg_ref", "sw_ref", "dropout_ref")
TOL64 = 1e-12
FAILS = []
COUNT = dict(f64=0, f32=0)


def load_old(rev, tmp):
    """The revision's modules under their own names; its oracle package as oracle_old."""
    pkg = os.path.join(tmp, "oracle_old")
    os.makedirs(pkg)
    open(os.path.join(pkg, "__init__.py"), "w").close()
    for name in ("model_ref_np", "model_ref_torch"):
        src = subprocess.check_output(["git", "-C", ROOT, "show", f"{rev}:oracle/{name}.py"], text=True)
        open(os.path.join(pkg, name + ".py"), "w").write(src)
    for name in OLD_TESTS:
        src = subprocess.check_output(["git", "-C", ROOT, "show", f"{rev}:tests/{name}.py"], text=True)
        open(os.path.join(tmp, name + ".py"), "w").write(src.replace("from oracle import", "from oracle_old import"))
    sys.path.insert(0, tmp)
    import oracle_old.model_ref_np as o1
    import oracle_old.model_ref_torch as o2
    mods = {name: __import__(name) for name in OLD_TESTS}
    return o1, o2, mods


def _suite_rel_err():
    """rel_err of the test suite's conftest (max |got - ref| / max |ref|)."""
    spec = importlib.util.spec_from_file_location("suite_conftest", os.path.join(ROOT, "tests", "conftest.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.rel_err


rel_err = _suite_rel_err()


def check64(tag, old, new, keys):
    for ko, kn in keys:
        COUNT["f64"] += 1
        e = rel_err(new[kn], old[ko])
        if not e <= TOL64:
            FAILS.append(f"{tag}: {ko} -> {kn}: float64 relative error {e:.3e}")


def check32(tag, old, new, keys):
    for ko, kn in keys:
        COUNT["f32"] += 1
        a, b = np.asarray(old[ko]), np.asarray(new[kn])
        if a.shape != b.shape or a.dtype != b.dtype or a.tobytes() != b.tobytes():
            FAILS.append(f"{tag}: {ko} -> {kn}: float32 results differ (max |d| {np.abs(a - b).max():.3e})")


def batches():
    """(graph-level batch, node-level batch): the test suite's small_case graphs."""
    from gcn_string_b200 import synthetic
    from oracle import batching_ref
    out = []
    for node_level in (False, True):
        ds = synthetic.make_dataset(8, seed=3, n_mean=60, deg=8, n_feat=12, node_level=node_level)
        (x, (idx, _, _), seg), _ = batching_ref.collate([ds.graph(i) for i in range(ds.n_graphs)])
        out.append((x, idx[:, 0], idx[:, 1], seg))
    return out


def labels(head, rows, c, rng):
    if head == "softmax":
        y = np.eye(c)[rng.integers(0, c, rows)]
        y[::5] = rng.random((y[::5].shape[0], c))                           # soft rows, sum != 1
        return y.astype(np.float32)
    if head == "sigmoid":
        return (rng.random((rows, c)) < 0.4).astype(np.float32)
    return rng.standard_normal((rows, c)).astype(np.float32)


def branches(O1, cfg, specs, w, s, x, rows, cols, seg, B, rng):
    """The float64 sides of PReLU's kink with 2 % of the elements moved to another side."""
    _, ctx = O1.forward(cfg, specs, w, s, x, rows, cols, seg, B, training=True)
    out = []
    for blk, c in zip(ctx["blocks"], ctx["caches"]):
        if blk.alpha is None:
            out.append(None)
            continue
        b = np.sign(c["z"]).astype(np.int8)
        flip = rng.random(b.shape) < 0.02
        b[flip] = rng.integers(-1, 2, int(flip.sum())).astype(np.int8)
        out.append(b)
    return out


def main(rev):
    import torch
    # the backward of a[cols] accumulates rows in a thread-dependent order: one thread makes float32 autograd
    # reproducible, so that a difference between old and new is a difference in the ops they run
    torch.set_num_threads(1)
    import gcn_string_b200 as g
    from gcn_string_b200.params import GNNConfig, block_specs
    from oracle import model_ref_np as O1, model_ref_torch as O2
    with tempfile.TemporaryDirectory() as tmp:
        o1, o2, M = load_old(rev, tmp)
        P, N, B, R, S, D = (M[k] for k in OLD_TESTS)
        graph, node = batches()
        n_cfg = 0
        for pool in ("sum", "avg", "attn_sum", None):
            x, rows, cols, seg = node if pool is None else graph
            n = x.shape[0]
            r_out = n if pool is None else 8
            for connectivity in ("cat", "sum", None):
                for agg in ("sum", "mean", "max"):
                    if agg == "max" and connectivity == "sum":
                        continue                                            # not a valid configuration
                    for head in O1.HEADS:
                        n_cfg += 1
                        rng = np.random.default_rng(n_cfg)
                        cfg = GNNConfig(in_features=12, output=3, activation=O1.activation(head), hidden=16,
                                        message_passing=2, connectivity=connectivity, pool=pool, aggregate=agg)
                        specs = block_specs(cfg)
                        w, s = g.init_params(cfg, seed=n_cfg, perturb=True)
                        y = labels(head, r_out, 3, rng)
                        sw = np.where(rng.random(r_out) < 0.3, 0.0, rng.uniform(0.25, 2.0, r_out))
                        ew = rng.uniform(0.5, 1.5, rows.shape[0])
                        gs = 1.0 / (3 * r_out)
                        br = branches(O1, cfg, specs, w, s, x, rows, cols, seg, 8, rng)
                        masks = D.model_masks(specs, cfg, n, r_out, 0.4, seed=5, step=n_cfg)
                        base = (cfg, specs, w, s, x, rows, cols, seg, y, 8)
                        reg = head in O1.LOSSES
                        tag = f"pool={pool} conn={connectivity} agg={agg} head={head}"
                        run_case(o1, o2, P, N, B, R, S, D, O1, O2, tag, base, head, reg, sw, ew, gs, br, masks)
    print(f"{n_cfg} configurations, {COUNT['f64']} float64 and {COUNT['f32']} float32 comparisons, "
          f"{len(FAILS)} failures")
    for f in FAILS:
        print("  ", f)
    return 1 if FAILS else 0


def run_case(o1, o2, P, N, B, R, S, D, O1, O2, tag, base, head, reg, sw, ew, gs, br, masks):
    cfg, specs, w, s, x, rows, cols, seg, y, nb = base
    pool = cfg.pool
    kw = dict(loss=head, delta=0.7) if reg else {}
    std = [("loss", "loss"), ("probs", "probs"), ("grads", "grads"), ("new_state", "new_state")]
    acc = std + [("acc", "metric")]
    # ---- the head's own float64 train step, and its inference forward
    for opts in ({}, dict(prelu_branch=br), dict(grad_scale=gs), dict(edge_weight=ew)):
        new = O1.loss_and_grads(*base, **kw, **opts)
        t = f"{tag} {sorted(opts)}"
        if head == "softmax" and pool == "sum" and "grad_scale" not in opts:
            old = o1.loss_and_grads(*base, **opts)
            check64("O1 " + t, old, new, acc)
            check64("O1 " + t, old["ctx"], new["ctx"], [("prelu_flips", "prelu_flips")])
        if "edge_weight" in opts:
            continue
        if head == "softmax" and pool in ("sum", "avg", "attn_sum") and "grad_scale" not in opts:
            check64("pool_ref " + t, P.loss_and_grads(*base, **opts), new, acc)
        if head == "softmax" and pool is None:
            check64("node_ref " + t, N.loss_and_grads(*base[:7], y, **opts), new, acc)
        if head == "sigmoid":
            check64("bce_ref " + t, B.loss_and_grads(*base, **opts), new, acc)
        if reg:
            check64("reg_ref " + t, R.loss_and_grads(*base, kind=head, delta=0.7, **opts), new,
                    std[:1] + std[2:] + [("mae", "metric"), ("pred", "logits"), ("pred", "probs")])
    new, _ = O1.forward(cfg, specs, w, s, x, rows, cols, seg, nb, training=False)
    old = {}
    if head == "softmax" and pool == "sum":
        old["O1"] = o1.forward(cfg, specs, w, s, x, rows, cols, seg, nb, training=False)[0]
    if head == "softmax" and pool is not None:
        old["pool_ref"] = P.forward(cfg, specs, w, s, x, rows, cols, seg, nb, training=False)[0]
    if head == "softmax" and pool is None:
        old["node_ref"] = N.forward(cfg, specs, w, s, x, rows, cols, training=False)[0]
    if head == "sigmoid":
        old["bce_ref"] = B.forward(cfg, specs, w, s, x, rows, cols, seg, nb, training=False)[0]
    if reg:
        old["reg_ref"] = R.forward(cfg, specs, w, s, x, rows, cols, seg, nb, training=False)[0]
    for k, v in old.items():
        check64(f"{k} forward {tag}", dict(out=v), dict(out=new), [("out", "out")])
    # ---- sample weights (sw_ref) and dropout (dropout_ref), every head
    for opts in ({}, dict(grad_scale=gs), dict(prelu_branch=br)):
        old = S.loss_and_grads(*base, sw, head, 0.7, **opts)
        new = O1.loss_and_grads(*base, loss=head, delta=0.7, sample_weight=sw, **opts)
        check64(f"sw_ref {tag} {sorted(opts)}", old, new,
                [("loss", "loss"), ("metric", "metric"), ("logits", "logits"), ("dlogits", "dlogits"), ("grads", "grads")])
    check64(f"sw_ref loss_at {tag}", dict(v=S.loss_at(*base, sw, head, 0.7)),
            dict(v=O1.loss_at(*base, loss=head, delta=0.7, sample_weight=sw)), [("v", "v")])
    loss = head if reg else None
    for opts in ({}, dict(sw=sw), dict(edge_weight=ew), dict(prelu_branch=br), dict(sw=sw, edge_weight=ew, prelu_branch=br)):
        old = D.loss_and_grads(*base, masks, 0.4, loss=loss, delta=0.7, **opts)
        nopts = {("sample_weight" if k == "sw" else k): v for k, v in opts.items()}
        new = O1.loss_and_grads(*base, masks=masks, rate=0.4, loss=loss, delta=0.7, **nopts)
        check64(f"dropout_ref {tag} {sorted(opts)}", old, new,
                [("loss", "loss"), ("metric", "metric"), ("logits", "logits"), ("grads", "grads"), ("new_state", "new_state")])
    check64(f"dropout_ref loss_at {tag}", dict(v=D.loss_at(*base, masks, 0.4, loss, sw, 0.7, ew)),
            dict(v=O1.loss_at(*base, masks=masks, rate=0.4, loss=loss, delta=0.7, sample_weight=sw, edge_weight=ew)),
            [("v", "v")])
    # ---- float32 autograd
    new = O2.loss_and_grads(*base, **kw)
    if head == "softmax" and pool == "sum":
        check32(f"O2 {tag}", o2.loss_and_grads(*base), new, std)
        check32(f"O2 prelu_branch {tag}", o2.loss_and_grads(*base, prelu_branch=br),
                O2.loss_and_grads(*base, prelu_branch=br), std)
    if head == "softmax" and pool is not None:
        check32(f"pool_ref torch {tag}", P.torch_loss_and_grads(*base), new, std)
    if head == "softmax" and pool is None:
        check32(f"node_ref torch {tag}", N.torch_loss_and_grads(*base[:7], y), new, std)
    if head == "sigmoid":
        check32(f"bce_ref torch {tag}", B.torch_loss_and_grads(*base), new, std)
    if reg:
        check32(f"reg_ref torch {tag}", R.torch_loss_and_grads(*base, kind=head, delta=0.7), new,
                [("loss", "loss"), ("pred", "logits"), ("grads", "grads"), ("new_state", "new_state")])
    check32(f"sw_ref torch {tag}", S.torch_loss_and_grads(*base, sw, head, 0.7),
            O2.loss_and_grads(*base, loss=head, delta=0.7, sample_weight=sw), [("loss", "loss"), ("grads", "grads")])
    import torch
    with torch.no_grad():
        old, _, _ = B.torch_logits(cfg, specs, w, s, x, rows, cols, seg, nb, False, requires_grad=False)
        new = O2.forward(cfg, O2.unpack(specs, w, s, requires_grad=False), *O2.tensors(x, rows, cols, seg), nb, False,
                         attn=O2.attn_leaf(cfg, specs, w, requires_grad=False))
    check32(f"torch_logits inference {tag}", dict(z=old.numpy()), dict(z=new.numpy()), [("z", "z")])


if __name__ == "__main__":
    sys.exit(main(sys.argv[1] if len(sys.argv) > 1 else "HEAD~1"))
