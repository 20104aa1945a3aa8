"""Bit-for-bit A/B of the loss entry points and the fused train step against another build of the library.

    GCS_LIB_PATH=gcn-string_b200/variants/libbase.so python scripts/loss_ab.py run OUT_DIR/base.npz
    python scripts/loss_ab.py run OUT_DIR/new.npz
    python scripts/loss_ab.py compare OUT_DIR/base.npz OUT_DIR/new.npz

`run` calls gcs_softmax_xent, gcs_softmax_xent_ws, gcs_sigmoid_bce and gcs_regression_loss (MSE, MAE, Huber) on seeded
inputs at rows x C in {0, 1x1, 1023x1, 1024x1, 1025x1, 5000x3, 65536x2, 65537x2, 508428 x {1, 2, 16, 64}} (the
softmax up to C = 64, the single-block gcs_softmax_xent up to 65 536 rows), with 16-byte aligned buffers and buffers
offset by one float, with and without loss_acc and dlogits, and without labels; then one fused train_step_grads
each for a node-level softmax, a graph-level sigmoid C = 3 and a graph-level linear Huber model.  Every output goes to
the .npz, the fp64 workspace partials too (loss_acc's float32 rounding can hide a change in them), arrays of more
than 2**20 elements as the SHA-256 of their bytes.  `compare` reports every array whose raw bits (uint32 views)
differ and exits 1 on any.
"""
from __future__ import annotations

import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = [(0, 1), (1, 1), (1023, 1), (1024, 1), (1025, 1), (5000, 3), (65536, 2), (65537, 2),
          (508_428, 1), (508_428, 2), (508_428, 16), (508_428, 64)]


def run(out_path):
    import torch
    import gcn_string_b200 as g
    from gcn_string_b200 import _lib, synthetic
    lib = _lib.load()
    st = _lib.stream_ptr()
    res = {}

    def keep(key, t):
        a = t.cpu().numpy()
        if a.size > 1 << 20:
            res[key + "_sha256"] = np.frombuffer(hashlib.sha256(a.tobytes()).digest(), dtype=np.uint32)
        else:
            res[key] = a

    def buf(n, off):                                    # n floats at a 16-byte aligned address, or one float past it
        return torch.zeros(n + 4, device="cuda")[off:off + n]

    def p(t):
        return t.data_ptr() if t is not None else None

    gen = torch.Generator(device="cuda").manual_seed(0)
    for rows, c in SHAPES:
        n = rows * c
        z_src = torch.randn(max(n, 1), device="cuda", generator=gen) * 3
        y_reg = torch.randn(max(n, 1), device="cuda", generator=gen)
        y_bin = (torch.rand(max(n, 1), device="cuda", generator=gen) > 0.5).float()
        y_hot = torch.nn.functional.one_hot(torch.randint(0, c, (max(rows, 1),), device="cuda", generator=gen),
                                            c).float().reshape(-1)
        gs = 1.0 / rows if rows else 0.0
        entries = [("bce", y_bin), ("mse", y_reg), ("mae", y_reg), ("huber", y_reg)]
        if c <= 64:
            entries.append(("xent_ws", y_hot))
            if rows <= 65536:
                entries.append(("xent", y_hot))
        for name, y_src in entries:
            for off in (0, 1):
                for want_loss, want_grad, labels in ((True, True, True), (True, False, True), (False, True, True),
                                                     (False, False, True), (False, False, False)):
                    z, y = buf(n, off), buf(n, off)
                    z.copy_(z_src[:n])
                    y.copy_(y_src[:n])
                    probs = buf(n, off).fill_(-7.0)
                    dl = buf(n, off).fill_(-7.0) if want_grad else None
                    la = torch.full((2,), -7.0, device="cuda") if want_loss else None
                    yp = p(y) if labels else None
                    if name == "xent":
                        ws_b = 0
                    elif name == "xent_ws":
                        ws_b = int(lib.gcs_softmax_xent_workspace_bytes(rows, c))
                    elif name == "bce":
                        ws_b = int(lib.gcs_sigmoid_bce_workspace_bytes(rows, c))
                    else:
                        ws_b = int(lib.gcs_regression_loss_workspace_bytes(rows, c))
                    ws = torch.empty(max(ws_b, 8), dtype=torch.uint8, device="cuda")
                    if name == "xent":
                        rc = lib.gcs_softmax_xent(p(z), yp, rows, c, p(probs), p(la), p(dl), gs, st)
                    elif name == "xent_ws":
                        rc = lib.gcs_softmax_xent_ws(p(z), yp, rows, c, p(probs), p(la), p(dl), gs, p(ws), ws_b, st)
                    elif name == "bce":
                        rc = lib.gcs_sigmoid_bce(p(z), yp, rows, c, p(probs), p(la), p(dl), gs, p(ws), ws_b, st)
                    else:
                        kind = {"mse": 1, "mae": 2, "huber": 3}[name]
                        rc = lib.gcs_regression_loss(kind, 0.7, p(z), yp, rows, c, p(probs), p(la), p(dl), gs, p(ws),
                                                     ws_b, st)
                    key = f"{name}_{rows}x{c}_off{off}_loss{int(want_loss)}_grad{int(want_grad)}_y{int(labels)}"
                    res[key + "_rc"] = np.array([rc], dtype=np.int32)
                    if rc != 0:
                        continue
                    torch.cuda.synchronize()
                    keep(key + "_probs", probs)
                    if dl is not None:
                        keep(key + "_dlogits", dl)
                    if la is not None:
                        keep(key + "_loss_acc", la)
                    if la is not None and ws_b > 0:           # the fp64 partials, which loss_acc's rounding can hide
                        keep(key + "_partials", ws[:ws_b])
        del z_src, y_reg, y_bin, y_hot

    # the fused train step: node-level softmax, graph-level sigmoid C = 3, graph-level linear Huber
    gl = synthetic.make_dataset_parallel(64, seed=1, n_mean=40, deg=6, n_feat=8)
    nl = synthetic.make_dataset_parallel(64, seed=1, n_mean=40, deg=6, n_feat=8, node_level=True)
    batches = {"graph": next(g.DisjointLoader(gl, batch_size=64, epochs=1, shuffle=False, symmetric=True)),
               "node": next(g.DisjointLoader(nl, batch_size=64, epochs=1, shuffle=False, node_level=True,
                                             symmetric=True))}
    for name, level, act, c, loss in (("node_softmax", "node", "softmax", 2, None),
                                      ("graph_sigmoid_c3", "graph", "sigmoid", 3, None),
                                      ("graph_linear_huber", "graph", None, 1, g.Huber(0.5))):
        (inputs, y2) = batches[level]
        gen = torch.Generator(device="cuda").manual_seed(2)
        rows = y2.shape[0]
        if act == "softmax":
            y = y2
        elif act == "sigmoid":
            y = (torch.rand(rows, c, device="cuda", generator=gen) > 0.5).float()
        else:
            y = torch.randn(rows, c, device="cuda", generator=gen)
        m = g.GeneralGNN(c, activation=act, hidden=32, message_passing=2, pool=None if level == "node" else "sum",
                         seed=3)
        m.build(8)
        la, probs = m.train_step_grads(inputs, y, loss=loss)
        torch.cuda.synchronize()
        keep(f"step_{name}_loss_acc", la)
        keep(f"step_{name}_probs", probs)
        keep(f"step_{name}_grads", m.grads)
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    np.savez(out_path, **res)
    print(f"{len(res)} arrays -> {out_path}")


def compare(a_path, b_path):
    a, b = np.load(a_path), np.load(b_path)
    bad = 0
    keys = sorted(set(a.files) | set(b.files))
    for k in keys:
        if k not in a.files or k not in b.files:
            print("missing in one side:", k)
            bad += 1
            continue
        x, y = a[k], b[k]
        if x.shape != y.shape or x.dtype != y.dtype:
            print("shape/dtype differs:", k, x.shape, y.shape)
            bad += 1
            continue
        nd = int((x.view(np.uint32) != y.view(np.uint32)).sum()) if x.size else 0
        if nd:
            print(f"{k}: {nd} of {x.size} elements differ")
            bad += 1
    print(f"{len(keys)} arrays compared, {bad} differ")
    return 1 if bad else 0


if __name__ == "__main__":
    if len(sys.argv) == 3 and sys.argv[1] == "run":
        run(sys.argv[2])
    elif len(sys.argv) == 4 and sys.argv[1] == "compare":
        sys.exit(compare(sys.argv[2], sys.argv[3]))
    else:
        sys.exit(__doc__)
