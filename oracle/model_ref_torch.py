"""O2 — PyTorch-CPU float32 restatement of the reference's op sequence with autograd
(TEST INFRASTRUCTURE; independent gradient check and the timed CPU baseline).

It executes what TensorFlow executes for /root/reference/src/scripts/gcn.py:328-340, op
by op and unfused (SURVEY.md §3.1): host scipy collate per step -> Dense / BN moments /
PReLU -> materialised ``gather`` of [nnz, H] messages -> segment sum (``index_add_``) ->
``Concatenate`` copies -> ``segment_sum`` pool -> post-MLP -> softmax cross-entropy ->
reverse-mode backward -> SGD apply.  It is a restatement ("port"), NOT TensorFlow; parity
is unpinned (oracle/__init__.py).  ``forward`` / ``loss_and_grads`` also take the other pools
('avg', 'attn_sum', None) and heads (sigmoid with binary_cross_entropy_with_logits; a linear
head with mse_loss, l1_loss or huber_loss) and sample weights, as model_ref_np does.
"""
from __future__ import annotations

import time

import numpy as np
import torch

from . import model_ref_np as O1


def unpack(specs, w, s, requires_grad=True):
    """Flat numpy buffers -> list of per-block dicts of leaf tensors (float32)."""
    out = []
    for sp_ in specs:
        def leaf(rng, shape=None, buf=w):
            o, n = rng
            if n == 0:
                return None
            t = torch.tensor(np.asarray(buf[o:o + n], dtype=np.float32))
            if shape:
                t = t.reshape(shape)
            return t
        d = dict(W=leaf(sp_.kernel, (sp_.k_in, sp_.m_out)), b=leaf(sp_.bias), gamma=leaf(sp_.gamma),
                 beta=leaf(sp_.beta), alpha=leaf(sp_.alpha),
                 mm=leaf(sp_.moving_mean, buf=s), mv=leaf(sp_.moving_variance, buf=s), spec=sp_)
        if requires_grad:
            for k in ("W", "b", "gamma", "beta", "alpha"):
                if d[k] is not None:
                    d[k].requires_grad_(True)
        out.append(d)
    return out


def _block(p, x, training, eps, stats=None, branch=None):
    h = x @ p["W"] + p["b"]
    if training:
        mean = h.mean(0)
        var = ((h - mean.detach()) ** 2).mean(0)           # tf.nn.moments
        if stats is not None:
            stats.append((mean.detach(), var.detach()))
    else:
        mean, var = p["mm"], p["mv"]
    inv = torch.rsqrt(var + eps) * p["gamma"]              # tf.nn.batch_normalization
    z = h * inv + (p["beta"] - mean * inv)
    if p["alpha"] is not None:
        if branch is not None:
            # PReLU with the side of the kink pinned per element (see model_ref_np.loss_and_grads): identical to the
            # line below wherever sign(z) agrees with the pinned branch, i.e. everywhere but within rounding of 0
            br = torch.as_tensor(branch)
            return z * (br > 0).to(z.dtype) + p["alpha"] * z * (br < 0).to(z.dtype)
        return torch.relu(z) - p["alpha"] * torch.relu(-z)  # Keras PReLU
    return z


def tensors(x, rows, cols, seg):
    """float32 features and int64 index tensors of a batch (``seg`` None: node-level, no pool)."""
    xt = torch.tensor(np.asarray(x, dtype=np.float32))
    rt, ct = (torch.tensor(np.asarray(v, dtype=np.int64)) for v in (rows, cols))
    return xt, rt, ct, None if seg is None else torch.tensor(np.asarray(seg, dtype=np.int64))


def attn_leaf(cfg, specs, w, requires_grad=True):
    """pool.attn_kernel [Wc, 1] as a float32 leaf, or None unless pool='attn_sum'."""
    if cfg.pool != "attn_sum":
        return None
    o, k = O1.pool_kernel_range(specs)
    return torch.tensor(np.asarray(w[o:o + k], dtype=np.float32)).reshape(k, 1).requires_grad_(requires_grad)


def forward(cfg, params, x, rows, cols, seg, n_graphs, training, stats=None, prelu_branch=None, attn=None):
    """Logits (before the head's activation); ``attn``: pool.attn_kernel (attn_leaf) for pool='attn_sum'."""
    P, L = cfg.pre_process, cfg.message_passing
    br = prelu_branch if prelu_branch is not None else [None] * len(params)
    out = x
    for k, p in enumerate(params[:P]):
        out = _block(p, out, training, cfg.bn_epsilon, stats, br[k])
    n = x.shape[0]
    for k, p in enumerate(params[P:P + L]):
        a = _block(p, out, training, cfg.bn_epsilon, stats, br[P + k])
        msgs = a[cols]                                      # tf.gather -> [nnz, H]
        z = torch.zeros(n, a.shape[1], dtype=a.dtype).index_add_(0, rows, msgs)
        out = torch.cat([z, out], dim=1) if cfg.connectivity == "cat" else (z + out if cfg.connectivity == "sum" else z)
    if cfg.pool in ("sum", "avg"):
        out = torch.zeros(n_graphs, out.shape[1], dtype=out.dtype).index_add_(0, seg, out)
        if cfg.pool == "avg":
            out = out / torch.bincount(seg, minlength=n_graphs).to(out.dtype).clamp(min=1.0)[:, None]
    elif cfg.pool == "attn_sum":
        sc = (out @ attn)[:, 0]
        mx = torch.zeros(n_graphs, dtype=out.dtype).scatter_reduce_(0, seg, sc.detach(), "amax", include_self=False)
        e = torch.exp(sc - mx[seg])
        den = torch.zeros(n_graphs, dtype=out.dtype).index_add_(0, seg, e)
        p = e / (den[seg] + 1e-9)
        out = torch.zeros(n_graphs, out.shape[1], dtype=out.dtype).index_add_(0, seg, p[:, None] * out)
    for k, p in enumerate(params[P + L:]):
        out = _block(p, out, training, cfg.bn_epsilon, stats, br[P + L + k])
    return out                                              # logits (pre-activation)


def _loss(head, z, y, delta, sample_weight):
    """The head's Keras loss on the logits z: mean over every element (= the mean over the columns, then the rows), or
    with ``sample_weight`` the weighted row losses summed and divided by the row count."""
    F = torch.nn.functional
    elementwise = dict(sigmoid=F.binary_cross_entropy_with_logits, mse=F.mse_loss, mae=F.l1_loss,
                       huber=lambda z, y, **kw: F.huber_loss(z, y, delta=delta, **kw))
    if sample_weight is None:
        if head == "softmax":
            return -(y * torch.log_softmax(z, dim=1)).sum(1).mean()
        return elementwise[head](z, y)
    wt = torch.tensor(np.asarray(sample_weight, dtype=np.float32).reshape(-1))
    if head == "softmax":
        l = torch.logsumexp(z, dim=1) * y.sum(dim=1) - (y * z).sum(dim=1)
    else:
        l = elementwise[head](z, y, reduction="none").mean(dim=1)
    return (wt * l).sum() / z.shape[0]


def loss_and_grads(cfg, specs, w, s, x, rows, cols, seg, y, n_graphs, *, loss=None, delta=1.0, sample_weight=None,
                   prelu_branch=None):
    """One training-mode step in float32 autograd, pool.attn_kernel a leaf; heads and arguments as in
    model_ref_np.loss_and_grads.  Returns dict(loss, probs, logits, grads, stats, new_state)."""
    params = unpack(specs, w, s)
    attn = attn_leaf(cfg, specs, w)
    xt, rt, ct, st = tensors(x, rows, cols, seg)
    yt = torch.tensor(np.asarray(y, dtype=np.float32))
    stats = []
    logits = forward(cfg, params, xt, rt, ct, st, n_graphs, True, stats, prelu_branch, attn)
    head = O1.head_of(cfg, loss)
    lval = _loss(head, logits, yt, delta, sample_weight)
    lval.backward()
    grads = np.zeros(w.shape[0], dtype=np.float32)
    for p in params:
        sp_ = p["spec"]
        for key, (o, n) in (("W", sp_.kernel), ("b", sp_.bias), ("gamma", sp_.gamma), ("beta", sp_.beta), ("alpha", sp_.alpha)):
            if n:
                grads[o:o + n] = p[key].grad.reshape(-1).numpy()
    if attn is not None:
        o, n = O1.pool_kernel_range(specs)
        grads[o:o + n] = attn.grad.reshape(-1).numpy()
    z = logits.detach()
    probs = torch.softmax(z, dim=1) if head == "softmax" else (torch.sigmoid(z) if head == "sigmoid" else z)
    new_state = np.asarray(s, dtype=np.float32).copy()      # Keras moving statistics: moving -= (moving - batch) * (1 - momentum)
    for p, (mean, var) in zip(params, stats):
        for rng, old, batch in ((p["spec"].moving_mean, p["mm"], mean), (p["spec"].moving_variance, p["mv"], var)):
            o, n = rng
            new_state[o:o + n] = (old - (old - batch) * (1.0 - cfg.bn_momentum)).numpy()
    return dict(loss=float(lval.detach()), probs=probs.numpy(), logits=z.numpy(), grads=grads, stats=stats,
                new_state=new_state)


def time_reference_path(cfg, specs, w, s, graphs, n_steps=3, warmup=1, train=True, lr=0.0002,
                        threads=None):
    """Timed CPU baseline: host scipy collate + forward (+ backward + SGD) per step on the
    same batch of ``graphs`` [(x, a, y)], as the reference does per batch.  Returns median
    seconds per step and the thread count used."""
    from . import batching_ref
    if threads:
        torch.set_num_threads(threads)
    params = unpack(specs, w, s, requires_grad=train)
    leaves = [p[k] for p in params for k in ("W", "b", "gamma", "beta", "alpha") if p[k] is not None]
    times = []
    for it in range(warmup + n_steps):
        t0 = time.perf_counter()
        (x, (indices, _vals, _shape), seg), y = batching_ref.collate(graphs)
        xt = torch.tensor(np.asarray(x, dtype=np.float32))
        rt = torch.tensor(indices[:, 0])
        ct = torch.tensor(indices[:, 1])
        st = torch.tensor(seg)
        yt = torch.tensor(np.asarray(y, dtype=np.float32))
        if train:
            logits = forward(cfg, params, xt, rt, ct, st, len(graphs), True)
            loss = -(yt * torch.log_softmax(logits, 1)).sum(1).mean()
            for t in leaves:
                t.grad = None
            loss.backward()
            with torch.no_grad():
                for t in leaves:
                    t -= lr * t.grad
        else:
            with torch.no_grad():
                forward(cfg, params, xt, rt, ct, st, len(graphs), False)
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    return float(np.median(times)), torch.get_num_threads()
