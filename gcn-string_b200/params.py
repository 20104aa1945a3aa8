"""GeneralGNN hyper-parameters and the flat parameter layout shared by the CUDA
library (csrc/model.cu computes the same offsets), the Python wrapper and the oracle.

Mirrors the keyword set of ``spektral.models.GeneralGNN.__init__`` as the reference
instantiates it (reference: src/scripts/gcn.py:320 — only ``output`` and
``activation`` are passed, everything else is the Spektral default; SURVEY.md §8 a2).

A "dense block" is the unit every stage is made of (SURVEY.md §8 a3/a4):
``Dense/K.dot + bias -> BatchNormalization -> Dropout(rate) -> PReLU | final activation`` (the rate is GeneralGNN's,
not part of this layout).
Blocks, in order: ``pre.0 .. pre.{P-1}``, ``gnn.0 .. gnn.{L-1}``, ``post.0 .. post.{Q-1}``.
Per block the trainable tensors are laid out ``kernel[K,M], bias[M], gamma[M], beta[M],
alpha[M]`` (no ``alpha`` on the last post block: its activation is the model's final
activation, not PReLU) in ONE flat fp32 buffer; with ``pool='attn_sum'`` the pool's
``attn_kernel [Wc, 1]`` follows the last block (every block offset stays as for 'sum'); the gradient buffer has the same layout
(it is the NCCL all-reduce bucket), and the non-trainable BatchNorm statistics
``moving_mean[M], moving_variance[M]`` per block live in a second flat buffer.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Optional, Tuple

CONNECTIVITY = {None: 0, "cat": 1, "sum": 2}
POOL = {None: 0, "sum": 1, "avg": 2, "attn_sum": 3}   # spektral GlobalSumPool / GlobalAvgPool / GlobalAttnSumPool
FINAL_ACT = {None: 0, "linear": 0, "softmax": 1, "sigmoid": 2}
AGGREGATE = {"sum": 0, "mean": 1, "max": 2}          # spektral scatter_sum / scatter_mean / scatter_max


@dataclass(frozen=True)
class GNNConfig:
    """Static description of one GeneralGNN (defaults = Spektral's)."""
    in_features: int
    output: int
    activation: Optional[str] = None
    hidden: int = 256
    message_passing: int = 4
    pre_process: int = 2
    post_process: int = 2
    connectivity: Optional[str] = "cat"
    batch_norm: bool = True
    dropout: float = 0.0
    aggregate: str = "sum"
    hidden_activation: str = "prelu"
    pool: Optional[str] = "sum"
    bn_momentum: float = 0.99      # Keras BatchNormalization defaults (SURVEY.md §8 a6)
    bn_epsilon: float = 1e-3

    def validate(self) -> None:
        """Raise for anything outside the native subset (no fallback; SURVEY.md §8b)."""
        if self.aggregate not in AGGREGATE:
            raise NotImplementedError("native path implements aggregate in {'sum', 'mean', 'max'}")
        if self.aggregate == "max" and self.connectivity == "sum":
            raise NotImplementedError("aggregate='max' with connectivity='sum' is not built")
        if self.pool not in POOL:
            raise NotImplementedError("native path implements pool in {'sum', 'avg', 'attn_sum', None}")
        if self.connectivity not in CONNECTIVITY:
            raise ValueError("connectivity must be 'cat', 'sum' or None")
        if self.dropout != 0.0:
            # the rate changes no parameter, state or workspace layout: GeneralGNN carries it into its training calls
            raise NotImplementedError("GNNConfig describes the layout, which dropout does not change: pass the rate as "
                                      "GeneralGNN(dropout=rate)")
        if self.hidden_activation != "prelu":
            raise NotImplementedError("native path implements hidden_activation='prelu' only")
        if not self.batch_norm:
            raise NotImplementedError("native path implements batch_norm=True only")
        if self.activation not in FINAL_ACT:
            raise NotImplementedError("final activation must be None/'linear'/'softmax'/'sigmoid'")
        if self.pre_process < 1 or self.post_process < 1 or self.message_passing < 1:
            raise NotImplementedError("pre_process, post_process, message_passing must be >= 1")
        if min(self.in_features, self.output, self.hidden) < 1:
            raise ValueError("feature widths must be positive")

    @property
    def cat_width(self) -> int:
        """Width of the node embedding entering the pool."""
        if self.connectivity == "cat":
            return self.hidden * (self.message_passing + 1)
        return self.hidden


def check_dropout_rate(rate) -> None:
    """Keras Dropout: ``0 <= rate < 1``; anything else (NaN included) is a ValueError."""
    if isinstance(rate, bool) or not isinstance(rate, (int, float)) or not (0.0 <= rate < 1.0):
        raise ValueError(f"dropout rate must be a number in [0, 1), got {rate!r}")


_U64 = (1 << 64) - 1


def dropout_seed(seed: int, rank: int = 0) -> int:
    """Key of the dropout mask stream of data-parallel rank ``rank`` for a model seeded with ``seed``: the splitmix64
    finaliser of ``seed + rank * 0x9E3779B97F4A7C15`` (mod 2^64).  The finaliser is a bijection and the odd increment
    makes ``seed + rank * inc`` distinct for every rank, so ranks draw independent masks; rank 0 is the single-device
    stream."""
    z = (int(seed) + int(rank) * 0x9E3779B97F4A7C15) & _U64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _U64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _U64
    return z ^ (z >> 31)


@dataclass(frozen=True)
class BlockSpec:
    name: str          # e.g. "gnn.2"
    k_in: int          # rows of kernel
    m_out: int         # cols of kernel
    has_alpha: bool    # PReLU follows
    offset: int        # float offset of kernel in the trainable buffer
    stat_offset: int   # float offset of moving_mean in the state buffer

    @property
    def kernel(self) -> Tuple[int, int]:
        return (self.offset, self.k_in * self.m_out)

    @property
    def bias(self) -> Tuple[int, int]:
        return (self.offset + self.k_in * self.m_out, self.m_out)

    @property
    def gamma(self) -> Tuple[int, int]:
        return (self.bias[0] + self.m_out, self.m_out)

    @property
    def beta(self) -> Tuple[int, int]:
        return (self.gamma[0] + self.m_out, self.m_out)

    @property
    def alpha(self) -> Tuple[int, int]:
        return (self.beta[0] + self.m_out, self.m_out if self.has_alpha else 0)

    @property
    def n_trainable(self) -> int:
        return self.k_in * self.m_out + (4 if self.has_alpha else 3) * self.m_out

    @property
    def moving_mean(self) -> Tuple[int, int]:
        return (self.stat_offset, self.m_out)

    @property
    def moving_variance(self) -> Tuple[int, int]:
        return (self.stat_offset + self.m_out, self.m_out)


def block_specs(cfg: GNNConfig) -> List[BlockSpec]:
    """Ordered dense blocks with their offsets (same arithmetic as csrc/model.cu)."""
    H = cfg.hidden
    blocks: List[Tuple[str, int, int, bool]] = []
    k = cfg.in_features
    for j in range(cfg.pre_process):
        blocks.append((f"pre.{j}", k, H, True))
        k = H
    for j in range(cfg.message_passing):
        k_in = H * (j + 1) if cfg.connectivity == "cat" else H
        blocks.append((f"gnn.{j}", k_in, H, True))
    k = cfg.cat_width
    for j in range(cfg.post_process):
        last = j == cfg.post_process - 1
        blocks.append((f"post.{j}", k, cfg.output if last else H, not last))
        k = H
    out, off, soff = [], 0, 0
    for name, k_in, m_out, has_alpha in blocks:
        spec = BlockSpec(name, k_in, m_out, has_alpha, off, soff)
        out.append(spec)
        off += spec.n_trainable
        soff += 2 * m_out
    return out


def pool_kernel_slice(cfg: GNNConfig) -> Optional[Tuple[int, int]]:
    """(offset, Wc) of ``pool.attn_kernel`` in the trainable buffer for ``pool='attn_sum'``, else None."""
    if cfg.pool != "attn_sum":
        return None
    last = block_specs(cfg)[-1]
    return (last.offset + last.n_trainable, cfg.cat_width)


def n_trainable(cfg: GNNConfig) -> int:
    pk = pool_kernel_slice(cfg)
    return sum(b.n_trainable for b in block_specs(cfg)) + (pk[1] if pk else 0)


def n_state(cfg: GNNConfig) -> int:
    return sum(2 * b.m_out for b in block_specs(cfg))


def named_slices(cfg: GNNConfig):
    """[(name, shape, offset, buffer)] with buffer in {'trainable', 'state'}; this is the
    order ``trainable_variables`` / ``get_weights`` use."""
    out = []
    for b in block_specs(cfg):
        out.append((f"{b.name}.kernel", (b.k_in, b.m_out), b.kernel[0], "trainable"))
        out.append((f"{b.name}.bias", (b.m_out,), b.bias[0], "trainable"))
        out.append((f"{b.name}.bn.gamma", (b.m_out,), b.gamma[0], "trainable"))
        out.append((f"{b.name}.bn.beta", (b.m_out,), b.beta[0], "trainable"))
        if b.has_alpha:
            out.append((f"{b.name}.prelu.alpha", (b.m_out,), b.alpha[0], "trainable"))
        out.append((f"{b.name}.bn.moving_mean", (b.m_out,), b.moving_mean[0], "state"))
        out.append((f"{b.name}.bn.moving_variance", (b.m_out,), b.moving_variance[0], "state"))
    pk = pool_kernel_slice(cfg)
    if pk:
        out.append(("pool.attn_kernel", (pk[1], 1), pk[0], "trainable"))
    return out


def init_params(cfg: GNNConfig, seed: int = 0, perturb: bool = False):
    """Keras-default initialisation as flat fp32 numpy buffers (trainable, state):
    glorot-uniform kernels, zero bias, gamma=1, beta=0, alpha=0, moving_mean=0,
    moving_variance=1 (SURVEY.md §8 a3/a6/a7); ``pool.attn_kernel`` glorot-uniform [Wc, 1], drawn after every
    block so that the blocks get the same values as with any other pool.  ``perturb=True`` moves gamma, beta,
    alpha, bias and the moving statistics off their defaults so every gradient path is
    exercised in parity tests (SURVEY.md §8d)."""
    import numpy as np
    rng = np.random.default_rng(seed)
    w = np.zeros(n_trainable(cfg), dtype=np.float32)
    s = np.zeros(n_state(cfg), dtype=np.float32)
    for b in block_specs(cfg):
        lim = np.sqrt(6.0 / (b.k_in + b.m_out))
        o, n = b.kernel
        w[o:o + n] = rng.uniform(-lim, lim, size=n).astype(np.float32)
        o, n = b.gamma
        w[o:o + n] = 1.0
        o, n = b.moving_variance
        s[o:o + n] = 1.0
        if perturb:
            o, n = b.bias
            w[o:o + n] = rng.normal(0, 0.1, n)
            o, n = b.gamma
            w[o:o + n] = rng.uniform(0.5, 1.5, n)
            o, n = b.beta
            w[o:o + n] = rng.normal(0, 0.2, n)
            o, n = b.alpha
            w[o:o + n] = rng.uniform(0.05, 0.45, n)
            o, n = b.moving_mean
            s[o:o + n] = rng.normal(0, 0.3, n)
            o, n = b.moving_variance
            s[o:o + n] = rng.uniform(0.5, 2.0, n)
    pk = pool_kernel_slice(cfg)
    if pk:
        o, n = pk
        lim = np.sqrt(6.0 / (n + 1))
        w[o:o + n] = rng.uniform(-lim, lim, size=n).astype(np.float32)
    return w, s
