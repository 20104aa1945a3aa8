"""linear_f16_pass256_kernel: the fp16-split forward / input-gradient GEMM for output widths that are multiples of 256
(one CTA-pair pass computes 256 output columns; the split A operand lives in shared memory).  Through the standalone
ops in debug mode 2 (fp16 everywhere, operand |max| by an extra pass) against float64 at 1e-5: widths 256 / 512 / 768,
reductions from one K block to a chunked 2048, ragged rows, strided A and C, accumulate, the four operand scalings of
test_fp16_split_tensor_core_gemm, and run-to-run bit identity."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from gcn_string_b200 import _lib, ops

from conftest import rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-5

# (M, K, N): every width with every reduction depth once, ragged row counts spread over them; the N = 256 cases of
# test_fp16_split_tensor_core_gemm are not repeated
CASES = [(1, 64, 256), (257, 256, 256), (33000, 1024, 256),
         (255, 64, 512), (1, 1280, 512), (257, 2048, 512), (33000, 256, 512),
         (257, 64, 768), (33000, 1280, 768), (255, 1024, 768), (1, 2048, 768)]


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.detach().cpu().numpy()


@pytest.mark.parametrize("M,K,N", CASES)
@pytest.mark.parametrize("scaling", ["unit", "tiny", "huge", "spread"])
def test_f16_gemm_256_column_pass(M, K, N, scaling):
    lib = _lib.load()
    rng = np.random.default_rng(7 * M + 3 * K + N + len(scaling))
    a_mag, w_mag = {"unit": (1.0, 1.0), "tiny": (1e-9, 1e-4), "huge": (3e4, 50.0), "spread": (1.0, 1.0)}[scaling]
    wideA = (rng.standard_normal((M, K + 64)) * a_mag).astype(np.float32)
    if scaling == "spread":
        wideA *= np.exp2(-rng.integers(0, 25, wideA.shape)).astype(np.float32)
    A = wideA[:, 32:32 + K]
    W = (rng.standard_normal((K, N)) / np.sqrt(K) * w_mag).astype(np.float32)
    b = (rng.standard_normal(N) * a_mag * w_mag).astype(np.float32)
    A64, W64 = A.astype(np.float64), W.astype(np.float64)
    dA = dev(wideA)[:, 32:32 + K]                                   # strided A
    try:
        lib.gcs_debug_set_param(7, 2)
        lib.gcs_debug_set_gemm_mode(2)
        out = torch.zeros(M, N + 128, device="cuda")
        y = ops.linear_fwd(dA, dev(W), dev(b), out=out[:, 128:])    # strided C
        assert rel_err(host(y), A64 @ W64 + b) < TOL
        assert float(out[:, :128].abs().max()) == 0.0               # nothing written left of the view
        y2 = ops.linear_fwd(dA, dev(W), dev(b))
        assert torch.equal(y2, y.contiguous())                      # bit-identical run to run, any C pitch
        # accumulate into an existing C: the input-gradient form with output width N and reduction K
        Wt = np.ascontiguousarray(W.T)
        base = (rng.standard_normal((M, N)) * a_mag * w_mag).astype(np.float32)
        acc = ops.linear_bwd_input(dA, dev(Wt), out=dev(base), accumulate=True)
        assert rel_err(host(acc), base + A64 @ W64) < TOL
        acc2 = ops.linear_bwd_input(dA, dev(Wt), out=dev(base), accumulate=True)
        assert torch.equal(acc, acc2)
    finally:
        lib.gcs_debug_set_gemm_mode(0)
        lib.gcs_debug_set_param(7, 1)
