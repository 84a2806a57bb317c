"""The tcgen05 projection kernel in isolation (through the C-ABI test hook) against a plain fp32 matmul of the same
rounded operands.  Covers both operand kinds (bf16; split bf16 hi/lo planes = the fp32-grade mode),
the plain epilogues, ragged M / N / K tiles.  The LayerNorm-fused epilogues are in test_gemm_ln_gpu.py."""

import numpy as np
import pytest
import torch

from openmpl_b200 import _lib

pytestmark = pytest.mark.gpu

SHAPES = [(128, 64, 64), (300, 256, 128), (1000, 1088, 1088), (777, 3264, 1088), (513, 2176, 1088), (2049, 1088, 2176),
          (130, 48, 32), (260, 544, 544), (4096, 96, 32), (64, 16, 8)]


def _split(x):
    """fp32 -> the two bf16 planes of the fp32-grade mode, [2, rows, cols]: hi = bf16(x), lo = bf16(x - hi)."""
    hi = x.to(torch.bfloat16)
    lo = (x - hi.float()).to(torch.bfloat16)
    return torch.stack([hi, lo]).contiguous()


def _gelu(x):
    return 0.5 * x * (1.0 + torch.erf(x / np.sqrt(2.0)))


def _run(M, N, K, dtype, epi):
    L = _lib.lib()
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N * 3 + K)
    A = torch.randn(M, K, device="cuda", generator=g)
    W = torch.randn(N, K, device="cuda", generator=g) / np.sqrt(K)
    bias = torch.randn(N, device="cuda", generator=g)
    if dtype == "bf16":
        Ad, Wd = A.to(torch.bfloat16), W.to(torch.bfloat16)
        Af, Wf = Ad.float(), Wd.float()
    else:
        # split mode: the kernel sees hi + lo of both operands and drops only the lo.lo product -> compare with the
        # exact product of the fp32 matrices (the 2^-16 operand error is part of what the mode promises)
        Ad, Wd = _split(A), _split(W)
        Af, Wf = A, W
    ref = Af.double() @ Wf.double().T + bias.double()
    out_fp32 = 0
    planes = (2,) if dtype == "tf32" else ()
    if epi == 0:
        Y = torch.empty(planes + (M, N), device="cuda", dtype=torch.bfloat16)
    elif epi == 1:
        ref = _gelu(ref)
        Y = torch.empty(planes + (M, N), device="cuda", dtype=torch.bfloat16)
    elif epi == 2:
        Y = torch.randn(M, N, device="cuda", generator=g)
        ref = ref + Y.double()
        out_fp32 = 1
    else:
        epi, out_fp32 = 0, 1
        Y = torch.empty(M, N, device="cuda", dtype=torch.float32)
    Y0 = Y.clone()
    stream = torch.cuda.current_stream().cuda_stream
    _lib.check(L.mpl_test_gemm(Ad.data_ptr(), Wd.data_ptr(), bias.data_ptr(), Y.data_ptr(), M, N, K,
                               _lib.PRECISIONS[dtype], epi, out_fp32, stream))
    torch.cuda.synchronize()
    del Y0
    out_is_bf16 = Y.dtype == torch.bfloat16 and not planes
    if planes and Y.dim() == 3:
        Y = Y[0].double() + Y[1].double()          # hi + lo planes
    err = (Y.double() - ref).abs().max().item() / max(ref.abs().max().item(), 1e-6)
    # split mode: 2^-16 operand error over a random-sign sum, plus 2^-17 of the split output
    tol = 6e-3 if out_is_bf16 else (4e-5 if dtype == "tf32" else 2e-5)
    assert err <= tol, f"M={M} N={N} K={K} {dtype} epi={epi}: rel err {err:.3e}"


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("dtype", ["bf16", "tf32"])
def test_gemm_cg2(shape, dtype):
    for epi in (0, 1, 2, 3):
        _run(*shape, dtype, epi)


def test_gemm_rejects_untileable_shapes():
    L = _lib.lib()
    x = torch.zeros(64, device="cuda")
    assert L.mpl_test_gemm(x.data_ptr(), x.data_ptr(), x.data_ptr(), x.data_ptr(), 4, 24, 8, 2, 0, 0, None) == _lib.MPL_ERR_UNSUPPORTED
    assert L.mpl_test_gemm(x.data_ptr(), x.data_ptr(), x.data_ptr(), x.data_ptr(), 4, 16, 12, 2, 0, 0, None) == _lib.MPL_ERR_UNSUPPORTED
