"""Unit tests of the CUDA kernels through the C ABI's diagnostic entry points (B200 only)."""
import ctypes as C

import pytest
import torch

from __graft_entry__ import load_package

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    pkg = load_package()
    import sys
    return sys.modules[pkg.__name__ + "._cabi"].load_library(), sys.modules[pkg.__name__ + "._cabi"]


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


@pytest.mark.parametrize("block_n", [64, 128, 256])
@pytest.mark.parametrize("M,N,K", [(180, 3072, 1024), (128, 256, 64), (100, 64, 64), (333, 1024, 4096), (1620, 512, 1088),
                                    (5760, 1024, 1024), (333, 1024, 1040)])    # K = 1040: a last K block of 16 columns (fmt_proj_create allows in_dim % 16)
def test_tcgen05_gemm_matches_torch(lib, M, N, K, block_n):
    L, cabi = lib
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N * 3 + K)
    A = torch.randn(M, K, device="cuda", generator=g).to(torch.bfloat16)
    W = (torch.randn(N, K, device="cuda", generator=g) * 0.05).to(torch.bfloat16)
    bias = torch.randn(N, device="cuda", generator=g)
    out = torch.full((M, N), float("nan"), device="cuda")
    cabi.check(L.fmt_debug_gemm_bf16(A.data_ptr(), W.data_ptr(), bias.data_ptr(), out.data_ptr(), M, N, K, block_n, _stream()), "gemm")
    torch.cuda.synchronize()
    ref = A.double() @ W.double().t() + bias.double()      # same bf16 operands, exact accumulation
    err = (out.double() - ref).abs().max().item()
    assert torch.isfinite(out).all()
    assert err <= 2e-3 * max(1.0, ref.abs().max().item()), err   # fp32 accumulation error only


@pytest.mark.parametrize("block_n", [512, 1024])     # CTA-pair kernel: 256 x 256 and 256 x 128 pair tiles
@pytest.mark.parametrize("M,N,K", [(5760, 1024, 1024), (512, 256, 64), (300, 512, 128), (1620, 3072, 1024), (5760, 1024, 4096),
                                    (51840, 512, 1088), (46080, 4096, 1024), (129, 256, 192)])
def test_cta_pair_gemm_matches_torch(lib, M, N, K, block_n):
    """cta_group::2 GEMM (two SMs per 256-row tile, B operand split across the pair)."""
    L, cabi = lib
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N * 3 + K)
    A = torch.randn(M, K, device="cuda", generator=g).to(torch.bfloat16)
    W = (torch.randn(N, K, device="cuda", generator=g) * 0.05).to(torch.bfloat16)
    bias = torch.randn(N, device="cuda", generator=g)
    out = torch.full((M, N), float("nan"), device="cuda")
    cabi.check(L.fmt_debug_gemm_bf16(A.data_ptr(), W.data_ptr(), bias.data_ptr(), out.data_ptr(), M, N, K, block_n, _stream()), "gemm")
    torch.cuda.synchronize()
    ref = A.float() @ W.float().t() + bias       # fp32 reference of the same bf16 operands (TF32 off by default for matmul)
    err = (out - ref).abs().max().item()
    assert torch.isfinite(out).all()
    assert err <= 4e-3 * max(1.0, ref.abs().max().item()), err


@pytest.mark.parametrize("M,N,K", [(180, 3072, 1024), (70, 68, 64), (360, 512, 1088)])
def test_fp32_simt_gemm_matches_torch(lib, M, N, K):
    L, cabi = lib
    g = torch.Generator(device="cuda").manual_seed(1)
    A = torch.randn(M, K, device="cuda", generator=g)
    W = torch.randn(N, K, device="cuda", generator=g) * 0.05
    bias = torch.randn(N, device="cuda", generator=g)
    out = torch.full((M, N), float("nan"), device="cuda")
    cabi.check(L.fmt_debug_gemm_fp32(A.data_ptr(), W.data_ptr(), bias.data_ptr(), out.data_ptr(), M, N, K, _stream()), "gemm")
    torch.cuda.synchronize()
    ref = A.double() @ W.double().t() + bias.double()
    rel = ((out.double() - ref).norm() / ref.norm()).item()
    assert rel <= 1e-6, rel
