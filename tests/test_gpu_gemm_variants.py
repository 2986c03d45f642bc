"""Do the sampler's GEMM kernel variants give the same bits on the same operands?  (B200 only.)

A StreamSampler step at partial occupancy replays a window graph captured for fewer slots, whose GEMMs have fewer rows, and the
sampler picks a GEMM variant from the row count M.  A step's frames are bitwise equal to a full-slot run only if every GEMM computes
each output element the same way whichever variant the bucket picks.  This test runs every GEMM shape of the model (synth dims) at
every variant - single-CTA tiles of block_n 64 / 128 / 256 and the CTA-pair tiles 256 x 256 / 256 x 128, no K slices - on the same
random operands, through fmt_debug_gemm_bf16 and fmt_debug_gemm_bf16x3, and asserts torch.equal between all of them.  The graphs
of an occupancy bucket choose their GEMM variants on their own row counts because of this (DESIGN.md section 4f)."""
import ctypes as C
import sys

import pytest
import torch

from __graft_entry__ import load_package

pytestmark = pytest.mark.gpu

VARIANTS = (64, 128, 256, 512, 1024)


@pytest.fixture(scope="module")
def lib():
    pkg = load_package()
    cabi = sys.modules[pkg.__name__ + "._cabi"]
    return cabi.load_library(), pkg.synth.FmtDims()


def model_gemms(d):
    """(name, N, K) of every Linear of a sampling window: x-embedder, condition embedder, AdaLN table, the four of a block, decoder."""
    kc = (d.dim_w + d.dim_a + d.dim_e + 63) // 64 * 64
    nt = d.fmt_depth * 6 * d.dim_h + 2 * d.dim_h
    return [("x_emb", d.dim_h, d.dim_w), ("c_emb", d.dim_h, kc), ("ada", nt, d.dim_h), ("qkv", 3 * d.dim_h, d.dim_h),
            ("proj", d.dim_h, d.dim_h), ("fc1", d.mlp_hidden, d.dim_h), ("fc2", d.dim_h, d.mlp_hidden), ("dec", d.dim_w, d.dim_h)]


def _run(L, fn, A, W, bias, M, N, K, block_n):
    out = torch.full((M, N), float("nan"), device="cuda")
    rc = fn(C.c_void_p(A.data_ptr()), C.c_void_p(W.data_ptr()), C.c_void_p(bias.data_ptr()), C.c_void_p(out.data_ptr()), M, N, K, block_n,
            C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, L.fmt_last_error().decode()
    torch.cuda.synchronize()
    return out


# rows: one slot's 3-way rows (180), a ragged count, and enough rows for several waves of every tile shape
@pytest.mark.parametrize("M", [180, 333, 2880])
@pytest.mark.parametrize("mode", ["bf16", "bf16x3"])
def test_gemm_variants_bitwise_equal(lib, mode, M):
    L, d = lib
    g = torch.Generator(device="cuda").manual_seed(M)
    differ = []
    for name, N, K in model_gemms(d):
        A = torch.randn(M, K, device="cuda", generator=g)
        W = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
        bias = torch.randn(N, device="cuda", generator=g)
        if mode == "bf16":
            fn, args = L.fmt_debug_gemm_bf16, (A.bfloat16(), W.bfloat16())
        else:
            fn, args = L.fmt_debug_gemm_bf16x3, (A, W)
        outs = {bn: _run(L, fn, *args, bias, M, N, K, bn) for bn in (0,) + VARIANTS}
        ref = outs[0]
        assert torch.isfinite(ref).all(), (name, mode, M)
        differ += [f"{name} (N={N}, K={K}) block_n {bn}: {(outs[bn] != ref).sum().item()} elements" for bn in VARIANTS
                   if not torch.equal(outs[bn], ref)]
    assert not differ, f"{mode} at M={M}, against the variant the sampler picks: " + "; ".join(differ)
