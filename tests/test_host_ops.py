"""CPU tests of what tests/test_gpu_ops.py relies on: its fp64 references restate the oracle's block exactly, and the ctypes
mirror of FmtDebugGemm has the header's layout."""
import ctypes as C
import os
import shutil
import subprocess
import sys
import tempfile

import pytest
import torch

import ops_ref as R
from __graft_entry__ import ROOT, load_package
from oracle import fmt_oracle as O


def _block_weights(H, mlp, g):
    p = "blocks.0."
    shapes = {"attn.qkv": (3 * H, H), "attn.proj": (H, H), "mlp.fc1": (mlp, H), "mlp.fc2": (H, mlp), "adaLN_modulation.1": (6 * H, H)}
    W = {}
    for name, (n, k) in shapes.items():
        W[p + name + ".weight"] = torch.randn(n, k, generator=g, dtype=torch.float64) / k ** 0.5
        W[p + name + ".bias"] = torch.randn(n, generator=g, dtype=torch.float64) * 0.1
    return W


@pytest.mark.parametrize("window", [0, 2, 7])
def test_references_compose_to_the_oracle_block(window):
    """lnmod -> qkv -> band attention -> proj (x += gate * .) -> lnmod -> fc1 (GELU) -> fc2 (x += gate * .), with the table
    offsets the sampler uses (shift, scale, gate = 0, H, 2H and 3H, 4H, 5H of a 6H row), equals O.fmt_block in fp64."""
    H, heads, mlp, N = 64, 4, 256, 13
    g = torch.Generator().manual_seed(window)
    W = _block_weights(H, mlp, g)
    x = torch.randn(1, N, H, generator=g, dtype=torch.float64)
    c_silu = torch.randn(1, N, H, generator=g, dtype=torch.float64)
    ref = O.fmt_block(W, 0, x, c_silu, O.band_mask(N, window), heads, O.Quant())

    def lin(name):
        return W["blocks.0." + name + ".weight"], W["blocks.0." + name + ".bias"]

    table = torch.nn.functional.linear(c_silu[0], *lin("adaLN_modulation.1"))          # (N, 6H): one table row per token row
    x0 = x[0]
    h = R.lnmod(x0, table, None, 0, H)
    wq, bq = lin("attn.qkv")
    a = R.band_attention(R.gemm_epilogue(R.STORE, h @ wq.t(), bq)[None], heads, window)[0]
    wp, bp = lin("attn.proj")
    x1 = R.gemm_epilogue(R.GATE_RES, a @ wp.t(), bp, x=x0, gate=table[:, 2 * H:3 * H])
    h2 = R.lnmod(x1, table, None, 3 * H, 4 * H)
    w1, b1 = lin("mlp.fc1")
    m = R.gemm_epilogue(R.GELU, h2 @ w1.t(), b1)
    w2, b2 = lin("mlp.fc2")
    x2 = R.gemm_epilogue(R.GATE_RES, m @ w2.t(), b2, x=x1, gate=table[:, 5 * H:6 * H])
    assert torch.allclose(x2, ref[0], rtol=0, atol=1e-12), (x2 - ref[0]).abs().max()


def test_band_attention_reference_matches_the_oracle_attention():
    H, heads, N = 96, 3, 11
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, N, H, generator=g, dtype=torch.float64)
    W = {"attn.qkv.weight": torch.randn(3 * H, H, generator=g, dtype=torch.float64), "attn.qkv.bias": torch.randn(3 * H, generator=g, dtype=torch.float64),
         "attn.proj.weight": torch.eye(H, dtype=torch.float64), "attn.proj.bias": torch.zeros(H, dtype=torch.float64)}
    qkv = torch.nn.functional.linear(x, W["attn.qkv.weight"], W["attn.qkv.bias"])
    for window in (0, 1, 4, 20):
        ref = O.attention(W, "", x, O.band_mask(N, window), heads, O.Quant())
        assert torch.allclose(R.band_attention(qkv, heads, window), ref, rtol=0, atol=1e-12)


def test_reference_gelu_is_the_tanh_approximation():
    x = torch.linspace(-8, 8, 1001, dtype=torch.float64)
    assert torch.allclose(R.gelu_tanh(x), torch.nn.functional.gelu(x, approximate="tanh"), rtol=0, atol=1e-15)
    assert (R.gelu_tanh(x) - torch.nn.functional.gelu(x)).abs().max() > 1e-4       # the exact-erf GELU is a different function


def test_pair_decoder_inverts_the_pair_layout():
    x = torch.randn(3, 128, dtype=torch.float32, generator=torch.Generator().manual_seed(0))
    hi = x.to(torch.bfloat16)
    lo = (x - hi.float()).to(torch.bfloat16)
    buf = torch.stack([hi.reshape(3, 2, 64), lo.reshape(3, 2, 64)], dim=2).reshape(3, 256)
    dec = R.decode_pairs(buf, 128)
    assert ((dec - x.double()).abs() <= R.PAIR_REPR * x.double().abs()).all()


def test_debug_gemm_struct_matches_the_header():
    cabi = sys.modules[load_package().__name__ + "._cabi"]
    G = cabi.FmtDebugGemm
    fields = [f[0] for f in G._fields_]
    assert fields == ["mode", "kind", "M", "N", "K", "block_n", "ksplit", "ldo", "out_f32", "frames", "A", "W", "bias", "out", "pos", "gate",
                      "urow", "ldg", "gate_off"]
    assert (cabi.FMT_EPI_STORE, cabi.FMT_EPI_GELU, cabi.FMT_EPI_POS, cabi.FMT_EPI_GATE_RES) == (R.STORE, R.GELU, R.POS, R.GATE_RES)
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no host C compiler for the offsetof probe")
    with tempfile.TemporaryDirectory() as tmp:
        src, exe = os.path.join(tmp, "probe.c"), os.path.join(tmp, "probe")
        with open(src, "w") as f:
            f.write('#include <stddef.h>\n#include <stdio.h>\n#include "fmt_b200.h"\nint main(void) {\n')
            for fld in fields:
                f.write(f'  printf("%zu ", offsetof(FmtDebugGemm, {fld}));\n')
            f.write('  printf("%zu %d %d %d %d\\n", sizeof(FmtDebugGemm), FMT_EPI_STORE, FMT_EPI_GELU, FMT_EPI_POS, FMT_EPI_GATE_RES);\n'
                    '  return 0;\n}\n')
        subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", exe, src], check=True)
        got = [int(v) for v in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [getattr(G, f).offset for f in fields] + [C.sizeof(G), R.STORE, R.GELU, R.POS, R.GATE_RES]
