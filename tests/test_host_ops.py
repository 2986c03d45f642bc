"""CPU tests of what tests/test_gpu_ops.py and tests/test_gpu_window_stages.py rely on: their fp64 references restate the oracle's
block, CFG combine and solvers exactly, the operand decoders invert the kernels' tiled layouts, the ctypes mirrors of
FmtDebugGemm / FmtDebugStage have the header's layout, and the stage entry points refuse bad shapes."""
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


def test_key_bias_does_not_change_band_attention():
    """q . (k_j + b_k) = q . k_j + q . b_k shifts every score of a query by the same amount, and softmax is shift-invariant: the
    key bias of the qkv projection cancels in attention, so the kernels' `+ bk` in the scores is exact arithmetic that no output
    can reveal (dropping it changes results by rounding only)."""
    heads, hd, N = 2, 32, 17
    g = torch.Generator().manual_seed(4)
    qkv = torch.randn(2, N, 3 * heads * hd, generator=g, dtype=torch.float64)
    kb = torch.zeros(3 * heads * hd, dtype=torch.float64)
    kb[heads * hd:2 * heads * hd] = torch.randn(heads * hd, generator=g, dtype=torch.float64) * 3
    for window in (0, 2, 7):
        assert torch.allclose(R.band_attention(qkv + kb, heads, window), R.band_attention(qkv, heads, window), rtol=0, atol=1e-12)


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


def test_tiled_decoders_invert_the_kernels_operand_layouts():
    """flow_tiled_off / win_tiled_off (flow.cuh, window.cuh), transcribed element by element, against the decoders."""
    def flow_off(c, r, col, nkb, CH):
        kb, cc = col >> 6, col & 63
        return (c * nkb + kb) * (CH * 64) + r * 64 + ((((cc >> 3) ^ (r & 7)) << 3) | (cc & 7))

    def win_off(r, col, Rp):
        kb, cc = col >> 6, col & 63
        return kb * Rp * 64 + r * 64 + ((((cc >> 3) ^ (r & 7)) << 3) | (cc & 7))

    g = torch.Generator().manual_seed(1)
    n_chunks, CH, cols = 3, 32, 192
    x = torch.randn(n_chunks * CH, cols, generator=g)
    buf = torch.empty(n_chunks * CH * cols)
    for c in range(n_chunks):
        for r in range(CH):
            for col in range(cols):
                buf[flow_off(c, r, col, cols // 64, CH)] = x[c * CH + r, col]
    assert torch.equal(R.flow_tiled_decode(buf, n_chunks, CH, cols), x)
    Rp = 128
    x = torch.randn(Rp, cols, generator=g)
    buf = torch.empty(Rp * cols)
    for r in range(Rp):
        for col in range(cols):
            buf[win_off(r, col, Rp)] = x[r, col]
    assert torch.equal(R.win_tiled_decode(buf, Rp, cols), x)


def test_cfg_and_rk_references_follow_the_oracle_and_the_solvers():
    """cfg_combine is forward_with_cfv's combine (branch order [uncond | all | audio-only], [truly-uncond | uncond | all |
    audio-only]); rk_stage walked over a step's stages is the solver's step: y0 + dt * sum_j b_j f(t, y_j)."""
    sampler = sys.modules[load_package().__name__ + ".sampler"]
    g = torch.Generator().manual_seed(2)
    vb = [torch.randn(5, generator=g, dtype=torch.float64) for _ in range(4)]
    a, r, e = 2.5, 1.5, 0.75
    u, c_all, a_only = vb[:3]
    assert torch.allclose(R.cfg_combine(vb[:3], a, r, e), u + a * (a_only - u) + e * (c_all - a_only))
    tu, u, c_all, a_only = vb
    assert torch.allclose(R.cfg_combine(vb, a, r, e), tu + r * (u - tu) + a * (a_only - u) + e * (c_all - a_only))
    assert R.clip_branches(4, 3) == [1, 2, 3] and R.clip_branches(4, 1) == [2] and R.clip_branches(3, 1) == [1]
    # dy/dt = -y: one step of every solver from y0 with the stage states rk_stage hands on, against its explicit formula
    y0, dt = torch.tensor([1.0, -2.0], dtype=torch.float64), 0.1
    for name, tab in sampler.SOLVERS.items():
        G, ks, y = len(tab["b"]), [], y0
        for st in range(G):
            ks.append(-y)
            y = R.rk_stage(y0, ks, st, dt, tab["a"], tab["b"])
        want = {"euler": 1 - dt, "midpoint": 1 - dt + dt ** 2 / 2, "heun2": 1 - dt + dt ** 2 / 2,
                "heun3": 1 - dt + dt ** 2 / 2 - dt ** 3 / 6, "rk4": 1 - dt + dt ** 2 / 2 - dt ** 3 / 6 + dt ** 4 / 24}[name]
        assert torch.allclose(y, y0 * want, rtol=1e-14, atol=0), name


def test_debug_stage_struct_matches_the_header():
    cabi = sys.modules[load_package().__name__ + "._cabi"]
    S = cabi.FmtDebugStage
    fields = [f[0] for f in S._fields_]
    assert (cabi.FMT_STAGE_ROW, cabi.FMT_STAGE_ATTN, cabi.FMT_STAGE_GELU, cabi.FMT_STAGE_COMB) == (0, 1, 2, 3)
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no host C compiler for the offsetof probe")
    with tempfile.TemporaryDirectory() as tmp:
        src, exe = os.path.join(tmp, "probe.c"), os.path.join(tmp, "probe")
        with open(src, "w") as f:
            f.write('#include <stddef.h>\n#include <stdio.h>\n#include "fmt_b200.h"\nint main(void) {\n')
            for fld in fields:
                f.write(f'  printf("%zu ", offsetof(FmtDebugStage, {fld}));\n')
            f.write('  printf("%zu %d %d %d %d\\n", sizeof(FmtDebugStage), FMT_STAGE_ROW, FMT_STAGE_ATTN, FMT_STAGE_GELU, FMT_STAGE_COMB);\n'
                    '  return 0;\n}\n')
        subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", exe, src], check=True)
        got = [int(v) for v in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [getattr(S, f).offset for f in fields] + [C.sizeof(S), 0, 1, 2, 3]


def _stage_desc(cabi, **kw):
    """A descriptor both entry points accept up to the shape checks (non-null pointers that are never dereferenced)."""
    d = cabi.FmtDebugStage(kind=cabi.FMT_STAGE_ROW, chunk_rows=64, n_branches=3, batch=1, n_frames=60, n_prev=10, H=256, heads=4,
                           window=2, mlp_hidden=1024, W=64, n_stages=1, ldt=14 * 256, shift_off=0, scale_off=256)
    for name in ("X", "Pacc", "QKVacc", "Hacc", "Vacc", "A1", "A2", "Hm", "ax", "table", "bias", "pos", "x_state", "kbuf", "ddt"):
        setattr(d, name, 256)
    for k, v in kw.items():
        setattr(d, k, v)
    return d


BAD_STAGES = [
    ("both", dict(kind=4)),
    ("both", dict(H=384)),                                  # no NV instance
    ("both", dict(n_branches=2)),
    ("both", dict(n_prev=60)),                              # no current frame
    ("both", dict(grid=-1)),
    ("both", dict(shift_off=13 * 256 + 4)),                 # a column past the table row
    ("both", dict(pos=None)),                               # mode 0 reads pos
    ("both", dict(kind=1, heads=3)),                        # head_dim 256 / 3
    ("both", dict(kind=1, H=1024, heads=4)),                # head_dim 256
    ("both", dict(kind=2, mlp_hidden=1000)),
    ("both", dict(kind=3, n_stages=2, stage=2)),
    ("both", dict(kind=3, n_stages=5)),
    ("both", dict(kind=3, n_stages=2, kbuf=None)),
    ("flow", dict(chunk_rows=48)),
    ("flow", dict(n_branches=4, batch=9)),                  # 36 chunks of 64 rows > 32
    ("flow", dict(grid=2)),                                 # 3 chunks need 3 CTAs
    ("flow", dict(kind=1, chunk_rows=32, window=33)),       # the band would reach past the neighbouring chunk
    ("window", dict(batch=2)),                              # 360 token rows > 256
    ("window", dict(urow=256)),
]


@pytest.mark.parametrize("which,bad", BAD_STAGES)
def test_stage_entry_points_refuse_bad_shapes_without_a_device(which, bad):
    """The shape checks run before any CUDA call, so they answer on a machine without a GPU too."""
    cabi = sys.modules[load_package().__name__ + "._cabi"]
    L = cabi.load_library()
    for kernel in (("flow", "window") if which == "both" else (which,)):
        fn = getattr(L, f"fmt_debug_{kernel}_stage")
        assert fn(C.byref(_stage_desc(cabi, **bad)), None) == -1, (kernel, bad)
        assert f"fmt_debug_{kernel}_stage" in L.fmt_last_error().decode()
    assert L.fmt_debug_flow_stage(None, None) == -1 and L.fmt_debug_window_stage(None, None) == -1
