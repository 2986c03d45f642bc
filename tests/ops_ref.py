"""fp64 references of the per-op kernels of the sampler step (fused GEMM epilogues, LayerNorm-modulate, band attention) and
decoders of the kernels' output types.  Each reference is the reference model's formula (oracle/fmt_oracle.py, FMT.py) evaluated
in fp64 on the operands the kernel saw."""
import math

import torch
import torch.nn.functional as F

from oracle import fmt_oracle as O

U32 = 2.0 ** -24                 # unit roundoff of fp32
BF16_HALF_ULP = 2.0 ** -8        # unit roundoff of bf16 (8 significant bits): half an ulp, relative
PAIR_REPR = 2.0 ** -16           # x - (hi + lo) of a bf16x3 pair: hi = bf16(x) leaves 2^-8 |x|, lo = bf16(x - hi) 2^-8 of that
TANH_APPROX = 2.0 ** -10.99      # tanh.approx.f32: maximum relative error (PTX ISA)

STORE, GELU, POS, GATE_RES = 0, 1, 2, 3


def gelu_tanh(x):
    """nn.GELU(approximate="tanh") (FMT.py:161), the formula of gelu_tanh / gelu_tanh_approx in gemm.cuh."""
    return 0.5 * x * (1.0 + torch.tanh(math.sqrt(2.0 / math.pi) * (x + 0.044715 * x ** 3)))


def gemm_epilogue(kind, acc, bias=None, pos=None, x=None, gate=None):
    """The epilogue applied to acc = A . W^T (M, N): bias, then GELU, + pos[m % frames] or x + gate * (.) (FMT.py:171-176).
    pos is (frames, N); gate holds the gate row of every output row (M, N)."""
    v = acc if bias is None else acc + bias
    if kind == GELU:
        return gelu_tanh(v)
    if kind == POS:
        rows = torch.arange(v.shape[0], device=v.device) % pos.shape[0]
        return v + pos[rows]
    if kind == GATE_RES:
        return x + gate * v
    return v


def table_rows(table, urow, rows):
    """Row r of an AdaLN table as the kernels address it: table[urow[r]] (urow None: table[r])."""
    return table[:rows] if urow is None else table[urow.long()]


def lnmod(X, table, urow, shift_off, scale_off):
    """LayerNorm (eps 1e-6, no affine) + modulate, FMT.py:157,168-169: LN(x) * (1 + scale) + shift, with shift and scale the
    H columns at shift_off / scale_off of the row's table row (table (U, ldt))."""
    H = X.shape[-1]
    t = table_rows(table, urow, X.shape[0])
    return F.layer_norm(X, (H,), eps=1e-6) * (1 + t[:, scale_off:scale_off + H]) + t[:, shift_off:shift_off + H]


def band_attention(qkv, heads, window):
    """softmax(masked q k^T hd^-1/2) v of every (sequence, head), FMT.py:15-19,69-88.  qkv (n_seq, N, 3 * heads * hd), columns
    [q | k | v] head-major; returns (n_seq, N, heads * hd)."""
    n_seq, N, C3 = qkv.shape
    hd = C3 // (3 * heads)
    q, k, v = qkv.reshape(n_seq, N, 3, heads, hd).permute(2, 0, 3, 1, 4)
    s = (q @ k.transpose(-2, -1)) * hd ** -0.5
    s = s.masked_fill(O.band_mask(N, window, device=qkv.device), float("-inf"))
    return (torch.softmax(s, dim=-1) @ v).transpose(1, 2).reshape(n_seq, N, heads * hd)


def decode_pairs(buf, ld):
    """A bf16x3 pair matrix (rows of 2 * ld bf16: every 64-column block of hi followed by the same block of lo) -> hi + lo, fp64."""
    rows = buf.shape[0]
    p = buf.view(torch.bfloat16).reshape(rows, ld // 64, 2, 64).double()
    return (p[:, :, 0] + p[:, :, 1]).reshape(rows, ld)
