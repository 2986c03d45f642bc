"""fp64 references of the per-op kernels of the sampler step (fused GEMM epilogues, LayerNorm-modulate, band attention) and of
the persistent window kernels' row-wise stages (CFG combine, Runge-Kutta bookkeeping), and decoders of the kernels' output types
and operand layouts.  Each reference is the reference model's formula (oracle/fmt_oracle.py, FMT.py) evaluated
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


def clip_branches(s_nb, nb):
    """Plan branches a clip reads when it combines nb of the plan's s_nb CFG branches: all of them; for nb = 1 the conditional
    branch ("all": index 1 of [uncond | all | audio-only], 2 of [truly-uncond | uncond | all | audio-only]); for 3 of 4 the last
    three, which carry the null masks of a 3-branch plan."""
    if nb == s_nb:
        return list(range(nb))
    if nb == 1:
        return [s_nb - 2]
    return [1, 2, 3]


def cfg_combine(vb, a, r, e):
    """CFG combine of forward_with_cfv (FMT.py:375-379,396-399; oracle forward_with_cfv) over the list of branch velocities vb."""
    if len(vb) == 1:
        return vb[0]
    if len(vb) == 3:
        u, c_all, a_only = vb
        return u + a * (a_only - u) + e * (c_all - a_only)
    tu, u, c_all, a_only = vb
    return tu + r * (u - tu) + a * (a_only - u) + e * (c_all - a_only)


def rk_stage(y0, k, g, dt, a, b):
    """Explicit Runge-Kutta bookkeeping once stage g's velocity k[g] is known (torchdiffeq fixed grid, Butcher tableau a / b of
    sampler.SOLVERS): the state stage g + 1 evaluates, y0 + dt * sum_{j <= g} a[g + 1][j] k_j, or after the last stage the
    step's result y0 + dt * sum_j b_j k_j.  Euler is a = [[0]], b = [1]."""
    c = b if g == len(b) - 1 else a[g + 1]
    acc = 0.0
    for j in range(g + 1):
        acc = acc + c[j] * k[j]
    return y0 + dt * acc


def _unswizzle(t):
    """Tiles (..., rows, 64) whose 16-byte chunk j of row r is stored at chunk j ^ (r % 8) (the 128-byte swizzle of a SW128
    K-major operand tile) -> the logical (..., rows, 64)."""
    rows = t.shape[-2]
    r = torch.arange(rows, device=t.device).view(rows, 1)
    p = torch.arange(64, device=t.device).view(1, 64)
    src = (((p >> 3) ^ (r & 7)) << 3) | (p & 7)
    return torch.gather(t, -1, src.expand(t.shape))


def flow_tiled_decode(buf, n_chunks, CH, cols):
    """Operand of the dataflow window kernel, [chunk][K block][CH][64] (flow_tiled_off) -> (n_chunks * CH, cols), padded rows."""
    t = _unswizzle(buf.reshape(n_chunks, cols // 64, CH, 64))
    return t.permute(0, 2, 1, 3).reshape(n_chunks * CH, cols)


def win_tiled_decode(buf, Rp, cols):
    """Operand of the barrier-stepped window kernel, [K block][Rp][64] (win_tiled_off) -> (Rp, cols)."""
    t = _unswizzle(buf.reshape(cols // 64, Rp, 64))
    return t.permute(1, 0, 2).reshape(Rp, cols)
