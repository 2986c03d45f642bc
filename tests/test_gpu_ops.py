"""The per-op kernels of the sampler step against fp64 references (tests/ops_ref.py), through the C ABI's diagnostic entry points:
the fused GEMM epilogues of the three GEMM kernels, the K-sliced gate epilogue, LayerNorm-modulate and both band-attention
kernels, in every precision mode (B200 only).

Each bound is derived from the arithmetic the kernel does after its inputs, in units of U32 (fp32 unit roundoff), and is tight
enough that a wrong constant, eps, approximation or predicate fails it.  The GEMM operands are small multiples of powers of two
(exact in bf16, with a zero lo part in bf16x3, and every partial sum exact in fp32), so the main loop is exact in every mode and
every kernel, whatever the order of its sums: what differs from the reference is the epilogue alone."""
import ctypes as C
import math
import sys

import pytest
import torch

import ops_ref as R
from __graft_entry__ import load_package

pytestmark = pytest.mark.gpu

U = R.U32
BF16, FP32, BF16X3 = 0, 1, 2
MODES = {"bf16": BF16, "fp32": FP32, "bf16x3": BF16X3}


@pytest.fixture(scope="module")
def lib():
    cabi = sys.modules[load_package().__name__ + "._cabi"]
    return cabi.load_library(), cabi


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return None if t is None else t.data_ptr()


# ------------------------------------------------------------------------------------------------ activation / table types
def _new_act(mode, rows, ld, out_f32=False):
    """A NaN-filled (rows, ld) buffer of the mode's activation type (fp32 if out_f32)."""
    if out_f32 or mode == FP32:
        return torch.full((rows, ld), float("nan"), device="cuda")
    if mode == BF16:
        return torch.full((rows, ld), float("nan"), device="cuda", dtype=torch.bfloat16)
    return torch.full((rows, 2 * ld), float("nan"), device="cuda", dtype=torch.bfloat16)    # bf16x3 pairs: 4 bytes per element


def _decode(mode, buf, ld, out_f32=False):
    if out_f32 or mode == FP32 or mode == BF16:
        return buf.double()
    return R.decode_pairs(buf, ld)


def _out_rounding(mode, out_f32=False):
    """Relative error of storing an fp32 value in the output type: bf16 rounding, the pair's representation error, or none."""
    if out_f32 or mode == FP32:
        return 0.0
    return R.BF16_HALF_ULP if mode == BF16 else R.PAIR_REPR


def _table(mode, t):
    """An AdaLN table / QKV tensor in the mode's table type (bf16 in bf16 mode, else fp32) and the values the kernel reads."""
    if mode == BF16:
        t = t.to(torch.bfloat16)
    else:
        t = t.float()
    return t, t.double()


# ------------------------------------------------------------------------------------------------ GEMM epilogues
def _exact_operands(M, N, K, g):
    """A = i / 8, W = j / 2^e with |i|, |j| <= 4: exact in bf16, every product a multiple of 2^-(3+e) and every partial sum below
    K * 2^(1-e) <= 2^16, so fp32 holds each sum exactly.  e spreads acc = A . W^T over about N(0, 1.5^2) for every K."""
    e = max(0, round(math.log2(0.55 * math.sqrt(K))))
    A = torch.randint(-4, 5, (M, K), device="cuda", generator=g).float() / 8
    W = torch.randint(-4, 5, (N, K), device="cuda", generator=g).float() / 2 ** e
    return A, W


def _run_gemm(L, cabi, mode, kind, M, N, K, block_n=0, ksplit=1, out_f32=0, urow=False, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed * 1000003 + M * 7919 + N * 31 + K + 17 * kind + 3 * block_n)
    A, W = _exact_operands(M, N, K, g)
    bias = torch.randn(N, device="cuda", generator=g)
    acc = A.double() @ W.double().t()
    ldo = (N // 64 + 1) * 64                      # guard columns [N, ldo) (a multiple of 64: pair outputs need it)
    GR = 3                                        # guard rows below M
    d = cabi.FmtDebugGemm(mode=mode, kind=kind, M=M, N=N, K=K, block_n=block_n, ksplit=ksplit, ldo=ldo, out_f32=out_f32)
    d.A, d.W, d.bias = A.data_ptr(), W.data_ptr(), bias.data_ptr()
    keep = {}
    v = acc + bias.double()
    if kind == R.POS:
        frames = 60                               # M is not a multiple of it: rows of the next sequence start mid-tile
        pos = torch.randn(frames, N, device="cuda", generator=g)
        d.pos, d.frames, keep["pos"] = pos.data_ptr(), frames, pos
        ref = R.gemm_epilogue(kind, acc, bias.double(), pos=pos.double())
        tol = 2 * U * (v.abs() + ref.abs())      # two fp32 additions: + bias, + pos
    elif kind == R.GATE_RES:
        # the table of the sampler's gate: rows of 6H per block for 2 blocks + 2H of the decoder, gate_mlp of block 1
        H = N
        ldg, gate_off = 6 * H * 2 + 2 * H, 6 * H + 5 * H
        n_rows = max(1, M // 3) if urow else M
        tab, tab64 = _table(mode, torch.randn(n_rows, ldg, device="cuda", generator=g))
        ur = torch.randint(0, n_rows, (M,), device="cuda", generator=g, dtype=torch.int32) if urow else None
        gate = R.table_rows(tab64, ur, M)[:, gate_off:gate_off + N]
        buf = torch.full((M + GR, ldo), float("nan"), device="cuda")
        buf[:M, :N] = torch.randn(M, N, device="cuda", generator=g) * 4
        x0 = buf[:M, :N].double()
        d.gate, d.urow, d.ldg, d.gate_off, keep["tab"], keep["ur"] = tab.data_ptr(), _ptr(ur), ldg, gate_off, tab, ur
        ref = R.gemm_epilogue(kind, acc, bias.double(), x=x0, gate=gate)
        if ksplit == 1:
            tol = 2 * U * (gate.abs() * v.abs() + ref.abs())           # fmaf(gate, fl(acc + bias), x): two roundings
        else:
            # x += gate * (partial + bias) and x += gate * partial in either order through fp32 RED: each slice's bias add,
            # product and RED round once; |partial_1| + |partial_2| <= sum_k |a_k w_k|
            S = A.double().abs() @ W.double().abs().t()
            tol = 4 * U * (gate.abs() * (S + bias.double().abs()) + x0.abs() + ref.abs())
    else:
        ref = R.gemm_epilogue(kind, acc, bias.double())
        if kind == R.GELU:
            # fl(acc + bias) moves GELU by <= 1.13 U |v|; the fp32 formula (cube, tanhf to 2 ulp, 1 + t, products) by < 6 U (|v| + |y|).
            # bf16 mode evaluates tanh with tanh.approx.f32, 2^-10.99 relative on t: 0.5 |v| |t| 2^-10.99 on y
            tol = 8 * U * (v.abs() + ref.abs())
            if mode == BF16:
                t = torch.tanh(math.sqrt(2.0 / math.pi) * (v + 0.044715 * v ** 3))
                tol = tol + 0.5 * v.abs() * t.abs() * R.TANH_APPROX
        else:
            tol = U * v.abs()                                            # fl(acc + bias)
    if kind != R.GATE_RES:
        buf = _new_act(mode, M + GR, ldo, out_f32)
        tol = tol + _out_rounding(mode, out_f32) * ref.abs()
    d.out = buf.data_ptr()
    cabi.check(L.fmt_debug_gemm_epilogue(C.byref(d), _stream()), "fmt_debug_gemm_epilogue")
    torch.cuda.synchronize()
    out = _decode(mode, buf, ldo, out_f32 or kind == R.GATE_RES)
    return out, ref, tol, M, N


def _check(out, ref, tol, M, N):
    got = out[:M, :N]
    err = (got - ref).abs()
    assert torch.isfinite(got).all(), "non-finite outputs"
    worst = (err / tol.clamp_min(1e-30)).max().item()
    assert (err <= tol).all(), f"max |err| {err.max().item():.3e}, {worst:.2f} x its bound"
    # guard rows below M and guard columns [N, ldo) keep their NaN fill: no store outside the output
    assert torch.isnan(out[M:]).all() and torch.isnan(out[:M, N:]).all(), "a store landed outside the (M, N) output"


# (mode, block_n): 0 = the sampler's choice; 64 / 128 / 256 single-CTA tcgen05 kernel, 512 / 1024 CTA-pair kernel; fp32 = SIMT only
GEMM_VARIANTS = [("bf16", b) for b in (0, 64, 128, 256, 512, 1024)] + [("bf16x3", b) for b in (0, 64, 128, 256, 512, 1024)] + [("fp32", 0)]
# (kind, out_f32, urow): the activation-typed store of the qkv / fc1 GEMMs, the fp32 store of the tables / decoder, GELU of fc1,
# + pos_embed of the x-embedder, x += gate * (.) of proj / fc2 with and without the condition-row indirection
EPILOGUES = [("store", 0, False), ("store_f32", 1, False), ("gelu", 0, False), ("pos", 1, False), ("gate", 1, False), ("gate_urow", 1, True)]
KINDS = {"store": R.STORE, "store_f32": R.STORE, "gelu": R.GELU, "pos": R.POS, "gate": R.GATE_RES, "gate_urow": R.GATE_RES}
# one clip (180 rows); a ragged tile with N % 256 != 0; 32 clips plus a ragged pair tile; N = 96 below one 128 / 256 tile
SHAPES = [(180, 96, 64), (333, 1056, 1088), (5820, 1056, 1024), (333, 96, 4096)]


@pytest.mark.parametrize("M,N,K", SHAPES)
@pytest.mark.parametrize("epilogue", [e[0] for e in EPILOGUES])
@pytest.mark.parametrize("mode,block_n", GEMM_VARIANTS)
def test_gemm_epilogue_matches_fp64(lib, mode, block_n, epilogue, M, N, K):
    L, cabi = lib
    _, out_f32, urow = next(e for e in EPILOGUES if e[0] == epilogue)
    _check(*_run_gemm(L, cabi, MODES[mode], KINDS[epilogue], M, N, K, block_n, out_f32=out_f32, urow=urow))


@pytest.mark.parametrize("urow", [False, True])
@pytest.mark.parametrize("M", [333, 5820])
@pytest.mark.parametrize("K", [1088, 4096])           # 17 K blocks: uneven slices of 8 and 9; 64 blocks: 32 and 32
@pytest.mark.parametrize("block_n", [512, 1024])
def test_k_sliced_gate_epilogue_matches_fp64(lib, block_n, K, M, urow):
    """The CTA-pair kernel with 2 K slices per tile: both slices' partial sums meet in x through fp32 RED, the bias once."""
    L, cabi = lib
    _check(*_run_gemm(L, cabi, BF16, R.GATE_RES, M, 1056, K, block_n, ksplit=2, out_f32=1, urow=urow))


@pytest.mark.parametrize("kind,K,block_n,mode", [(R.GATE_RES, 64, 512, BF16),      # 1 K block, 2 slices: one would be empty
                                                 (R.GATE_RES, 64, 1024, BF16),
                                                 (R.GELU, 1024, 512, BF16),        # slices only add into x
                                                 (R.GATE_RES, 1024, 256, BF16),    # the single-CTA kernel is never sliced
                                                 (R.GATE_RES, 1024, 0, FP32)])
def test_k_slicing_rejects_what_it_cannot_run(lib, kind, K, block_n, mode):
    L, cabi = lib
    M, N = 300, 256
    A = torch.zeros(M, K, device="cuda")
    W = torch.zeros(N, K, device="cuda")
    tab = torch.zeros(M, N, device="cuda", dtype=torch.bfloat16 if mode == BF16 else torch.float32)
    out = torch.zeros(M, N, device="cuda")
    d = cabi.FmtDebugGemm(mode=mode, kind=kind, M=M, N=N, K=K, block_n=block_n, ksplit=2, ldo=N, out_f32=1)
    d.A, d.W, d.out, d.gate, d.ldg = A.data_ptr(), W.data_ptr(), out.data_ptr(), tab.data_ptr(), N
    with pytest.raises(ValueError):
        cabi.check(L.fmt_debug_gemm_epilogue(C.byref(d), _stream()), "fmt_debug_gemm_epilogue")
    torch.cuda.synchronize()
    assert (out == 0).all()


# ------------------------------------------------------------------------------------------------ LayerNorm-modulate
def _ln_rows(rows, H, g):
    X = torch.randn(rows, H, device="cuda", generator=g) * 2 + 0.5
    X[0] = 100 + 0.1 * torch.randn(H, device="cuda", generator=g)    # large mean, small spread: a one-pass variance is ~6 % off
    X[1] = -100 + 0.1 * torch.randn(H, device="cuda", generator=g)
    X[2] = 1e-3 * torch.randn(H, device="cuda", generator=g)         # variance ~1e-6 = eps: eps 1e-5 would change rstd 2.3x
    X[3] = 0.7                                                       # constant row: variance 0, rstd = eps^-1/2
    X[rows - 1] = 1e-3 * torch.randn(H, device="cuda", generator=g) + 3.0
    return X


@pytest.mark.parametrize("urow", [False, True])
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("H", [128, 256, 512, 1024])
def test_lnmod_matches_fp64(lib, H, mode, urow):
    L, cabi = lib
    m = MODES[mode]
    rows = 4 * 37 + 3                                # not a multiple of the 4 rows (warps) of a block
    g = torch.Generator(device="cuda").manual_seed(H + 7 * m + int(urow))
    X = _ln_rows(rows, H, g)
    ldt = 6 * H * 2 + 2 * H                          # the sampler's table row; block 1's shift_mlp / scale_mlp
    shift_off, scale_off = 6 * H + 3 * H, 6 * H + 4 * H
    n_rows = rows // 3 if urow else rows
    tab, tab64 = _table(m, torch.randn(n_rows, ldt, device="cuda", generator=g) * 0.5)
    ur = torch.randint(0, n_rows, (rows,), device="cuda", generator=g, dtype=torch.int32) if urow else None
    out = _new_act(m, rows + 1, H)
    cabi.check(L.fmt_debug_lnmod(m, X.data_ptr(), rows, H, tab.data_ptr(), _ptr(ur), ldt, shift_off, scale_off, out.data_ptr(), _stream()),
               "fmt_debug_lnmod")
    torch.cuda.synchronize()
    got = _decode(m, out, H)
    X64 = X.double()
    ref = R.lnmod(X64, tab64, ur, shift_off, scale_off)
    # mean: a per-lane sum of H/128 float4 then 5 shuffle levels, (H/128 + 7) roundings deep: |d mean| <= c U mean|x|, which moves
    # z = (x - mean) rstd by c U mean|x| rstd.  Two-pass variance, rsqrtf and (x - mean) * rstd: relative c U on z.
    c = 2 * (H // 128 + 8)
    var = X64.var(dim=1, unbiased=False, keepdim=True)
    rstd = (var + 1e-6).rsqrt()
    z = (X64 - X64.mean(dim=1, keepdim=True)) * rstd
    sc = R.table_rows(tab64, ur, rows)[:, scale_off:scale_off + H]
    err_z = c * U * (X64.abs().mean(dim=1, keepdim=True) * rstd + z.abs())
    # fmaf(z, fl(1 + scale), shift): two more roundings, then the output type's
    tol = (1 + sc).abs() * (err_z + U * z.abs()) + U * ref.abs() + _out_rounding(m) * ref.abs()
    err = (got[:rows] - ref).abs()
    assert torch.isfinite(got[:rows]).all()
    assert (err <= tol).all(), f"max |err| {err.max().item():.3e} in row {int(err.max(dim=1).values.argmax())}"
    assert torch.isnan(got[rows:]).all()


def test_lnmod_rejects_unsupported_widths(lib):
    L, cabi = lib
    X = torch.zeros(4, 384, device="cuda")
    out = torch.zeros(4, 384, device="cuda")
    with pytest.raises(ValueError):
        cabi.check(L.fmt_debug_lnmod(FP32, X.data_ptr(), 4, 384, X.data_ptr(), None, 384, 0, 0, out.data_ptr(), _stream()), "lnmod")


# ------------------------------------------------------------------------------------------------ band attention
WARP, TILE = 1, 2


def _variants(mode, N, hd):
    tile = mode == BF16 and hd in (64, 128) and 2 * N * hd * 2 <= 48 * 1024
    return [WARP, TILE] if tile else [WARP]


def _bits(t):
    return t.view(torch.int16 if t.element_size() == 2 else torch.int32)


def _attention(L, cabi, mode, qkv, n_seq, N, heads, hd, window, variant):
    out = _new_act(mode, n_seq * N + 1, heads * hd)
    rc = L.fmt_debug_band_attention(mode, qkv.data_ptr(), n_seq, N, heads, hd, window, out.data_ptr(), variant, _stream())
    cabi.check(rc, "fmt_debug_band_attention")
    torch.cuda.synchronize()
    return out


def _attention_check(mode, out, ref, qkv64, heads, window):
    n_seq, N, C3 = qkv64.shape
    hd = C3 // (3 * heads)
    Hd = heads * hd
    got = _decode(mode, out, Hd)
    assert torch.isnan(got[n_seq * N:]).all()
    got = got[:n_seq * N].reshape(n_seq, N, Hd)
    q, k, v = qkv64.reshape(n_seq, N, 3, heads, hd).permute(2, 0, 3, 1, 4)
    # scores: fp32 dot products <= 32 roundings deep (per-lane FMAs + shuffle tree; the tile kernel also rounds q * scale):
    # |d s| <= 32 U scale sum_d |q_d k_d|.  Softmax moves o by <= 2 max|v| max|d s| (d o / d s_j = p_j (v_j - o)); the
    # exponentials (expf / __expf of arguments <= 0) and the online sums add (16 + 4 (2w + 1)) U max|v|.
    blocked = R.O.band_mask(N, window, device=qkv64.device)
    ds = 32 * U * hd ** -0.5 * (q.abs() @ k.abs().transpose(-2, -1)).masked_fill(blocked, 0).amax(dim=-1, keepdim=True)
    vrow = v.abs().amax(dim=-1)[:, :, None, :].expand(-1, -1, N, -1)                        # max |v_j| for (row i, key j)
    vmax = vrow.masked_fill(blocked, 0).amax(dim=-1, keepdim=True)                             # (n_seq, heads, N, 1)
    tol_h = vmax * (2 * ds + (16 + 4 * (2 * window + 1)) * U)                                # (n_seq, heads, N, 1)
    tol = tol_h.expand(-1, -1, -1, hd).transpose(1, 2).reshape(n_seq, N, Hd) + _out_rounding(mode) * ref.abs()
    err = (got - ref).abs()
    assert torch.isfinite(got).all(), "non-finite outputs"
    assert (err <= tol).all(), f"max |err| {err.max().item():.3e}, {(err / tol).max().item():.2f} x its bound"


@pytest.mark.parametrize("window", [0, 1, 2, 3, 4, 7])
@pytest.mark.parametrize("N", [1, 3, 5, 60, 61, 96])
@pytest.mark.parametrize("hd", [32, 64, 128])
@pytest.mark.parametrize("mode", list(MODES))
def test_band_attention_matches_fp64(lib, mode, hd, N, window):
    """Both kernels where they run: bands wider than one 5-key batch (window >= 3) merge batches online; rows whose band ends
    early skip batches (tile kernel); N = 61 leaves a partial group of 4 rows; hd 128 at N = 96 fills the tile kernel's 48 KB."""
    L, cabi = lib
    m = MODES[mode]
    heads, n_seq = 2, 3
    g = torch.Generator(device="cuda").manual_seed(hd * 131 + N * 7 + window + 1000 * m)
    qkv, qkv64 = _table(m, torch.randn(n_seq, N, 3 * heads * hd, device="cuda", generator=g) * 1.5)
    ref = R.band_attention(qkv64, heads, window)
    for variant in _variants(m, N, hd):
        _attention_check(m, _attention(L, cabi, m, qkv, n_seq, N, heads, hd, window, variant), ref, qkv64, heads, window)


@pytest.mark.parametrize("hd", [64, 128])
@pytest.mark.parametrize("mode", list(MODES))
def test_band_attention_is_stable_at_scores_of_100(lib, mode, hd):
    """Scores of +-100 after scaling: exp(100) overflows fp32, only the running-max subtraction keeps the softmax finite."""
    L, cabi = lib
    m = MODES[mode]
    heads, n_seq, N, window = 2, 3, 61, 7
    g = torch.Generator(device="cuda").manual_seed(hd + 10 * m)
    x = torch.randn(n_seq, N, 3, heads, hd, device="cuda", generator=g) * 0.5
    sign = torch.randint(0, 2, (n_seq, N, heads), device="cuda", generator=g).float() * 2 - 1
    x[:, :, 0, :, 0] = 16.0                                        # q_0
    x[:, :, 1, :, 0] = sign * 100.0 * math.sqrt(hd) / 16.0           # k_0: q_0 k_0 / sqrt(hd) = +-100
    qkv, qkv64 = _table(m, x.reshape(n_seq, N, 3 * heads * hd))
    assert (qkv64.reshape(n_seq, N, 3, heads, hd)[:, :, 1, :, 0].abs() * 16 / math.sqrt(hd)).min() > 99    # after bf16 rounding too
    ref = R.band_attention(qkv64, heads, window)
    for variant in _variants(m, N, hd):
        _attention_check(m, _attention(L, cabi, m, qkv, n_seq, N, heads, hd, window, variant), ref, qkv64, heads, window)


@pytest.mark.parametrize("mode", list(MODES))
def test_band_attention_selects_the_sampler_kernel(lib, mode):
    """Variant 0 is the sampler's choice: the tile kernel in bf16 once sequences x heads >= 2 x SMs, else the warp kernel."""
    L, cabi = lib
    m = MODES[mode]
    heads, hd, N, window = 8, 64, 60, 2
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    hi = -(-2 * sms // heads)
    g = torch.Generator(device="cuda").manual_seed(5)
    for n_seq, want in ((hi, TILE if m == BF16 else WARP), (hi - 1, WARP)):
        qkv, _ = _table(m, torch.randn(n_seq, N, 3 * heads * hd, device="cuda", generator=g))
        auto = _attention(L, cabi, m, qkv, n_seq, N, heads, hd, window, 0)
        forced = {v: _attention(L, cabi, m, qkv, n_seq, N, heads, hd, window, v) for v in _variants(m, N, hd)}
        assert torch.equal(_bits(auto), _bits(forced[want]))
        if len(forced) == 2:                        # the two kernels round differently: the comparison above tells them apart
            assert not torch.equal(_bits(forced[WARP]), _bits(forced[TILE]))


@pytest.mark.parametrize("mode,N,hd", [(FP32, 60, 64), (BF16X3, 60, 64), (BF16, 60, 32), (BF16, 97, 128)])
def test_band_attention_rejects_an_impossible_tile_kernel(lib, mode, N, hd):
    """The tile kernel exists for bf16 with head_dim 64 or 128 and K / V of a head within 48 KB (N = 97 at hd 128 is 48.5 KB)."""
    L, cabi = lib
    heads = 2
    qkv, _ = _table(mode, torch.zeros(1, N, 3 * heads * hd, device="cuda"))
    out = _new_act(mode, N, heads * hd)
    assert L.fmt_debug_band_attention(mode, qkv.data_ptr(), 1, N, heads, hd, 2, out.data_ptr(), TILE, _stream()) == -1
    torch.cuda.synchronize()
    assert torch.isnan(out.float()).all()
