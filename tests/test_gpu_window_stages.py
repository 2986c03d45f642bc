"""The row-wise stages of the two persistent window kernels against fp64 references (tests/ops_ref.py), through
fmt_debug_flow_stage (dataflow kernel, flow.cuh) and fmt_debug_window_stage (barrier-stepped kernel, window.cuh).  Both run the
kernels' own stage functions in the production thread layout and tables, one stage kind over every chunk / row (B200 only).

Neither kernel calls the per-op kernels of tests/test_gpu_ops.py: each has its own residual update, LayerNorm-modulate, band
attention, GELU, CFG combine and ODE update, which the end-to-end comparisons (2e-2) cannot resolve.  Each stage here runs on
inputs the test builds and is compared with fp64 applied to those same inputs.  Each bound is derived from the arithmetic the
stage does after its inputs, in units of U32, and reuses test_gpu_ops.py's bound where the arithmetic is the same.  Every
buffer a stage must not touch starts NaN-filled and must still be NaN afterwards; every accumulator it consumes must read back
exactly 0.  The kernels' GEMM engines are not covered here."""
import ctypes as C
import math
import sys

import pytest
import torch

import ops_ref as R
from __graft_entry__ import load_package

pytestmark = pytest.mark.gpu

U = R.U32
B8 = R.BF16_HALF_ULP
FLOW, WIN = "flow", "window"
ROW, ATTN, GELU, COMB = 0, 1, 2, 3


@pytest.fixture(scope="module")
def lib():
    cabi = sys.modules[load_package().__name__ + "._cabi"]
    return cabi.load_library(), cabi


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _nan(*shape, dtype=torch.float32):
    return torch.full(shape, float("nan"), device="cuda", dtype=dtype)


class Geo:
    """Token rows of n_branches x batch sequences of N frames (P context frames) as each kernel lays them out: the flow kernel in
    chunks of CH rows padded per sequence to NPs rows, the window kernel unpadded (operands padded to Rp rows)."""

    def __init__(self, kernel, nb, B, N, P=10, CH=64):
        self.kernel, self.nb, self.B, self.N, self.P, self.CH = kernel, nb, B, N, P, CH
        self.seqs = nb * B
        if kernel == FLOW:
            nsub = -(-N // CH)
            self.NPs, self.n_chunks = nsub * CH, self.seqs * nsub
            self.rows = self.n_chunks * CH
        else:
            self.NPs = N
            self.rows = self.seqs * N
            self.Rp = -(-self.rows // 64) * 64
        self.prow = (torch.arange(self.seqs, device="cuda")[:, None] * self.NPs + torch.arange(N, device="cuda")[None]).reshape(-1)
        self.valid = torch.zeros(self.rows, dtype=torch.bool, device="cuda")
        self.valid[self.prow] = True

    def desc(self, cabi, kind, grid=0, **kw):
        d = cabi.FmtDebugStage(kind=kind, grid=grid, chunk_rows=self.CH if self.kernel == FLOW else 0, n_branches=self.nb, batch=self.B,
                               n_frames=self.N, n_prev=self.P, H=128, heads=2, n_stages=1)
        for k, v in kw.items():
            setattr(d, k, v)
        return d

    def operand(self, cols):
        """A NaN-filled bf16 operand of `cols` columns in the kernel's tiled layout."""
        n = self.n_chunks * self.CH if self.kernel == FLOW else self.Rp
        return _nan(n * cols, dtype=torch.bfloat16)

    def decode(self, buf, cols):
        """Tiled operand -> (padded rows, cols) fp64, and its rows no token row maps to (must keep their NaN fill)."""
        if self.kernel == FLOW:
            full = R.flow_tiled_decode(buf, self.n_chunks, self.CH, cols).double()
            return full, full[~self.valid]
        full = R.win_tiled_decode(buf, self.Rp, cols).double()
        return full[:self.rows], full[self.rows:]

    def padded(self, x, fill=float("nan")):
        """(seqs * N, cols) token rows -> (rows, cols) in the kernel's row layout, padding rows NaN."""
        out = torch.full((self.rows, x.shape[1]), fill, device="cuda", dtype=x.dtype)
        out[self.prow] = x
        return out


def _run(L, cabi, geo, d):
    fn = L.fmt_debug_flow_stage if geo.kernel == FLOW else L.fmt_debug_window_stage
    cabi.check(fn(C.byref(d), _stream()), "fmt_debug_%s_stage" % geo.kernel)
    torch.cuda.synchronize()


def _assert_within(got, ref, tol, what):
    err = (got - ref).abs()
    assert torch.isfinite(got).all(), f"{what}: non-finite values"
    assert (err <= tol).all(), f"{what}: max |err| {err.max().item():.3e}, {(err / tol.clamp_min(1e-30)).max().item():.2f} x its bound"


def _bf16_tol(ref, tol):
    """bf16(y) for an fp32 y within tol of ref: |bf16(y) - y| <= 2^-8 |y| <= 2^-8 (|ref| + tol)."""
    return tol + B8 * (ref.abs() + tol)


# ------------------------------------------------------------------------------------------------ ROW
def _hard_rows(n, H, g):
    """Target residual rows as hard as test_gpu_ops._ln_rows: mean +-100 with spread 0.1, variance ~eps, a constant row."""
    X = torch.randn(n, H, device="cuda", generator=g) * 2 + 0.5
    X[0] = 100 + 0.1 * torch.randn(H, device="cuda", generator=g)
    X[1] = -100 + 0.1 * torch.randn(H, device="cuda", generator=g)
    X[2] = 1e-3 * torch.randn(H, device="cuda", generator=g)
    X[3] = 0.7
    X[n - 1] = 1e-3 * torch.randn(H, device="cuda", generator=g) + 3.0     # the ragged last chunk of the last sequence
    return X


# (kernel, rows per chunk, frames): 60 and 61 frames leave a ragged last chunk of 28 / 29 rows (32-row chunks) or 60 / 61 (64)
ROW_GEOS = [(FLOW, 64, 60), (FLOW, 32, 61), (WIN, 0, 60), (WIN, 0, 61)]
# the stage after the x-embedder (mode 0, block 0's msa modulation), after proj (gate_msa, mlp modulation; the window kernel
# also zeroes the QKV accumulator) and after fc2 (gate_mlp, then the decoder's shift / scale); table rows of 2 blocks + decoder
ROW_STAGES = {"x_emb": (0, 0, 0, 1), "proj": (1, 8, 9, 10), "fc2": (1, 11, 12, 13)}     # mode, gate / shift / scale column in units of H


def _row_case(L, cabi, kernel, CH, N, H, stage, urow, grid=0, seed=0):
    geo = Geo(kernel, 3, 1, N, CH=CH)
    mode, gq, sq, cq = ROW_STAGES[stage]
    g = torch.Generator(device="cuda").manual_seed(H * 7 + N + CH + 100 * mode + gq + int(urow) + 1000 * seed)
    T, ldt = geo.seqs * N, 14 * H
    n_tab = T // 3 if urow else T
    tab = (torch.randn(n_tab, ldt, device="cuda", generator=g) * 0.5).to(torch.bfloat16)
    ur = torch.randint(0, n_tab, (T,), device="cuda", generator=g, dtype=torch.int32) if urow else None
    t64 = R.table_rows(tab.double(), ur, T)
    acc = torch.randn(T, H, device="cuda", generator=g)
    bias = torch.randn(H, device="cuda", generator=g)
    target = _hard_rows(T, H, g)
    pos = torch.randn(N, H, device="cuda", generator=g)
    frame = torch.arange(T, device="cuda") % N
    if mode == 0:
        acc = target - bias - pos[frame]
        X0 = _nan(T, H)
    else:
        gate = t64[:, gq * H:(gq + 1) * H].float()
        X0 = target - gate * (acc + bias)
    X, Pacc = geo.padded(X0), geo.padded(acc)
    QKV = _nan(2 * geo.rows, 3 * H)
    A1 = geo.operand(H)
    zero_qkv = int(kernel == WIN and stage == "proj")
    d = geo.desc(cabi, ROW, grid, H=H, heads=H // 64, row_mode=mode, zero_qkv=zero_qkv, ldt=ldt, gate_off=gq * H, shift_off=sq * H,
                 scale_off=cq * H)
    d.X, d.Pacc, d.QKVacc, d.A1, d.table, d.bias, d.pos = X.data_ptr(), Pacc.data_ptr(), QKV.data_ptr(), A1.data_ptr(), tab.data_ptr(), \
        bias.data_ptr(), pos.data_ptr()
    d.urow = None if ur is None else ur.data_ptr()
    _run(L, cabi, geo, d)

    a64, b64, X064 = acc.double(), bias.double(), X0.double()
    if mode == 0:
        p64 = pos.double()[frame]
        x_ref = a64 + b64 + p64
        e_x = 2 * U * (a64.abs() + b64.abs() + p64.abs())                 # (acc + bias) + pos: two fp32 additions
    else:
        gate64 = t64[:, gq * H:(gq + 1) * H]
        x_ref = X064 + gate64 * (a64 + b64)
        e_x = 2 * U * (gate64.abs() * (a64.abs() + b64.abs()) + X064.abs())  # fmaf(gate, fl(acc + bias), x): two roundings
    _assert_within(X.double()[geo.prow], x_ref, e_x, "X")
    assert torch.isnan(X[~geo.valid]).all(), "X: a padding row was written"
    assert (Pacc[geo.prow] == 0).all(), "Pacc: the consumed accumulator rows are not zero"
    assert torch.isnan(Pacc[~geo.valid]).all(), "Pacc: a padding row was written"
    if zero_qkv:
        assert (QKV[:geo.rows] == 0).all() and torch.isnan(QKV[geo.rows:]).all(), "QKVacc: rows not zeroed (or beyond them written)"
    else:
        assert torch.isnan(QKV).all(), "QKVacc was written"

    ref = R.lnmod(x_ref, t64, None, sq * H, cq * H)
    # After x: the bound of test_gpu_ops.test_lnmod_matches_fp64 (the same per-lane float4 sums, 5 shuffle levels and up to 4
    # warps per row through shared memory: at most H/128 + 8 roundings deep; two-pass variance, rsqrtf, fmaf(z, 1 + scale, shift)).
    c = 2 * (H // 128 + 8)
    var = x_ref.var(dim=1, unbiased=False, keepdim=True)
    rstd = (var + 1e-6).rsqrt()
    z = (x_ref - x_ref.mean(dim=1, keepdim=True)) * rstd
    err_z = c * U * (x_ref.abs().mean(dim=1, keepdim=True) * rstd + z.abs())
    # x itself is fp32-rounded (e_x): to first order a row perturbation dx moves z_i by <= rstd max|dx| (2 + 2 |z_i|)
    # (the mean by max|dx|, the standard deviation by 2 max|dx|)
    err_z = err_z + rstd * e_x.amax(dim=1, keepdim=True) * (2 + 2 * z.abs())
    sc = t64[:, cq * H:(cq + 1) * H]
    tol = _bf16_tol(ref, (1 + sc).abs() * (err_z + U * z.abs()) + U * ref.abs())
    got, pad = geo.decode(A1, H)
    _assert_within(got[geo.prow], ref, tol, "A1")
    assert torch.isnan(pad).all(), "A1: a padding row was written"


@pytest.mark.parametrize("urow", [False, True])
@pytest.mark.parametrize("stage", list(ROW_STAGES))
@pytest.mark.parametrize("H", [128, 256, 512, 1024])      # NV = 1, 2, 4, 8: 1, 2, 4 and 4 warps per row
@pytest.mark.parametrize("kernel,CH,N", ROW_GEOS)
def test_row_stage_matches_fp64(lib, kernel, CH, N, H, stage, urow):
    if urow and kernel == WIN:
        pytest.skip("the window kernel's AdaLN table has one row per token row")
    _row_case(*lib, kernel, CH, N, H, stage, urow)


@pytest.mark.parametrize("kernel,CH,N,grid", [(FLOW, 32, 61, 7), (WIN, 0, 61, 5)])
@pytest.mark.parametrize("H", [256, 1024])
def test_row_stage_on_a_small_grid(lib, kernel, CH, N, grid, H):
    """One CTA per chunk (flow) or 5 CTAs for 183 rows (window): each CTA walks many rows."""
    _row_case(*lib, kernel, CH, N, H, "proj", kernel == FLOW, grid=grid, seed=1)


# ------------------------------------------------------------------------------------------------ ATTN
def _attn_case(L, cabi, kernel, hd, window, parity=0, grid=0, big=False):
    heads = 128 // hd if hd < 128 else 2                  # H = 128 or 256
    H, N = heads * hd, 61
    geo = Geo(kernel, 1, 3, N, CH=32)                      # 32-row chunks: the band crosses into the neighbouring chunk; 29 rows last
    g = torch.Generator(device="cuda").manual_seed(hd * 131 + window * 7 + parity + 3 * grid + 1000 * int(big))
    x = torch.randn(geo.seqs, N, 3, heads, hd, device="cuda", generator=g) * 1.5
    bias = torch.randn(3 * H, device="cuda", generator=g) * 0.5
    if big:                                               # as test_band_attention_is_stable_at_scores_of_100
        x *= 1 / 3
        sign = torch.randint(0, 2, (geo.seqs, N, heads), device="cuda", generator=g).float() * 2 - 1
        x[:, :, 0, :, 0] = 16.0
        x[:, :, 1, :, 0] = sign * 100.0 * math.sqrt(hd) / 16.0
        bias.view(3, heads, hd)[:2, :, 0] = 0.0
    qkv = x.reshape(geo.seqs * N, 3 * H)
    if kernel == FLOW:
        QKV = _nan(2, geo.rows, 3 * H)
        QKV[parity] = geo.padded(qkv)
        QKV[parity ^ 1] = geo.padded(torch.randn(geo.seqs * N, 3 * H, device="cuda", generator=g))    # slices the stage must zero
        before = QKV[parity].clone()
    else:
        QKV = geo.padded(qkv)
        before = QKV.clone()
    A2 = geo.operand(H)
    d = geo.desc(cabi, ATTN, grid, H=H, heads=heads, window=window, parity=parity)
    d.QKVacc, d.A2, d.bias = QKV.data_ptr(), A2.data_ptr(), bias.data_ptr()
    _run(L, cabi, geo, d)

    qkv64 = qkv.double().reshape(geo.seqs, N, 3 * H)
    ref = R.band_attention(qkv64 + bias.double(), heads, window)
    q, k, _ = (qkv64 + bias.double()).reshape(geo.seqs, N, 3, heads, hd).permute(2, 0, 3, 1, 4)
    v = qkv64.reshape(geo.seqs, N, 3, heads, hd)[:, :, 2].transpose(1, 2)
    # Scores: q + b_q, k + b_k and the scale rsqrtf(hd) (2 ulp) round; the dot product is an FMA chain over hd/16 (flow, 16 lanes
    # per row) or hd/32 (window, 32 lanes) elements per lane plus 4 or 5 shuffle levels: |d s| <= c U scale sum_d |q_d k_d| with
    # c = hd/16 + 4 + 3 + 4 (flow) or hd/32 + 5 + 3 + 4 (window).  After that the bound of test_gpu_ops._attention_check:
    # softmax moves o by <= 2 max|v| max|d s|; the exponentials (__expf of arguments <= 0), the online merge of batches and
    # __fdividef(1, den) add (16 + 4 (2w + 1)) U max|v|.  The value bias is added last by one fmaf: U |o|.
    c = hd // 16 + 11 if kernel == FLOW else hd // 32 + 12
    blocked = R.O.band_mask(N, window, device=qkv64.device)
    ds = c * U * hd ** -0.5 * (q.abs() @ k.abs().transpose(-2, -1)).masked_fill(blocked, 0).amax(dim=-1, keepdim=True)
    vrow = v.abs().amax(dim=-1)[:, :, None, :].expand(-1, -1, N, -1)
    vmax = vrow.masked_fill(blocked, 0).amax(dim=-1, keepdim=True)
    tol_h = vmax * (2 * ds + (16 + 4 * (2 * window + 1)) * U)
    tol = tol_h.expand(-1, -1, -1, hd).transpose(1, 2).reshape(geo.seqs, N, H) + U * ref.abs()
    got, pad = geo.decode(A2, H)
    _assert_within(got[geo.prow].reshape(geo.seqs, N, H), ref, _bf16_tol(ref, tol), "A2")
    assert torch.isnan(pad).all(), "A2: a padding row was written"
    if kernel == FLOW:
        assert torch.equal(QKV[parity].view(torch.int32), before.view(torch.int32)), "the QKV buffer read was modified"
        other = QKV[parity ^ 1]
        assert (other[geo.prow] == 0).all(), "the other parity's q / k / v slices of the chunk's rows are not zero"
        assert torch.isnan(other[~geo.valid]).all(), "a padding row of the other parity was written"
    else:
        assert torch.equal(QKV.view(torch.int32), before.view(torch.int32)), "QKVacc was modified"


@pytest.mark.parametrize("parity", [0, 1])
@pytest.mark.parametrize("window", [0, 1, 2, 3, 4, 7])    # >= 3: several 5-key batches merged online (flow), win_attn_wide (window)
@pytest.mark.parametrize("hd", [32, 64, 128])
@pytest.mark.parametrize("kernel", [FLOW, WIN])
def test_attention_stage_matches_fp64(lib, kernel, hd, window, parity):
    if parity and kernel == WIN:
        pytest.skip("the window kernel has one QKV buffer")
    _attn_case(*lib, kernel, hd, window, parity)


@pytest.mark.parametrize("hd", [32, 128])
@pytest.mark.parametrize("kernel,grid", [(FLOW, 7), (WIN, 3)])
def test_attention_stage_on_a_small_grid(lib, kernel, grid, hd):
    """Flow: 7 CTAs for 6 chunks, one CTA per chunk serves every head of it (the qkv bias is reloaded per head); window: 3 CTAs."""
    _attn_case(*lib, kernel, hd, 3, parity=1, grid=grid)


@pytest.mark.parametrize("hd", [64, 128])
@pytest.mark.parametrize("kernel", [FLOW, WIN])
def test_attention_stage_is_stable_at_scores_of_100(lib, kernel, hd):
    """Scores of +-100 after scaling: exp(100) overflows fp32, only the running-max subtraction keeps the softmax finite."""
    _attn_case(*lib, kernel, hd, 7, parity=1, big=True)


# ------------------------------------------------------------------------------------------------ GELU
@pytest.mark.parametrize("grid", [0, 5])
@pytest.mark.parametrize("M4", [4096, 1088])              # 1088 = 17 x 64: the last 1024-column slab of a row is partial
@pytest.mark.parametrize("kernel", [FLOW, WIN])
def test_gelu_stage_matches_fp64(lib, kernel, M4, grid):
    L, cabi = lib
    geo = Geo(kernel, 1, 3, 60, CH=64)
    if kernel == FLOW and grid:
        grid = geo.n_chunks + 2
    g = torch.Generator(device="cuda").manual_seed(M4 + grid + (kernel == FLOW))
    T = geo.seqs * geo.N
    acc = torch.randn(T, M4, device="cuda", generator=g) * 4
    acc[0, :8] = torch.tensor([12.0, -12.0, 30.0, -30.0, 10.5, -10.5, 60.0, -60.0], device="cuda")     # arguments beyond +-10
    acc[T - 1, -8:] = torch.tensor([-14.0, 14.0, -11.0, 11.0, 25.0, -25.0, 0.0, -0.0], device="cuda")
    bias = torch.randn(M4, device="cuda", generator=g) * 0.5
    bias[:8] = 0.0
    bias[-8:] = 0.0
    Hacc = geo.padded(acc)
    Hm = geo.operand(M4)
    d = geo.desc(cabi, GELU, grid, H=128, heads=2, mlp_hidden=M4)
    d.Hacc, d.Hm, d.bias = Hacc.data_ptr(), Hm.data_ptr(), bias.data_ptr()
    _run(L, cabi, geo, d)
    v = acc.double() + bias.double()
    ref = R.gelu_tanh(v)
    # test_gpu_ops' bound of the GELU epilogue in bf16 mode (the same fl(acc + bias) and gelu_tanh_fast with tanh.approx.f32)
    t = torch.tanh(math.sqrt(2.0 / math.pi) * (v + 0.044715 * v ** 3))
    tol = 8 * U * (v.abs() + ref.abs()) + 0.5 * v.abs() * t.abs() * R.TANH_APPROX
    got, pad = geo.decode(Hm, M4)
    _assert_within(got[geo.prow], ref, _bf16_tol(ref, tol), "Hm")
    assert torch.isnan(pad).all(), "Hm: a padding row was written"
    assert (Hacc[geo.prow] == 0).all(), "Hacc: the consumed accumulator rows are not zero"
    assert torch.isnan(Hacc[~geo.valid]).all(), "Hacc: a padding row was written"


@pytest.mark.parametrize("kernel", [FLOW, WIN])
def test_gelu_stage_is_bitwise_the_per_op_gelu_epilogue(lib, kernel):
    """tanh.approx.f32 may err by 2^-11 relative, and that allowance covers the gap between the tanh and the exact-erf GELU at
    every argument (at most 0.95 of it), so no bound derived from its documented accuracy can tell the two apart.  The bf16 GELU
    epilogue of the per-op GEMM (gelu_tanh_approx, gemm.cuh) evaluates the same formula with the same instruction: on the same
    fp32 pre-activation fl(acc + bias) both must give the same bits.  acc = A . W^T of exactly representable operands
    (test_gpu_ops._exact_operands) is exact in fp32 in either kernel."""
    from test_gpu_ops import _exact_operands
    L, cabi = lib
    geo = Geo(kernel, 1, 3, 60, CH=64)
    T, M4, K = geo.seqs * geo.N, 1088, 256
    g = torch.Generator(device="cuda").manual_seed(11 + (kernel == FLOW))
    A, Wt = _exact_operands(T, M4, K, g)
    acc = (A.double() @ Wt.double().t()).float()
    bias = torch.randn(M4, device="cuda", generator=g) * 0.5
    bias[:6] = torch.tensor([12.0, -12.0, 30.0, -30.0, 10.5, -10.5], device="cuda")      # arguments beyond +-10
    ref = torch.full((T, M4), float("nan"), device="cuda", dtype=torch.bfloat16)
    e = cabi.FmtDebugGemm(mode=0, kind=cabi.FMT_EPI_GELU, M=T, N=M4, K=K, block_n=0, ksplit=1, ldo=M4, out_f32=0)
    e.A, e.W, e.bias, e.out = A.data_ptr(), Wt.data_ptr(), bias.data_ptr(), ref.data_ptr()
    cabi.check(L.fmt_debug_gemm_epilogue(C.byref(e), _stream()), "fmt_debug_gemm_epilogue")
    Hacc = geo.padded(acc)
    Hm = geo.operand(M4)
    d = geo.desc(cabi, GELU, H=128, heads=2, mlp_hidden=M4)
    d.Hacc, d.Hm, d.bias = Hacc.data_ptr(), Hm.data_ptr(), bias.data_ptr()
    _run(L, cabi, geo, d)
    if kernel == FLOW:
        got = R.flow_tiled_decode(Hm, geo.n_chunks, geo.CH, M4)[geo.prow]
    else:
        got = R.win_tiled_decode(Hm, geo.Rp, M4)[:T]
    assert torch.isfinite(ref.float()).all()
    same = got.view(torch.int16) == ref.view(torch.int16)
    assert same.all(), f"{int((~same).sum())} of {same.numel()} elements differ from the per-op GELU epilogue"


# ------------------------------------------------------------------------------------------------ COMB
SOLVER_STAGES = [("euler", 0), ("heun2", 0), ("heun2", 1), ("heun3", 0), ("heun3", 1), ("heun3", 2),
                 ("rk4", 0), ("rk4", 1), ("rk4", 2), ("rk4", 3)]
SLOT_BRANCHES = {1: [1, 1, 1], 3: [3, 1, 3], 4: [4, 3, 1]}    # per clip of 3 (slot_branch0: which plan branches a clip reads)
PLAN_SCALES = (2.5, 1.5, 0.75)
SLOT_SCALES = [(1.75, 2.25, 1.25), (3.0, 0.5, 1.5), (0.5, 2.0, 2.5)]


def _f32(x):
    return float(torch.tensor(x, dtype=torch.float32))


@pytest.mark.parametrize("solver,stage", SOLVER_STAGES)
@pytest.mark.parametrize("slots", [False, True])
@pytest.mark.parametrize("nb", [1, 3, 4])
@pytest.mark.parametrize("kernel", [FLOW, WIN])
def test_comb_stage_matches_fp64(lib, kernel, nb, slots, solver, stage):
    L, cabi = lib
    sampler = sys.modules[load_package().__name__ + ".sampler"]
    tab = sampler.SOLVERS[solver]
    a32 = [[_f32(x) for x in row] for row in tab["a"]]
    b32 = [_f32(x) for x in tab["b"]]
    G = len(b32)
    B, W, step = 3, 64, 1
    N, P = (60, 10) if kernel == FLOW else (20, 5)             # the window kernel serves at most 256 token rows: 4 x 3 x 20
    Lc = N - P
    geo = Geo(kernel, nb, B, N, P=P, CH=32)                # 32-row chunks: the current frames of a clip span two chunks
    g = torch.Generator(device="cuda").manual_seed(nb * 100 + 10 * int(slots) + 17 * G + stage + (kernel == FLOW))
    V = _nan(nb, B, geo.NPs, W)
    V[:, :, :N] = torch.randn(nb, B, N, W, device="cuda", generator=g) * 2
    V0 = V.clone()
    bias = torch.randn(W, device="cuda", generator=g) * 0.5
    x0 = torch.randn(B, Lc, W, device="cuda", generator=g)
    x_state = x0.clone()
    kbuf = _nan(G, B, Lc, W)
    kbuf[:stage] = torch.randn(stage, B, Lc, W, device="cuda", generator=g)
    k0 = kbuf.clone()
    ddt = torch.tensor([0.05, 1.0 / 9.0, 0.3], device="cuda")
    ax = _nan(nb, B, N, W, dtype=torch.bfloat16)
    d = geo.desc(cabi, COMB, W=W, n_stages=G, stage=stage, step=step, a_scale=PLAN_SCALES[0], r_scale=PLAN_SCALES[1], e_scale=PLAN_SCALES[2])
    for i in range(G):
        for j in range(G):
            d.rk_a[i * G + j] = a32[i][j]
        d.rk_b[i] = b32[i]
    d.Vacc, d.bias, d.x_state, d.kbuf, d.ddt, d.ax = V.data_ptr(), bias.data_ptr(), x_state.data_ptr(), kbuf.data_ptr(), ddt.data_ptr(), ax.data_ptr()
    if slots:
        sb = (C.c_int32 * B)(*SLOT_BRANCHES[nb])
        ss = (C.c_float * (3 * B))(*[s for t in SLOT_SCALES for s in t])
        d.slot_branches, d.slot_scales = C.cast(sb, C.c_void_p), C.cast(ss, C.c_void_p)
    _run(L, cabi, geo, d)

    vb = V0[:, :, P:N].double() + bias.double()                 # (nb, B, Lc, W)
    v_ref = torch.empty(B, Lc, W, dtype=torch.float64, device="cuda")
    tol_v = torch.empty_like(v_ref)
    for b in range(B):
        nbc, (ca, cr, ce) = (SLOT_BRANCHES[nb][b], SLOT_SCALES[b]) if slots else (nb, PLAN_SCALES)
        br = R.clip_branches(nb, nbc)
        vs = [vb[i, b] for i in br]
        v_ref[b] = R.cfg_combine(vs, ca, cr, ce)
        # fl(v + decoder bias), one difference, one product and one addition per guidance term: nb + 2 roundings, each <= U S
        m = [x.abs() for x in vs]
        if nbc == 1:
            S = m[0]
        elif nbc == 3:
            S = m[0] + abs(ca) * (m[2] + m[0]) + abs(ce) * (m[1] + m[2])
        else:
            S = m[0] + abs(cr) * (m[1] + m[0]) + abs(ca) * (m[3] + m[1]) + abs(ce) * (m[2] + m[3])
        tol_v[b] = (nbc + 2) * U * S
    dt = ddt[step].double().item()
    ks = [k0[j].double() for j in range(stage)] + [v_ref]
    y_ref = R.rk_stage(x0.double(), ks, stage, dt, a32, b32)
    c = b32 if stage == G - 1 else a32[stage + 1]
    # acc = sum_j fmaf(c_j, k_j, acc): stage + 1 roundings of at most U sum_j |c_j k_j|, plus |c_g| tol_v; y = fmaf(dt, acc, y0)
    err_acc = (stage + 1) * U * sum(abs(c[j]) * ks[j].abs() for j in range(stage + 1)) + abs(c[stage]) * tol_v
    tol_y = U * y_ref.abs() + abs(dt) * err_acc
    last = stage == G - 1

    cur = V[:, :, P:N]
    assert (cur == 0).all(), "Vacc: the consumed current frames are not zero"
    assert torch.isnan(V[:, :, N:]).all(), "Vacc: a padding row was written"
    if kernel == FLOW:
        assert torch.equal(V[:, :, :P], V0[:, :, :P]), "Vacc: context frames (never read) were modified"
    else:
        assert (V[:, :, :P] == 0).all(), "Vacc: the context frames are not zero"
    if G > 1:
        _assert_within(kbuf[stage].double(), v_ref, tol_v, "kbuf[stage]")
        assert torch.equal(kbuf[:stage], k0[:stage]), "kbuf of an earlier stage was modified"
        assert torch.isnan(kbuf[stage + 1:]).all(), "kbuf of a later stage was written"
    else:
        assert torch.isnan(kbuf).all(), "kbuf was written by an Euler step"
    if last:
        _assert_within(x_state.double(), y_ref, tol_y, "x_state")
    else:
        assert torch.equal(x_state, x0), "x_state was written before the last stage"
    got = ax[:, :, P:].double()
    for br in range(nb):
        _assert_within(got[br], y_ref, _bf16_tol(y_ref, tol_y), f"ax of branch {br}")
        if last:
            assert torch.equal(ax[br, :, P:], x_state.to(torch.bfloat16)), "ax is not bf16 of the new state"
    assert torch.isnan(ax[:, :, :P].float()).all(), "ax: a context frame was written"
