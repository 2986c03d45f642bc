"""bf16x3 precision mode (FMT_MODE_BF16X3) on the B200: split-bf16 tcgen05 GEMMs held to the fp32 validation mode's gates.

Every GEMM operand is split as x = hi + lo (hi = bf16(x), lo = bf16(x - hi)) and the GEMM sums Ah.Wh + Ah.Wl + Al.Wh in fp32 on
the tensor pipe.  An emulation with exact products (fp64 sums) gives a relative GEMM error of 4.4e-6 and latents of configs[1]
within 6.6e-6 of the oracle; the bounds below are about 3x those, since how the tensor pipe rounds its fp32 accumulation is not
part of the emulation.  Measured on a B200: GEMM errors of 4.8e-6 (K = 512) growing to 1.47e-5 (K = 4096) and 3.2e-5 (K = 9216),
configs[1] latents 1.26e-5 max-abs from the oracle, 32 clips 2.6e-6 relative.
"""
import ctypes as C
import sys

import pytest
import torch

import cases
from __graft_entry__ import load_package
from oracle import fmt_oracle as O
from test_gpu_parity import CFV_CASES, CLIP_CASES, PROJ_CASES, _projection_layer, model_for, run_node
from test_gpu_psnr import _configs1

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
MODE = "bf16x3"


@pytest.fixture(scope="module")
def pkg():
    return load_package()


@pytest.fixture(scope="module")
def lib(pkg):
    cabi = sys.modules[pkg.__name__ + "._cabi"]
    return cabi.load_library(), cabi


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


# ---------------------------------------------------------------------------------------------- the split GEMM
@pytest.mark.parametrize("block_n", [64, 128, 256, 512, 1024])
@pytest.mark.parametrize("M", [180, 5820])              # one clip with 3-way CFG; 32 clips + a ragged 60-row tile
@pytest.mark.parametrize("K", [512, 1024, 1088, 4096, 9216])
def test_bf16x3_gemm_against_fp64(lib, M, K, block_n):
    L, cabi = lib
    N = 512
    g = torch.Generator(device="cuda").manual_seed(M * 7 + K + block_n)
    A = torch.randn(M, K, device="cuda", generator=g)
    W = torch.randn(N, K, device="cuda", generator=g)
    bias = torch.randn(N, device="cuda", generator=g)
    ref = A.double() @ W.double().t() + bias.double()
    out = torch.full((M, N), float("nan"), device="cuda")
    cabi.check(L.fmt_debug_gemm_bf16x3(A.data_ptr(), W.data_ptr(), bias.data_ptr(), out.data_ptr(), M, N, K, block_n, _stream()), "gemm_bf16x3")
    A16, W16 = A.to(torch.bfloat16), W.to(torch.bfloat16)
    out16 = torch.full((M, N), float("nan"), device="cuda")
    cabi.check(L.fmt_debug_gemm_bf16(A16.data_ptr(), W16.data_ptr(), bias.data_ptr(), out16.data_ptr(), M, N, K, block_n, _stream()), "gemm_bf16")
    torch.cuda.synchronize()
    assert torch.isfinite(out).all()
    rel = ((out.double() - ref).norm() / ref.norm()).item()
    rel16 = ((out16.double() - ref).norm() / ref.norm()).item()
    print(f"M={M} K={K} block_n={block_n}: bf16x3 {rel:.2e}, bf16 {rel16:.2e}")
    # The error grows with K beyond the emulation's: the tensor pipe rounds its fp32 accumulator once per MMA, and the split GEMM
    # issues three MMAs per 16-wide K step.  K = 9216 occurs only in the audio projection (the FMT's GEMMs have K <= 4096): there a
    # B200 measured 3.2e-5, about 70x below bf16.
    tol, gain = (1.5e-5, 100) if K <= 4096 else (5e-5, 40)
    assert rel <= tol, rel
    assert rel * gain <= rel16, (rel, rel16)


def test_bf16x3_gemm_rejects_ragged_k(lib):
    L, cabi = lib
    A, W, out = torch.zeros(128, 96, device="cuda"), torch.zeros(64, 96, device="cuda"), torch.zeros(128, 64, device="cuda")
    assert L.fmt_debug_gemm_bf16x3(A.data_ptr(), W.data_ptr(), None, out.data_ptr(), 128, 64, 96, 0, _stream()) != 0


# ---------------------------------------------------------------------------------------------- the fixtures of the fp32 mode's gates
@pytest.mark.parametrize("name", CLIP_CASES)
def test_bf16x3_clips_match_reference(pkg, name):
    ref = cases.golden(name)
    out = run_node(pkg, name, MODE)
    assert out.shape == ref.shape
    rel = cases.rel_err(out, ref)
    assert rel <= 1e-4, (name, rel)
    big = ref.abs() > 1e-2
    per_elem = ((out - ref).abs()[big] / ref.abs()[big]).max().item()
    assert per_elem <= 2e-2, (name, per_elem)


@pytest.mark.parametrize("name", CFV_CASES)
def test_bf16x3_single_evaluation_matches_forward_with_cfv(pkg, name):
    rec = cases.CASES[name]
    d = cases.dims_of(rec)
    be = pkg.backend_for(model_for(pkg, rec["dims"]), DEV)
    r_s, wa, we = [t.to(DEV) for t in cases.case_inputs(rec)]
    x, prev_x, prev_wa, prev_we = [t.to(DEV).contiguous() for t in cases.cfv_extra_inputs(rec)]
    L = d.frames_per_clip
    dynamic = we.shape[1] > 1
    nb = pkg.n_branches_for(rec["a"], rec["r"], rec["e"], rec.get("include_r_cfg", False))
    nfe = 11                                                          # a grid point k / 10 equals the fixture's t
    k = round(rec["t"] * (nfe - 1))
    assert abs(k / (nfe - 1) - rec["t"]) < 1e-6
    be.configure(rec["B"], nb, dynamic, nfe, "euler", MODE)
    v = be.velocity(k, x, wa[:, :L].contiguous(), r_s, (we[:, :L] if dynamic else we).contiguous(), prev_x, prev_wa,
                    prev_we if dynamic else None, rec["a"], rec["r"], rec["e"]).cpu()
    ref = cases.golden(name)
    assert v.shape == ref.shape
    assert cases.rel_err(v, ref) <= 1e-4, cases.rel_err(v, ref)


@pytest.mark.parametrize("name", PROJ_CASES)
def test_bf16x3_audio_projection_matches_reference(pkg, name):
    rec = cases.CASES[name]
    ref = cases.golden(name)
    (out,) = pkg.FloatApplyAudioProjection().apply_projection(cases.projection_input(rec), _projection_layer(pkg, rec), _mode=MODE)
    assert out.device.type == "cpu" and out.shape == ref.shape
    assert cases.rel_err(out, ref) <= 1e-4, cases.rel_err(out, ref)


# ---------------------------------------------------------------------------------------------- against the oracle, determinism
def test_bf16x3_configs1_matches_oracle_and_is_deterministic(pkg):
    """configs[1] (1 clip, 100 frames, nfe 10, a_cfg 2): the per-op graph path (the window kernels are bf16-only)."""
    (r_s, wa, we, noise), _, ref = _configs1()
    model = model_for(pkg, "full")
    node = pkg.FloatSampleMotionSequenceRD_VA()
    args = (2.0, 1.0, 1.0, False, 10, "euler", 1e-5, 1e-5, 0.1, 0.1, 0.1, True, 15)
    a = node.sample_rd_sequence_va(r_s, wa, we, 100, model, *args, _mode=MODE, _noise=noise)[0]
    b = node.sample_rd_sequence_va(r_s, wa, we, 100, model, *args, _mode=MODE, _noise=noise)[0]
    assert pkg.backend_for(model, DEV).window_kernel_status() == -1
    err = cases.max_abs(a, ref)
    print(f"configs[1] bf16x3: max-abs {err:.3e}, rel {cases.rel_err(a, ref):.3e}")
    assert err <= 2e-5, err
    assert torch.equal(a, b)


def test_bf16x3_32_clips_matches_oracle_and_is_deterministic(pkg):
    """32 clips x 200 frames (5760 token rows per window): the CTA-pair split GEMMs."""
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    from oracle.synth import synth_inputs
    B, T, nfe = 32, 200, 10
    r_s, wa, we = synth_inputs(d, B, T, seed=321)
    g = torch.Generator().manual_seed(11)
    noise = torch.stack([torch.randn(B, d.frames_per_clip, d.dim_w, generator=g) for _ in range(-(-T // d.frames_per_clip))])
    node = pkg.FloatSampleMotionSequenceRD_VA()
    args = (2.0, 1.0, 1.0, False, nfe, "euler", 1e-5, 1e-5, 0.1, 0.1, 0.1, True, 11)
    a = node.sample_rd_sequence_va(r_s, wa, we, T, model, *args, _mode=MODE, _noise=noise)[0]
    b = node.sample_rd_sequence_va(r_s, wa, we, T, model, *args, _mode=MODE, _noise=noise)[0]
    tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            ref = O.sample_loop({k: v.to(DEV) for k, v in cases.weights("full").items()}, d, r_s.to(DEV), wa.to(DEV), we.to(DEV), T, nfe=nfe,
                                a_cfg_scale=2.0, r_cfg_scale=1.0, e_cfg_scale=1.0, noise=noise.to(DEV)).cpu()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = tf32
    assert a.shape == ref.shape == (B, T, d.dim_w)
    rel = cases.rel_err(a, ref)
    print(f"32 clips bf16x3: rel {rel:.3e}, max-abs {cases.max_abs(a, ref):.3e}")
    assert rel <= 1e-4, rel
    assert torch.equal(a, b)


# ---------------------------------------------------------------------------------------------- decoded frames
def test_bf16x3_psnr_gate(pkg, monkeypatch):
    """The fp32 mode's PSNR gate (tests/test_gpu_psnr.py) for bf16x3 latents of configs[1], through the reference decoder.  The
    repository does not carry that decoder: without a copy the test prints the latent error it would decode and skips."""
    from oracle import refshim
    import importlib
    from test_gpu_psnr import FRAMES, T, _psnr
    (r_s, wa, we, noise), _, ref = _configs1()
    lat = pkg.FloatSampleMotionSequenceRD_VA().sample_rd_sequence_va(
        r_s, wa, we, T, model_for(pkg, "full"), 2.0, 1.0, 1.0, False, 10, "euler", 1e-5, 1e-5, 0.1, 0.1, 0.1, True, 15, _mode=MODE, _noise=noise)[0]
    print(f"bf16x3 configs[1] latents: max-abs {cases.max_abs(lat, ref):.3e}, rms {float((lat - ref).pow(2).mean().sqrt()):.3e}")
    if not refshim.reference_available():
        pytest.skip("no copy of the reference decoder (oracle/_ref: run __graft_entry__.build())")
    d = cases.FmtDims()
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    with torch.no_grad():
        ref_cpu = O.sample_loop(cases.weights("full"), d, r_s, wa, we, T, nfe=10, a_cfg_scale=2.0, e_cfg_scale=1.0, noise=noise)
    refshim.load_reference()
    Generator = importlib.import_module("refnodes.models.float.generator").Generator
    torch.manual_seed(0)
    gen = Generator(512, 512, 20).eval().to(DEV)
    img = torch.rand(1, 3, 512, 512, generator=torch.Generator().manual_seed(3)) * 2 - 1
    with torch.no_grad():
        s_r, _, feats = gen.enc(img.to(DEV), None, None)

        def frames_of(r_d):
            r_d = r_d.to(DEV)
            return [((gen.dec(s_r + r_d[:, t], None, feats)[0].clamp(-1, 1) + 1) / 2).cpu() for t in FRAMES]
        fr_ref = frames_of(ref)
        psnr = min(_psnr(a, b) for a, b in zip(frames_of(lat), fr_ref))
        floor = min(_psnr(a, b) for a, b in zip(frames_of(ref_cpu), fr_ref))
    print(f"bf16x3 PSNR {psnr:.1f} dB on the worst frame; the reference's CPU-vs-GPU floor {floor:.1f} dB")
    assert psnr >= min(40.0, floor - 6.0), (psnr, floor)
