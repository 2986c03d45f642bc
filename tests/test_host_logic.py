"""CPU tests of the host side: C-ABI library exports, solver schedules, branch selection, option plumbing, loud failure
without a GPU.  No compute call is made through the library here (no GPU in the build container)."""
import ctypes as C
import os
import re
import sys

import pytest
import torch

import cases
from __graft_entry__ import ROOT, load_package
from oracle import fmt_oracle as O


@pytest.fixture(scope="module")
def pkg():
    return load_package()


def _cabi(pkg):
    return sys.modules[pkg.__name__ + "._cabi"]


def test_library_exports_every_symbol_of_the_header(pkg):
    hdr = open(os.path.join(ROOT, "include", "fmt_b200.h")).read()
    declared = set(re.findall(r"FMT_API\s+[\w\s\*]+?\b(fmt_\w+)\s*\(", hdr))
    assert {"fmt_create", "fmt_destroy", "fmt_configure", "fmt_sample_clip", "fmt_velocity", "fmt_last_error"} <= declared
    sys.modules[pkg.__name__ + ".build"].build()
    lib = _cabi(pkg).load_library()
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/fmt_b200.h but not exported"
    assert set(_cabi(pkg)._SIGNATURES) == declared           # the ctypes binding covers exactly the header
    assert lib.fmt_abi_version() == _cabi(pkg).FMT_ABI_VERSION


def test_struct_layouts_match_the_header(pkg):
    cabi = _cabi(pkg)
    assert C.sizeof(cabi.FmtDims) == 40
    assert C.sizeof(cabi.FmtPlan) == 24 + 4 * 8
    assert cabi.FmtClip.noise.offset == 32 and cabi.FmtClip.T_wa.offset == 48 and cabi.FmtClip.progress.offset == 72
    assert len(cabi.GLOBAL_KEYS) == cabi.FMT_W_NUM_GLOBAL and len(cabi.BLOCK_KEYS) == cabi.FMT_W_PER_BLOCK


def test_no_cpu_fallback(pkg):
    """Without a CUDA device the product path must fail loudly (never route through the oracle / eager torch)."""
    model = pkg.FmtModel(cases.weights("small"), target_device="cpu")
    with pytest.raises(pkg.FmtError):
        pkg.backend_for(model, "cpu")
    if not torch.cuda.is_available():
        d = cases.SMALL_DIMS
        sd = cases.weights("small")
        dims = pkg.Dims.from_options({}, sd)
        with pytest.raises((pkg.FmtError, RuntimeError, AssertionError)):
            pkg.FmtBackend(sd, dims, "cuda:0")
    src = open(os.path.join(ROOT, "comfyui-float_optimized_b200", "sampler.py")).read()
    src += open(os.path.join(ROOT, "comfyui-float_optimized_b200", "nodes.py")).read()
    assert "oracle" not in src


@pytest.mark.parametrize("method", ["euler", "midpoint", "heun2", "heun3", "rk4"])
@pytest.mark.parametrize("nfe", [1, 2, 5, 10])
def test_schedule_reproduces_torchdiffeq_fixed_grid(pkg, method, nfe):
    """The Butcher-tableau schedule handed to the C ABI integrates dy/dt = f(t, y) exactly like the oracle's restatement
    of torchdiffeq's fixed-grid solvers (same evaluation times, same combination weights)."""
    s = pkg.build_schedule(nfe, method)
    assert s["n_steps"] == max(0, nfe - 1) and len(s["t_eval"]) == s["n_steps"] * s["n_stages"]
    f = lambda t, y: torch.sin(3.0 * t) * y + torch.cos(y) * t      # noqa: E731
    y0 = torch.linspace(-1, 1, 7, dtype=torch.float64)
    ref = O.odeint_fixed(f, y0, torch.linspace(0, 1, nfe, dtype=torch.float32).double(), method)
    G, y = s["n_stages"], y0.clone()
    for i in range(s["n_steps"]):
        ks = []
        for g in range(G):
            yg = y + s["dt"][i] * sum(s["a"][g * G + j] * ks[j] for j in range(g)) if g else y
            ks.append(f(torch.tensor(s["t_eval"][i * G + g], dtype=torch.float64), yg))
        y = y + s["dt"][i] * sum(s["b"][j] * ks[j] for j in range(G))
    assert torch.allclose(y, ref, rtol=1e-6, atol=1e-7), (y - ref).abs().max()


@pytest.mark.parametrize("method,order", [("euler", 1), ("midpoint", 2), ("heun2", 2), ("heun3", 3), ("rk4", 4)])
def test_solver_tableaux_satisfy_the_order_conditions(pkg, method, order):
    """torchdiffeq is not installed here, so the fixtures of the non-Euler solvers come from a restatement of its fixed-grid
    steppers (tests/golden/refshim.py).  This test pins the tableaux to something that restatement cannot influence: the
    Runge-Kutta order conditions of the method each name stands for (explicit midpoint, Heun's 2nd- and 3rd-order methods, the
    3/8-rule RK4 of torchdiffeq's rk4_alt_step_func), and the observed convergence order on an ODE with a closed-form solution."""
    import numpy as np
    from float_fmt_b200.sampler import SOLVERS
    t = SOLVERS[method]
    a, b, c = np.array(t["a"], dtype=np.float64), np.array(t["b"], dtype=np.float64), np.array(t["c"], dtype=np.float64)
    assert np.allclose(np.triu(a), 0)                                   # explicit
    assert np.allclose(a.sum(1), c) and np.isclose(b.sum(), 1.0)        # row-sum condition, order 1
    if order >= 2:
        assert np.isclose(b @ c, 1 / 2)
    if order >= 3:
        assert np.isclose(b @ c ** 2, 1 / 3) and np.isclose(b @ a @ c, 1 / 6)
    if order >= 4:
        assert np.isclose(b @ c ** 3, 1 / 4) and np.isclose((b * c) @ a @ c, 1 / 8)
        assert np.isclose(b @ a @ c ** 2, 1 / 12) and np.isclose(b @ a @ a @ c, 1 / 24)
    if order < 4:                                                       # ... and not one order more
        nxt = {1: np.isclose(b @ c, 1 / 2), 2: np.isclose(b @ c ** 2, 1 / 3) and np.isclose(b @ a @ c, 1 / 6),
               3: np.isclose(b @ c ** 3, 1 / 4) and np.isclose((b * c) @ a @ c, 1 / 8)}[order]
        assert not nxt
    # observed order on y' = -2 t y^2, y(0) = 1  ->  y(t) = 1 / (1 + t^2), through the schedule the C ABI receives
    def err(nfe):
        s_ = pkg.build_schedule(nfe, method)
        G, y = s_["n_stages"], 1.0
        for i in range(s_["n_steps"]):
            ks = []
            for g in range(G):
                yg = y + s_["dt"][i] * sum(s_["a"][g * G + j] * ks[j] for j in range(g))
                tg = s_["t_eval"][i * G + g]
                ks.append(-2.0 * tg * yg * yg)
            y = y + s_["dt"][i] * sum(s_["b"][j] * ks[j] for j in range(G))
        return abs(y - 0.5)
    e1, e2 = err(11), err(21)
    assert abs(np.log2(e1 / e2) - order) < 0.35, (e1, e2)


def test_unknown_solver_raises(pkg):
    with pytest.raises(ValueError):
        pkg.build_schedule(10, "dopri5")


def test_branch_selection_mirrors_forward_with_cfv(pkg):
    assert pkg.n_branches_for(1.0, 1.0, 1.0, False) == 1 and pkg.n_branches_for(1.0, 1.0, 1.0, True) == 1   # FMT.py:346,400
    assert pkg.n_branches_for(2.0, 1.0, 1.0, False) == 3 and pkg.n_branches_for(1.0, 1.0, 3.0, False) == 3
    assert pkg.n_branches_for(2.0, 1.0, 1.0, True) == 4 and pkg.n_branches_for(1.0, 0.5, 1.0, True) == 4


def test_dims_follow_the_checkpoint(pkg):
    sd = cases.weights("small")
    d, s = pkg.Dims.from_options(pkg.BaseOptions(), sd), cases.SMALL_DIMS
    assert (d.dim_h, d.dim_w, d.dim_a, d.fmt_depth, d.mlp_hidden) == (s.dim_h, s.dim_w, s.dim_a, s.fmt_depth, s.mlp_hidden)
    full = pkg.Dims.from_options(pkg.BaseOptions())
    assert (full.dim_h, full.frames_per_clip, full.num_prev_frames, full.attention_window) == (1024, 50, 10, 2)


def test_node_surface_matches_reference(pkg):
    """UNIQUE_NAME / FUNCTION / RETURN_TYPES / input names of nodes_vadv.py:534-623 and nodes_adv.py:697-723."""
    va = pkg.FloatSampleMotionSequenceRD_VA
    assert va.UNIQUE_NAME == "FloatSampleMotionSequenceRD_VA" and va.FUNCTION == "sample_rd_sequence_va"
    assert va.RETURN_TYPES == ("TORCH_TENSOR", "FLOAT_FMT_MODEL") and va.CATEGORY == "FLOAT/Very Advanced"
    req = va.INPUT_TYPES()["required"]
    assert list(req) == ["r_s_latent", "wa_latent", "audio_num_frames", "we_latent", "float_fmt_model", "a_cfg_scale", "r_cfg_scale",
                         "e_cfg_scale", "include_r_cfg", "nfe", "torchdiffeq_ode_method", "ode_atol", "ode_rtol", "audio_dropout_prob",
                         "ref_dropout_prob", "emotion_dropout_prob", "fix_noise_seed", "seed"]
    assert req["torchdiffeq_ode_method"][0] == ["euler", "midpoint", "rk4", "heun2", "heun3"]
    assert req["nfe"][1] == {"default": 10, "min": 1, "max": 1000} and req["seed"][1]["default"] == 15
    adv = pkg.FloatSampleMotionSequenceRD
    assert adv.UNIQUE_NAME == "FloatSampleMotionSequenceRD" and adv.FUNCTION == "sample_rd_sequence"
    assert list(adv.INPUT_TYPES()["required"]) == ["r_s_latent", "wa_latent", "audio_num_frames", "we_latent", "float_pipe", "a_cfg_scale",
                                                   "e_cfg_scale", "seed"]
    # nodes_vadv.py:147-166
    ap = pkg.FloatApplyAudioProjection
    assert ap.UNIQUE_NAME == "FloatApplyAudioProjection" and ap.FUNCTION == "apply_projection" and ap.CATEGORY == "FLOAT/Very Advanced"
    assert ap.RETURN_TYPES == ("TORCH_TENSOR",) and ap.RETURN_NAMES == ("wa_latent",)
    req = ap.INPUT_TYPES()["required"]
    assert list(req) == ["wav2vec_features", "projection_layer"] and req["projection_layer"][0] == "AUDIO_PROJECTION_LAYER"
    assert set(pkg.NODE_CLASS_MAPPINGS) == {"FloatSampleMotionSequenceRD_VA", "FloatSampleMotionSequenceRD", "FloatProcessOpt",
                                            "FloatApplyAudioProjection"}
    # nodes.py:146-168 - the simple node
    fp = pkg.FloatProcess
    assert fp.UNIQUE_NAME == "FloatProcessOpt" and fp.DISPLAY_NAME == "FLOAT Process (Opt)" and fp.FUNCTION == "floatprocess"
    assert fp.RETURN_TYPES == ("IMAGE", "AUDIO", "FLOAT") and fp.RETURN_NAMES == ("images", "ref_audio", "fps") and fp.CATEGORY == "FLOAT"
    assert list(fp.INPUT_TYPES()["required"]) == ["ref_image", "ref_audio", "float_pipe", "a_cfg_scale", "e_cfg_scale", "fps", "emotion",
                                                  "face_align", "seed"]
    # the widgets this backend adds are optional, so saved reference workflows load unchanged; keep_on_device defaults to the
    # reference's behaviour (CPU tensors between nodes)
    for cls in (va, adv):
        assert list(cls.INPUT_TYPES()["optional"]) == ["precision", "keep_on_device"]
        assert cls.INPUT_TYPES()["optional"]["keep_on_device"][1]["default"] is False
    assert list(fp.INPUT_TYPES()["optional"]) == ["precision"]
    assert list(ap.INPUT_TYPES()["optional"]) == ["keep_on_device"] and ap.INPUT_TYPES()["optional"]["keep_on_device"][1]["default"] is False


def test_required_inputs_equal_the_reference_classes(pkg):
    """INPUT_TYPES()["required"] of the three sampler nodes, compared entry by entry with the reference's own classes as stored in
    tests/golden/node_surface.json (type / enum, default, min, max, step, forceInput; RETURN_TYPES, FUNCTION, UNIQUE_NAME)."""
    import json
    from golden.make_golden import NODE_SURFACE, node_surface
    want = json.load(open(os.path.join(cases.GOLDEN_DIR, "node_surface.json")))
    for name in NODE_SURFACE:
        ours, ref = node_surface(getattr(pkg, name)), want[name]
        assert [r[0] for r in ours["required"]] == [r[0] for r in ref["required"]], name
        for a, b in zip(ours["required"], ref["required"]):
            assert a == b, (name, a, b)
        assert (ours["RETURN_TYPES"], ours["FUNCTION"], ours["UNIQUE_NAME"]) == (ref["RETURN_TYPES"], ref["FUNCTION"], ref["UNIQUE_NAME"]), name


def test_precision_mode_resolution(pkg, monkeypatch):
    monkeypatch.delenv("FMT_MODE", raising=False)
    assert pkg.resolve_mode(None) == "bf16" and pkg.resolve_mode("default") == "bf16" and pkg.resolve_mode("fp32") == "fp32"
    monkeypatch.setenv("FMT_MODE", "fp32")
    assert pkg.resolve_mode(None) == "fp32" and pkg.resolve_mode("default") == "fp32" and pkg.resolve_mode("bf16") == "bf16"
    with pytest.raises(ValueError):
        pkg.resolve_mode("fp8")


def test_float_process_swaps_the_sampler_and_restores_it(pkg):
    """FLOAT Process (Opt): G.sample is this backend only inside the call; a CPU pipe has no fallback (FmtError), and the
    (image, audio) pairing / seed + i policy of nodes.py:178-205 is kept."""
    import types
    calls = []

    class G:
        def __init__(self):
            self.opt = None

        def sample(self, data, **kw):
            return "reference sampler"

    g = G()
    with pkg.use_b200_sampler(g, "bf16"):
        assert "sample" in vars(g)
    assert "sample" not in vars(g) and g.sample({}) == "reference sampler"

    def run_inference(_p, img, audio, a_cfg_scale, r_cfg_scale, e_cfg_scale, emo, no_crop, seed):
        calls.append((tuple(img.shape), tuple(audio["waveform"].shape), emo, no_crop, seed, "sample" in vars(g)))
        return torch.zeros(3, 4, 4, 3)

    opt = types.SimpleNamespace(cudnn_benchmark_enabled=False, r_cfg_scale=1.0, fps=25.0)
    pipe = types.SimpleNamespace(G=g, rank=torch.device("cpu"), opt=opt, run_inference=run_inference)
    imgs, audio, fps = pkg.FloatProcess().floatprocess(torch.zeros(1, 8, 8, 3), {"waveform": torch.zeros(2, 1, 100), "sample_rate": 16000}, pipe,
                                                      2.0, 1.0, 30.0, "none", True, 7)
    assert imgs.shape == (6, 4, 4, 3) and fps == 30.0 and opt.fps == 30.0 and audio["waveform"].shape == (1, 1, 200)
    assert calls == [((1, 8, 8, 3), (1, 1, 100), None, False, 7, True), ((1, 8, 8, 3), (1, 1, 100), None, False, 8, True)]
    assert "sample" not in vars(g)


def test_node_validation_runs_before_any_device_work(pkg):
    model = pkg.FmtModel(cases.weights("small"), target_device="cpu")
    node = pkg.FloatSampleMotionSequenceRD_VA()
    r_s, wa, we = torch.zeros(2, 32), torch.zeros(2, 20, 32), torch.zeros(2, 1, 7)
    args = (2.0, 1.0, 1.0, False, 2, "euler", 1e-5, 1e-5, 0.3, 0.3, 0.3, True, 3)
    with pytest.raises(TypeError):
        node.sample_rd_sequence_va(r_s.numpy(), wa, we, 20, model, *args)
    with pytest.raises(ValueError):
        node.sample_rd_sequence_va(r_s[:1], wa, we, 20, model, *args)
    before = (model.opt.audio_dropout_prob, model.opt.ref_dropout_prob, model.opt.emotion_dropout_prob)
    with pytest.raises(pkg.FmtError):          # CPU target: no fallback; dropout probs restored (nodes_vadv.py:729-735)
        node.sample_rd_sequence_va(r_s, wa, we, 20, model, *args)
    assert before == (model.opt.audio_dropout_prob, model.opt.ref_dropout_prob, model.opt.emotion_dropout_prob)


def test_audio_projection_validation_mirrors_reference(pkg):
    """nodes_vadv.py:170-181: TypeErrors for non-tensor / non-module / wrong rank / wrong feature size, raised before any device
    work; a CPU target has no fallback."""
    node = pkg.FloatApplyAudioProjection()
    layer = pkg.AudioProjectionLayer(768, 512, target_device="cpu")
    x = torch.zeros(1, 10, 768)
    with pytest.raises(TypeError):
        node.apply_projection(x.numpy(), layer)
    with pytest.raises(TypeError):
        node.apply_projection(x, "not a module")
    with pytest.raises(TypeError):
        node.apply_projection(x[0], layer)
    with pytest.raises(TypeError, match="only_last_features"):
        node.apply_projection(torch.zeros(1, 10, 9216), layer)
    with pytest.raises(pkg.FmtError):
        node.apply_projection(x, layer)


def test_distinct_condition_rows(pkg):
    """The AdaLN tables hold one row per DISTINCT condition row of forward_with_cfv's batched forward (FMT.py:360-392); this is the
    host-only view of that map (no GPU): checked against a direct construction of the condition rows from symbolic inputs."""
    import ctypes as C
    import numpy as np
    cabi = sys.modules[pkg.__name__ + "._cabi"]
    lib = cabi.load_library()
    N, P = 60, 10

    def reference_map(nb, B, dynamic):
        # symbolic condition row of (branch, clip, frame): what cat[wr, wa, we] holds, with the per-branch nulling of FMT.py:360-392
        null = {1: [(0, 0, 0)], 3: [(0, 1, 1), (0, 0, 0), (0, 0, 1)], 4: [(1, 1, 1), (0, 1, 1), (0, 0, 0), (0, 0, 1)]}[nb]   # (zr, za, ze)
        rows = []
        for br in range(nb):
            zr, za, ze = null[br]
            for b in range(B):
                for f in range(N):
                    ctx = f < P
                    wr = ("wr", b) if not zr else 0
                    wa = ("prev_wa", b, f) if ctx else (("wa", b, f) if not za else 0)         # prev_wa is never nulled (:366,388)
                    if ze:
                        we = 0
                    elif not dynamic:
                        we = ("we", b)                                                          # static emotion covers the context frames (:325-326)
                    else:
                        we = ("prev_we", b, f) if ctx else ("we", b, f)
                    rows.append((wr, wa, we))
        first = {}
        return [first.setdefault(r, len(first)) for r in rows], len(first)

    for nb, B, dynamic in [(3, 1, 0), (3, 2, 1), (4, 3, 0), (4, 1, 1), (1, 2, 0)]:
        out = (C.c_int32 * (nb * B * N))()
        U = lib.fmt_debug_condition_rows(nb, B, N, P, dynamic, out)
        ref, U_ref = reference_map(nb, B, dynamic)
        assert U == U_ref and list(out) == ref, (nb, B, dynamic, U, U_ref)
    assert lib.fmt_debug_condition_rows(3, 1, N, P, 0, None) == 2 * N + 1          # 121 of 180 rows per clip with 3-way CFG
    assert lib.fmt_debug_condition_rows(1, 4, N, P, 0, None) == 4 * N             # a single branch has nothing to share
    assert lib.fmt_debug_condition_rows(5, 1, N, P, 0, None) < 0
