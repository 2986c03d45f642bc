"""Per-clip guidance in sample_clips on the B200: each clip's own a/r/e scales and include_r_cfg in one call.

Pins: per-clip settings equal to the call's == today's call bitwise; a clip's result does not depend on the other clips' settings
(bitwise, same plan); mixed 1-, 3- and 4-branch clips against the oracle run on each clip alone with its own settings (fp32 /
bf16x3 1e-4 relative; bf16 2e-2 max-abs and 1e-2 of the clip sampled alone), on the per-op path and, with short windows, in the
persistent kernels; launch count and determinism of mixed calls.
"""
import pytest
import torch

import cases
from __graft_entry__ import load_package
from oracle import fmt_oracle as O
from test_gpu_multiclip import LENGTHS, make_clips, oracle, solo
from test_gpu_parity import model_for

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
A = (2.0, 1.0, 1.0, False)                       # 3 branches
B = (2.0, 0.5, 1.5, True)                        # 4 branches
MIX = [(2.0, 1.0, 1.0, False), (1.0, 1.0, 3.0, False), (2.0, 0.5, 1.5, True), (1.0, 1.0, 1.0, False)]   # 3, 3, 4, 1 branches
KEYS = ("a_cfg_scale", "r_cfg_scale", "e_cfg_scale", "include_r_cfg")


@pytest.fixture(scope="module")
def pkg():
    return load_package()


def with_guidance(clips, settings):
    return [dict(c, **dict(zip(KEYS, g))) for c, g in zip(clips, settings)]


def guidance_kw(g, **kw):
    return dict(kw, **dict(zip(KEYS, g)))


def slot_args(clips, dev=DEV):
    return [[c[k].to(dev).contiguous() for c in clips] for k in ("r_s", "wa", "we")] + [[c["noise"].to(dev) for c in clips]]


@pytest.mark.parametrize("mode,call", [("bf16", A), ("fp32", B)])
def test_per_clip_settings_equal_to_the_call_are_bitwise_today(pkg, mode, call):
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    clips = make_clips(d, LENGTHS, seed=200)
    kw = guidance_kw(call, nfe=3, method="euler", mode=mode)
    today = pkg.sample_clips(model, clips, device=DEV, **kw)
    per_clip = pkg.sample_clips(model, with_guidance(clips, [call] * len(clips)), device=DEV, **guidance_kw((1.0, 1.0, 1.0, False), **kw))
    for i, (x, y) in enumerate(zip(today, per_clip)):
        assert torch.equal(x, y), i


@pytest.mark.parametrize("mode", ["bf16", "bf16x3", "fp32"])
def test_a_clip_does_not_depend_on_the_other_clips_settings(pkg, mode):
    """LENGTHS with A for the even clips and B for the odd ones, then A for all on the same (4-branch) plan: the A clips agree."""
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    clips = make_clips(d, LENGTHS, seed=210)
    n = len(clips)
    mixed = [A if i % 2 == 0 else B for i in range(n)]
    outs = pkg.sample_clips(model, with_guidance(clips, mixed), device=DEV, nfe=3, method="euler", mode=mode)
    sch = pkg.clip_schedule([-(-T // d.frames_per_clip) for T in LENGTHS])
    be = pkg.backend_for(model, DEV)
    be.configure(sch.slots, 4, False, 3, "euler", mode)                    # the plan of the mixed call
    r_s, wa, we, noise = slot_args(clips)
    all_a = be.sample_clips(r_s, wa, we, LENGTHS, noise, [A[0]] * n, [A[1]] * n, [A[2]] * n, n_branches=[3] * n)
    for i in range(0, n, 2):
        assert torch.equal(outs[i], all_a[i]), i


MIXED = [  # mode, dynamic emotion, method, nfe
    ("fp32", False, "euler", 3),
    ("bf16x3", True, "midpoint", 3),
    ("bf16x3", False, "euler", 3),
    ("bf16", False, "euler", 4),
    ("bf16", True, "heun2", 3),
]


@pytest.mark.parametrize("mode,dynamic,method,nfe", MIXED)
def test_mixed_guidance_matches_the_oracle_per_clip(pkg, mode, dynamic, method, nfe):
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    clips = make_clips(d, LENGTHS, seed=220 + nfe, dynamic=dynamic)
    settings = [MIX[i % len(MIX)] for i in range(len(clips))]
    sch = pkg.clip_schedule([-(-T // d.frames_per_clip) for T in LENGTHS])
    assert max(sch.start) > 0                                               # some clips start mid-call in a reused slot
    outs = pkg.sample_clips(model, with_guidance(clips, settings), device=DEV, nfe=nfe, method=method, mode=mode)
    for i, (c, g, o) in enumerate(zip(clips, settings, outs)):
        kw = guidance_kw(g, nfe=nfe, method=method, mode=mode)
        o = o.cpu()
        ref = oracle(d, c, **kw)
        assert o.shape == ref.shape == (1, c["audio_num_frames"], d.dim_w)
        if mode == "bf16":
            assert cases.max_abs(o, ref) <= 2e-2, (i, g, sch.start[i], cases.max_abs(o, ref))
            alone = solo(pkg, model, c, **kw)
            assert cases.max_abs(o, alone) <= 1e-2, (i, g, sch.start[i], cases.max_abs(o, alone))
        else:
            assert cases.rel_err(o, ref) <= 1e-4, (i, g, sch.start[i], cases.rel_err(o, ref))


def _short_window_model(pkg, d, W):
    opt = pkg.BaseOptions()
    for k, v in d.as_dict().items():
        if hasattr(opt, k):
            setattr(opt, k, v)
    return pkg.FmtModel(W, opt, target_device=DEV)


@pytest.mark.parametrize("window_flag", ["3", "1"])
@pytest.mark.parametrize("settings", [[B, A, MIX[1]], [A, MIX[3], MIX[1]]], ids=["3and4", "1and3"])
def test_persistent_kernels_combine_per_slot(pkg, monkeypatch, window_flag, settings):
    """N = 32 frames: two slots of 4 branches are 256 token rows, so the whole window runs in one persistent kernel (the dataflow
    kernel, or the barrier-stepped one with FMT_WINDOW=1) with different guidance in its two slots."""
    from oracle.synth import FmtDims, synth_state_dict
    d = FmtDims(num_prev_frames=6, wav2vec_sec=1.04, fmt_depth=3)
    assert d.total_frames == 32
    W = synth_state_dict(d, seed=5)
    lengths = [70, 45, 20]                                                  # 3, 2, 1 windows of 26 frames: 2 slots, one refill
    sch = pkg.clip_schedule([-(-T // d.frames_per_clip) for T in lengths])
    assert sch.slots == 2 and max(sch.start) > 0
    clips = with_guidance(make_clips(d, lengths, seed=230), settings)
    nfe, plan_nb = 3, max(pkg.n_branches_for(*g) for g in settings)
    monkeypatch.setenv("FMT_WINDOW", window_flag)
    model = _short_window_model(pkg, d, W)
    be = pkg.backend_for(model, DEV)
    be.configure(sch.slots, plan_nb, False, nfe, "euler", "bf16")
    assert be.window_kernel_status() == 0
    outs = [o.cpu() for o in pkg.sample_clips(model, clips, device=DEV, nfe=nfe, method="euler", mode="bf16")]
    assert be.window_kernel_status() == 0
    monkeypatch.setenv("FMT_WINDOW", "0")
    per_op_model = _short_window_model(pkg, d, W)
    per_op = pkg.sample_clips(per_op_model, clips, device=DEV, nfe=nfe, method="euler", mode="bf16")
    assert pkg.backend_for(per_op_model, DEV).window_kernel_status() == -1
    torch.backends.cuda.matmul.allow_tf32 = False
    Wd = {k: v.to(DEV) for k, v in W.items()}
    for i, (c, g, o, p) in enumerate(zip(clips, settings, outs, per_op)):
        with torch.no_grad():
            ref = O.sample_loop(Wd, d, c["r_s"].to(DEV), c["wa"].to(DEV), c["we"].to(DEV), c["audio_num_frames"], nfe=nfe,
                                noise=c["noise"].unsqueeze(1).to(DEV), **dict(zip(KEYS, g))).cpu()
        assert cases.max_abs(o, ref) <= 2e-2, (i, g, cases.max_abs(o, ref))
        assert cases.max_abs(o, p.cpu()) <= 1e-2, (i, g, cases.max_abs(o, p.cpu()))


def test_mixed_launch_count_determinism_and_bad_branch_counts(pkg):
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    clips = make_clips(d, LENGTHS, seed=240)
    n = len(clips)
    n_win = [-(-T // d.frames_per_clip) for T in LENGTHS]
    sch = pkg.clip_schedule(n_win)
    settings = [MIX[i % len(MIX)] for i in range(n)]
    a, r, e, _ = zip(*settings)
    nb = [pkg.n_branches_for(*g) for g in settings]
    be = pkg.backend_for(model, DEV)
    be.configure(sch.slots, 4, False, 3, "euler", "bf16")
    r_s, wa, we, noise = slot_args(clips)
    be.launch_count(reset=True)
    first = [o.clone() for o in be.sample_clips(r_s, wa, we, LENGTHS, noise, a, r, e, n_branches=nb)]
    torch.cuda.synchronize()
    assert be.launch_count() == sch.makespan * (1 + be.graph_kernel_nodes())
    again = be.sample_clips(r_s, wa, we, LENGTHS, noise, a, r, e, n_branches=nb)
    for i, (x, y) in enumerate(zip(first, again)):
        assert torch.equal(x, y), i
    for bad in ([2] * n, [5] * n):
        with pytest.raises(ValueError):
            be.sample_clips(r_s, wa, we, LENGTHS, noise, a, r, e, n_branches=bad)
    be.configure(sch.slots, 3, False, 3, "euler", "bf16")
    with pytest.raises(ValueError):                                         # more branches than the plan
        be.sample_clips(r_s, wa, we, LENGTHS, noise, a, r, e, n_branches=nb)
    be.configure(sch.slots, 1, False, 3, "euler", "bf16")
    with pytest.raises(ValueError):                                         # a 1-branch plan takes 1-branch clips only
        be.sample_clips(r_s, wa, we, LENGTHS, noise, 2.0, 1.0, 1.0, n_branches=[3] + [1] * (n - 1))
