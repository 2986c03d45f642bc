"""sample_clips on the B200: many clips of different lengths on refilled batch slots, each held to the gates of a one-clip call.

Pins: equal lengths == the batched fmt_sample_clip bitwise; one clip == the B = 1 dataflow kernel bitwise.  Mixed lengths: every
clip against the oracle run on that clip alone with the same noise (fp32 / bf16x3 1e-4 relative; bf16 2e-2 max-abs and 1e-2 of
the clip sampled alone), including clips that start mid-call in a slot another clip used before.
"""
import pytest
import torch

import cases
from __graft_entry__ import load_package
from test_gpu_parity import _oracle_on_gpu, model_for

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
LENGTHS = [23, 50, 51, 100, 149, 260, 300]


@pytest.fixture(scope="module")
def pkg():
    return load_package()


def make_clips(d, lengths, seed, dynamic=False):
    from oracle.synth import synth_inputs
    clips = []
    for i, T in enumerate(lengths):
        r_s, wa, we = synth_inputs(d, 1, T, seed=seed + i, dynamic_we=dynamic)
        g = torch.Generator().manual_seed(seed * 1000 + i)
        noise = torch.randn(-(-T // d.frames_per_clip), d.frames_per_clip, d.dim_w, generator=g)
        clips.append(dict(r_s=r_s, wa=wa, we=we, audio_num_frames=T, noise=noise))
    return clips


def solo(pkg, model, c, **kw):
    """The clip alone through the existing one-call path (perform_ode_sampling_loop, batch 1)."""
    d = pkg.backend_for(model, DEV).dims
    return pkg.perform_ode_sampling_loop(model, c["r_s"].to(DEV), c["wa"].to(DEV), c["we"].to(DEV), c["audio_num_frames"], d.num_prev_frames,
                                         d.frames_per_clip, d.dim_w, kw["nfe"], kw["method"], 1e-5, 1e-5, DEV, kw["a_cfg_scale"],
                                         kw["r_cfg_scale"], kw["e_cfg_scale"], kw["include_r_cfg"], None, mode=kw["mode"],
                                         noise=c["noise"].unsqueeze(1)).cpu()


def oracle(d, c, **kw):
    return _oracle_on_gpu(d, c["r_s"], c["wa"], c["we"], c["audio_num_frames"], c["noise"].unsqueeze(1), nfe=kw["nfe"], method=kw["method"],
                          a_cfg_scale=kw["a_cfg_scale"], r_cfg_scale=kw["r_cfg_scale"], e_cfg_scale=kw["e_cfg_scale"],
                          include_r_cfg=kw["include_r_cfg"])


def test_equal_lengths_equal_the_batched_call(pkg):
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    clips = make_clips(d, [100, 100, 100], seed=50)
    kw = dict(nfe=3, method="euler", a_cfg_scale=2.0, r_cfg_scale=1.0, e_cfg_scale=1.0, include_r_cfg=False, mode="bf16")
    outs = pkg.sample_clips(model, clips, device=DEV, **kw)
    assert pkg.clip_schedule([2, 2, 2]).slots == 3
    be = pkg.backend_for(model, DEV)
    be.configure(3, 3, False, 3, "euler", "bf16")
    cat = lambda k: torch.cat([c[k] for c in clips]).to(DEV).contiguous()          # noqa: E731
    noise = torch.stack([c["noise"] for c in clips], dim=1).to(DEV).contiguous()
    ref = be.sample_clip(cat("r_s"), cat("wa"), cat("we"), 100, noise, 2.0, 1.0, 1.0).cpu()
    for i, o in enumerate(outs):
        assert o.shape == (1, 100, d.dim_w) and torch.equal(o.cpu(), ref[i:i + 1]), i


def test_one_clip_equals_the_single_clip_call(pkg):
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    (c,) = make_clips(d, [149], seed=60)
    kw = dict(nfe=4, method="euler", a_cfg_scale=2.0, r_cfg_scale=1.0, e_cfg_scale=1.0, include_r_cfg=False, mode="bf16")
    (out,) = pkg.sample_clips(model, [c], device=DEV, **kw)
    assert pkg.backend_for(model, DEV).window_kernel_status() == 0          # one clip, 3-way CFG: the dataflow window kernel
    assert torch.equal(out.cpu(), solo(pkg, model, c, **kw))


MIXED = [  # mode, dynamic emotion, (a, r, e, include_r_cfg), method, nfe
    ("fp32", False, (2.0, 1.0, 1.0, False), "euler", 3),
    ("bf16x3", True, (2.0, 0.5, 1.5, True), "midpoint", 3),
    ("bf16x3", False, (2.0, 1.0, 1.0, False), "euler", 4),
    ("bf16", False, (2.0, 1.0, 1.0, False), "euler", 4),
    ("bf16", True, (2.0, 0.5, 1.5, True), "heun2", 3),
]


@pytest.mark.parametrize("mode,dynamic,scales,method,nfe", MIXED)
def test_mixed_lengths_match_the_oracle_per_clip(pkg, mode, dynamic, scales, method, nfe):
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    a, r, e, inc = scales
    kw = dict(nfe=nfe, method=method, a_cfg_scale=a, r_cfg_scale=r, e_cfg_scale=e, include_r_cfg=inc, mode=mode)
    clips = make_clips(d, LENGTHS, seed=70 + nfe, dynamic=dynamic)
    sch = pkg.clip_schedule([-(-T // d.frames_per_clip) for T in LENGTHS])
    assert sch.slots == 4 and sch.makespan == 6 and max(sch.start) > 0       # some clips start mid-call in a reused slot
    outs = pkg.sample_clips(model, clips, device=DEV, **kw)
    for i, (c, o) in enumerate(zip(clips, outs)):
        o = o.cpu()
        ref = oracle(d, c, **kw)
        assert o.shape == ref.shape == (1, c["audio_num_frames"], d.dim_w)
        if mode == "bf16":
            assert cases.max_abs(o, ref) <= 2e-2, (i, sch.start[i], cases.max_abs(o, ref))
            alone = solo(pkg, model, c, **kw)
            assert cases.max_abs(o, alone) <= 1e-2, (i, sch.start[i], cases.max_abs(o, alone))
        else:
            assert cases.rel_err(o, ref) <= 1e-4, (i, sch.start[i], cases.rel_err(o, ref))


def test_refilled_slot_starts_from_zero_context(pkg):
    """[300, 50 x 6]: two slots; the six short clips run one after another in slot 1, each with its own zero context."""
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    lengths = [300] + [50] * 6
    sch = pkg.clip_schedule([-(-T // d.frames_per_clip) for T in lengths])
    assert sch.slots == 2 and sch.start[1:] == (0, 1, 2, 3, 4, 5)
    clips = make_clips(d, lengths, seed=90)
    kw = dict(nfe=4, method="euler", a_cfg_scale=2.0, r_cfg_scale=1.0, e_cfg_scale=1.0, include_r_cfg=False, mode="bf16")
    outs = pkg.sample_clips(model, clips, device=DEV, **kw)
    for i, (c, o) in enumerate(zip(clips, outs)):
        o = o.cpu()
        assert cases.max_abs(o, oracle(d, c, **kw)) <= 2e-2, i
        assert cases.max_abs(o, solo(pkg, model, c, **kw)) <= 1e-2, i
    kw32 = dict(kw, mode="bf16x3")
    outs = pkg.sample_clips(model, clips, device=DEV, **kw32)
    for i, (c, o) in enumerate(zip(clips, outs)):
        assert cases.rel_err(o.cpu(), oracle(d, c, **kw32)) <= 1e-4, i


def test_exact_writes_work_and_determinism(pkg):
    """Outputs are views into one NaN-filled buffer with guard rows between clips: every clip's frames are written, no guard row is.
    The call costs the schedule's windows and nothing more, and it is bitwise reproducible."""
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    clips = make_clips(d, LENGTHS, seed=110)
    n_win = [-(-T // d.frames_per_clip) for T in LENGTHS]
    sch = pkg.clip_schedule(n_win)
    be = pkg.backend_for(model, DEV)
    be.configure(sch.slots, 3, False, 4, "euler", "bf16")
    guard = 3
    offs, o = [], guard
    for T in LENGTHS:
        offs.append(o)
        o += T + guard
    buf = torch.full((o, d.dim_w), float("nan"), device=DEV)
    views = [buf[s:s + T] for s, T in zip(offs, LENGTHS)]
    r_s, wa, we = ([c[k].to(DEV).contiguous() for c in clips] for k in ("r_s", "wa", "we"))
    noise = [c["noise"].to(DEV) for c in clips]
    ticks = []
    be.launch_count(reset=True)
    be.sample_clips(r_s, wa, we, LENGTHS, noise, 2.0, 1.0, 1.0, progress=lambda w, n: ticks.append((w, n)), out=views)
    torch.cuda.synchronize()
    launches = be.launch_count()
    assert sch.makespan == max(n_win)                                        # short clips add no windows
    assert launches == sch.makespan * (1 + be.graph_kernel_nodes()), (launches, sch.makespan, be.graph_kernel_nodes())
    assert ticks == [(w, sch.makespan) for w in range(sch.makespan)]
    written = torch.zeros(o, dtype=torch.bool)
    for s, T in zip(offs, LENGTHS):
        written[s:s + T] = True
    host = buf.cpu()
    assert torch.isfinite(host[written]).all()
    assert torch.isnan(host[~written]).all()
    first = host.clone()
    again = be.sample_clips(r_s, wa, we, LENGTHS, noise, 2.0, 1.0, 1.0)
    for s, T, x in zip(offs, LENGTHS, again):
        assert torch.equal(x.cpu()[0], first[s:s + T])
