"""StreamSampler on the B200: clips fed audio in pieces, one window per step on shared slots.

Pins: streams fed in random pieces == sample_clips bitwise on the same plan; one stream on one slot == the one-clip call bitwise
(dataflow window kernel); per-stream guidance, dynamic emotion and midpoint against the oracle (fp32 / bf16x3 1e-4 relative);
streams that join mid-flight in slots other streams used, writing nothing but their own frames; a 30-window stream with a bounded
buffer; launches and slot-record copies per step; seeded streams == sample_clips with the same seeds.
"""
import random

import pytest
import torch

import cases
from __graft_entry__ import load_package
from test_gpu_guidance import B, MIX, guidance_kw, with_guidance
from test_gpu_multiclip import LENGTHS, make_clips, oracle, solo
from test_gpu_parity import model_for

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
KW = dict(nfe=4, method="euler", a_cfg_scale=2.0, r_cfg_scale=1.0, e_cfg_scale=1.0, include_r_cfg=False)
GUIDANCE = ("a_cfg_scale", "r_cfg_scale", "e_cfg_scale", "include_r_cfg")


@pytest.fixture(scope="module")
def pkg():
    return load_package()


def open_clip(sm, c, dynamic=False):
    own = {k: c[k] for k in GUIDANCE if k in c}
    return sm.open(c["r_s"].to(DEV), None if dynamic else c["we"].to(DEV), noise=c["noise"], **own)


def run_streams(sm, clips, seed, dynamic=False, max_chunk=120):
    """Feeds every clip in seeded random pieces of 1..max_chunk frames, interleaved across streams, stepping after each round;
    returns each clip's frames, concatenated in window order."""
    rng = random.Random(seed)
    streams = [open_clip(sm, c, dynamic) for c in clips]
    fed = [0] * len(clips)
    got = {s: [] for s in streams}
    while not all(s.done for s in streams):
        order = list(range(len(clips)))
        rng.shuffle(order)
        for i in order:
            T = clips[i]["audio_num_frames"]
            if fed[i] < T:
                t = min(T - fed[i], rng.randint(1, max_chunk))
                sm.feed(streams[i], clips[i]["wa"][:, fed[i]:fed[i] + t].to(DEV),
                        clips[i]["we"][:, fed[i]:fed[i] + t].to(DEV) if dynamic else None)
                fed[i] += t
                if fed[i] == T:
                    sm.finish(streams[i])
        for s, o in sm.step().items():
            got[s].append(o)
    outs = [torch.cat(got[s], dim=1).cpu() for s in streams]
    for s in streams:
        sm.close(s)
    return outs


@pytest.mark.parametrize("mode", ["bf16", "bf16x3"])
def test_streams_equal_sample_clips_bitwise(pkg, mode):
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    clips = make_clips(d, LENGTHS, seed=300)
    kw = dict(KW, mode=mode)
    ref = [o.cpu() for o in pkg.sample_clips(model, clips, device=DEV, **kw)]
    slots = pkg.clip_schedule([-(-T // d.frames_per_clip) for T in LENGTHS]).slots
    sm = pkg.StreamSampler(model, slots=slots, device=DEV, **kw)
    outs = run_streams(sm, clips, seed=1)
    for i, (o, r) in enumerate(zip(outs, ref)):
        assert o.shape == r.shape and torch.equal(o, r), (i, (o - r).abs().max().item())


def test_one_stream_equals_the_single_clip_call(pkg):
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    (c,) = make_clips(d, [149], seed=310)
    kw = dict(KW, mode="bf16")
    sm = pkg.StreamSampler(model, slots=1, device=DEV, **kw)
    (out,) = run_streams(sm, [c], seed=2)
    assert pkg.backend_for(model, DEV).window_kernel_status() == 0          # one slot, 3-way CFG: the dataflow window kernel
    assert torch.equal(out, solo(pkg, model, c, **kw))


@pytest.mark.parametrize("mode,dynamic,method", [("fp32", False, "euler"), ("bf16x3", True, "midpoint")])
def test_mixed_guidance_streams_match_the_oracle(pkg, mode, dynamic, method):
    """Per-stream guidance of 3, 3, 4 and 1 branches on a 4-branch plan."""
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    clips = make_clips(d, LENGTHS[:4], seed=320, dynamic=dynamic)
    clips = with_guidance(clips, MIX)
    kw = guidance_kw(B, nfe=3, method=method, mode=mode)
    sm = pkg.StreamSampler(model, slots=3, we_dynamic=dynamic, device=DEV, **kw)
    assert sm.n_branches == 4
    outs = run_streams(sm, clips, seed=3, dynamic=dynamic)
    for i, (c, o, g) in enumerate(zip(clips, outs, MIX)):
        ref = oracle(d, c, **guidance_kw(g, nfe=3, method=method, mode=mode))
        assert o.shape == ref.shape and cases.rel_err(o, ref) <= 1e-4, (i, cases.rel_err(o, ref))


class GuardedOutputs:
    """Backend proxy: every window's outputs go to one NaN-filled buffer with guard rows around each stream's frames."""
    guard = 3

    def __init__(self, be):
        self.be, self.device, self.dims = be, be.device, be.dims
        self.clean = True

    def configure(self, *plan):
        self.be.configure(*plan)

    def sample_windows(self, r_s, wa, we, x0, ctx, out, *rest):
        g, rows = self.guard, [o.shape[1] for o in out]
        buf = torch.full((sum(rows) + g * (len(rows) + 1), self.dims.dim_w), float("nan"), device=self.device)
        starts = [g + sum(rows[:i]) + g * i for i in range(len(rows))]
        views = [buf[s:s + n] for s, n in zip(starts, rows)]
        self.be.sample_windows(r_s, wa, we, x0, ctx, views, *rest)
        written = torch.zeros(buf.shape[0], dtype=torch.bool)
        for s, n in zip(starts, rows):
            written[s:s + n] = True
        host = buf.cpu()
        self.clean &= bool(torch.isfinite(host[written]).all()) and bool(torch.isnan(host[~written]).all())
        for o, v in zip(out, views):
            o.copy_(v.view_as(o))


def test_streams_join_mid_flight(pkg):
    """Two long streams run alone for three steps; then shorter ones open and take the slots as the first streams move and finish."""
    d = cases.FmtDims()
    L = d.frames_per_clip
    model = model_for(pkg, "full")
    clips = make_clips(d, [300, 120, 100, 149, 51, 23], seed=330)
    kw = dict(KW, nfe=3, mode="bf16x3")
    sm = pkg.StreamSampler(model, slots=3, device=DEV, **kw)
    proxy = GuardedOutputs(sm._be)
    sm._be = proxy
    got = {}
    first = [open_clip(sm, c) for c in clips[:2]]
    for s, c in zip(first, clips[:2]):
        sm.feed(s, c["wa"].to(DEV))
        sm.finish(s)
    slot_of = []
    for _ in range(3):
        slot_of.append(sm.ready())
        for s, o in sm.step().items():
            got.setdefault(s, []).append(o)
    late = [open_clip(sm, c) for c in clips[2:]]
    for s, c in zip(late, clips[2:]):
        sm.feed(s, c["wa"].to(DEV))
        sm.finish(s)
    streams = first + late
    while not all(s.done for s in streams):
        slot_of.append(sm.ready())
        for s, o in sm.step().items():
            got.setdefault(s, []).append(o)
    assert slot_of[:3] == [first] * 3
    assert slot_of[3] == [first[0], late[0], late[1]]          # late[0] takes slot 1, which first[1] ran in
    assert slot_of[4] == [late[2], late[3], first[0]]          # first[0] moves from slot 0 to slot 2, its context with it
    assert proxy.clean
    for i, (s, c) in enumerate(zip(streams, clips)):
        o = torch.cat(got[s], dim=1).cpu()
        assert o.shape == (1, c["audio_num_frames"], d.dim_w) and len(got[s]) == -(-c["audio_num_frames"] // L)
        assert cases.rel_err(o, oracle(d, c, **kw)) <= 1e-4, (i, cases.rel_err(o, oracle(d, c, **kw)))


def test_long_stream_is_bounded_and_equals_the_offline_call(pkg):
    """configs[2]'s 60 s clip (1500 frames, 30 windows) fed 50 frames at a time."""
    d = cases.FmtDims()
    L, P = d.frames_per_clip, d.num_prev_frames
    model = model_for(pkg, "full")
    (c,) = make_clips(d, [1500], seed=340)
    kw = dict(KW, nfe=10, mode="bf16")
    (ref,) = pkg.sample_clips(model, [c], device=DEV, **kw)
    sm = pkg.StreamSampler(model, slots=1, device=DEV, **kw)
    s = open_clip(sm, c)
    parts, peak = [], 0
    for k in range(0, 1500, 50):
        sm.feed(s, c["wa"][:, k:k + 50].to(DEV))
        if k + 50 == 1500:
            sm.finish(s)
        parts += list(sm.step().values())
        peak = max(peak, s.buffered_frames)
    assert s.done and len(parts) == 30
    assert peak <= P + L
    assert torch.equal(torch.cat(parts, dim=1).cpu(), ref.cpu())


def test_cost_per_step_and_seeded_noise(pkg):
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    clips = make_clips(d, LENGTHS, seed=350)
    seeded = [dict({k: v for k, v in c.items() if k != "noise"}, seed=1000 + i) for i, c in enumerate(clips)]
    kw = dict(KW, mode="bf16")
    ref = [o.cpu() for o in pkg.sample_clips(model, seeded, device=DEV, **kw)]
    slots = pkg.clip_schedule([-(-T // d.frames_per_clip) for T in LENGTHS]).slots
    sm = pkg.StreamSampler(model, slots=slots, device=DEV, **kw)
    be = pkg.backend_for(model, DEV)
    streams = [sm.open(c["r_s"].to(DEV), c["we"].to(DEV), seed=c["seed"]) for c in seeded]
    for s, c in zip(streams, seeded):
        sm.feed(s, c["wa"].to(DEV))
        sm.finish(s)
    got = {s: [] for s in streams}
    torch.cuda.synchronize()
    be.launch_count(reset=True)
    n_steps = 0
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        while not all(s.done for s in streams):
            for s, o in sm.step().items():
                got[s].append(o)
            n_steps += 1
        torch.cuda.synchronize()
    assert be.launch_count() == n_steps * (1 + be.graph_kernel_nodes()), (be.launch_count(), n_steps, be.graph_kernel_nodes())
    h2d = [e for e in prof.events() if e.name.startswith("Memcpy HtoD")]
    assert len(h2d) == n_steps, [e.name for e in h2d]
    assert sum(len(v) for v in got.values()) == sum(-(-T // d.frames_per_clip) for T in LENGTHS)
    for i, (s, r) in enumerate(zip(streams, ref)):
        assert torch.equal(torch.cat(got[s], dim=1).cpu(), r), i
