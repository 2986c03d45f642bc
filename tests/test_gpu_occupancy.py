"""StreamSampler steps at partial occupancy on the B200: a step with k ready streams replays the window graph of occupancy_slots(S, k)
slots, and every stream's frames stay bitwise equal to the plan's full graph.

Pins: a 16-slot sampler stepped through occupancies 16, 1, 2, 3, 5 and 9 == each clip through FmtBackend.sample_clips on the same
16-slot plan (every slot busy), bf16 and bf16x3, with last_window_slots() == occupancy_slots(16, k) after each step, launches of
1 + graph_kernel_nodes() and one host-to-device copy per step, and the same bits again after another plan took the backend; per-stream
guidance of 1, 3 and 4 branches on a 4-branch plan, dynamic emotion and per-stream schedules (the per-slot graph's buckets) == the
full-graph call, fp32 also against the oracle; plans whose window graph is the dataflow kernel keep their one graph at every
occupancy.
"""
import pytest
import torch

import cases
from __graft_entry__ import load_package
from test_gpu_guidance import MIX, guidance_kw, with_guidance
from test_gpu_multiclip import make_clips, oracle
from test_gpu_parity import model_for
from test_gpu_schedules import SCHEDULES, with_schedules

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
S = 16
OCCUPANCY = [16, 1, 2, 3, 5, 9]                     # 16 first, while every stream still has a window left
LENGTHS = [101 + 3 * i for i in range(S)]           # 3 windows each: sample_clips schedules them on 16 slots, one clip per slot
KW = dict(nfe=3, method="euler", a_cfg_scale=2.0, r_cfg_scale=1.0, e_cfg_scale=1.0, include_r_cfg=False)
R_CFG = (2.0, 0.5, 1.5, True)                       # 4 branches


@pytest.fixture(scope="module")
def pkg():
    return load_package()


def on_device(clips):
    """The clips' tensors on the device, so that feeding and stepping copy nothing from the host but the slot records."""
    return [{k: v.to(DEV) if torch.is_tensor(v) else v for k, v in c.items()} for c in clips]


def run_occupancies(pkg, sm, clips, occupancy=OCCUPANCY, dynamic=()):
    """Steps sm so that step j has exactly occupancy[j % len(occupancy)] ready streams (all that are left, at the end): before each step
    the chosen streams get exactly their next window's frames (and finish with their last).  The choice rotates over the streams
    that are left, so a stream runs in different slots.  Returns each clip's frames and (k, last_window_slots()) of every step."""
    L = sm.dims.frames_per_clip
    be = sm._be
    streams = []
    for i, c in enumerate(clips):
        own = {k: c[k] for k in ("a_cfg_scale", "r_cfg_scale", "e_cfg_scale", "include_r_cfg", "nfe", "method") if k in c}
        dyn = i in dynamic
        streams.append(sm.open(c["r_s"], None if dyn else c["we"], noise=c["noise"], we_dynamic=dyn, **own))
    fed = [0] * len(clips)
    got = {s: [] for s in streams}
    seen = []
    j = 0
    while not all(s.done for s in streams):
        live = [i for i, c in enumerate(clips) if fed[i] < c["audio_num_frames"]]
        k = min(occupancy[j % len(occupancy)], len(live))
        for t in range(k):
            i = live[(j + t) % len(live)]
            T = clips[i]["audio_num_frames"]
            n = min(L, T - fed[i])
            sm.feed(streams[i], clips[i]["wa"][:, fed[i]:fed[i] + n], clips[i]["we"][:, fed[i]:fed[i] + n] if i in dynamic else None)
            fed[i] += n
            if fed[i] == T:
                sm.finish(streams[i])
        ran = sm.step()
        assert len(ran) == k, (j, k, len(ran))
        seen.append((k, be.last_window_slots()))
        for s, o in ran.items():
            got[s].append(o)
        j += 1
    outs = [torch.cat(got[s], dim=1).cpu() for s in streams]
    for s in streams:
        sm.close(s)
    return outs, seen


@pytest.mark.parametrize("mode", ["bf16", "bf16x3"])
def test_partial_occupancy_equals_the_full_graph(pkg, mode):
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    clips = on_device(make_clips(d, LENGTHS, seed=600))
    kw = dict(KW, mode=mode)
    assert pkg.clip_schedule([-(-T // d.frames_per_clip) for T in LENGTHS]).slots == S
    ref = [o.cpu() for o in pkg.sample_clips(model, clips, device=DEV, **kw)]
    be = pkg.backend_for(model, DEV)
    sm = pkg.StreamSampler(model, slots=S, device=DEV, **kw)
    assert be.window_kernel_status() == -1                                  # 16 slots x 3 branches: one kernel per op
    torch.cuda.synchronize()
    be.launch_count(reset=True)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        outs, seen = run_occupancies(pkg, sm, clips)
        torch.cuda.synchronize()
    n_steps = len(seen)
    assert {k for k, _ in seen} >= set(OCCUPANCY)
    assert all(slots == pkg.occupancy_slots(S, k) for k, slots in seen), seen
    assert be.launch_count() == n_steps * (1 + be.graph_kernel_nodes()), (be.launch_count(), n_steps, be.graph_kernel_nodes())
    h2d = [e for e in prof.events() if e.name.startswith("Memcpy HtoD")]
    assert len(h2d) == n_steps, [e.name for e in h2d]
    for i, (o, r) in enumerate(zip(outs, ref)):
        assert o.shape == r.shape and torch.equal(o, r), (i, (o - r).abs().max().item())

    # another plan takes the backend (its own buckets), then this sampler's plan comes back with buckets captured anew
    other = pkg.StreamSampler(model, slots=8, device=DEV, **dict(kw, nfe=2))
    run_occupancies(pkg, other, clips[:5], occupancy=[3, 1])
    again, seen2 = run_occupancies(pkg, sm, clips, occupancy=OCCUPANCY[::-1])
    assert all(slots == pkg.occupancy_slots(S, k) for k, slots in seen2), seen2
    for i, (o, r) in enumerate(zip(again, ref)):
        assert torch.equal(o, r), (i, (o - r).abs().max().item())


@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_per_stream_settings_at_partial_occupancy(pkg, mode):
    """Guidance of 3, 3, 4 and 1 branches on a 4-branch plan, every third stream on dynamic emotion and streams on five schedules:
    steps that mix schedules replay the per-slot window graph of their bucket."""
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    dynamic = {i for i in range(S) if i % 3 == 1}
    static, dyn = make_clips(d, LENGTHS, seed=610), make_clips(d, LENGTHS, seed=610, dynamic=True)
    clips = [dict(dyn[i], we_dynamic=True) if i in dynamic else dict(static[i], we_dynamic=False) for i in range(S)]
    clips = with_guidance(clips, [MIX[i % len(MIX)] for i in range(S)])
    schedules = [(n_, m) for m, n_ in (SCHEDULES[i % len(SCHEDULES)] for i in range(S))]
    clips = on_device(with_schedules(clips, schedules))
    kw = guidance_kw(R_CFG, nfe=2, method="rk4", mode=mode)                # the plan: 4 branches, 8 evaluations (rk4 x 2)
    ref = [o.cpu() for o in pkg.sample_clips(model, clips, device=DEV, **kw)]
    be = pkg.backend_for(model, DEV)
    assert be._plan_key[:2] == (S, 4) and be._plan_key[3:5] == (2, "rk4")
    sm = pkg.StreamSampler(model, slots=S, device=DEV, **kw)
    outs, seen = run_occupancies(pkg, sm, clips, dynamic=dynamic)
    assert be.ode_graph_kernel_nodes() > 0
    assert all(slots == pkg.occupancy_slots(S, k) for k, slots in seen), seen
    for i, (o, r) in enumerate(zip(outs, ref)):
        assert o.shape == r.shape and torch.equal(o, r), (i, (o - r).abs().max().item())
    if mode == "fp32":
        for i in (0, 1, 2, 3, 7):                                           # 3, 3 (dynamic), 4 and 1 branches; rk4, euler, heun2, ...
            c = {k: v.cpu() if torch.is_tensor(v) else v for k, v in clips[i].items()}
            g = MIX[i % len(MIX)]
            ref_o = oracle(d, c,
                           **guidance_kw(g, nfe=schedules[i][0], method=schedules[i][1]))
            assert cases.rel_err(outs[i], ref_o) <= 1e-4, (i, cases.rel_err(outs[i], ref_o))


@pytest.mark.parametrize("slots,guidance", [(1, (2.0, 1.0, 1.0, False)), (4, (1.0, 1.0, 1.0, False))])
def test_dataflow_plans_keep_their_one_graph(pkg, slots, guidance):
    """slots=1 with 3-way CFG and a 1-branch plan of 4 slots run the dataflow window kernel at every occupancy."""
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    clips = on_device(make_clips(d, LENGTHS[:slots], seed=620))
    kw = guidance_kw(guidance, nfe=3, method="euler", mode="bf16")
    ref = [o.cpu() for o in pkg.sample_clips(model, clips, device=DEV, **kw)]
    be = pkg.backend_for(model, DEV)
    assert be._plan_key[0] == slots and be.window_kernel_status() == 0
    sm = pkg.StreamSampler(model, slots=slots, device=DEV, **kw)
    statuses = []
    L = d.frames_per_clip
    streams = [sm.open(c["r_s"], c["we"], noise=c["noise"]) for c in clips]
    fed, got, seen, j = [0] * slots, {s: [] for s in streams}, [], 0
    while not all(s.done for s in streams):
        live = [i for i, c in enumerate(clips) if fed[i] < c["audio_num_frames"]]
        for t in range(min(1 + j % slots, len(live))):
            i = live[(j + t) % len(live)]
            n = min(L, clips[i]["audio_num_frames"] - fed[i])
            sm.feed(streams[i], clips[i]["wa"][:, fed[i]:fed[i] + n])
            fed[i] += n
            if fed[i] == clips[i]["audio_num_frames"]:
                sm.finish(streams[i])
        ran = sm.step()
        seen.append((len(ran), be.last_window_slots()))
        statuses.append(be.window_kernel_status())
        for s, o in ran.items():
            got[s].append(o)
        j += 1
    assert statuses and all(st == 0 for st in statuses), statuses
    assert all(n == slots for _, n in seen) and {k for k, _ in seen} == set(range(1, slots + 1)), seen
    for i, (s, r) in enumerate(zip(streams, ref)):
        assert torch.equal(torch.cat(got[s], dim=1).cpu(), r), i
