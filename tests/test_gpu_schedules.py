"""Per-clip and per-stream ODE schedules (nfe and solver) on the B200: the per-slot window graph.

Pins: every clip on the plan's own schedule through the per-slot graph == the plan's graph bitwise (euler's fused combine and a
multi-stage solver, bf16 and bf16x3); in a mixed call, the clips of each schedule == a uniform call on that schedule bitwise (4-branch
plan: the per-slot condition rows); every clip against the oracle run on it alone with its own nfe, solver and guidance (all five
solvers, nfe 1 to 5; fp32 / bf16x3 1e-4 relative, bf16 2e-2 max-abs); a 1-branch plan of <= 256 token rows runs a mixed call one
kernel per op; streams on different schedules == the mixed sample_clips call bitwise; guard rows, launches, and the t-embedding
cache.
"""
import random

import pytest
import torch

import cases
from __graft_entry__ import load_package
from test_gpu_guidance import MIX, guidance_kw, slot_args, with_guidance
from test_gpu_multiclip import LENGTHS, make_clips, oracle
from test_gpu_parity import model_for

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
R_CFG = (2.0, 0.5, 1.5, True)                     # 4 branches


@pytest.fixture(scope="module")
def pkg():
    return load_package()


def with_schedules(clips, schedules):
    return [dict(c, nfe=n, method=m) for c, (n, m) in zip(clips, schedules)]


def n_win(d, lengths):
    return [-(-T // d.frames_per_clip) for T in lengths]


@pytest.mark.parametrize("mode", ["bf16", "bf16x3"])
@pytest.mark.parametrize("method,nfe", [("euler", 4), ("heun3", 3)])
def test_plan_schedule_per_slot_equals_the_plan_graph(pkg, mode, method, nfe):
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    clips = make_clips(d, LENGTHS, seed=400)
    kw = dict(nfe=nfe, method=method, a_cfg_scale=2.0, r_cfg_scale=1.0, e_cfg_scale=1.0, include_r_cfg=False, mode=mode)
    ref = [o.cpu() for o in pkg.sample_clips(model, clips, device=DEV, **kw)]
    sch = pkg.clip_schedule(n_win(d, LENGTHS))
    assert 3 * sch.slots * d.total_frames > 256                              # the plan's graph runs one kernel per op too
    be = pkg.backend_for(model, DEV)
    be.configure(sch.slots, 3, False, nfe, method, mode)
    n = len(clips)
    r_s, wa, we, noise = slot_args(clips)
    outs = be.sample_clips(r_s, wa, we, LENGTHS, noise, 2.0, 1.0, 1.0, schedules=[(nfe, method)] * n)
    assert be.ode_graph_kernel_nodes() > 0                                   # the per-slot graph ran
    for i, (o, r) in enumerate(zip(outs, ref)):
        assert torch.equal(o.cpu(), r), (i, (o.cpu() - r).abs().max().item())


# schedules of 3, 4, 4, 2 and 3 evaluations; the keyword's (rk4, 2) sets the plan
SCHEDULES = [("euler", 4), ("midpoint", 3), ("rk4", 2), ("heun2", 2), ("heun3", 2)]


@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_mixed_call_equals_uniform_calls_per_schedule(pkg, mode):
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    clips = make_clips(d, LENGTHS, seed=410)
    n = len(clips)
    settings = [R_CFG if i % 3 == 0 else MIX[i % 2] for i in range(n)]      # 4- and 3-branch clips: a 4-branch plan
    schedules = [(n_, m) for m, n_ in (SCHEDULES[(i + 1) % len(SCHEDULES)] for i in range(n))]
    assert len(set(schedules[i] for i in range(n))) >= 4 and schedules[0] != schedules[1]
    clips = with_guidance(clips, settings)
    mixed = [o.cpu() for o in pkg.sample_clips(model, with_schedules(clips, schedules), device=DEV, nfe=2, method="rk4", mode=mode)]
    be = pkg.backend_for(model, DEV)
    assert be._plan_key[1] == 4 and be._plan_key[3:5] == (2, "rk4") and be.window_kernel_status() == -1
    for sc in sorted(set(schedules)):
        uniform = pkg.sample_clips(model, clips, device=DEV, nfe=sc[0], method=sc[1], mode=mode)
        assert be._plan_key[:2] == (pkg.clip_schedule(n_win(d, LENGTHS)).slots, 4)
        for i in (i for i in range(n) if schedules[i] == sc):
            assert torch.equal(mixed[i], uniform[i].cpu()), (sc, i, (mixed[i] - uniform[i].cpu()).abs().max().item())


# all five solvers, nfe 1 to 5: 0, 1, 4, 4, 4, 4 and 6 evaluations per window
ORACLE_SCHEDULES = [("euler", 1), ("euler", 2), ("midpoint", 3), ("heun2", 3), ("rk4", 2), ("euler", 5), ("heun3", 3)]


@pytest.mark.parametrize("mode,dynamic", [("fp32", False), ("bf16x3", True), ("bf16x3", False), ("bf16", False), ("bf16", True)])
def test_mixed_schedules_match_the_oracle_per_clip(pkg, mode, dynamic):
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    clips = make_clips(d, LENGTHS, seed=420 + dynamic, dynamic=dynamic)
    settings = [MIX[i % len(MIX)] for i in range(len(clips))]
    schedules = [(n_, m) for m, n_ in ORACLE_SCHEDULES]
    if dynamic:
        schedules = schedules[::-1]
    clips = with_schedules(with_guidance(clips, settings), schedules)
    outs = pkg.sample_clips(model, clips, device=DEV, nfe=3, method="euler", mode=mode)
    assert pkg.backend_for(model, DEV)._plan_key[3:5] == (3, "heun3")
    for i, (c, g, sc, o) in enumerate(zip(clips, settings, schedules, outs)):
        o = o.cpu()
        ref = oracle(d, c, **guidance_kw(g, nfe=sc[0], method=sc[1]))
        assert o.shape == ref.shape == (1, c["audio_num_frames"], d.dim_w)
        if sc[0] == 1:
            assert torch.equal(o[0], c["noise"].reshape(-1, d.dim_w)[:c["audio_num_frames"]])          # nfe 1 returns the noise
        if mode == "bf16":
            assert cases.max_abs(o, ref) <= 2e-2, (i, g, sc, cases.max_abs(o, ref))
        else:
            assert cases.rel_err(o, ref) <= 1e-4, (i, g, sc, cases.rel_err(o, ref))


def test_small_plan_runs_mixed_schedules_per_op(pkg):
    """One branch and three slots are 180 token rows: the plan's graph is the dataflow window kernel, a mixed call runs the
    per-slot graph one kernel per op."""
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    lengths = [100, 60, 50, 149]
    assert pkg.clip_schedule(n_win(d, lengths)).slots * d.total_frames <= 256
    clips = make_clips(d, lengths, seed=430)
    unguided = (1.0, 1.0, 1.0, False)
    kw = guidance_kw(unguided, nfe=4, method="euler", mode="bf16")
    pkg.sample_clips(model, clips, device=DEV, **kw)
    be = pkg.backend_for(model, DEV)
    assert be.window_kernel_status() == 0
    schedules = [(4, "euler"), (2, "rk4"), (3, "midpoint"), (2, "heun3")]
    outs = pkg.sample_clips(model, with_schedules(clips, schedules), device=DEV, **kw)
    assert be.window_kernel_status() == -1 and be._plan_key[3:5] == (2, "rk4")
    for i, (c, sc, o) in enumerate(zip(clips, schedules, outs)):
        ref = oracle(d, c, **guidance_kw(unguided, nfe=sc[0], method=sc[1]))
        assert cases.max_abs(o.cpu(), ref) <= 2e-2, (i, sc, cases.max_abs(o.cpu(), ref))


def test_streams_on_their_own_schedules_equal_the_mixed_call(pkg):
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    clips = make_clips(d, LENGTHS, seed=440)
    schedules = [(n_, m) for m, n_ in (SCHEDULES[i % len(SCHEDULES)] for i in range(len(clips)))]
    clips = with_schedules(clips, schedules)
    kw = dict(nfe=2, method="rk4", a_cfg_scale=2.0, r_cfg_scale=1.0, e_cfg_scale=1.0, include_r_cfg=False, mode="bf16")
    ref = [o.cpu() for o in pkg.sample_clips(model, clips, device=DEV, **kw)]
    slots = pkg.clip_schedule(n_win(d, LENGTHS)).slots
    assert slots >= 2 and 3 * slots * d.total_frames > 256
    sm = pkg.StreamSampler(model, slots=slots, device=DEV, **kw)
    with pytest.raises(ValueError):                                           # 5 evaluations, the plan runs 4
        sm.open(clips[0]["r_s"].to(DEV), clips[0]["we"].to(DEV), noise=clips[0]["noise"], nfe=6, method="euler")
    rng = random.Random(5)
    streams = [sm.open(c["r_s"].to(DEV), c["we"].to(DEV), noise=c["noise"], nfe=c["nfe"], method=c["method"]) for c in clips]
    fed, got = [0] * len(clips), {s: [] for s in streams}
    while not all(s.done for s in streams):
        for i in rng.sample(range(len(clips)), len(clips)):
            T = clips[i]["audio_num_frames"]
            if fed[i] < T:
                t = min(T - fed[i], rng.randint(1, 120))
                sm.feed(streams[i], clips[i]["wa"][:, fed[i]:fed[i] + t].to(DEV))
                fed[i] += t
                if fed[i] == T:
                    sm.finish(streams[i])
        for s, o in sm.step().items():
            got[s].append(o)
    for i, (s, r) in enumerate(zip(streams, ref)):
        o = torch.cat(got[s], dim=1).cpu()
        assert o.shape == r.shape and torch.equal(o, r), (i, (o - r).abs().max().item())


def test_guard_rows_launches_and_the_t_embedding_cache(pkg):
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    clips = make_clips(d, LENGTHS, seed=450)
    n = len(clips)
    sch = pkg.clip_schedule(n_win(d, LENGTHS))
    be = pkg.backend_for(model, DEV)
    be.configure(sch.slots, 3, False, 7, "euler", "bf16")                    # 6 evaluations per window
    schedules = [[(7, "euler"), (4, "heun2"), (4, "midpoint")][i % 3] for i in range(n)]   # two schedules no other test uses
    r_s, wa, we, noise = slot_args(clips)
    g = 2
    rows = [T for T in LENGTHS]
    buf = torch.full((sum(rows) + g * (n + 1), d.dim_w), float("nan"), device=DEV)
    starts = [g + sum(rows[:i]) + g * i for i in range(n)]
    views = [buf[s:s + T] for s, T in zip(starts, rows)]
    torch.cuda.synchronize()
    be.launch_count(reset=True)
    first = [o.clone() for o in be.sample_clips(r_s, wa, we, LENGTHS, noise, 2.0, 1.0, 1.0, out=views, schedules=schedules)]
    torch.cuda.synchronize()
    nodes = be.ode_graph_kernel_nodes()
    assert nodes > 0
    assert be.launch_count(reset=True) == sch.makespan * (1 + nodes) + 2 * 3          # + the t-embeddings of the two new schedules
    written = torch.zeros(buf.shape[0], dtype=torch.bool)
    for s, T in zip(starts, rows):
        written[s:s + T] = True
    host = buf.cpu()
    assert torch.isfinite(host[written]).all() and torch.isnan(host[~written]).all()
    again = be.sample_clips(r_s, wa, we, LENGTHS, noise, 2.0, 1.0, 1.0, schedules=schedules)
    torch.cuda.synchronize()
    assert be.launch_count() == sch.makespan * (1 + nodes)                           # cached: no t-embedding work
    for i, (x, y) in enumerate(zip(first, again)):
        assert torch.equal(x.view_as(y), y), i
    with pytest.raises(ValueError):                                                  # more evaluations than the plan
        be.sample_clips(r_s, wa, we, LENGTHS, noise, 2.0, 1.0, 1.0, schedules=[(8, "euler")] + schedules[1:])
