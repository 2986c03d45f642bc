"""Per-clip and per-stream emotion modes on the B200: static and dynamic clips in one call, on one plan.

Pins: in a call that mixes the modes, every clip == a uniform call of its own mode on the same plan bitwise (the plan's graph, the
per-slot graph with mixed schedules and guidance, and a 1-branch plan that runs the dataflow window kernel), in bf16, bf16x3 and fp32;
every clip of a mixed call against the oracle run on it alone (fp32 / bf16x3 1e-4 relative, bf16 2e-2 max-abs); one StreamSampler
holding static and dynamic streams == the mixed call bitwise, with the launches and graph of a uniform sampler; guard rows.
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
A = (2.0, 1.0, 1.0, False)                        # 3 branches


@pytest.fixture(scope="module")
def pkg():
    return load_package()


def both_modes(d, lengths, seed, dynamic_of):
    """The clips with static and with dynamic emotion (same r_s, wa and noise), and the mixed set: clip i dynamic iff dynamic_of(i),
    each declaring its mode."""
    static, dynamic = make_clips(d, lengths, seed), make_clips(d, lengths, seed, dynamic=True)
    mixed = [dict(dynamic[i] if dynamic_of(i) else static[i], we_dynamic=bool(dynamic_of(i))) for i in range(len(lengths))]
    return static, dynamic, mixed


def check_oracle(d, clips, outs, mode, settings, schedules=None):
    for i, (c, o) in enumerate(zip(clips, outs)):
        nfe, method = schedules[i] if schedules else (c.get("nfe", 3), c.get("method", "euler"))
        ref = oracle(d, c, **guidance_kw(settings[i], nfe=nfe, method=method))
        o = o.cpu()
        assert o.shape == ref.shape
        if mode == "bf16":
            assert cases.max_abs(o, ref) <= 2e-2, (i, cases.max_abs(o, ref))
        else:
            assert cases.rel_err(o, ref) <= 1e-4, (i, cases.rel_err(o, ref))


def assert_each_equals_its_uniform_call(mixed_out, static_out, dynamic_out, dynamic_of):
    for i, o in enumerate(mixed_out):
        r = (dynamic_out if dynamic_of(i) else static_out)[i]
        assert torch.equal(o.cpu(), r.cpu()), (i, dynamic_of(i), (o.cpu() - r.cpu()).abs().max().item())


@pytest.mark.parametrize("mode", ["bf16", "bf16x3", "fp32"])
def test_mixed_call_on_the_plan_graph(pkg, mode):
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    dyn = lambda i: i % 2 == 1                                              # noqa: E731  clip 0 static: the plan's mode
    static, dynamic, mixed = both_modes(d, LENGTHS, 500, dyn)
    kw = guidance_kw(A, nfe=3, method="euler", mode=mode)
    be = pkg.backend_for(model, DEV)
    out = pkg.sample_clips(model, mixed, device=DEV, **kw)
    assert be._plan_key[2] is False
    nodes = be.graph_kernel_nodes()
    s_out = pkg.sample_clips(model, static, device=DEV, **kw)
    d_out = pkg.sample_clips(model, dynamic, device=DEV, **kw)
    assert be.graph_kernel_nodes() == nodes
    assert_each_equals_its_uniform_call(out, s_out, d_out, dyn)
    check_oracle(d, mixed, out, mode, [A] * len(mixed))


SCHEDULES = [(4, "euler"), (3, "midpoint"), (2, "rk4"), (2, "heun2"), (2, "heun3"), (3, "euler"), (4, "euler")]


@pytest.mark.parametrize("mode", ["bf16", "bf16x3", "fp32"])
def test_mixed_call_on_the_per_slot_graph_with_schedules_and_guidance(pkg, mode):
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    dyn = lambda i: i % 3 != 1                                              # noqa: E731
    settings = [MIX[i % len(MIX)] for i in range(len(LENGTHS))]            # 3, 3, 4 and 1 branches: a 4-branch plan
    own = lambda cl: [dict(c, nfe=n, method=m) for c, (n, m) in zip(with_guidance(cl, settings), SCHEDULES)]   # noqa: E731
    static, dynamic, mixed = (own(x) for x in both_modes(d, LENGTHS, 510, dyn))
    kw = dict(nfe=2, method="rk4", mode=mode)
    be = pkg.backend_for(model, DEV)
    out = pkg.sample_clips(model, mixed, device=DEV, **kw)
    assert be._plan_key[1] == 4 and be._plan_key[3:5] == (2, "rk4") and be.window_kernel_status() == -1
    nodes = be.ode_graph_kernel_nodes()
    assert nodes > 0
    s_out = pkg.sample_clips(model, static, device=DEV, **kw)
    d_out = pkg.sample_clips(model, dynamic, device=DEV, **kw)
    assert be.ode_graph_kernel_nodes() == nodes
    assert_each_equals_its_uniform_call(out, s_out, d_out, dyn)
    check_oracle(d, mixed, out, mode, settings, SCHEDULES)


def test_mixed_call_in_the_dataflow_window_kernel(pkg):
    """One branch and three slots are 180 token rows: the plan's graph is the dataflow window kernel, which builds the condition rows
    with the same cond_gather_kernel."""
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    lengths = [100, 60, 50, 149]
    unguided = (1.0, 1.0, 1.0, False)
    dyn = lambda i: i in (0, 3)                                             # noqa: E731  the plan is dynamic here
    static, dynamic, mixed = both_modes(d, lengths, 520, dyn)
    kw = guidance_kw(unguided, nfe=4, method="euler", mode="bf16")
    be = pkg.backend_for(model, DEV)
    out = pkg.sample_clips(model, mixed, device=DEV, **kw)
    assert be.window_kernel_status() == 0 and be._plan_key[:3] == (3, 1, True)
    s_out = pkg.sample_clips(model, static, device=DEV, **kw)
    assert be.window_kernel_status() == 0
    d_out = pkg.sample_clips(model, dynamic, device=DEV, **kw)
    assert be.window_kernel_status() == 0
    assert_each_equals_its_uniform_call(out, s_out, d_out, dyn)
    check_oracle(d, mixed, out, "bf16", [unguided] * len(mixed), [(4, "euler")] * len(mixed))


class GuardedOutputs:
    """Backend proxy: every window's outputs go to one NaN-filled buffer with guard rows around each stream's frames."""
    guard = 3

    def __init__(self, be):
        self.be, self.device, self.dims = be, be.device, be.dims
        self.clean, self.mixed_steps = True, 0

    def configure(self, *plan):
        self.be.configure(*plan)

    def sample_windows(self, r_s, wa, we, x0, ctx, out, *rest, **kw):
        g, rows = self.guard, [o.shape[1] for o in out]
        buf = torch.full((sum(rows) + g * (len(rows) + 1), self.dims.dim_w), float("nan"), device=self.device)
        starts = [g + sum(rows[:i]) + g * i for i in range(len(rows))]
        views = [buf[s:s + n] for s, n in zip(starts, rows)]
        self.be.sample_windows(r_s, wa, we, x0, ctx, views, *rest, **kw)
        self.mixed_steps += "we_dynamic" in kw
        written = torch.zeros(buf.shape[0], dtype=torch.bool)
        for s, n in zip(starts, rows):
            written[s:s + n] = True
        host = buf.cpu()
        self.clean &= bool(torch.isfinite(host[written]).all()) and bool(torch.isnan(host[~written]).all())
        for o, v in zip(out, views):
            o.copy_(v.view_as(o))


def run_mixed_streams(sm, clips, dyn, seed):
    rng = random.Random(seed)
    streams = [sm.open(c["r_s"].to(DEV), None if dyn(i) else c["we"].to(DEV), noise=c["noise"], we_dynamic=dyn(i))
               for i, c in enumerate(clips)]
    fed, got, n_steps = [0] * len(clips), {s: [] for s in streams}, 0
    while not all(s.done for s in streams):
        for i in rng.sample(range(len(clips)), len(clips)):
            T = clips[i]["audio_num_frames"]
            if fed[i] < T:
                t = min(T - fed[i], rng.randint(1, 120))
                sm.feed(streams[i], clips[i]["wa"][:, fed[i]:fed[i] + t].to(DEV),
                        clips[i]["we"][:, fed[i]:fed[i] + t].to(DEV) if dyn(i) else None)
                fed[i] += t
                if fed[i] == T:
                    sm.finish(streams[i])
        ran = sm.step()
        for s, o in ran.items():
            got[s].append(o)
        n_steps += bool(ran)
    return [torch.cat(got[s], dim=1).cpu() for s in streams], n_steps


def test_one_stream_sampler_holds_static_and_dynamic_streams(pkg):
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    dyn = lambda i: i % 2 == 0                                              # noqa: E731
    _, _, mixed = both_modes(d, LENGTHS, 530, dyn)
    kw = guidance_kw(A, nfe=3, method="euler", mode="bf16")
    ref = [o.cpu() for o in pkg.sample_clips(model, mixed, device=DEV, **kw)]
    slots = pkg.clip_schedule([-(-T // d.frames_per_clip) for T in LENGTHS]).slots
    be = pkg.backend_for(model, DEV)
    uniform = pkg.StreamSampler(model, slots=slots, device=DEV, **kw)      # static: every stream of the uniform sampler
    nodes = be.graph_kernel_nodes()
    sm = pkg.StreamSampler(model, slots=slots, device=DEV, **kw)
    proxy = GuardedOutputs(be)
    sm._be = proxy
    torch.cuda.synchronize()
    be.launch_count(reset=True)
    outs, n_steps = run_mixed_streams(sm, mixed, dyn, seed=9)
    torch.cuda.synchronize()
    assert be.launch_count() == n_steps * (1 + nodes)                        # no re-capture, no extra launches
    assert be.graph_kernel_nodes() == nodes and proxy.clean and proxy.mixed_steps > 0
    for i, (o, r) in enumerate(zip(outs, ref)):
        assert o.shape == r.shape and torch.equal(o, r), (i, dyn(i), (o - r).abs().max().item())
    del uniform


def test_guard_rows_of_a_mixed_call(pkg):
    d = cases.FmtDims()
    model = model_for(pkg, "full")
    dyn = lambda i: i % 2 == 1                                              # noqa: E731
    _, _, mixed = both_modes(d, LENGTHS, 540, dyn)
    n = len(mixed)
    be = pkg.backend_for(model, DEV)
    be.configure(pkg.clip_schedule([-(-T // d.frames_per_clip) for T in LENGTHS]).slots, 3, False, 3, "euler", "bf16")
    r_s, wa, we, noise = slot_args(mixed)
    g = 2
    buf = torch.full((sum(LENGTHS) + g * (n + 1), d.dim_w), float("nan"), device=DEV)
    starts = [g + sum(LENGTHS[:i]) + g * i for i in range(n)]
    views = [buf[s:s + T] for s, T in zip(starts, LENGTHS)]
    modes = [dyn(i) for i in range(n)]
    be.sample_clips(r_s, wa, we, LENGTHS, noise, 2.0, 1.0, 1.0, out=views, we_dynamic=modes)
    be.sample_clips(r_s, wa, we, LENGTHS, noise, 2.0, 1.0, 1.0, out=views, we_dynamic=modes, schedules=[(3, "euler")] * n)
    written = torch.zeros(buf.shape[0], dtype=torch.bool)
    for s, T in zip(starts, LENGTHS):
        written[s:s + T] = True
    host = buf.cpu()
    assert torch.isfinite(host[written]).all() and torch.isnan(host[~written]).all()
    with pytest.raises(ValueError):                                        # a mode that contradicts the clip's we
        be.sample_clips(r_s, wa, we, LENGTHS, noise, 2.0, 1.0, 1.0, we_dynamic=[not m for m in modes])
