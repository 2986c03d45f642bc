"""CPU tests of per-clip and per-stream ODE schedules: validation of the nfe / method keys before any device call, the plan a
mixed call configures, the StreamSampler capacity check, the per-slot condition-row deduplication, and the C ABI of FmtClipOde."""
import ctypes as C
import os
import shutil
import subprocess
import sys
import tempfile

import pytest
import torch

from __graft_entry__ import ROOT, load_package
from test_host_multiclip import _small_model


@pytest.fixture(scope="module")
def pkg():
    p = load_package()
    sys.modules[p.__name__ + ".build"].build()
    return p


class _RecordingBackend:
    """Stands in for FmtBackend: records what sample_clips configures and passes down, and does no device work."""

    def __init__(self, dims):
        self.dims, self.device, self.calls = dims, torch.device("cpu"), []

    def configure(self, batch, n_branches, we_dynamic, nfe, method, mode):
        self.calls.append(("configure", nfe, method))

    def sample_clips(self, r_s, wa, we, T, noise, a, r, e, progress=None, out=None, n_branches=None, schedules=None):
        self.calls.append(("sample_clips", None if schedules is None else tuple(schedules)))
        return [torch.zeros(1, t, self.dims.dim_w) for t in T]


def _clip(d, T=30, **kw):
    c = dict(r_s=torch.zeros(1, d.dim_w), wa=torch.zeros(1, T, d.dim_a), we=torch.zeros(1, 1, d.dim_e), seed=1)
    c.update(kw)
    return c


def _resolve(pkg, monkeypatch, clips, **call):
    sampler = sys.modules[pkg.__name__ + ".sampler"]
    model, d = _small_model(pkg)
    be = _RecordingBackend(d)
    monkeypatch.setattr(sampler, "backend_for", lambda *a, **k: be)
    kw = dict(nfe=3, method="euler", mode="bf16", device="cpu")
    kw.update(call)
    pkg.sample_clips(model, [_clip(d, **c) for c in clips], **kw)
    (_, nfe, method), (_, schedules) = be.calls
    return (nfe, method), schedules


def test_evaluation_counts(pkg):
    stages = {"euler": 1, "midpoint": 2, "heun2": 2, "heun3": 3, "rk4": 4}
    for method, g in stages.items():
        for nfe in (1, 2, 5, 10):
            assert pkg.n_evals(nfe, method) == (nfe - 1) * g
            sc = pkg.build_schedule(nfe, method)
            assert sc["n_steps"] * sc["n_stages"] == pkg.n_evals(nfe, method) == len(sc["t_eval"])
    # the workloads of tools/schedule_bench.py
    assert [pkg.n_evals(n, m) for m, n in (("euler", 10), ("heun3", 4), ("midpoint", 5), ("rk4", 3))] == [9, 9, 8, 8]


def test_plan_takes_the_schedule_that_needs_the_most_evaluations(pkg, monkeypatch):
    # one schedule for every clip: the call's, through the plan's window graph as before
    assert _resolve(pkg, monkeypatch, [{}, {}]) == ((3, "euler"), None)
    assert _resolve(pkg, monkeypatch, [dict(nfe=3), dict(method="euler")]) == ((3, "euler"), None)
    # a clip that needs more than the keyword schedule sets the plan; every clip's schedule goes down
    plan, sch = _resolve(pkg, monkeypatch, [{}, dict(nfe=5, method="heun2"), dict(method="rk4")])
    assert plan == (5, "heun2") and sch == ((3, "euler"), (5, "heun2"), (3, "rk4"))
    # tie (8 evaluations each): the keyword schedule when some clip runs it, else the first in input order
    plan, sch = _resolve(pkg, monkeypatch, [dict(nfe=3, method="rk4"), {}, dict(nfe=9, method="euler")], nfe=5, method="midpoint")
    assert plan == (5, "midpoint") and sch == ((3, "rk4"), (5, "midpoint"), (9, "euler"))
    plan, sch = _resolve(pkg, monkeypatch, [dict(nfe=3, method="rk4"), dict(nfe=9, method="euler")], nfe=5, method="midpoint")
    assert plan == (3, "rk4") and sch == ((3, "rk4"), (9, "euler"))
    plan, sch = _resolve(pkg, monkeypatch, [dict(nfe=3, method="rk4"), dict(nfe=9, method="euler")], nfe=2, method="euler")
    assert plan == (3, "rk4") and sch == ((3, "rk4"), (9, "euler"))
    # every clip on one schedule that ties the keyword's: the plan is that schedule, and the plan's window graph runs
    assert _resolve(pkg, monkeypatch, [dict(nfe=4, method="heun3")] * 2, nfe=10, method="euler") == ((4, "heun3"), None)
    # every clip on one schedule that is not the keyword's: the plan is that schedule, no per-clip schedules
    assert _resolve(pkg, monkeypatch, [dict(nfe=4, method="heun3")] * 2) == ((4, "heun3"), None)
    # nfe 1 (no evaluation) with another clip's solver
    plan, sch = _resolve(pkg, monkeypatch, [dict(nfe=1, method="rk4"), {}], nfe=1, method="euler")
    assert plan == (1, "euler") and sch == ((1, "rk4"), (1, "euler"))


def test_bad_schedule_keys_raise_before_any_device_call(pkg, monkeypatch):
    sampler = sys.modules[pkg.__name__ + ".sampler"]
    model, d = _small_model(pkg)

    def no_device(*a, **k):
        raise AssertionError("device work before validation")

    monkeypatch.setattr(sampler, "backend_for", no_device)
    bad = [
        (dict(nfe=2.0), TypeError),
        (dict(nfe="3"), TypeError),
        (dict(nfe=True), TypeError),
        (dict(nfe=None), TypeError),
        (dict(nfe=torch.tensor(3)), TypeError),
        (dict(nfe=0), ValueError),
        (dict(nfe=-2), ValueError),
        (dict(method="dopri5"), ValueError),
        (dict(method=None), ValueError),
        (dict(method=["euler"]), ValueError),
    ]
    for over, exc in bad:
        with pytest.raises(exc):
            pkg.sample_clips(model, [_clip(d), _clip(d, **over)], nfe=3, method="euler", mode="bf16", device="cpu")


class _StubBackend:
    def __init__(self, dims):
        self.dims, self.device = dims, torch.device("cpu")

    def configure(self, *a):
        pass


def test_stream_capacity_and_keys(pkg, monkeypatch):
    sampler = sys.modules[pkg.__name__ + ".sampler"]
    model, d = _small_model(pkg)
    monkeypatch.setattr(sampler, "backend_for", lambda *a, **k: _StubBackend(d))
    sm = pkg.StreamSampler(model, slots=2, nfe=4, method="midpoint", device="cpu")          # 6 evaluations per window
    assert sm.capacity == 6
    r_s, we = torch.zeros(1, d.dim_w), torch.zeros(1, 1, d.dim_e)
    for ok in (dict(nfe=7, method="euler"), dict(nfe=3, method="heun3"), dict(nfe=1, method="rk4"), dict(method="heun2"), {}):
        st = sm.open(r_s, we, seed=1, **ok)
        assert st.schedule == (ok.get("nfe", 4), ok.get("method", "midpoint"))
    for over in (dict(nfe=8, method="euler"), dict(nfe=3, method="rk4"), dict(nfe=5)):
        with pytest.raises(ValueError, match="evaluations"):
            sm.open(r_s, we, seed=1, **over)
    for over, exc in ((dict(nfe=2.5), TypeError), (dict(nfe=False), TypeError), (dict(nfe=0), ValueError), (dict(method="rk45"), ValueError),
                      (dict(solver="euler"), TypeError)):
        with pytest.raises(exc):
            sm.open(r_s, we, seed=1, **over)
    assert len(sm._streams) == 5                                      # the refused opens left nothing behind


def test_per_slot_condition_rows_never_span_two_slots(pkg):
    lib = sys.modules[pkg.__name__ + "._cabi"].load_library()
    B, N, P = 3, 12, 4
    for nb in (1, 3, 4):
        for dyn in (0, 1):
            plan = (C.c_int32 * (nb * B * N))()
            own = (C.c_int32 * (nb * B * N))()
            U = lib.fmt_debug_condition_rows(nb, B, N, P, dyn, plan)
            sU = lib.fmt_debug_condition_rows_ode(nb, B, N, P, dyn, 1, own)
            assert lib.fmt_debug_condition_rows_ode(nb, B, N, P, dyn, 0, None) == U
            assert sU == U + (B - 1 if nb == 4 else 0), (nb, dyn, U, sU)
            slot_of = {}
            for row in range(nb * B * N):
                b = (row // N) % B
                assert slot_of.setdefault(own[row], b) == b, (nb, dyn, row)
            # within one slot the per-slot rows are the plan's rows
            for b in range(B):
                rows = [br * B * N + b * N + f for br in range(nb) for f in range(N)]
                pairs = {(plan[r], own[r]) for r in rows}
                assert len({p for p, _ in pairs}) == len({o for _, o in pairs}) == len(pairs)


def test_ode_entry_points_are_exported_with_the_header_layout(pkg):
    cabi = sys.modules[pkg.__name__ + "._cabi"]
    lib = cabi.load_library()
    for name in ("fmt_sample_clips_ode", "fmt_sample_windows_ode", "fmt_ode_graph_kernel_nodes", "fmt_debug_condition_rows_ode"):
        assert callable(getattr(lib, name))
    O = cabi.FmtClipOde
    fields = ["n_steps", "n_stages", "t_eval", "dt", "rk_a", "rk_b"]
    assert [f[0] for f in O._fields_] == fields
    p = C.sizeof(C.c_void_p)
    assert [getattr(O, f).offset for f in fields] == [i * p for i in range(6)] and C.sizeof(O) == 6 * p
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no host C compiler for the offsetof probe")
    with tempfile.TemporaryDirectory() as tmp:
        src, exe = os.path.join(tmp, "probe.c"), os.path.join(tmp, "probe")
        with open(src, "w") as f:
            f.write('#include <stddef.h>\n#include <stdio.h>\n#include "fmt_b200.h"\nint main(void) {\n')
            for fld in fields:
                f.write(f'  printf("%zu ", offsetof(FmtClipOde, {fld}));\n')
            f.write('  printf("%zu\\n", sizeof(FmtClipOde));\n  return 0;\n}\n')
        subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", exe, src], check=True)
        got = [int(x) for x in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [getattr(O, f).offset for f in fields] + [C.sizeof(O)]
    assert cabi.FMT_ABI_VERSION == 2 and lib.fmt_abi_version() == 2


def test_backend_schedule_list_is_checked(pkg):
    be = sys.modules[pkg.__name__ + ".sampler"].FmtBackend
    ode, keep = be._clip_ode([(3, "euler"), (2, "rk4"), (1, "heun3")], 3)
    assert list(ode.n_steps[:3]) == [2, 1, 0] and list(ode.n_stages[:3]) == [1, 4, 3]
    assert [ode.rk_b[1][j] for j in range(4)] == [0.125, 0.375, 0.375, 0.125]
    for bad in ([(3, "euler")], [(0, "euler"), (3, "euler")], [(True, "euler"), (3, "euler")], [(3, "rk45"), (3, "euler")]):
        with pytest.raises(ValueError):
            be._clip_ode(bad, 2)
