"""CPU tests of per-clip guidance in sample_clips: how per-clip settings resolve to branch counts and to the plan, validation
before any device call, and the C ABI of fmt_sample_clips_guided / FmtClipGuidance."""
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
        self.calls.append(("configure", batch, n_branches))

    def sample_clips(self, r_s, wa, we, T, noise, a, r, e, progress=None, out=None, n_branches=None):
        self.calls.append(("sample_clips", tuple(a), tuple(r), tuple(e), tuple(n_branches)))
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
    kw = dict(nfe=3, method="euler", a_cfg_scale=2.0, r_cfg_scale=1.0, e_cfg_scale=1.0, include_r_cfg=False, mode="bf16", device="cpu")
    kw.update(call)
    pkg.sample_clips(model, [_clip(d, **c) for c in clips], **kw)
    (_, _, plan_nb), (_, a, r, e, nb) = be.calls
    return plan_nb, list(zip(a, r, e, nb))


def test_per_clip_settings_resolve_to_branch_counts(pkg, monkeypatch):
    # no per-clip settings: the call's guidance for every clip, as before
    assert _resolve(pkg, monkeypatch, [{}, {}]) == (3, [(2.0, 1.0, 1.0, 3)] * 2)
    # the mix of one call: 3-, 1- and 4-branch clips, r != 1 without include_r_cfg (3 branches, r unused); the plan takes 4
    plan, per = _resolve(pkg, monkeypatch, [{}, dict(a_cfg_scale=1.0), dict(r_cfg_scale=0.5, e_cfg_scale=1.5, include_r_cfg=True),
                                            dict(r_cfg_scale=0.5), dict(a_cfg_scale=1, e_cfg_scale=3)])
    assert plan == 4
    assert per == [(2.0, 1.0, 1.0, 3), (1.0, 1.0, 1.0, 1), (2.0, 0.5, 1.5, 4), (2.0, 0.5, 1.0, 3), (1.0, 1.0, 3.0, 3)]
    # a per-clip key overrides the call's keyword for that clip only
    plan, per = _resolve(pkg, monkeypatch, [dict(a_cfg_scale=2.0), {}], a_cfg_scale=1.0, r_cfg_scale=1.0, e_cfg_scale=1.0)
    assert (plan, per) == (3, [(2.0, 1.0, 1.0, 3), (1.0, 1.0, 1.0, 1)])
    plan, per = _resolve(pkg, monkeypatch, [dict(include_r_cfg=True), {}], r_cfg_scale=0.5)
    assert (plan, per) == (4, [(2.0, 0.5, 1.0, 4), (2.0, 0.5, 1.0, 3)])
    # every clip unguided: a 1-branch plan; include_r_cfg alone adds no branch
    assert _resolve(pkg, monkeypatch, [dict(a_cfg_scale=1.0, include_r_cfg=True)] * 2) == (1, [(1.0, 1.0, 1.0, 1)] * 2)


def test_bad_per_clip_guidance_raises_before_any_device_call(pkg, monkeypatch):
    sampler = sys.modules[pkg.__name__ + ".sampler"]
    model, d = _small_model(pkg)

    def no_device(*a, **k):
        raise AssertionError("device work before validation")

    monkeypatch.setattr(sampler, "backend_for", no_device)
    kw = dict(nfe=3, method="euler", a_cfg_scale=2.0, r_cfg_scale=1.0, e_cfg_scale=1.0, include_r_cfg=False, mode="bf16", device="cpu")
    bad = [
        (dict(a_cfg_scale="2"), TypeError),
        (dict(r_cfg_scale=None), TypeError),
        (dict(e_cfg_scale=True), TypeError),
        (dict(a_cfg_scale=torch.tensor(2.0)), TypeError),
        (dict(include_r_cfg=1), TypeError),
        (dict(include_r_cfg="yes"), TypeError),
        (dict(a_cfg_scale=float("nan")), ValueError),
        (dict(r_cfg_scale=float("inf")), ValueError),
        (dict(e_cfg_scale=-float("inf")), ValueError),
    ]
    for over, exc in bad:
        with pytest.raises(exc):
            pkg.sample_clips(model, [_clip(d), _clip(d, **over)], **kw)


def test_guided_entry_point_is_exported_with_the_header_layout(pkg):
    cabi = sys.modules[pkg.__name__ + "._cabi"]
    lib = cabi.load_library()
    assert callable(lib.fmt_sample_clips_guided) and callable(lib.fmt_sample_clips)
    G = cabi.FmtClipGuidance
    fields = ["a_cfg_scale", "r_cfg_scale", "e_cfg_scale", "n_branches"]
    assert [f[0] for f in G._fields_] == fields
    # four host pointers, in header order
    p = C.sizeof(C.c_void_p)
    assert [getattr(G, f).offset for f in fields] == [0, p, 2 * p, 3 * p] and C.sizeof(G) == 4 * p
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no host C compiler for the offsetof probe")
    with tempfile.TemporaryDirectory() as tmp:
        src, exe = os.path.join(tmp, "probe.c"), os.path.join(tmp, "probe")
        with open(src, "w") as f:
            f.write('#include <stddef.h>\n#include <stdio.h>\n#include "fmt_b200.h"\nint main(void) {\n')
            for fld in fields:
                f.write(f'  printf("%zu ", offsetof(FmtClipGuidance, {fld}));\n')
            f.write('  printf("%zu\\n", sizeof(FmtClipGuidance));\n  return 0;\n}\n')
        subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", exe, src], check=True)
        got = [int(x) for x in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [getattr(G, f).offset for f in fields] + [C.sizeof(G)]


def test_abi_version_is_unchanged(pkg):
    cabi = sys.modules[pkg.__name__ + "._cabi"]
    assert cabi.FMT_ABI_VERSION == 2 and cabi.load_library().fmt_abi_version() == 2
