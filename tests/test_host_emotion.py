"""CPU tests of per-clip and per-stream emotion modes (static or dynamic we): the condition-row map that every mix of modes shares,
validation before any device call, how sample_clips and StreamSampler resolve each clip's mode and what they pass down, and the C
ABI of the general sampling entries."""
import ctypes as C
import itertools
import random
import sys

import pytest
import torch

from __graft_entry__ import load_package
from test_host_multiclip import _small_model


@pytest.fixture(scope="module")
def pkg():
    p = load_package()
    sys.modules[p.__name__ + ".build"].build()
    return p


def _lib(pkg):
    return sys.modules[pkg.__name__ + "._cabi"].load_library()


N, P = 60, 10
NULLS = {1: [(0, 0, 0)], 3: [(0, 1, 1), (0, 0, 0), (0, 0, 1)], 4: [(1, 1, 1), (0, 1, 1), (0, 0, 0), (0, 0, 1)]}   # (zr, za, ze), FMT.py:360-392


def reference_map(nb, modes, per_slot):
    """test_host_logic.py's symbolic condition rows with slot b's own emotion mode; per_slot: rows of different slots are distinct."""
    rows = []
    for br in range(nb):
        zr, za, ze = NULLS[nb][br]
        for b, dynamic in enumerate(modes):
            for f in range(N):
                ctx = f < P
                wr = ("wr", b) if not zr else 0
                wa = ("prev_wa", b, f) if ctx else (("wa", b, f) if not za else 0)
                if ze:
                    we = 0
                elif not dynamic:
                    we = ("we", b)
                else:
                    we = ("prev_we", b, f) if ctx else ("we", b, f)
                rows.append((wr, wa, we, b if per_slot else None))
    first = {}
    return [first.setdefault(r, len(first)) for r in rows], len(first)


def slot_map(lib, nb, modes, per_slot):
    B = len(modes)
    out = (C.c_int32 * (nb * B * N))()
    U = lib.fmt_debug_condition_rows_slots(nb, B, N, P, (C.c_int32 * B)(*modes), per_slot, out)
    return list(out), U


def test_condition_rows_are_the_same_for_every_mix_of_modes(pkg):
    lib = _lib(pkg)
    rng = random.Random(11)
    for nb, B, per_slot in itertools.product((1, 3, 4), (1, 2, 3, 5, 8), (0, 1)):
        mixes = list(itertools.product((0, 1), repeat=B)) if B <= 3 else [tuple(rng.randint(0, 1) for _ in range(B)) for _ in range(6)]
        uniform = slot_map(lib, nb, [0] * B, per_slot)
        for modes in mixes:
            got = slot_map(lib, nb, list(modes), per_slot)
            assert got == uniform, (nb, B, per_slot, modes)
            ref, U_ref = reference_map(nb, modes, per_slot)
            assert got == (ref, U_ref), (nb, B, per_slot, modes)
        # the uniform entries are the per-slot entry with one mode for every slot
        out = (C.c_int32 * (nb * B * N))()
        assert lib.fmt_debug_condition_rows_ode(nb, B, N, P, 1, per_slot, out) == uniform[1] and list(out) == uniform[0]
    assert lib.fmt_debug_condition_rows_slots(3, 2, N, P, None, 0, None) < 0


def test_the_emotion_key_never_splits_a_row():
    """Why the map does not depend on the modes: in every branch that keeps the emotion, the row's audio term is already keyed by
    (clip, frame) - a context frame's prev_wa (never nulled) or the current frame's wa - so static or dynamic emotion, a function of
    (clip, frame), adds nothing to the key."""
    for nb, nulls in NULLS.items():
        for zr, za, ze in nulls:
            assert ze or not za, (nb, zr, za, ze)


class _RecordingBackend:
    """Stands in for FmtBackend: records the plan and what sample_clips / sample_windows pass down; no device work."""

    def __init__(self, dims):
        self.dims, self.device, self.plans, self.calls = dims, torch.device("cpu"), [], []

    def configure(self, *plan):
        self.plans.append(plan)

    def sample_clips(self, r_s, wa, we, T, noise, a, r, e, progress=None, out=None, n_branches=None, schedules=None, **kw):
        self.calls.append(dict(kw, we_frames=[t.shape[1] for t in we]))
        return [torch.zeros(1, t, self.dims.dim_w) for t in T]

    def sample_windows(self, r_s, wa, we, x0, ctx, out, first_window, a, r, e, nb, **kw):
        self.calls.append(dict(kw, we=[t.clone() for t in we]))


def _clip(d, T=30, we_T=1, **kw):
    c = dict(r_s=torch.zeros(1, d.dim_w), wa=torch.zeros(1, T, d.dim_a), we=torch.zeros(1, we_T, d.dim_e), audio_num_frames=T, seed=1)
    c.update(kw)
    return c


@pytest.fixture()
def recording(pkg, monkeypatch):
    sampler = sys.modules[pkg.__name__ + ".sampler"]
    model, d = _small_model(pkg)
    be = _RecordingBackend(d)
    monkeypatch.setattr(sampler, "backend_for", lambda *a, **k: be)
    return model, d, be


KW = dict(nfe=3, method="euler", mode="bf16", device="cpu")


def test_sample_clips_resolves_each_clips_mode(pkg, recording):
    model, d, be = recording
    L = d.frames_per_clip
    static, dynamic = dict(T=30), dict(T=2 * L, we_T=2 * L)
    cases = [
        # clips, call keyword -> the plan's we_dynamic, the per-clip modes passed down (None: not passed)
        ([static, static], None, False, None),
        ([dynamic, dynamic], None, True, None),
        ([dynamic, dict(static, we_dynamic=False)], None, True, [True, False]),
        ([dict(static, we_dynamic=False), dynamic, dynamic], None, False, [False, True, True]),
        ([dict(dynamic, we_dynamic=True), static], False, True, [True, False]),
        ([static, dynamic], True, None, None),                  # the keyword makes the static clip dynamic: its we contradicts it
        ([dynamic, dynamic], True, True, None),
        ([dict(static, we_dynamic=False), dict(static, we_dynamic=False)], True, False, None),
    ]
    for clips, keyword, plan_mode, passed in cases:
        be.plans.clear(), be.calls.clear()
        call = dict(KW, we_dynamic=keyword)
        if plan_mode is None:
            with pytest.raises(ValueError):
                pkg.sample_clips(model, [_clip(d, **c) for c in clips], **call)
            assert not be.plans and not be.calls
            continue
        pkg.sample_clips(model, [_clip(d, **c) for c in clips], **call)
        (plan,), (sent,) = be.plans, be.calls
        slots = pkg.clip_schedule([-(-c["T"] // L) for c in clips]).slots
        assert plan == (slots, 3, plan_mode, 3, "euler", "bf16"), (clips, keyword)
        assert sent.get("we_dynamic") == passed, (clips, keyword, sent)
        assert sent["we_frames"] == [c.get("we_T", 1) for c in clips]


def test_validation_before_any_device_call(pkg, monkeypatch):
    sampler = sys.modules[pkg.__name__ + ".sampler"]
    model, d = _small_model(pkg)
    L = d.frames_per_clip

    def no_device(*a, **k):
        raise AssertionError("device work before validation")

    monkeypatch.setattr(sampler, "backend_for", no_device)
    good_dyn = _clip(d, T=2 * L, we_T=2 * L, we_dynamic=True)
    bad = {
        "declared dynamic, 1-frame we": ([_clip(d, we_dynamic=True), good_dyn], ValueError),
        "declared static, per-frame we": ([good_dyn, _clip(d, T=2 * L, we_T=2 * L, we_dynamic=False)], ValueError),
        "non-bool mode": ([_clip(d, we_dynamic=1), good_dyn], TypeError),
        "string mode": ([_clip(d), _clip(d, T=2 * L, we_T=2 * L, we_dynamic="yes")], TypeError),
        "dynamic we short of the last window": ([_clip(d), _clip(d, T=2 * L + 1, we_T=2 * L, we_dynamic=True)], ValueError),
        "undeclared clips disagree": ([good_dyn, _clip(d), _clip(d, T=L, we_T=L)], ValueError),
    }
    for name, (clips, exc) in bad.items():
        with pytest.raises(exc):
            pkg.sample_clips(model, clips, **KW)
    with pytest.raises(TypeError):
        pkg.sample_clips(model, [_clip(d)], **dict(KW, we_dynamic=0))


@pytest.fixture()
def streams(pkg, monkeypatch):
    sampler = sys.modules[pkg.__name__ + ".sampler"]
    model, d = _small_model(pkg)
    be = _RecordingBackend(d)
    monkeypatch.setattr(sampler, "backend_for", lambda *a, **k: be)

    def make(**kw):
        return pkg.StreamSampler(model, **dict(dict(slots=3, nfe=3, method="euler", mode="bf16", device="cpu"), **kw))
    return make, be, d


def test_stream_validation(pkg, streams):
    make, be, d = streams
    r_s, we = torch.zeros(1, d.dim_w), torch.zeros(1, 1, d.dim_e)
    sm = make()                                           # static by default
    with pytest.raises(ValueError):
        sm.open(r_s, we, seed=1, we_dynamic=True)         # a dynamic stream's we arrives with feed()
    with pytest.raises(ValueError):
        sm.open(r_s, seed=1, we_dynamic=False)
    with pytest.raises(TypeError):
        sm.open(r_s, we, seed=1, we_dynamic=0)
    dyn, stat = sm.open(r_s, seed=1, we_dynamic=True), sm.open(r_s, we, seed=2)
    wa = torch.zeros(1, 5, d.dim_a)
    with pytest.raises(ValueError):
        sm.feed(stat, wa, torch.zeros(1, 5, d.dim_e))     # static stream fed we
    with pytest.raises(ValueError):
        sm.feed(dyn, wa)                                  # dynamic stream fed without we
    with pytest.raises(ValueError):
        sm.feed(dyn, wa, torch.zeros(1, 4, d.dim_e))
    assert dyn.fed == stat.fed == 0 and not be.calls
    dyn_sm = make(we_dynamic=True)
    with pytest.raises(ValueError):
        dyn_sm.open(r_s, we, seed=1)                      # the constructor's mode is the default
    dyn_sm.open(r_s, we, seed=1, we_dynamic=False)


def test_streams_resolve_their_modes(pkg, streams):
    make, be, d = streams
    L = d.frames_per_clip
    for default in (False, True):
        be.plans.clear(), be.calls.clear()
        sm = make(we_dynamic=default)
        assert be.plans == [(3, 3, default, 3, "euler", "bf16")]          # the plan keeps the constructor's mode
        r_s = torch.zeros(1, d.dim_w)
        s_we = torch.full((1, 1, d.dim_e), 7.0)
        stat = sm.open(r_s, s_we, seed=1, we_dynamic=False)
        dyn = sm.open(r_s, seed=2, we_dynamic=True)
        own = sm.open(r_s, None if default else s_we, seed=3)       # the sampler's mode
        assert (stat.we_dynamic, dyn.we_dynamic, own.we_dynamic) == (False, True, default)
        d_we = torch.arange(L + 5, dtype=torch.float32).reshape(1, -1, 1).expand(1, L + 5, d.dim_e).contiguous()
        sm.feed(stat, torch.zeros(1, L, d.dim_a))
        sm.feed(dyn, torch.zeros(1, L + 5, d.dim_a), d_we)
        sm.feed(own, torch.zeros(1, L, d.dim_a), d_we[:, :L] if default else None)
        sm.step()
        (sent,) = be.calls
        assert sent["we_dynamic"] == [False, True, default]         # mixed: every stream's mode goes down
        assert torch.equal(sent["we"][0], s_we) and torch.equal(sent["we"][1], d_we[0])
        assert all(p == be.plans[0] for p in be.plans)
        # a step whose streams all have the plan's mode passes none
        for s in (stat, dyn, own):
            sm.close(s)
        only = sm.open(r_s, None if default else s_we, seed=4)
        sm.feed(only, torch.zeros(1, L, d.dim_a), d_we[:, :L] if default else None)
        sm.step()
        assert "we_dynamic" not in be.calls[-1]


def test_c_abi_of_the_general_entries(pkg):
    lib = _lib(pkg)
    cabi = sys.modules[pkg.__name__ + "._cabi"]
    i32p = C.POINTER(C.c_int32)
    assert lib.fmt_sample_clip_set.argtypes == [C.c_void_p, C.POINTER(cabi.FmtClipSet), C.POINTER(cabi.FmtClipGuidance),
                                                C.POINTER(cabi.FmtClipOde), i32p, C.c_void_p]
    assert lib.fmt_sample_window_set.argtypes == [C.c_void_p, C.POINTER(cabi.FmtWindowSet), C.POINTER(cabi.FmtClipGuidance),
                                                  C.POINTER(cabi.FmtClipOde), i32p, C.c_void_p]
    assert lib.fmt_debug_condition_rows_slots.argtypes[4] == i32p
    # host-side argument checks, no device work
    assert lib.fmt_sample_clip_set(None, None, None, None, None, None) == -1
    assert lib.fmt_sample_window_set(None, None, None, None, None, None) == -1
    assert b"null argument" in lib.fmt_last_error()
