"""CPU tests of StreamSampler's host side: the readiness rule and slot order, the window each stream hands to the library, its
seeded noise, its bounded buffer and the validation that runs before any device call.  The backend is a recording stand-in."""
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


class FakeBackend:
    """Records every configure() and every window of sample_windows(); writes the step number into the outputs."""

    def __init__(self, dims):
        self.dims, self.device = dims, torch.device("cpu")
        self.plans, self.calls = [], []
        self.live = True

    def configure(self, *plan):
        assert self.live, "device work before validation"
        self.plans.append(plan)

    def sample_windows(self, r_s, wa, we, x0, ctx, out, first_window, a, r, e, nb):
        assert self.live, "device work before validation"
        self.calls.append([dict(wa=w.clone(), we=v.clone(), x0=x.clone(), first=f, n_out=o.shape[1], guidance=g)
                           for w, v, x, o, f, *g in zip(wa, we, x0, out, first_window, a, r, e, nb)])
        for o in out:
            o.fill_(len(self.calls))


@pytest.fixture()
def rig(pkg, monkeypatch):
    sampler = sys.modules[pkg.__name__ + ".sampler"]
    model, d = _small_model(pkg)
    fake = FakeBackend(d)
    monkeypatch.setattr(sampler, "backend_for", lambda m, dev, dims=None: fake)

    def make(**kw):
        args = dict(slots=2, nfe=3, method="euler", mode="bf16", device="cpu")
        args.update(kw)
        return pkg.StreamSampler(model, **args)
    return make, fake, d


def audio(d, t, seed=0):
    return torch.randn(1, t, d.dim_a, generator=torch.Generator().manual_seed(seed))


def opened(sm, d, seed, **kw):
    return sm.open(torch.zeros(1, d.dim_w), torch.zeros(1, 1, d.dim_e), seed=seed, **kw)


def test_readiness_and_selection_order(rig):
    make, fake, d = rig
    L = d.frames_per_clip
    sm = make(slots=2)
    a, b, c = (opened(sm, d, seed=i) for i in range(3))
    sm.feed(a, audio(d, 2 * L))
    sm.feed(b, audio(d, L - 1))
    sm.feed(c, audio(d, L))
    assert sm.ready() == [a, c]                                # b lacks a frame; a and c became ready together: open order
    out = sm.step()
    assert list(out) == [a, c] and all(o.shape == (1, L, d.dim_w) for o in out.values())
    sm.feed(b, audio(d, 1))
    assert sm.ready() == [a, b]                               # a's window 1 became ready before b's window 0
    sm2 = make(slots=1)
    x, y = opened(sm2, d, 1), opened(sm2, d, 2)
    sm2.feed(x, audio(d, 3 * L))
    sm2.feed(y, audio(d, L))
    assert list(sm2.step()) == [x]
    assert sm2.ready() == [y]                                  # y has waited longer than x's next window
    assert list(sm2.step()) == [y] and list(sm2.step()) == [x] and list(sm2.step()) == [x] and sm2.step() == {}
    assert not x.done                                          # 3 L frames but not finished: a 4th window may still come
    sm2.finish(x)
    assert sm2.ready() == [] and x.done                       # finished with exactly 3 L frames: no 4th window


def test_ragged_last_window_and_finish_edges(rig):
    make, fake, d = rig
    L = d.frames_per_clip
    sm = make(slots=4)
    ragged, short, exact = (opened(sm, d, seed=i) for i in range(3))
    sm.feed(ragged, audio(d, L + 7))
    sm.feed(short, audio(d, 5))
    sm.feed(exact, audio(d, 2 * L))
    assert sm.ready() == [ragged, exact]
    sm.step()
    assert sm.ready() == [exact]                               # ragged's 7 frames wait for more audio or finish()
    sm.finish(ragged)
    sm.finish(short)
    sm.finish(exact)
    assert sm.ready() == [exact, ragged, short]               # exact's window 1 was ready before finish() made the others ready
    out = sm.step()
    assert [o.shape[1] for o in out.values()] == [L, 7, 5]
    assert [w["first"] for w in fake.calls[-1]] == [0, 0, 1] and [w["n_out"] for w in fake.calls[-1]] == [L, 7, 5]
    assert all(s.done for s in (ragged, short, exact)) and sm.step() == {}
    with pytest.raises(ValueError):
        sm.feed(exact, audio(d, 1))                             # feed after finish


def test_each_window_sees_its_frames_and_the_clip_noise(pkg, rig):
    """Fed in random pieces, window w gets wa frames [w L - P, fed) (from 0 in window 0) and the w-th window of clip_noise(seed)."""
    make, fake, d = rig
    L, P = d.frames_per_clip, d.num_prev_frames
    rng = random.Random(3)
    T = [5 * L + 3, 2 * L, 1, 3 * L - 1]
    full = [audio(d, t, seed=10 + i) for i, t in enumerate(T)]
    sm = make(slots=3, we_dynamic=True)
    streams = [sm.open(torch.zeros(1, d.dim_w), seed=40 + i) for i in range(len(T))]
    fed = [0] * len(T)
    seen = {s: [] for s in streams}
    while any(not s.done for s in streams):
        for i, s in enumerate(streams):
            if fed[i] < T[i]:
                t = min(T[i] - fed[i], rng.randint(1, 2 * L))
                sm.feed(s, full[i][:, fed[i]:fed[i] + t], we=full[i][:, fed[i]:fed[i] + t, :d.dim_e])
                fed[i] += t
                if fed[i] == T[i]:
                    sm.finish(s)
        before = [s.fed for s in streams]
        out = sm.step()
        for s, win in zip(out, fake.calls[-1]):
            i, w = streams.index(s), len(seen[s])
            start = 0 if w == 0 else w * L - P
            assert torch.equal(win["wa"], full[i][0, start:before[i]]), (i, w)
            assert torch.equal(win["we"], full[i][0, start:before[i], :d.dim_e]), (i, w)
            assert win["first"] == int(w == 0) and win["n_out"] == min(L, T[i] - w * L)
            seen[s].append(win["x0"])
    for i, s in enumerate(streams):
        n_win = -(-T[i] // L)
        assert len(seen[s]) == n_win
        assert torch.equal(torch.stack(seen[s]), pkg.clip_noise(40 + i, d, n_win, "cpu"))
    assert len(set(fake.plans)) == 1 and fake.plans[0] == (3, 3, True, 3, "euler", "bf16")


def test_buffer_stays_bounded(rig):
    make, fake, d = rig
    L, P = d.frames_per_clip, d.num_prev_frames
    sm = make(slots=1)
    s = opened(sm, d, seed=5)
    chunk = 7
    peak = 0
    for k in range(30 * L // chunk):
        sm.feed(s, audio(d, chunk, seed=k))
        sm.step()
        assert s.buffered_frames == s.fed - max(0, s.windows_run * L - P)
        peak = max(peak, s.buffered_frames)
    assert s.windows_run >= 29 and peak <= P + L + chunk         # independent of the stream's length
    sm.close(s)
    with pytest.raises(ValueError):
        sm.feed(s, audio(d, 1))


def test_validation_before_any_device_call(pkg, rig, monkeypatch):
    make, fake, d = rig
    L = d.frames_per_clip
    sampler = sys.modules[pkg.__name__ + ".sampler"]
    model = _small_model(pkg)[0]
    no = dict(slots=2, nfe=3, method="euler", mode="bf16", device="cpu")
    bad_ctor = [(dict(no, slots=0), ValueError), (dict(no, slots=257), ValueError), (dict(no, slots=2.0), ValueError),
                (dict(no, nfe=0), ValueError), (dict(no, method="dopri5"), ValueError), (dict(no, mode="fp16"), ValueError),
                (dict(no, we_dynamic=1), TypeError), (dict(no, a_cfg_scale="2"), TypeError),
                (dict(no, e_cfg_scale=float("nan")), ValueError), (dict(no, include_r_cfg=1), TypeError)]
    with monkeypatch.context() as m:
        m.setattr(sampler, "backend_for", lambda *a, **k: pytest.fail("device work before validation"))
        for kw, exc in bad_ctor:
            with pytest.raises(exc):
                pkg.StreamSampler(model, **kw)

    sm = make()                                                # 3 branches
    dyn = make(we_dynamic=True)
    s = opened(sm, d, 1)
    sd = dyn.open(torch.zeros(1, d.dim_w), seed=1)
    sn = sm.open(torch.zeros(1, d.dim_w), torch.zeros(1, 1, d.dim_e), noise=torch.zeros(2, L, d.dim_w))
    fake.live = False
    r_s, we = torch.zeros(1, d.dim_w), torch.zeros(1, 1, d.dim_e)
    bad = {
        "r_s shape": lambda: sm.open(torch.zeros(2, d.dim_w), we, seed=1),
        "r_s dtype": (lambda: sm.open(torch.zeros(1, d.dim_w, dtype=torch.int64), we, seed=1), TypeError),
        "static without we": lambda: sm.open(r_s, seed=1),
        "static we shape": lambda: sm.open(r_s, torch.zeros(1, 2, d.dim_e), seed=1),
        "dynamic we at open": lambda: dyn.open(r_s, we, seed=1),
        "seed and noise": lambda: sm.open(r_s, we, seed=1, noise=torch.zeros(1, L, d.dim_w)),
        "neither seed nor noise": lambda: sm.open(r_s, we),
        "noise shape": lambda: sm.open(r_s, we, noise=torch.zeros(1, L + 1, d.dim_w)),
        "noise not a tensor": (lambda: sm.open(r_s, we, noise=[0.0]), TypeError),
        "more branches than the plan": lambda: sm.open(r_s, we, seed=1, r_cfg_scale=0.5, include_r_cfg=True),
        "unknown keyword": (lambda: sm.open(r_s, we, seed=1, cfg=2.0), TypeError),
        "bad scale": (lambda: sm.open(r_s, we, seed=1, a_cfg_scale=None), TypeError),
        "wa not a tensor": (lambda: sm.feed(s, [[0.0]]), TypeError),
        "wa dtype": (lambda: sm.feed(s, torch.zeros(1, 3, d.dim_a, dtype=torch.int32)), TypeError),
        "wa batch 2": lambda: sm.feed(s, torch.zeros(2, 3, d.dim_a)),
        "wa dim_a": lambda: sm.feed(s, torch.zeros(1, 3, d.dim_a + 1)),
        "wa empty": lambda: sm.feed(s, torch.zeros(1, 0, d.dim_a)),
        "we to a static stream": lambda: sm.feed(s, torch.zeros(1, 3, d.dim_a), torch.zeros(1, 3, d.dim_e)),
        "dynamic without we": lambda: dyn.feed(sd, torch.zeros(1, 3, d.dim_a)),
        "dynamic we length": lambda: dyn.feed(sd, torch.zeros(1, 3, d.dim_a), torch.zeros(1, 2, d.dim_e)),
        "beyond the given noise": lambda: sm.feed(sn, torch.zeros(1, 2 * L + 1, d.dim_a)),
        "finish with no audio": lambda: sm.finish(s),
        "another sampler's stream": lambda: dyn.feed(s, torch.zeros(1, 3, d.dim_a)),
    }
    for name, case in bad.items():
        fn, exc = case if isinstance(case, tuple) else (case, ValueError)
        with pytest.raises(exc):
            fn()
        assert s.fed == 0 and sd.fed == 0 and sn.fed == 0, name
    assert sm.step() == {} and fake.calls == []
    sm.feed(sn, torch.zeros(1, L, d.dim_a))
    with pytest.raises(ValueError):
        sm.finish(sn)                                           # 1 window of audio, 2 of noise
    sm.feed(s, torch.zeros(1, 3, d.dim_a))
    sm.finish(s)
    with pytest.raises(ValueError):
        sm.finish(s)
    with pytest.raises(ValueError):
        sm.feed(s, torch.zeros(1, 3, d.dim_a))
    assert fake.calls == []
    # a 4-branch plan takes 1-, 3- and 4-branch streams
    fake.live = True
    wide = make(a_cfg_scale=2.0, r_cfg_scale=0.5, include_r_cfg=True)
    assert wide.n_branches == 4
    for g in (dict(a_cfg_scale=1.0), dict(), dict(include_r_cfg=False), dict(a_cfg_scale=1.0, r_cfg_scale=1.0, include_r_cfg=False)):
        st = opened(wide, d, 1, **g)
        wide.feed(st, torch.zeros(1, L, d.dim_a))
    wide.step()
    assert [w["guidance"][3] for w in fake.calls[-1]] == [4, 4]
    wide.step()
    assert [w["guidance"][3] for w in fake.calls[-1]] == [3, 1]
