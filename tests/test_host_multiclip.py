"""CPU tests of sample_clips' host side: the slot schedule (fmt_clip_schedule, host-only), per-clip seeded noise and the
validation that runs before any device call."""
import random
import sys

import pytest
import torch

import cases
from __graft_entry__ import load_package


@pytest.fixture(scope="module")
def pkg():
    p = load_package()
    sys.modules[p.__name__ + ".build"].build()
    return p


def _small_model(pkg):
    """The small synthetic FMT with options that match its weights (window geometry included), on the CPU."""
    opt = pkg.BaseOptions()
    for k, v in cases.SMALL_DIMS.as_dict().items():
        if hasattr(opt, k):
            setattr(opt, k, v)
    model = pkg.FmtModel(cases.weights("small"), opt, target_device="cpu")
    return model, pkg.Dims.from_options(opt, model.state_dict())


def _check_schedule(n_win, sch):
    """Every clip gets exactly its windows, in one slot, back to back; no slot runs two clips in one window."""
    S, makespan = sch.slots, sch.makespan
    busy = {}
    for i, nw in enumerate(n_win):
        assert 0 <= sch.slot[i] < S and sch.start[i] >= 0
        for w in range(sch.start[i], sch.start[i] + nw):
            assert (sch.slot[i], w) not in busy, (i, busy.get((sch.slot[i], w)))
            busy[(sch.slot[i], w)] = i
    assert makespan == max(sch.start[i] + nw for i, nw in enumerate(n_win))
    assert len(busy) == sum(n_win)


def test_schedule_lengths_minimal_and_deterministic(pkg):
    rng = random.Random(7)
    for trial in range(200):
        n = rng.randint(1, 40)
        n_win = [rng.randint(1, rng.choice([2, 6, 12])) for _ in range(n)]
        sch = pkg.clip_schedule(n_win)
        _check_schedule(n_win, sch)
        assert sch.makespan == max(n_win), (n_win, sch)
        # minimal: every smaller slot count, scheduled the same way, takes longer than the longest clip
        for s in range(1, sch.slots):
            smaller = pkg.clip_schedule(n_win, n_slots=s)
            _check_schedule(n_win, smaller)
            assert smaller.slots == s and smaller.makespan > max(n_win), (n_win, s, smaller)
        assert pkg.clip_schedule(n_win) == sch                        # deterministic


def test_schedule_order_and_refill(pkg):
    # [300, 50 x 6] frames at L = 50: a 6-window clip and six 1-window clips fill 2 slots in 6 windows
    n_win = [6, 1, 1, 1, 1, 1, 1]
    sch = pkg.clip_schedule(n_win)
    assert sch.slots == 2 and sch.makespan == 6
    assert sch.slot[0] == 0 and sch.start[0] == 0
    assert [sch.slot[i] for i in range(1, 7)] == [1] * 6 and [sch.start[i] for i in range(1, 7)] == list(range(6))  # refills in input order
    # longest first, ties in input order
    sch = pkg.clip_schedule([2, 5, 2, 5])
    assert sch.slots == 3 and sch.makespan == 5
    assert list(zip(sch.slot, sch.start)) == [(2, 0), (0, 0), (2, 2), (1, 0)]


def test_schedule_edge_cases(pkg):
    for n in (1, 2, 5, 64, 256):
        for w in (1, 3):
            sch = pkg.clip_schedule([w] * n)
            assert sch.slots == n and sch.makespan == w and sorted(sch.slot) == list(range(n)) and set(sch.start) == {0}
    assert pkg.clip_schedule([9]) == pkg.ClipSchedule(1, (0,), (0,), 9)
    # more clips than 256 slots of the longest clip's length can hold: 256 slots, a longer makespan
    sch = pkg.clip_schedule([2] * 600)
    _check_schedule([2] * 600, sch)
    assert sch.slots == 256 and sch.makespan == 6
    with pytest.raises(ValueError):
        pkg.clip_schedule([])
    with pytest.raises(ValueError):
        pkg.clip_schedule([3, 0])
    with pytest.raises(ValueError):
        pkg.clip_schedule([3], n_slots=257)


def test_seeded_noise_is_the_single_clip_node_draw(pkg, monkeypatch):
    """A clip's seed draws what the VA node draws for that clip alone (batch 1, fix_noise_seed) on the same device."""
    nodes = sys.modules[pkg.__name__ + ".nodes"]
    model, d = _small_model(pkg)
    drawn = {}

    def fake_loop(**kw):
        n_win = -(-kw["audio_num_frames"] // kw["model_num_frames_for_clip"])
        drawn["noise"] = pkg.draw_window_noise(1, d, n_win, kw["target_device"], kw["noise_seed_generator"])
        return torch.zeros(1, kw["audio_num_frames"], d.dim_w)

    monkeypatch.setattr(nodes, "perform_ode_sampling_loop", fake_loop)
    L = d.frames_per_clip
    for seed, T in ((15, 3 * L - 7), (123456789, L)):
        r_s, wa, we = torch.zeros(1, d.dim_w), torch.zeros(1, T, d.dim_a), torch.zeros(1, 1, d.dim_e)
        nodes.FloatSampleMotionSequenceRD_VA().sample_rd_sequence_va(r_s, wa, we, T, model, 2.0, 1.0, 1.0, False, 3, "euler", 1e-5, 1e-5,
                                                                     0.1, 0.1, 0.1, True, seed)
        mine = pkg.clip_noise(seed, d, -(-T // L), "cpu")
        assert mine.shape == (-(-T // L), 1, L, d.dim_w) and torch.equal(mine, drawn["noise"])


def test_validation_before_any_device_call(pkg, monkeypatch):
    sampler = sys.modules[pkg.__name__ + ".sampler"]
    model, d = _small_model(pkg)
    L = d.frames_per_clip

    def clip(T=30, T_wa=None, we_T=1, B=1, **kw):
        c = dict(r_s=torch.zeros(B, d.dim_w), wa=torch.zeros(B, T_wa or T, d.dim_a), we=torch.zeros(B, we_T, d.dim_e),
                 audio_num_frames=T, seed=1)
        c.update(kw)
        return c

    def no_device(*a, **k):
        raise AssertionError("device work before validation")

    monkeypatch.setattr(sampler, "backend_for", no_device)
    kw = dict(nfe=3, method="euler", a_cfg_scale=2.0, r_cfg_scale=1.0, e_cfg_scale=1.0, include_r_cfg=False, mode="bf16", device="cpu")
    bad = {
        "mixed emotion": ([clip(), clip(T=2 * L, we_T=2 * L)], ValueError),
        "short wa": ([clip(T=2 * L + 1, T_wa=2 * L)], ValueError),
        "short dynamic we": ([clip(T=2 * L + 1, we_T=2 * L)], ValueError),
        "batch 2": ([clip(B=2)], ValueError),
        "empty": ([], ValueError),
        "not a list": (clip(), TypeError),
        "not a mapping": ([torch.zeros(3)], TypeError),
        "not tensors": ([clip(wa=[[0.0]])], TypeError),
        "seed and noise": ([clip(noise=torch.zeros(1, L, d.dim_w))], ValueError),
        "bad noise": ([clip(seed=None, noise=torch.zeros(2, L, d.dim_w))], ValueError),
        "wrong dim_a": ([clip(wa=torch.zeros(1, 30, d.dim_a + 1))], ValueError),
        "zero frames": ([clip(audio_num_frames=0)], ValueError),
    }
    for name, (clips, exc) in bad.items():
        with pytest.raises(exc):
            pkg.sample_clips(model, clips, **kw)
    with pytest.raises(ValueError):
        pkg.sample_clips(model, [clip()], **dict(kw, method="dopri5"))
    # valid clips reach the backend, and a CPU device has no fallback
    monkeypatch.undo()
    with pytest.raises(pkg.FmtError):
        pkg.sample_clips(model, [clip(), clip(T=2 * L - 3), clip(T=L, noise=torch.zeros(1, L, d.dim_w), seed=None)], **kw)
