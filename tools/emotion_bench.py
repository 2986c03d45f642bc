"""Static and dynamic emotion in one call against one call per mode and one call per clip, and one StreamSampler holding both kinds
of stream against two samplers (one per mode) stepping alternately on one backend, alternated in one process.

  python tools/emotion_bench.py [--out FILE] [--reps N]

Workload: the 64 clips of tools/multiclip_bench.py (same seeded lengths, inputs and noise seeds; nfe 10, euler, a_cfg 2 = 3-way CFG,
synthetic weights of bench.py), the odd-numbered half with dynamic emotion (one SER-like vector per 50-frame chunk), in the bf16 and
bf16x3 modes.  Clip arms, each on its own backend so that plans stay captured:
  mixed     one sample_clips call of all 64 clips
  per_mode  one call with the 32 static clips, then one with the 32 dynamic clips
  per_clip  one call per clip (batch 1)
Stream arms, on the slot count of the mixed call, all audio fed up front, stepped until drained (noise drawn from the seeds inside
the timed region): one StreamSampler with both kinds of stream, and a static and a dynamic sampler stepping in turn on one backend.
Each arm is timed with a host clock from a device synchronise to a device synchronise (256 MiB memset before each, outside the
timing); reported are the median wall time over --reps and sum(T_i) / wall.  The card (name, power limit, max SM clock) is read in
the same run.
"""
import argparse
import json
import math
import os
import random
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from __graft_entry__ import load_package  # noqa: E402

N_CLIPS, T_MIN, T_MAX, NFE, A_CFG = 64, 50, 300, 10, 2.0


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


class _Model:
    """The synthetic FMT as the module StreamSampler and backend_for take: state_dict() and options."""

    def __init__(self, sd, opt):
        self._sd, self.opt, self.target_device = sd, opt, "cuda:0"

    def state_dict(self):
        return self._sd


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON result here")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("emotion_bench: needs a CUDA device (B200); there is nothing to measure without one")
    pkg = load_package()
    dev = torch.device("cuda:0")
    fd = pkg.synth.FmtDims()
    sd = pkg.synth.synth_state_dict(fd, seed=0)
    dims = pkg.Dims.from_options(pkg.BaseOptions(), sd)
    L, W = dims.frames_per_clip, dims.dim_w
    rng = random.Random(4)
    lengths = [rng.randint(T_MIN, T_MAX) for _ in range(N_CLIPS)]
    n_win = [math.ceil(T / L) for T in lengths]
    T_pad = max(lengths)
    r_s, wa, we_s = [t.to(dev) for t in pkg.synth.synth_inputs(fd, N_CLIPS, T_pad, seed=7)]
    we_d = pkg.synth.synth_inputs(fd, N_CLIPS, T_pad, seed=7, dynamic_we=True)[2].to(dev)
    dyn = [i % 2 == 1 for i in range(N_CLIPS)]
    clip_rs = [r_s[i:i + 1].contiguous() for i in range(N_CLIPS)]
    clip_wa = [wa[i:i + 1, :T].contiguous() for i, T in enumerate(lengths)]
    clip_we = [(we_d[i:i + 1, :T] if dyn[i] else we_s[i:i + 1]).contiguous() for i, T in enumerate(lengths)]
    noise = [pkg.clip_noise(1000 + i, dims, nw, dev) for i, nw in enumerate(n_win)]
    groups = {m: [i for i in range(N_CLIPS) if dyn[i] == m] for m in (False, True)}
    sched = pkg.clip_schedule(n_win)
    sched_mode = {m: pkg.clip_schedule([n_win[i] for i in g]) for m, g in groups.items()}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    frames = sum(lengths)
    res = dict(card=card(), note=__doc__.strip().splitlines()[0], n_clips=N_CLIPS, n_dynamic=sum(dyn), lengths=lengths,
               sum_frames=frames, nfe=NFE, n_branches=3,
               schedule=dict(mixed=[sched.slots, sched.makespan], static=[sched_mode[False].slots, sched_mode[False].makespan],
                             dynamic=[sched_mode[True].slots, sched_mode[True].makespan]))
    model = _Model(sd, pkg.BaseOptions())

    bes = {arm: pkg.FmtBackend(sd, dims, dev) for arm in ("mixed", "static", "dynamic", "per_clip")}
    for mode in ("bf16", "bf16x3"):
        bes["mixed"].configure(sched.slots, 3, False, NFE, "euler", mode)
        for m, name in ((False, "static"), (True, "dynamic")):
            bes[name].configure(sched_mode[m].slots, 3, m, NFE, "euler", mode)
        bes["per_clip"].configure(1, 3, False, NFE, "euler", mode)
        outs = [torch.empty(1, T, W, device=dev) for T in lengths]

        def mixed():
            bes["mixed"].sample_clips(clip_rs, clip_wa, clip_we, lengths, noise, A_CFG, 1.0, 1.0, out=outs, we_dynamic=dyn)

        def per_mode():
            for m, name in ((False, "static"), (True, "dynamic")):
                g = groups[m]
                bes[name].sample_clips(*[[x[i] for i in g] for x in (clip_rs, clip_wa, clip_we, lengths, noise)], A_CFG, 1.0, 1.0,
                                       out=[outs[i] for i in g])

        def per_clip():
            be = bes["per_clip"]
            for i in range(N_CLIPS):
                be.sample_clips([clip_rs[i]], [clip_wa[i]], [clip_we[i]], [lengths[i]], [noise[i]], A_CFG, 1.0, 1.0, out=[outs[i]],
                                we_dynamic=[dyn[i]])

        kw = dict(nfe=NFE, method="euler", mode=mode, a_cfg_scale=A_CFG, r_cfg_scale=1.0, e_cfg_scale=1.0, include_r_cfg=False,
                  device=dev)

        def feed_all(sm, idx):
            sts = []
            for i in idx:
                st = sm.open(clip_rs[i], None if dyn[i] else clip_we[i], seed=1000 + i, we_dynamic=dyn[i])
                sm.feed(st, clip_wa[i], clip_we[i] if dyn[i] else None)
                sm.finish(st)
                sts.append(st)
            return sts

        def one_sampler():
            sm = pkg.StreamSampler(model, slots=sched.slots, **kw)
            sts = feed_all(sm, range(N_CLIPS))
            while not all(s.done for s in sts):
                sm.step()

        def two_samplers():
            sms = {m: pkg.StreamSampler(model, slots=sched.slots, we_dynamic=m, **kw) for m in (False, True)}
            sts = {m: feed_all(sms[m], groups[m]) for m in (False, True)}
            while not all(s.done for m in sts for s in sts[m]):
                for m in (False, True):
                    sms[m].step()

        arms = {"mixed": mixed, "per_mode": per_mode, "per_clip": per_clip, "stream_one_sampler": one_sampler,
                "stream_two_samplers": two_samplers}
        for fn in arms.values():                           # warm-up
            fn()
        torch.cuda.synchronize()
        walls = {a: [] for a in arms}
        for _ in range(args.reps):
            for a, fn in arms.items():
                flush.zero_()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn()
                torch.cuda.synchronize()
                walls[a].append(time.perf_counter() - t0)
        r = {}
        for a in arms:
            w = sorted(walls[a])
            med = w[len(w) // 2]
            r[a] = dict(wall_s_median=med, wall_s_min=w[0], wall_s_max=w[-1], frames_per_s=frames / med)
        res[mode] = r
    for be in bes.values():
        be.close()
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        json.dump(res, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
