"""Clips with different ODE schedules (nfe, solver): one sample_clips call with per-clip schedules against one call per schedule
(and, for the first workload, one call per clip), alternated in one process.

  python tools/schedule_bench.py [--out FILE] [--reps N]

Clips: the 64 of tools/multiclip_bench.py (same seeded lengths of 50-300 frames, inputs and per-clip noise seeds), 3-way CFG
(a_cfg 2), static emotion, synthetic weights of bench.py, in the bf16 and bf16x3 modes.  Workloads:
  (i)  (euler, 10), (heun3, 4), (midpoint, 5), (rk4, 3) assigned round-robin: 9, 9, 8 and 8 evaluations per window.  Arms: one
       mixed call (plan: euler 10, the per-slot window graph), one sample_clips call per schedule (four), one call per clip.
  (ii) 8 of the 64 clips (every 8th) at (euler, 20), 19 evaluations, the rest at (euler, 10), 9.  Arms: one mixed call (every slot
       padded to 19 evaluations), and two calls (the euler-20 clips, then the euler-10 clips, each through its plan's graph).
Each call of an arm has its own backend, so every plan and graph stays captured.  Per rep the arms run one after another, each
timed with a host clock from a device synchronise to a device synchronise (256 MiB memset before each, outside the timing).
Reported per arm: the median wall time of --reps, sum(T_i) / wall, the slots and window graphs of each call, and the card (name,
power limit, max SM clock) read in the same run.
"""
import argparse
import json
import math
import os
import random
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from __graft_entry__ import load_package  # noqa: E402
from multiclip_bench import A_CFG, N_CLIPS, T_MAX, T_MIN, card  # noqa: E402

SCHEDULES_I = [(10, "euler"), (4, "heun3"), (5, "midpoint"), (3, "rk4")]
LONG, BASE = (20, "euler"), (10, "euler")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON result here")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("schedule_bench: needs a CUDA device (B200); there is nothing to measure without one")
    pkg = load_package()
    dev = torch.device("cuda:0")
    fd = pkg.synth.FmtDims()
    sd = pkg.synth.synth_state_dict(fd, seed=0)
    dims = pkg.Dims.from_options(pkg.BaseOptions(), sd)
    L, W = dims.frames_per_clip, dims.dim_w
    rng = random.Random(4)
    lengths = [rng.randint(T_MIN, T_MAX) for _ in range(N_CLIPS)]
    n_win = [math.ceil(T / L) for T in lengths]
    r_s, wa, we = [t.to(dev) for t in pkg.synth.synth_inputs(fd, N_CLIPS, max(lengths), seed=7)]
    clip_rs = [r_s[i:i + 1].contiguous() for i in range(N_CLIPS)]
    clip_wa = [wa[i:i + 1, :T].contiguous() for i, T in enumerate(lengths)]
    clip_we = [we[i:i + 1].contiguous() for i in range(N_CLIPS)]
    noise = [pkg.clip_noise(1000 + i, dims, nw, dev) for i, nw in enumerate(n_win)]
    outs = [torch.empty(1, T, W, device=dev) for T in lengths]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    frames = sum(lengths)
    workloads = {
        "i_near_equal_evaluations": [SCHEDULES_I[i % len(SCHEDULES_I)] for i in range(N_CLIPS)],
        "ii_8_of_64_at_euler_20": [LONG if i % 8 == 0 else BASE for i in range(N_CLIPS)],
    }
    res = dict(card=card(), note=__doc__.strip().splitlines()[0], n_clips=N_CLIPS, lengths=lengths, sum_frames=frames, a_cfg_scale=A_CFG)

    def call_on(idx, schedules):
        """One sample_clips call over the clips idx, on a backend of its own: per-clip schedules unless they are all one."""
        sch = pkg.clip_schedule([n_win[i] for i in idx])
        own = [schedules[i] for i in idx]
        plan = pkg.plan_schedule(own, *own[0])
        be = pkg.FmtBackend(sd, dims, dev)
        pick = lambda xs: [xs[i] for i in idx]                  # noqa: E731
        kw = {} if all(s == plan for s in own) else dict(schedules=own)

        def fn():
            be.sample_clips(pick(clip_rs), pick(clip_wa), pick(clip_we), pick(lengths), pick(noise), A_CFG, 1.0, 1.0, out=pick(outs), **kw)
        return be, sch, plan, fn, bool(kw)

    for wl, schedules in workloads.items():
        groups = {}
        for i, s in enumerate(schedules):
            groups.setdefault(s, []).append(i)
        calls = {"mixed": [call_on(list(range(N_CLIPS)), schedules)],
                 "grouped": [call_on(idx, schedules) for idx in sorted(groups.values(), key=lambda ix: -pkg.n_evals(*schedules[ix[0]]))]}
        per_clip_be = {s: pkg.FmtBackend(sd, dims, dev) for s in groups} if wl.startswith("i_") else None
        res[wl] = dict(schedules={f"{m} {n}": len(ix) for (n, m), ix in groups.items()})
        for mode in ("bf16", "bf16x3"):
            for arm in calls.values():
                for be, sch, plan, _, _ in arm:
                    be.configure(sch.slots, 3, False, *plan, mode)
            fns = {name: (lambda arm=arm: [c[3]() for c in arm]) for name, arm in calls.items()}
            if per_clip_be is not None:
                for s, be in per_clip_be.items():
                    be.configure(1, 3, False, *s, mode)

                def per_clip():
                    for i, T in enumerate(lengths):
                        per_clip_be[schedules[i]].sample_clip(clip_rs[i], clip_wa[i], clip_we[i], T, noise[i], A_CFG, 1.0, 1.0, out=outs[i])
                fns["per_clip"] = per_clip
            for fn in fns.values():                            # warm-up: graphs captured, t-embeddings cached
                fn()
            torch.cuda.synchronize()
            walls = {a: [] for a in fns}
            for _ in range(args.reps):
                for a, fn in fns.items():
                    flush.zero_()
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    fn()
                    torch.cuda.synchronize()
                    walls[a].append(time.perf_counter() - t0)
            r = {}
            for a, w in walls.items():
                w = sorted(w)
                med = w[len(w) // 2]
                r[a] = dict(wall_s_median=med, wall_s_min=w[0], wall_s_max=w[-1], frames_per_s=frames / med)
                if a in calls:
                    r[a]["calls"] = [dict(clips=len(sch.slot), plan=f"{plan[1]} {plan[0]}", evaluations=pkg.n_evals(*plan), slots=sch.slots,
                                          window_graphs=sch.makespan, per_slot_graph=per_slot) for _, sch, plan, _, per_slot in calls[a]]
                else:
                    r[a]["calls"] = dict(n=N_CLIPS, slots=1, window_graphs=sum(n_win))
            r["speedup_mixed_over_grouped"] = r["grouped"]["wall_s_median"] / r["mixed"]["wall_s_median"]
            r["faster"] = "mixed" if r["speedup_mixed_over_grouped"] > 1 else "grouped"
            if "per_clip" in r:
                r["speedup_mixed_over_per_clip"] = r["per_clip"]["wall_s_median"] / r["mixed"]["wall_s_median"]
            res[wl][mode] = r
        for arm in calls.values():
            for be, _, _, _, _ in arm:
                be.close()
        for be in (per_clip_be or {}).values():
            be.close()
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        json.dump(res, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
