"""Clips with different guidance settings: one sample_clips call with per-clip guidance against one call per settings group (and,
for the first workload, one call per clip), alternated in one process.

  python tools/guidance_bench.py [--out FILE] [--reps N]

Clips: the 64 of tools/multiclip_bench.py (same seeded lengths of 50-300 frames, inputs and per-clip noise seeds), nfe 10, euler,
static emotion, synthetic weights of bench.py, in the bf16 and bf16x3 modes.  Workloads:
  (i)  four 3-branch settings (a_cfg, e_cfg) = (2, 1), (1, 3), (1.5, 1.5), (2.5, 0.5), assigned round-robin.  Arms: one mixed
       call, one sample_clips call per settings group (four), one call per clip.
  (ii) 8 of the 64 clips (every 8th) use include_r_cfg with r_cfg 0.5 (4 branches), the rest a_cfg 2 (3 branches).  Arms: one
       mixed call on a 4-branch plan, and two grouped calls (the 4-branch clips, then the 3-branch clips).
Each call of an arm has its own backend, so every plan stays captured.  Per rep the arms run one after another, each timed with
a host clock from a device synchronise to a device synchronise (256 MiB memset before each, outside the timing).  Reported per
arm: the median wall time of --reps, sum(T_i) / wall, the slots and window graphs of each call, and the card (name, power limit,
max SM clock) read in the same run.
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
from multiclip_bench import N_CLIPS, NFE, T_MAX, T_MIN, card  # noqa: E402

SETTINGS_I = [(2.0, 1.0, 1.0, False), (1.0, 1.0, 3.0, False), (1.5, 1.0, 1.5, False), (2.5, 1.0, 0.5, False)]
R_CFG, BASE = (2.0, 0.5, 1.0, True), (2.0, 1.0, 1.0, False)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON result here")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("guidance_bench: needs a CUDA device (B200); there is nothing to measure without one")
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
        "i_four_3branch_settings": [SETTINGS_I[i % len(SETTINGS_I)] for i in range(N_CLIPS)],
        "ii_8_of_64_include_r_cfg": [R_CFG if i % 8 == 0 else BASE for i in range(N_CLIPS)],
    }
    res = dict(card=card(), note=__doc__.strip().splitlines()[0], n_clips=N_CLIPS, lengths=lengths, sum_frames=frames, nfe=NFE)

    def call_on(idx, settings, plan_nb=None):
        """One sample_clips call over the clips idx, on a backend of its own; returns (fn, info)."""
        sch = pkg.clip_schedule([n_win[i] for i in idx])
        nb = [pkg.n_branches_for(*settings[i]) for i in idx]
        be = pkg.FmtBackend(sd, dims, dev)
        pick = lambda xs: [xs[i] for i in idx]                  # noqa: E731
        a, r, e = ([settings[i][k] for i in idx] for k in range(3))

        def fn():
            be.sample_clips(pick(clip_rs), pick(clip_wa), pick(clip_we), pick(lengths), pick(noise), a, r, e, out=pick(outs), n_branches=nb)
        return be, sch, plan_nb or max(nb), fn

    for wl, settings in workloads.items():
        groups = {}
        for i, g in enumerate(settings):
            groups.setdefault(g, []).append(i)
        calls = {"mixed": [call_on(list(range(N_CLIPS)), settings)],
                 "grouped": [call_on(idx, settings) for idx in sorted(groups.values(), key=lambda ix: -pkg.n_branches_for(*settings[ix[0]]))]}
        per_clip_be = pkg.FmtBackend(sd, dims, dev) if wl.startswith("i_") else None
        res[wl] = dict(settings={str(g): len(ix) for g, ix in groups.items()})
        for mode in ("bf16", "bf16x3"):
            for arm in calls.values():
                for be, sch, nb, _ in arm:
                    be.configure(sch.slots, nb, False, NFE, "euler", mode)
            fns = {name: (lambda arm=arm: [c[3]() for c in arm]) for name, arm in calls.items()}
            if per_clip_be is not None:
                per_clip_be.configure(1, 3, False, NFE, "euler", mode)

                def per_clip():
                    for i, T in enumerate(lengths):
                        per_clip_be.sample_clip(clip_rs[i], clip_wa[i], clip_we[i], T, noise[i], *settings[i][:3], out=outs[i])
                fns["per_clip"] = per_clip
            for fn in fns.values():                            # warm-up
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
                    r[a]["calls"] = [dict(clips=len(sch.slot), plan_branches=nb, slots=sch.slots, window_graphs=sch.makespan)
                                     for _, sch, nb, _ in calls[a]]
                else:
                    r[a]["calls"] = dict(n=N_CLIPS, plan_branches=3, slots=1, window_graphs=sum(n_win))
            r["speedup_mixed_over_grouped"] = r["grouped"]["wall_s_median"] / r["mixed"]["wall_s_median"]
            r["faster"] = "mixed" if r["speedup_mixed_over_grouped"] > 1 else "grouped"
            if "per_clip" in r:
                r["speedup_mixed_over_per_clip"] = r["per_clip"]["wall_s_median"] / r["mixed"]["wall_s_median"]
            res[wl][mode] = r
        for arm in calls.values():
            for be, _, _, _ in arm:
                be.close()
        if per_clip_be is not None:
            per_clip_be.close()
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        json.dump(res, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
