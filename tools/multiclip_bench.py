"""Many clips of different lengths: one call per clip, sample_clips on refilled slots, and (for context) one batched call with every
clip padded to the longest, alternated in one process.

  python tools/multiclip_bench.py [--out FILE] [--reps N]

Workload: 64 clips with seeded lengths between 50 and 300 frames (25 fps), nfe 10, euler, a_cfg 2 (3-way CFG), static emotion,
synthetic weights and inputs of bench.py, in the bf16 and bf16x3 modes.  Each arm has its own backend (plans stay captured); per rep
the arms run one after another, each timed with a host clock from a device synchronise to a device synchronise (256 MiB memset
before each, outside the timing).  Reported per arm: the median wall time, sum(T_i) / wall, the slot count and makespan of the
schedule, the window graphs replayed, and the card (name, power limit, max SM clock) read in the same run.
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON result here")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("multiclip_bench: needs a CUDA device (B200); there is nothing to measure without one")
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
    r_s, wa, we = [t.to(dev) for t in pkg.synth.synth_inputs(fd, N_CLIPS, T_pad, seed=7)]
    clip_rs = [r_s[i:i + 1].contiguous() for i in range(N_CLIPS)]
    clip_wa = [wa[i:i + 1, :T].contiguous() for i, T in enumerate(lengths)]
    clip_we = [we[i:i + 1].contiguous() for i in range(N_CLIPS)]
    noise = [pkg.clip_noise(1000 + i, dims, nw, dev) for i, nw in enumerate(n_win)]
    # padded arm: every clip replicate-padded to the longest (its own windows see the same wa; the noise of its extra windows is new)
    wa_pad = torch.cat([torch.cat([w, w[:, -1:].expand(1, T_pad - w.shape[1], -1)], dim=1) for w in clip_wa]).contiguous()
    nw_pad = math.ceil(T_pad / L)
    noise_pad = torch.randn(nw_pad, N_CLIPS, L, W, device=dev, generator=torch.Generator(dev).manual_seed(5))
    sched = pkg.clip_schedule(n_win)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    frames = sum(lengths)
    res = dict(card=card(), note=__doc__.strip().splitlines()[0], n_clips=N_CLIPS, lengths=lengths, sum_frames=frames, nfe=NFE,
               n_branches=3, schedule=dict(slots=sched.slots, makespan=sched.makespan, windows_of_all_clips=sum(n_win)))

    bes = {arm: pkg.FmtBackend(sd, dims, dev) for arm in ("per_clip", "sample_clips", "padded")}
    for mode in ("bf16", "bf16x3"):
        bes["per_clip"].configure(1, 3, False, NFE, "euler", mode)
        bes["sample_clips"].configure(sched.slots, 3, False, NFE, "euler", mode)
        bes["padded"].configure(N_CLIPS, 3, False, NFE, "euler", mode)
        outs = [torch.empty(1, T, W, device=dev) for T in lengths]
        out_pad = torch.empty(N_CLIPS, T_pad, W, device=dev)

        def per_clip():
            be = bes["per_clip"]
            for i, T in enumerate(lengths):
                be.sample_clip(clip_rs[i], clip_wa[i], clip_we[i], T, noise[i], A_CFG, 1.0, 1.0, out=outs[i])

        def multi():
            bes["sample_clips"].sample_clips(clip_rs, clip_wa, clip_we, lengths, noise, A_CFG, 1.0, 1.0, out=outs)

        def padded():
            bes["padded"].sample_clip(r_s, wa_pad, we, T_pad, noise_pad, A_CFG, 1.0, 1.0, out=out_pad)

        arms = {"per_clip": (per_clip, 1, sum(n_win)), "sample_clips": (multi, sched.slots, sched.makespan),
                "padded": (padded, N_CLIPS, nw_pad)}
        for fn, _, _ in arms.values():                     # warm-up
            fn()
        torch.cuda.synchronize()
        walls = {a: [] for a in arms}
        for _ in range(args.reps):
            for a, (fn, _, _) in arms.items():
                flush.zero_()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn()
                torch.cuda.synchronize()
                walls[a].append(time.perf_counter() - t0)
        r = {}
        for a, (_, batch, graphs) in arms.items():
            w = sorted(walls[a])
            med = w[len(w) // 2]
            r[a] = dict(wall_s_median=med, wall_s_min=w[0], wall_s_max=w[-1], frames_per_s=frames / med, batch_slots=batch,
                        windows_makespan=graphs, window_graphs_replayed=graphs)
        r["speedup_sample_clips_over_per_clip"] = r["per_clip"]["wall_s_median"] / r["sample_clips"]["wall_s_median"]
        r["speedup_sample_clips_over_padded"] = r["padded"]["wall_s_median"] / r["sample_clips"]["wall_s_median"]
        res[mode] = r
    for be in bes.values():
        be.close()
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        json.dump(res, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
