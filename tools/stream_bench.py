"""Streams (StreamSampler) against the offline calls, alternated in one process.

  python tools/stream_bench.py [--out FILE] [--steps N] [--reps N]

1. Step latency: S in {1, 8, 32, 64, 128, 256} streams, all with their next window ready (bf16, nfe 10, euler, a_cfg 2 = 3-way CFG,
   static emotion).  Each step is timed with a host clock from a device synchronise to a device synchronise, alternating with one
   window of fmt_sample_clip at batch S (its own backend, the same plan).  Reported: the medians over --steps steps, their
   difference (the cost of streaming: slot records, per-stream noise draw, buffer trimming, the Python bookkeeping) and the
   derived number of real-time streams, S * floor(2 s / t_step) (a window is 50 frames = 2 s of video at 25 fps).
2. Continuous batching: the 64 clips of tools/multiclip_bench.py (same lengths, inputs and seeds) through StreamSampler(slots=44)
   with all audio fed up front and stepped until drained, against sample_clips (44 slots, 6 windows), in bf16 and bf16x3.  Both
   arms draw their noise from the clips' seeds inside the timed region; wall time is the median of --reps, arms alternated.
The card (name, power limit, max SM clock) is read in the same run.
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
SLOT_COUNTS = (1, 8, 32, 64, 128, 256)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def median(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON result here")
    ap.add_argument("--steps", type=int, default=25, help="timed steps per slot count (median)")
    ap.add_argument("--reps", type=int, default=3, help="repetitions of the continuous-batching workload (median)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stream_bench: needs a CUDA device (B200); there is nothing to measure without one")
    pkg = load_package()
    dev = torch.device("cuda:0")
    fd = pkg.synth.FmtDims()
    sd = pkg.synth.synth_state_dict(fd, seed=0)
    opt = pkg.BaseOptions()
    model = pkg.FmtModel(sd, opt, target_device=dev)
    dims = pkg.Dims.from_options(opt, sd)
    L, W = dims.frames_per_clip, dims.dim_w
    res = dict(card=card(), note=__doc__.strip().splitlines()[0], nfe=NFE, n_branches=3)

    # ---- 1. step latency
    window_be = pkg.FmtBackend(sd, dims, dev)
    n_win = args.steps + 2                                  # 2 warm-up steps
    lat = {}
    for S in SLOT_COUNTS:
        r_s, wa, we = [t.to(dev) for t in pkg.synth.synth_inputs(fd, S, n_win * L, seed=11)]
        sm = pkg.StreamSampler(model, slots=S, nfe=NFE, method="euler", mode="bf16", a_cfg_scale=A_CFG, device=dev)
        streams = [sm.open(r_s[i:i + 1], we[i:i + 1], seed=i) for i in range(S)]
        for i, s in enumerate(streams):
            sm.feed(s, wa[i:i + 1])
        window_be.configure(S, 3, False, NFE, "euler", "bf16")
        win_wa = wa[:, :L].contiguous()
        noise = torch.randn(1, S, L, W, device=dev, generator=torch.Generator(dev).manual_seed(3))
        out = torch.empty(S, L, W, device=dev)
        t_stream, t_window = [], []
        for k in range(n_win):
            ts, ran = timed(sm.step)
            assert len(ran) == S
            tw, _ = timed(lambda: window_be.sample_clip(r_s, win_wa, we, L, noise, A_CFG, 1.0, 1.0, out=out))
            if k >= 2:
                t_stream.append(ts)
                t_window.append(tw)
        ms, mw = median(t_stream), median(t_window)
        lat[str(S)] = dict(step_ms_median=ms * 1e3, step_ms_min=min(t_stream) * 1e3, step_ms_max=max(t_stream) * 1e3,
                           sample_clip_window_ms_median=mw * 1e3, streaming_cost_ms=(ms - mw) * 1e3,
                           realtime_streams_derived=S * math.floor(2.0 / ms))
        for s in streams:
            sm.close(s)
        del sm, streams, r_s, wa, we
        torch.cuda.empty_cache()
    window_be.close()
    res["step_latency"] = dict(steps_timed=args.steps, by_streams=lat,
                               realtime_streams_note="derived: S * floor(2 s / median step time), not a measured real-time run")

    # ---- 2. continuous batching: the workload of tools/multiclip_bench.py
    rng = random.Random(4)
    lengths = [rng.randint(T_MIN, T_MAX) for _ in range(N_CLIPS)]
    r_s, wa, we = [t.to(dev) for t in pkg.synth.synth_inputs(fd, N_CLIPS, max(lengths), seed=7)]
    clips = [dict(r_s=r_s[i:i + 1].contiguous(), wa=wa[i:i + 1, :T].contiguous(), we=we[i:i + 1].contiguous(), seed=1000 + i)
             for i, T in enumerate(lengths)]
    sched = pkg.clip_schedule([math.ceil(T / L) for T in lengths])
    frames = sum(lengths)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    cb = dict(n_clips=N_CLIPS, sum_frames=frames, slots=sched.slots, sample_clips_makespan=sched.makespan)
    for mode in ("bf16", "bf16x3"):
        sm = pkg.StreamSampler(model, slots=sched.slots, nfe=NFE, method="euler", mode=mode, a_cfg_scale=A_CFG, device=dev)

        def offline():
            return pkg.sample_clips(model, clips, nfe=NFE, method="euler", a_cfg_scale=A_CFG, mode=mode, device=dev)

        def streamed():
            streams = [sm.open(c["r_s"], c["we"], seed=c["seed"]) for c in clips]
            for s, c in zip(streams, clips):
                sm.feed(s, c["wa"])
                sm.finish(s)
            got, steps = {s: [] for s in streams}, 0
            while not all(s.done for s in streams):
                for s, o in sm.step().items():
                    got[s].append(o)
                steps += 1
            for s in streams:
                sm.close(s)
            return [torch.cat(got[s], dim=1) for s in streams], steps

        offline(), streamed()                              # warm-up
        walls = {"sample_clips": [], "stream": []}
        for _ in range(args.reps):
            flush.zero_()
            t, ref = timed(offline)
            walls["sample_clips"].append(t)
            flush.zero_()
            t, (outs, steps) = timed(streamed)
            walls["stream"].append(t)
        r = {a: dict(wall_s_median=median(w), wall_s_min=min(w), wall_s_max=max(w), frames_per_s=frames / median(w))
             for a, w in walls.items()}
        r["stream"]["steps_run"] = steps
        r["sample_clips"]["windows_run"] = sched.makespan
        r["outputs_bitwise_equal"] = all(torch.equal(a, b) for a, b in zip(outs, ref))
        cb[mode] = r
    res["continuous_batching"] = cb
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        json.dump(res, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
