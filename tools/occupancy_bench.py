"""StreamSampler steps at partial occupancy: a 256-slot sampler with k ready streams against a sampler of k slots, in one process.

  python tools/occupancy_bench.py [--out FILE] [--steps N]

For k in {1, 8, 32, 64, 128, 256}: k streams with every next window ready (bf16, nfe 10, euler, a_cfg 2 = 3-way CFG, static emotion)
step on StreamSampler(slots=256), which replays the window graph of occupancy_slots(256, k) slots, alternating step by step with the
same streams (same inputs and seeds) on StreamSampler(slots=k).  The two samplers run on two backends (two model objects with the
same weights), so neither re-captures when the other steps.  Each step is timed with a host clock from a device synchronise to a
device synchronise; reported are the medians over --steps steps after 2 warm-up steps, and the first step of the 256-slot sampler
at each k, which captures that bucket's graph (minus the median: the capture cost).  The card (name, power limit, max SM clock) is
read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from __graft_entry__ import load_package  # noqa: E402

NFE, A_CFG, SLOTS = 10, 2.0, 256
READY = (1, 8, 32, 64, 128, 256)


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
    ap.add_argument("--steps", type=int, default=25, help="timed steps per ready count (median)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("occupancy_bench: needs a CUDA device (B200); there is nothing to measure without one")
    pkg = load_package()
    dev = torch.device("cuda:0")
    fd = pkg.synth.FmtDims()
    sd = pkg.synth.synth_state_dict(fd, seed=0)
    opt = pkg.BaseOptions()
    big_model, own_model = pkg.FmtModel(sd, opt, target_device=dev), pkg.FmtModel(sd, opt, target_device=dev)
    L = pkg.Dims.from_options(opt, sd).frames_per_clip
    kw = dict(nfe=NFE, method="euler", mode="bf16", a_cfg_scale=A_CFG, device=dev)
    res = dict(card=card(), note=__doc__.strip().splitlines()[0], nfe=NFE, n_branches=3, plan_slots=SLOTS, steps_timed=args.steps,
               timing="host clock, device synchronise to device synchronise, median of the timed steps")
    t0, big = timed(lambda: pkg.StreamSampler(big_model, slots=SLOTS, **kw))
    res["construct_256_slots_ms"] = t0 * 1e3
    n_win = args.steps + 2
    by_k = {}
    for k in READY:
        r_s, wa, we = [t.to(dev) for t in pkg.synth.synth_inputs(fd, k, n_win * L, seed=11)]
        t_own, own = timed(lambda: pkg.StreamSampler(own_model, slots=k, **kw))
        arms = {}
        for name, sm in (("bucket", big), ("own", own)):
            streams = [sm.open(r_s[i:i + 1], we[i:i + 1], seed=i) for i in range(k)]
            for i, s in enumerate(streams):
                sm.feed(s, wa[i:i + 1])
            arms[name] = (sm, streams, [])
        first = None
        for j in range(n_win):
            for name, (sm, streams, ts) in arms.items():
                t, ran = timed(sm.step)
                assert len(ran) == k
                if name == "bucket" and j == 0:
                    first = t
                if j >= 2:
                    ts.append(t)
        mb, mo = median(arms["bucket"][2]), median(arms["own"][2])
        by_k[str(k)] = dict(bucket_slots=pkg.occupancy_slots(SLOTS, k), last_window_slots=big._be.last_window_slots(),
                            step_ms_median=mb * 1e3, step_ms_min=min(arms["bucket"][2]) * 1e3, step_ms_max=max(arms["bucket"][2]) * 1e3,
                            own_sampler_step_ms_median=mo * 1e3, own_sampler_step_ms_min=min(arms["own"][2]) * 1e3,
                            own_sampler_step_ms_max=max(arms["own"][2]) * 1e3, ratio_to_own_sampler=mb / mo,
                            own_sampler_window_kernel_status=own._be.window_kernel_status(),
                            first_step_ms=first * 1e3, first_use_capture_ms=(first - mb) * 1e3, own_sampler_construct_ms=t_own * 1e3)
        print(k, json.dumps(by_k[str(k)]), flush=True)
        for sm, streams, _ in arms.values():
            for s in streams:
                sm.close(s)
        del own, arms, r_s, wa, we
        torch.cuda.empty_cache()
    res["by_ready_streams"] = by_k
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        json.dump(res, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
