"""Per-step time of the three precision modes (bf16, bf16x3, fp32) and the isolated GEMMs of bf16 against bf16x3, in one run.

  python tools/precision_bench.py [--out FILE]

Step times: device events around fmt_sample_clip (all windows of the workload, 256 MiB memset between timed calls as in bench.py),
divided by windows x ODE steps; one backend per arm, arms alternated rep by rep so that drift on a shared card hits them alike.
Workloads: configs[1] (1 clip x 100 frames) and 32 clips x 200 frames, nfe 10, a_cfg 2, 3-way CFG, euler, synthetic weights and
inputs of bench.py.  At configs[1] bf16 runs twice: on the dataflow window kernel (its default) and one kernel per op
(FMT_WINDOW=0), which is the path bf16x3 and fp32 take there.
GEMMs: qkv / proj / fc1 / fc2 at 32 clips (M = 5760) through fmt_debug_gemm_bench (bf16 operands, bf16 output) and
fmt_debug_gemm_bench_bf16x3 (pair operands, fp32 output), back to back with L2-warm operands; block_n 0 is the kernel the sampler
picks, the others are the explicit variants.
"""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from __graft_entry__ import load_package  # noqa: E402

NFE, A_CFG = 10, 2.0


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def step_times(pkg, dims, sd, dev, B, T, arms, reps, iters):
    L = dims.frames_per_clip
    n_win = math.ceil(T / L)
    r_s, wa, we = [t.to(dev) for t in pkg.synth.synth_inputs(pkg.synth.FmtDims(), B, T, seed=7)]
    noise = pkg.draw_window_noise(B, dims, n_win, dev, torch.Generator(dev).manual_seed(15))
    out = torch.empty(B, T, dims.dim_w, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    bes = {}
    for name, mode, window in arms:
        os.environ["FMT_WINDOW"] = window                          # read when the handle is created
        be = pkg.FmtBackend(sd, dims, dev)
        be.configure(B, 3, False, NFE, "euler", mode)
        for _ in range(2):
            be.sample_clip(r_s, wa, we, T, noise, A_CFG, 1.0, 1.0, out=out)
        bes[name] = be
    os.environ.pop("FMT_WINDOW", None)
    times = {name: [] for name in bes}
    for _ in range(reps):
        for name, be in bes.items():
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
            torch.cuda.synchronize()
            for e0, e1 in evs:
                flush.zero_()
                e0.record()
                be.sample_clip(r_s, wa, we, T, noise, A_CFG, 1.0, 1.0, out=out)
                e1.record()
            torch.cuda.synchronize()
            times[name].append(1e3 * sum(e0.elapsed_time(e1) for e0, e1 in evs) / iters / (n_win * (NFE - 1)))
    res = {}
    for name, be in bes.items():
        t = sorted(times[name])
        res[name] = dict(us_per_ode_step_median=t[len(t) // 2], us_per_ode_step_min=t[0], us_per_ode_step_max=t[-1],
                         window_kernel=be.window_kernel_status())
        be.close()
    return res


def pair(x):
    """fp32 (rows, K) -> bf16 bits (rows, 2K) in the pair layout: [hi 0:64 | lo 0:64 | hi 64:128 | lo 64:128 | ...]."""
    hi = x.to(torch.bfloat16)
    lo = (x - hi.float()).to(torch.bfloat16)
    r, k = x.shape
    return torch.stack([hi.view(r, k // 64, 64), lo.view(r, k // 64, 64)], dim=2).reshape(r, 2 * k).contiguous()


def gemm_times(L, dev, M, iters=50):
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    shapes = [("qkv", 3072, 1024), ("proj", 1024, 1024), ("fc1", 4096, 1024), ("fc2", 1024, 4096)]
    res = {}

    def timed(fn):
        fn(3)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        fn(iters)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / iters

    for name, N, K in shapes:
        g = torch.Generator(device=dev).manual_seed(N + K)
        A = torch.randn(M, K, device=dev, generator=g)
        W = torch.randn(N, K, device=dev, generator=g) * 0.05
        bias = torch.zeros(N, device=dev)
        out = torch.empty(M, N, device=dev)
        A16, W16, A3, W3 = A.to(torch.bfloat16), W.to(torch.bfloat16), pair(A), pair(W)
        r = dict(M=M, N=N, K=K)
        for bn in (0, 128, 512):
            r[f"bf16_us_bn{bn}"] = timed(lambda n: L.fmt_debug_gemm_bench(A16.data_ptr(), W16.data_ptr(), bias.data_ptr(), out.data_ptr(), M, N, K, bn, n, st))
        for bn in (0, 64, 128, 512, 1024):
            r[f"bf16x3_us_bn{bn}"] = timed(lambda n: L.fmt_debug_gemm_bench_bf16x3(A3.data_ptr(), W3.data_ptr(), bias.data_ptr(), out.data_ptr(), M, N, K,
                                                                                  bn, n, st))
        r["ratio_bf16x3_over_bf16"] = r["bf16x3_us_bn0"] / r["bf16_us_bn0"]
        r["bf16x3_tflops"] = 2 * 3 * M * N * K / r["bf16x3_us_bn0"] / 1e6
        res[name] = r
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON result here")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    pkg = load_package()
    cabi = sys.modules[pkg.__name__ + "._cabi"]
    L = cabi.load_library()
    dev = torch.device("cuda:0")
    sd = pkg.synth.synth_state_dict(pkg.synth.FmtDims(), seed=0)
    dims = pkg.Dims.from_options(pkg.BaseOptions(), sd)
    res = dict(card=card(), note=__doc__.strip().splitlines()[0])
    res["configs1_1clip_100frames"] = step_times(pkg, dims, sd, dev, 1, 100, [("bf16", "bf16", "3"), ("bf16_per_op", "bf16", "0"), ("bf16x3", "bf16x3", "3"),
                                                                            ("fp32", "fp32", "3")], args.reps, 20)
    res["b32_32clips_200frames"] = step_times(pkg, dims, sd, dev, 32, 200, [("bf16", "bf16", "3"), ("bf16x3", "bf16x3", "3"), ("fp32", "fp32", "3")],
                                              args.reps, 2)
    for k in ("configs1_1clip_100frames", "b32_32clips_200frames"):
        r = res[k]
        r["ratio_bf16x3_over_bf16"] = r["bf16x3"]["us_per_ode_step_median"] / r["bf16"]["us_per_ode_step_median"]
        r["ratio_fp32_over_bf16x3"] = r["fp32"]["us_per_ode_step_median"] / r["bf16x3"]["us_per_ode_step_median"]
    res["gemms_32clips"] = gemm_times(L, dev, 32 * 3 * 60)
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        json.dump(res, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
