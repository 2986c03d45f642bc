#!/usr/bin/env python
"""Benchmark of the FMT motion-latent sampling path (BASELINE.json metric: motion-latent frames/s, FMT, nfe=10).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--frames T] [--dump-outputs DIR]

One "step" = one sampler call (= ``_perform_ode_sampling_loop``) over one batch of synthetic clips:
``ceil(T/50)`` windows x ``nfe-1`` Euler steps x 3-way CFG.  Default workload = BASELINE.json configs[1]:
1 clip, 4 s -> 100 frames, nfe=10, a_cfg=2, e_cfg=1, bf16.  ``--batch 32 --frames 200`` gives the tensor-pipe
regime of configs[3] (per GPU).  For N > 1 (torchrun) every rank samples its own clips (data parallel, weak
scaling) and the step ends with one NCCL all-gather of the motion latents.

Prints ONE JSON line (rank 0).  ``value`` = frames/s with inputs resident in HBM, timed with CUDA events, max over
ranks; ``e2e`` = the same through the node class with CPU tensors in / CPU tensor out (H2D, noise draw, D2H inside
the timed region); ``roofline`` = algorithmic bytes (or FLOPs) of one window launch / its measured duration against
MEASURED_PEAKS.json; ``cpu_baseline`` = the UNMODIFIED reference node (oracle/_ref copy, torch fp32 eager) on the host cores
(the oracle port only when no copy of the reference exists); ``large_batch`` = configs[3] on the same GPUs: 256 clips x 200
frames in total, 256/N clips per GPU (strong scaling of a fixed job, tensor-pipe regime) with its own roofline / e2e / clocks.

The product arm imports nothing from ``oracle/``: the seeded synthetic weights and inputs come from the package's ``synth``
module; ``oracle/`` is executed by the baseline legs alone (``cpu_baseline``, ``gpu_eager_baseline``, ``--impl reference``).

``--dump-outputs DIR`` writes the motion latents the timed path returned in its last timed step to ``DIR/r_d.npy`` (float32,
(clips, frames, dim_w); with N GPUs the gathered latents of all ranks; ``--impl reference``: the first window's frames).  Weights,
inputs and noise are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NFE, A_CFG, E_CFG, R_CFG = 10, 2.0, 1.0, 1.0
DUMP_BYTES = 60_000_000          # --dump-outputs stays below 64 MB including the .npy header


def dump_outputs(out_dir, r_d):
    """Writes ``r_d`` as ``out_dir/r_d.npy`` (float32).  Latents larger than DUMP_BYTES are cut to a fixed sample of their
    frame rows (seed 0, kept in row order), shape (rows, dim_w), so that runs with the same arguments stay comparable."""
    import numpy as np
    r_d = r_d.detach().float().cpu()
    rows = r_d.reshape(-1, r_d.shape[-1])
    keep = DUMP_BYTES // (4 * rows.shape[1])
    if rows.shape[0] > keep:
        r_d = rows[torch.randperm(rows.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "r_d.npy"), r_d.contiguous().numpy())


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"], bf16_tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


def measured_traffic(key):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` captures (profiles/r02_traffic.json,
    else round 1's)."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            rec = json.load(open(p)).get(key)
            if rec:
                return rec
    return {}


def algorithmic_work(dims, B, nb, S):
    """Per-window algorithmic bytes / FLOPs (DESIGN.md §4, SURVEY.md §8d), bf16 weights, AdaLN tables hoisted."""
    H, W, M, D, N = dims.dim_h, dims.dim_w, dims.mlp_hidden, dims.fmt_depth, dims.total_frames
    Kc = dims.dim_w + dims.dim_a + dims.dim_e
    NT = D * 6 * H + 2 * H
    step_params = D * (3 * H * H + H * H + 2 * H * M) + H * W + W * H          # qkv, proj, fc1, fc2, x_embedder, decoder.linear
    rows = nb * B * N
    table_bytes = rows * NT * 2                                                 # bf16 shift/scale/gate rows of one evaluation
    step_bytes = 2 * step_params + table_bytes
    prep_bytes = 2 * (NT * H + H * Kc) + S * table_bytes                        # adaLN + c_embedder weights once, table written once
    macs_row = step_params + NT * H + H * Kc                                    # every Linear, per token row (hoisting moves, not removes)
    attn_flops_row = 4 * N * H                                                  # dense-equivalent QK^T + PV, as the reference computes
    flops_step = rows * (2 * macs_row + attn_flops_row)
    # What the product executes: the AdaLN projections run once per DISTINCT condition row (the unconditional branch's current frames
    # share one row per clip and its context rows equal the audio-only branch's: 2N + 1 of 3N rows with 3-way CFG), everything else per
    # token row.  Reported beside the algorithmic (reference-equivalent) count, which is what the roofline fraction is defined on.
    distinct = B * (2 * N + 1) if nb == 3 and os.environ.get("FMT_DEDUP", "1") != "0" else rows
    flops_step_exec = rows * (2 * step_params + attn_flops_row) + distinct * 2 * (NT * H + H * Kc)
    return dict(step_bytes=step_bytes, window_bytes=S * step_bytes + prep_bytes, window_flops=S * flops_step, rows=rows,
                window_flops_executed=S * flops_step_exec, distinct_condition_rows=distinct)


class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(gpu_index)],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, reasons = [], set()
        for r in rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1]))
                out["sm_max_mhz"] = float(r[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.strip().lower() == "active":
                    reasons.add(name)
        if sm:
            sm.sort()
            out["sm_mhz"] = sm[len(sm) // 2]
        out["reasons"], out["samples"] = sorted(reasons), len(sm)
        return out


def synth_module():
    """The package's seeded synthetic weights / inputs (SURVEY.md §8d) - no algorithm of the path, nothing from oracle/."""
    from __graft_entry__ import load_package
    load_package()
    return sys.modules["float_fmt_b200.synth"]


def workload_inputs(dims, B, T, rank):
    return synth_module().synth_inputs(dims, B, T, seed=7 + 1000 * rank)


def cpu_reference_clip(W, dims, r_s, wa, we, T, noise):
    """The reference algorithm with injected noise: oracle/fmt_oracle.py (used by the eager-GPU comparator only)."""
    from oracle import fmt_oracle as O
    with torch.no_grad():
        return O.sample_loop(W, dims, r_s, wa, we, T, nfe=NFE, a_cfg_scale=A_CFG, r_cfg_scale=R_CFG, e_cfg_scale=E_CFG, noise=noise)


def time_cpu_baseline(W, dims, B, T, budget_s, reps=3):
    """The reference node itself (oracle/_ref, unmodified; port only if absent) on the host cores, on a bounded sample."""
    from oracle import ref_arm
    kind, run = ref_arm.make_cpu_sampler(W, dims, NFE, A_CFG, R_CFG, E_CFG)
    r_s, wa, we = workload_inputs(dims, B, T, 0)
    L = dims.frames_per_clip
    n_win = math.ceil(T / L)
    # bounded sample: the whole clip if one pass fits the budget, else its first window
    t0 = time.perf_counter()
    run(r_s, wa[:, :L], we[:, :L] if we.shape[1] > 1 else we, L, 15)
    t_win = time.perf_counter() - t0
    frames, sample = (T, f"whole workload: {B} clip(s) x {T} frames, {n_win} windows x {NFE - 1} steps, 3-way CFG") \
        if t_win * n_win * (reps + 0.5) <= budget_s else (L, f"first window only: {B} clip(s) x {L} frames, {NFE - 1} steps, 3-way CFG")
    best = float("inf")
    for _ in range(reps):
        t0 = time.perf_counter()
        run(r_s, wa[:, :frames], we[:, :frames] if we.shape[1] > 1 else we, frames, 15)
        best = min(best, time.perf_counter() - t0)
        if best * reps > budget_s:
            break
    return dict(value=B * frames / best, unit="frames/s", cores=torch.get_num_threads(), kind=kind, sample=sample + "; " + ref_arm.describe(kind),
                ms_per_ode_step=1e3 * best / (math.ceil(frames / L) * (NFE - 1)))


def time_gpu_eager_baseline(W, dims, B, T, dev, reps=3):
    """The same oracle port run eagerly on the B200 in fp32 (TF32 off): what the reference's PyTorch code does when its
    target device is the GPU (BASELINE.md §3).  Reported beside the CPU baseline; never a gate."""
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    Wd = {k: v.to(dev) for k, v in W.items()}
    r_s, wa, we = [t.to(dev) for t in workload_inputs(dims, B, T, 0)]
    L = dims.frames_per_clip
    n_win = math.ceil(T / L)
    g = torch.Generator(dev).manual_seed(15)
    noise = torch.stack([torch.randn(B, L, dims.dim_w, generator=g, device=dev) for _ in range(n_win)])
    best = float("inf")
    for i in range(reps + 1):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        cpu_reference_clip(Wd, dims, r_s, wa, we, T, noise)
        torch.cuda.synchronize()
        if i > 0:
            best = min(best, time.perf_counter() - t0)
    return dict(value=B * T / best, unit="frames/s", kind="port", device="cuda:0, torch eager fp32 (TF32 off)",
                ms_per_ode_step=1e3 * best / (n_win * (NFE - 1)))


def measure_handoff(pkg, model, dims, B, T, dev, iters=10):
    """SURVEY.md 8f rank 2: FloatApplyAudioProjection -> sampler node, end to end from CPU wav2vec features to CPU motion latents,
    with the reference's CPU hand-off between the two nodes (nodes_vadv.py:197,692-694) and with the device-resident one
    (keep_on_device).  Wall clock, synchronised; bf16 mode."""
    synth = pkg.synth
    layer = pkg.AudioProjectionLayer(9216, dims.dim_w, target_device=dev)
    g = torch.Generator().manual_seed(62)
    with torch.no_grad():
        for prm in layer.parameters():
            prm.copy_(torch.randn(prm.shape, generator=g) * (0.01 if prm.ndim == 2 else 0.1) + (1.0 if prm.ndim == 1 and prm is layer[1].weight else 0.0))
    feats = synth.synth_wav2vec_features(B, T, 9216, seed=5).pin_memory()
    r_s, _, we = workload_inputs(dims, B, T, 0)
    r_s, we = r_s.pin_memory(), we.pin_memory()
    proj, samp = pkg.FloatApplyAudioProjection(), pkg.FloatSampleMotionSequenceRD_VA()
    args = (A_CFG, R_CFG, E_CFG, False, NFE, "euler", 1e-5, 1e-5, 0.1, 0.1, 0.1, True, 15)
    out = {}
    for keep in (False, True):
        def run():
            (wa,) = proj.apply_projection(feats, layer, keep_on_device=keep)
            r_d, _ = samp.sample_rd_sequence_va(r_s, wa, we, T, model, *args)
            return r_d
        for _ in range(3):
            run()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(iters):
            run()
        torch.cuda.synchronize()
        out["device_resident_ms" if keep else "cpu_handoff_ms"] = 1e3 * (time.perf_counter() - t0) / iters
    out.update(workload=f"{B} clip(s) x {T} frames: CPU wav2vec features (B, T, 9216) -> FloatApplyAudioProjection -> "
                        "FloatSampleMotionSequenceRD_VA -> CPU latents", handoff_bytes=B * T * dims.dim_w * 4,
               value=B * T / (out["device_resident_ms"] * 1e-3), unit="frames/s")
    return out


def measure_product(pkg, be, model, dims, B, T, rank, world, dev, dist, steps, warmup, e2e_iters, keep_output=False):
    """Times the product path on this rank's B clips x T frames: resident (CUDA events) and end to end (node, CPU tensors).
    With ``keep_output`` the result's ``output`` holds the latents of the last timed resident step (gathered over ranks), on the CPU."""
    L = dims.frames_per_clip
    n_win = math.ceil(T / L)
    be.configure(B, 3, False, NFE, "euler", "bf16")
    r_s, wa, we = workload_inputs(dims, B, T, rank)
    r_s_d, wa_d, we_d = r_s.to(dev), wa.to(dev), we.to(dev)
    g = torch.Generator(dev).manual_seed(15 + rank)
    noise_d = pkg.draw_window_noise(B, be.dims, n_win, dev, g)
    out_d = torch.empty(B, T, dims.dim_w, device=dev)
    gathered = torch.empty(world * B, T, dims.dim_w, device=dev) if world > 1 else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def step_resident():
        be.sample_clip(r_s_d, wa_d, we_d, T, noise_d, A_CFG, R_CFG, E_CFG, out=out_d)
        if world > 1:
            dist.all_gather_into_tensor(gathered, out_d)        # the only collective of the path: final gather of r_d

    node = pkg.FloatSampleMotionSequenceRD_VA()
    r_s_p, wa_p, we_p = r_s.pin_memory(), wa.pin_memory(), we.pin_memory()

    def step_e2e():
        out, _ = node.sample_rd_sequence_va(r_s_p, wa_p, we_p, T, model, A_CFG, R_CFG, E_CFG, False, NFE, "euler", 1e-5, 1e-5,
                                            0.1, 0.1, 0.1, True, 15 + rank)
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n, wall=False):
        """n iterations; device time from CUDA event pairs around each iteration (L2 flushed outside the pairs)."""
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        barrier()
        t_wall = 0.0
        for e0, e1 in evs:
            flush.zero_()
            if wall:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
            e0.record()
            fn()
            e1.record()
            if wall:
                torch.cuda.synchronize()
                t_wall += time.perf_counter() - t0
        barrier()
        t_dev = sum(e0.elapsed_time(e1) for e0, e1 in evs) * 1e-3
        t = torch.tensor([t_wall if wall else t_dev], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    clocks = ClockSampler(dev.index) if rank == 0 else None
    for _ in range(warmup):
        step_resident()
    be.launch_count(reset=True)
    t_res = timed(step_resident, steps)
    launches = be.launch_count(reset=True)
    output = (gathered if world > 1 else out_d).cpu() if keep_output else None
    for _ in range(min(3, warmup)):
        step_e2e()
    t_e2e = timed(step_e2e, e2e_iters, wall=True)        # host-visible latency: the call returns a CPU tensor
    clk = clocks.stop() if clocks else None
    h2d = (r_s.numel() + wa.numel() + we.numel()) * 4
    d2h = B * T * dims.dim_w * 4
    del flush, gathered, out_d, noise_d
    return dict(t_step=t_res / steps, t_e2e=t_e2e / e2e_iters, launches=int(launches), clocks=clk, h2d=h2d, d2h=d2h, n_win=n_win,
                window_kernel=be.window_kernel_status(), output=output)


def roofline_record(dims, B, T, t_step, n_win, pk):
    S = NFE - 1
    work = algorithmic_work(dims, B, 3, S)
    t_window = t_step / n_win
    hbm_achieved = work["window_bytes"] / t_window / 1e9
    tf_achieved = work["window_flops"] / t_window / 1e12
    hbm_frac, tf_frac = hbm_achieved / pk["hbm_gbs"], tf_achieved / pk["bf16_tflops_sustained"]
    # Which roofline binds is a property of the workload (SURVEY.md §8d): <= 2 clips stream the weights (180 flop/B per clip
    # against a ridge of ~210), >= 8 clips are dense-contraction bound.
    # <= 256 token rows run the persistent window kernel: the dataflow kernel (csrc/flow.cuh) unless FMT_WINDOW selects round 1's
    small = "b1_flow" if os.environ.get("FMT_WINDOW", "3") == "3" else "b1_window"
    prof = measured_traffic(small if work["rows"] <= 256 else "b32")
    if work["rows"] <= 512:
        roof = dict(bound="hbm", achieved=hbm_achieved, peak=pk["hbm_gbs"], unit="GB/s", frac=hbm_frac, traffic=prof.get("dram_bytes_per_launch"))
    else:
        roof = dict(bound="tensor", achieved=tf_achieved, peak=pk["bf16_tflops_sustained"], unit="TFLOP/s", frac=tf_frac, traffic=prof.get("dram_bytes_per_launch"))
    roof.update(peak_source=pk["source"], launch="one captured window graph = prepare + %d ODE steps" % S, dominant_kernel=prof.get("kernel"),
                traffic_source=prof.get("source"),
                us_per_ode_step=1e6 * t_window / S, algorithmic_bytes_per_window=work["window_bytes"],
                algorithmic_flops_per_window=work["window_flops"], other_bound_frac=min(hbm_frac, tf_frac),
                executed_flops_per_window=work["window_flops_executed"], distinct_condition_rows=work["distinct_condition_rows"],
                token_rows=work["rows"], executed_tflops=work["window_flops_executed"] / t_window / 1e12)
    return roof


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=1, help="clips per GPU")
    ap.add_argument("--frames", type=int, default=100, help="frames per clip (25 fps)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--large-clips", type=int, default=256, help="total clips of the large_batch record (configs[3]); 0 = skip it")
    ap.add_argument("--large-frames", type=int, default=200)
    ap.add_argument("--force-port", action="store_true", help="reference arm: time the oracle port even when the reference copy exists")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the latents of the last timed step to DIR/r_d.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    synth = synth_module()
    dims = synth.FmtDims()
    B, T = args.batch, args.frames
    L = dims.frames_per_clip
    n_win = math.ceil(T / L)
    S = NFE - 1
    workload = (f"configs[1]: {B} clip x {T} frames (4 s @25 fps), nfe={NFE}, a_cfg={A_CFG}, e_cfg={E_CFG}, 3-way CFG, euler, bf16"
                if (B, T) == (1, 100) else f"{B} clips/GPU x {T} frames, nfe={NFE}, a_cfg={A_CFG}, e_cfg={E_CFG}, 3-way CFG, euler, bf16")
    config = dict(workload=workload, clips_per_gpu=B, frames_per_clip=T, windows=n_win, ode_steps_per_window=S, cfg_branches=3,
                  parallelism=f"dp{world}", l2="256 MiB memset between timed iterations (L2 flush)")

    # ------------------------------------------------------------------ reference arm: the reference node on the host cores, rank 0 only
    if args.impl == "reference":
        if rank != 0:
            return
        from oracle import ref_arm
        W = synth.synth_state_dict(dims, seed=0)
        kind, run = ref_arm.make_cpu_sampler(W, dims, NFE, A_CFG, R_CFG, E_CFG, force_port=args.force_port)
        r_s, wa, we = workload_inputs(dims, B, T, 0)
        t0 = time.perf_counter()
        run(r_s, wa[:, :L], we, L, 15)
        t_win = time.perf_counter() - t0
        total = args.steps + args.warmup
        frames = T if t_win * n_win * total <= 150 else L
        sample = (f"whole workload per step ({B} clip x {T} frames)" if frames == T else
                  f"first window per step ({B} clip x {L} frames, {S} ODE steps)") + "; " + ref_arm.describe(kind)
        for _ in range(max(0, args.warmup - 1)):
            run(r_s, wa[:, :frames], we, frames, 15)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            r_d = run(r_s, wa[:, :frames], we, frames, 15)
        el = time.perf_counter() - t0
        if args.dump_outputs:
            # whether a step covers the whole clip or its first window depends on this host's speed: dump the first window,
            # which both compute alike, so that the file's shape follows from the arguments
            dump_outputs(args.dump_outputs, r_d[:, :L])
        v = args.steps * B * frames / el
        print(json.dumps(dict(impl="reference", metric="motion-latent frames/s (FMT, nfe=10)", value=v, unit="frames/s", n_gpus=args.gpus,
                              steps=args.steps, warmup=args.warmup, ms_per_step=1e3 * el / args.steps, higher_is_better=True, scaling="weak",
                              vs_baseline=None, dtype="f32", data="synthetic", config=config, cpu_processes=1,
                              note="ONE CPU process (rank 0, all host cores) on one GPU's share of the workload, whatever --gpus says: "
                                   "compare it with the product arm's per-GPU value, not with its N-GPU aggregate",
                              cpu_baseline=dict(value=v, unit="frames/s", cores=torch.get_num_threads(), kind=kind, sample=sample),
                              e2e=dict(value=v, unit="frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))))
        return

    # ------------------------------------------------------------------ our arm
    from __graft_entry__ import load_package
    pkg = load_package()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    W = synth.synth_state_dict(dims, seed=0)
    model = pkg.FmtModel(W, target_device=dev)
    be = pkg.backend_for(model, dev)
    pk = peaks()

    m = measure_product(pkg, be, model, dims, B, T, rank, world, dev, dist, args.steps, max(3, args.warmup), max(10, args.steps // 4),
                        keep_output=bool(args.dump_outputs) and rank == 0)
    graph_nodes = be.graph_kernel_nodes()

    # ---- configs[3]: a fixed job of 256 clips x 200 frames split over the GPUs (strong scaling; tensor-pipe regime)
    large = None
    if args.large_clips > 0:
        Bl, Tl = -(-args.large_clips // world), args.large_frames
        try:
            ml = measure_product(pkg, be, model, dims, Bl, Tl, rank, world, dev, dist, 3, 3, 3)
            roof_l = roofline_record(dims, Bl, Tl, ml["t_step"], ml["n_win"], pk)
            large = dict(workload=f"configs[3]: {world * Bl} clips x {Tl} frames in total, {Bl} clips per GPU, nfe={NFE}, 3-way CFG, euler, bf16",
                         clips_total=world * Bl, clips_per_gpu=Bl, frames_per_clip=Tl, scaling="strong (fixed 256-clip job)",
                         value=world * Bl * Tl / ml["t_step"], unit="frames/s", ms_per_step=1e3 * ml["t_step"], steps=3, warmup=3,
                         us_per_ode_step=roof_l["us_per_ode_step"], roofline=roof_l, gpu_launches=ml["launches"], clocks=ml["clocks"],
                         e2e=dict(value=world * Bl * Tl / ml["t_e2e"], unit="frames/s", h2d_bytes_per_step=ml["h2d"], d2h_bytes_per_step=ml["d2h"],
                                  ms_per_step=1e3 * ml["t_e2e"]))
        except Exception as e:          # e.g. not enough free HBM for the 256-clip tables next to another tenant
            large = dict(error=f"{type(e).__name__}: {e}"[:300])

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    t_step = m["t_step"]
    frames_total = world * B * T
    roof = roofline_record(dims, B, T, t_step, n_win, pk)
    res = dict(metric="motion-latent frames/s (FMT, nfe=10)", value=frames_total / t_step, unit="frames/s", n_gpus=world, steps=args.steps,
               warmup=max(3, args.warmup), ms_per_step=1e3 * t_step, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="bf16",
               data="synthetic", config=config, us_per_ode_step=roof["us_per_ode_step"],
               e2e=dict(value=frames_total / m["t_e2e"], unit="frames/s", h2d_bytes_per_step=m["h2d"], d2h_bytes_per_step=m["d2h"],
                        ms_per_step=1e3 * m["t_e2e"], api="FloatSampleMotionSequenceRD_VA.sample_rd_sequence_va (CPU tensors in/out)"),
               gpu_launches=m["launches"], graph_kernel_nodes=graph_nodes, window_kernel_status=m["window_kernel"], roofline=roof, clocks=m["clocks"])
    if large is not None:
        res["large_batch"] = large
    if world == 1 and B <= 32:
        try:
            res["handoff"] = measure_handoff(pkg, model, dims, B, T, dev)
        except Exception as e:
            res["handoff"] = dict(error=f"{type(e).__name__}: {e}"[:300])
    if not args.no_cpu_baseline and world == 1:
        res["cpu_baseline"] = time_cpu_baseline(W, dims, B, T, budget_s=25.0)
        if B <= 32:
            res["gpu_eager_baseline"] = time_gpu_eager_baseline(W, dims, B, T, dev)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, m["output"])
    print(json.dumps(res))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
