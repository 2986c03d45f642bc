"""bench.py contract checks: the reference arm (the oracle port on the host cores) prints ONE JSON line with the result's keys
and dumps the latents of its last timed step; the algorithmic-work formulas match SURVEY.md §8d.  The product arm's dump is
checked on the GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_reference_arm_prints_the_contract_line(tmp_path):
    d = run_bench("--impl", "reference", "--steps", "1", "--warmup", "1", "--frames", "50", "--dump-outputs", str(tmp_path))
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["higher_is_better"] is True and d["scaling"] == "weak"
    assert d["metric"].startswith("motion-latent frames/s") and d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]
    # --dump-outputs: the latents of the timed call, recomputed here from the same seeded weights, inputs and noise
    from oracle import fmt_oracle as O
    from oracle.synth import FmtDims, synth_inputs, synth_state_dict
    dims = FmtDims()
    r_d = np.load(tmp_path / "r_d.npy")
    assert r_d.dtype == np.float32 and r_d.shape == (1, 50, dims.dim_w)
    r_s, wa, we = synth_inputs(dims, 1, 50, seed=7)
    noise = torch.randn(1, 1, dims.frames_per_clip, dims.dim_w, generator=torch.Generator().manual_seed(15))
    with torch.no_grad():
        ref = O.sample_loop(synth_state_dict(dims, seed=0), dims, r_s, wa, we, 50, nfe=10, a_cfg_scale=2.0, e_cfg_scale=1.0, noise=noise)
    assert float((torch.from_numpy(r_d) - ref).abs().max()) <= 2e-4


def test_steps_must_be_positive():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode != 0 and "--steps" in res.stderr


@pytest.mark.gpu
def test_product_arm_dumps_the_latents_of_its_last_timed_step(tmp_path, monkeypatch):
    """--steps K times K sampler calls (K times the launches of one), and the product arm's r_d.npy is the output of its timed
    path for the bench's seeded inputs and noise: the same for any K, and equal to the oracle on the same device within the bf16
    tolerance of the parity tests."""
    common = ("--warmup", "1", "--frames", "60", "--large-clips", "0", "--no-cpu-baseline", "--dump-outputs")
    one = run_bench("--steps", "1", *common, str(tmp_path / "k1"))
    three = run_bench("--steps", "3", *common, str(tmp_path / "k3"))
    assert one["steps"] == 1 and three["steps"] == 3 and one["value"] > 0 and three["value"] > 0
    assert one["gpu_launches"] > 0 and three["gpu_launches"] == 3 * one["gpu_launches"]
    from __graft_entry__ import load_package
    from oracle import fmt_oracle as O
    pkg = load_package()
    dims, dev = pkg.synth.FmtDims(), torch.device("cuda:0")
    r_d = np.load(tmp_path / "k3" / "r_d.npy")
    assert r_d.dtype == np.float32 and r_d.shape == (1, 60, dims.dim_w)
    assert np.array_equal(r_d, np.load(tmp_path / "k1" / "r_d.npy"))
    r_s, wa, we = pkg.synth.synth_inputs(dims, 1, 60, seed=7)
    noise = pkg.draw_window_noise(1, pkg.Dims(), 2, dev, torch.Generator(dev).manual_seed(15))
    W = {k: v.to(dev) for k, v in pkg.synth.synth_state_dict(dims, seed=0).items()}
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    with torch.no_grad():
        ref = O.sample_loop(W, dims, r_s.to(dev), wa.to(dev), we.to(dev), 60, nfe=10, a_cfg_scale=2.0, e_cfg_scale=1.0, noise=noise).cpu()
    assert float((torch.from_numpy(r_d) - ref).abs().max()) <= 2e-2


def test_algorithmic_work_matches_the_survey():
    sys.path.insert(0, ROOT)
    import bench
    from oracle.synth import FmtDims
    w = bench.algorithmic_work(FmtDims(), 1, 3, 9)
    # SURVEY.md §8d: 203.4 MB of step weights + 18.43 MB of AdaLN table rows per clip and step; 155 196 416 MACs per token row
    assert abs(w["step_bytes"] - (203.4e6 + 18.43e6)) / 221.8e6 < 2e-3
    assert w["rows"] == 180
    macs_row = (w["window_flops"] / 9 / 180 - 4 * 60 * 1024) / 2
    assert macs_row == 155_196_416
