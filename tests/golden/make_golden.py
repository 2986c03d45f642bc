"""Generate the committed golden fixtures by running the REAL reference in this container.

    python tests/golden/make_golden.py            # writes tests/golden/*.npz + manifest.json + node_surface.json

The reference (``/root/reference/src/nodes``) is imported in place through ``refshim.py`` and
fed the seeded synthetic weights / inputs from ``oracle/synth.py``; its node entry points are
called exactly as ComfyUI would call them (CPU tensors in, CPU tensors out).  The fixtures pin
``oracle/fmt_oracle.py`` (tests/test_oracle_golden.py) and, on the GPU box where /root/reference
does not exist, the CUDA path (tests/test_gpu_parity.py).

Every case stores its inputs' *recipe* (seeds, shapes, scales) in manifest.json, never the
weights (627 MB): both sides regenerate them from ``synth_state_dict(seed)``.
"""
import importlib
import json
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

from oracle.synth import FmtDims, SMALL_DIMS, synth_state_dict, synth_inputs, synth_projection, synth_wav2vec_features  # noqa: E402
import refshim  # noqa: E402

FULL = FmtDims()

# name -> recipe.  "entry": which reference entry point produced the fixture.
CASES = {
    # BASELINE.json configs[0]: 1 clip, 4 s -> 100 frames, nfe 10, a=2, e=1, seed 15
    "va_config1": dict(entry="va", dims="full", B=1, T=100, nfe=10, a=2.0, r=1.0, e=1.0, seed=15),
    "va_dynamic": dict(entry="va", dims="full", B=2, T=130, nfe=5, a=1.0, r=1.0, e=3.0, seed=16, dynamic_we=True),
    "va_rcfg": dict(entry="va", dims="full", B=1, T=60, nfe=4, a=2.0, r=1.5, e=1.5, seed=17, include_r_cfg=True),
    "va_single": dict(entry="va", dims="full", B=1, T=50, nfe=10, a=1.0, r=1.0, e=1.0, seed=18),
    "va_nfe1": dict(entry="va", dims="full", B=1, T=70, nfe=1, a=2.0, r=1.0, e=1.0, seed=19),
    "va_ragged": dict(entry="va", dims="full", B=1, T=110, T_wa=120, nfe=3, a=2.0, r=1.0, e=1.0, seed=20),
    "va_short_wa": dict(entry="va", dims="full", B=1, T=100, T_wa=90, nfe=3, a=2.0, r=1.0, e=1.0, seed=21),
    "adv_node": dict(entry="adv", dims="full", B=1, T=75, nfe=10, a=2.5, r=1.0, e=1.2, seed=1234),
    "legacy_sample": dict(entry="legacy", dims="full", B=1, T=100, nfe=10, a=2.0, r=1.0, e=1.0, seed=62064758300528,
                          onehot_we=True),
    "cfv_step3": dict(entry="cfv", dims="full", B=2, t=0.3, a=2.0, r=1.0, e=1.5, seed=30, dynamic_we=True),
    "cfv_step4": dict(entry="cfv", dims="full", B=1, t=0.7, a=2.0, r=0.5, e=1.5, seed=31, include_r_cfg=True),
    "cfv_step1": dict(entry="cfv", dims="full", B=1, t=0.0, a=1.0, r=1.0, e=1.0, seed=32),
    "va_midpoint": dict(entry="va", dims="full", B=1, T=50, nfe=4, a=2.0, r=1.0, e=1.0, seed=40, method="midpoint"),
    "va_rk4": dict(entry="va", dims="full", B=1, T=50, nfe=3, a=2.0, r=1.0, e=1.0, seed=41, method="rk4"),
    "va_heun2": dict(entry="va", dims="full", B=1, T=50, nfe=4, a=2.0, r=1.0, e=1.0, seed=42, method="heun2"),
    "va_heun3": dict(entry="va", dims="full", B=1, T=50, nfe=3, a=2.0, r=1.0, e=1.0, seed=43, method="heun3"),
    # small architecture (loader-inferred dims, nodes_vadv_loader.py:655-866): fast CPU-side host-logic tests
    "small_static": dict(entry="va", dims="small", B=3, T=31, nfe=6, a=2.0, r=1.0, e=1.0, seed=50),
    "small_dynamic": dict(entry="va", dims="small", B=2, T=40, nfe=4, a=1.5, r=1.0, e=2.0, seed=51, dynamic_we=True),
    "small_rcfg": dict(entry="va", dims="small", B=2, T=24, nfe=5, a=2.0, r=2.0, e=1.0, seed=52, include_r_cfg=True),
    # SURVEY.md §8f rank 2: FloatApplyAudioProjection (nodes_vadv.py:147-198) on 12 stacked wav2vec layers / the last layer only
    "proj_stacked": dict(entry="proj", dims="full", B=2, T=37, in_dim=9216, seed=60),
    "proj_last": dict(entry="proj", dims="full", B=1, T=100, in_dim=768, seed=61),
}


# node_surface.json: what a saved ComfyUI workflow depends on in the three sampler nodes (class name -> reference module)
NODE_SURFACE = {"FloatSampleMotionSequenceRD_VA": "nodes_vadv", "FloatSampleMotionSequenceRD": "nodes_adv", "FloatProcess": "nodes"}
SURFACE_FIELDS = ("default", "min", "max", "step", "forceInput")


def node_surface(cls) -> dict:
    """UNIQUE_NAME, FUNCTION, RETURN_TYPES and, in order, [name, type or enum, {default/min/max/step/forceInput}] of every
    INPUT_TYPES()["required"] entry, as plain JSON values."""
    req = cls.INPUT_TYPES()["required"]
    rows = [[k, v[0], {f: v[1][f] for f in SURFACE_FIELDS if len(v) > 1 and f in v[1]}] for k, v in req.items()]
    return json.loads(json.dumps(dict(UNIQUE_NAME=cls.UNIQUE_NAME, FUNCTION=cls.FUNCTION, RETURN_TYPES=list(cls.RETURN_TYPES), required=rows)))


def write_node_surface():
    refshim.load_reference()
    surface = {name: node_surface(getattr(importlib.import_module("refnodes." + mod), name)) for name, mod in NODE_SURFACE.items()}
    surface["_meta"] = dict(source="the reference's node classes, imported in place via tests/golden/refshim.py")
    json.dump(surface, open(os.path.join(HERE, "node_surface.json"), "w"), indent=1)


def dims_of(rec):
    return FULL if rec["dims"] == "full" else SMALL_DIMS


def case_inputs(rec):
    d = dims_of(rec)
    T_in = rec.get("T_wa", rec.get("T", d.frames_per_clip))
    return synth_inputs(d, rec["B"], T_in, seed=100 + rec["seed"] % 1000, dynamic_we=rec.get("dynamic_we", False),
                        onehot_we=rec.get("onehot_we", False))


def cfv_extra_inputs(rec):
    """x, prev_x, prev_wa, prev_we for the single-evaluation cases."""
    d = dims_of(rec)
    g = torch.Generator().manual_seed(rec["seed"] + 5000)
    B, L, P = rec["B"], d.frames_per_clip, d.num_prev_frames
    x = torch.randn(B, L, d.dim_w, generator=g)
    prev_x = torch.randn(B, P, d.dim_w, generator=g)
    prev_wa = torch.randn(B, P, d.dim_a, generator=g).sigmoid()
    prev_we = torch.softmax(torch.randn(B, P, d.dim_e, generator=g), dim=-1)
    return x, prev_x, prev_wa, prev_we


_models = {}


def ref_model(dims_name):
    if dims_name not in _models:
        d = FULL if dims_name == "full" else SMALL_DIMS
        sd = synth_state_dict(d, seed=0)
        overrides = {} if dims_name == "full" else d.as_dict()
        _models[dims_name] = refshim.build_reference_fmt(sd, **overrides)
    return _models[dims_name]


def projection_layer(rec):
    """The module LoadAudioProjectionLayer builds (nodes_vadv_loader.py:233-257), with the seeded weights."""
    layer = torch.nn.Sequential(torch.nn.Linear(rec["in_dim"], FULL.dim_a), torch.nn.LayerNorm(FULL.dim_a), torch.nn.SiLU())
    layer.load_state_dict(synth_projection(rec["in_dim"], FULL.dim_a, seed=rec["seed"]))
    layer.inferred_input_feature_dim = rec["in_dim"]
    layer.target_device = torch.device("cpu")
    return layer.eval()


@torch.no_grad()
def run_case(name, rec):
    if rec["entry"] == "proj":
        refshim.load_reference()
        node = importlib.import_module("refnodes.nodes_vadv").FloatApplyAudioProjection()
        x = synth_wav2vec_features(rec["B"], rec["T"], rec["in_dim"], seed=rec["seed"])
        (out,) = node.apply_projection(x, projection_layer(rec))
        return out.detach().cpu().float().numpy()
    ref, model, opt = ref_model(rec["dims"])
    d = dims_of(rec)
    r_s, wa, we = case_inputs(rec)
    entry = rec["entry"]
    if entry == "va":
        node = importlib.import_module("refnodes.nodes_vadv").FloatSampleMotionSequenceRD_VA()
        out, _ = node.sample_rd_sequence_va(
            r_s_latent=r_s, wa_latent=wa, we_latent=we, audio_num_frames=rec["T"], float_fmt_model=model,
            a_cfg_scale=rec["a"], r_cfg_scale=rec["r"], e_cfg_scale=rec["e"], include_r_cfg=rec.get("include_r_cfg", False),
            nfe=rec["nfe"], torchdiffeq_ode_method=rec.get("method", "euler"), ode_atol=1e-5, ode_rtol=1e-5,
            audio_dropout_prob=0.1, ref_dropout_prob=0.1, emotion_dropout_prob=0.1, fix_noise_seed=True, seed=rec["seed"])
    elif entry == "adv":
        node = importlib.import_module("refnodes.nodes_adv").FloatSampleMotionSequenceRD()
        pipe_opt = type(opt)()
        pipe_opt.rank = torch.device("cpu")
        pipe_opt.nfe = rec["nfe"]
        G = types.SimpleNamespace(fmt=model, num_prev_frames=d.num_prev_frames, num_frames_for_clip=d.frames_per_clip)
        pipe = types.SimpleNamespace(opt=pipe_opt, G=G)
        out, _ = node.sample_rd_sequence(r_s, wa, rec["T"], we, pipe, rec["a"], rec["e"], rec["seed"])
    elif entry == "legacy":
        FLOATmod = importlib.import_module("refnodes.models.float.FLOAT")
        lopt = type(opt)()
        lopt.rank = torch.device("cpu")
        lopt.nfe = rec["nfe"]
        emo_idx = int(we[0, 0].argmax())
        fake_self = types.SimpleNamespace(
            opt=lopt, fmt=model, num_frames_for_clip=d.frames_per_clip, num_prev_frames=d.num_prev_frames,
            audio_encoder=types.SimpleNamespace(inference=lambda a, seq_len: wa),
            emotion_encoder=types.SimpleNamespace(label2id={"x": emo_idx}, predict_emotion=None),
            odeint_kwargs={"atol": 1e-5, "rtol": 1e-5, "method": "euler"}, first_run=False, pbar=None)
        # a: (B, samples) with ceil(samples*fps/sr) == T
        a = torch.zeros(rec["B"], int(rec["T"] * lopt.sampling_rate / lopt.fps))
        out = FLOATmod.FLOAT.sample(fake_self, {"r_s": r_s, "a": a}, a_cfg_scale=rec["a"], r_cfg_scale=rec["r"],
                                    e_cfg_scale=rec["e"], emo="x", nfe=999, seed=rec["seed"])
    elif entry == "cfv":
        x, prev_x, prev_wa, prev_we = cfv_extra_inputs(rec)
        L = d.frames_per_clip
        wa_c = wa[:, :L]
        we_c = we[:, :L] if we.shape[1] > 1 else we
        out = model.forward_with_cfv(t=torch.tensor([rec["t"]]), x=x, wa=wa_c, wr=r_s, we=we_c, prev_x=prev_x,
                                     prev_wa=prev_wa, prev_we=prev_we, a_cfg_scale=rec["a"], r_cfg_scale=rec["r"],
                                     e_cfg_scale=rec["e"], include_r_cfg=rec.get("include_r_cfg", False))
    else:
        raise KeyError(entry)
    return out.detach().cpu().float().numpy()


def main():
    assert refshim.reference_available(), "run this in the build container (needs /root/reference)"
    torch.manual_seed(0)
    only = set(sys.argv[1:])
    manifest_path = os.path.join(HERE, "manifest.json")
    manifest = json.load(open(manifest_path)) if os.path.exists(manifest_path) else {}
    for name, rec in CASES.items():
        if only and name not in only:
            continue
        out = run_case(name, rec)
        np.savez_compressed(os.path.join(HERE, name + ".npz"), out=out)
        manifest[name] = dict(rec, shape=list(out.shape), std=float(out.std()), absmax=float(np.abs(out).max()))
        print(f"{name:16s} shape={out.shape} std={out.std():.4f} absmax={np.abs(out).max():.4f}", flush=True)
    manifest["_meta"] = dict(torch=torch.__version__, weights="oracle.synth.synth_state_dict(dims, seed=0)",
                             inputs="oracle.synth.synth_inputs(dims, B, T_wa or T, seed=100 + seed % 1000, ...)",
                             reference="/root/reference v1.1.2, imported in place via tests/golden/refshim.py")
    json.dump(manifest, open(manifest_path, "w"), indent=1, sort_keys=True)
    if not only or "node_surface" in only:
        write_node_surface()


if __name__ == "__main__":
    main()
