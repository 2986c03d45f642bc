"""ComfyUI node classes for the FMT sampling path - same UNIQUE_NAMEs, INPUT_TYPES, RETURN_TYPES and FUNCTION names as
the reference nodes they replace, backed by libfmt_b200.so instead of eager PyTorch + torchdiffeq.

  FloatSampleMotionSequenceRD_VA   <- src/nodes/nodes_vadv.py:534-735
  FloatSampleMotionSequenceRD      <- src/nodes/nodes_adv.py:697-820
  FloatProcess ("FLOAT Process (Opt)") <- src/nodes/nodes.py:146-222: same node; for the duration of the call the pipe's
                                      ``G.sample`` (FLOAT.py:172-253) is this backend, everything else (face crop, wav2vec /
                                      SER encoders, image encoder / decoder) stays the reference code of the pipe.
Tensors cross node edges on the CPU, as in the reference (nodes_vadv.py:197,719).
"""
import logging

import torch

from .options import BaseOptions, TORCHDIFFEQ_FIXED_STEP_SOLVERS
from .sampler import PRECISION_MODES, perform_ode_sampling_loop, resolve_mode, use_b200_sampler

NODES_NAME = "FLOAT_Optimized"
logger = logging.getLogger(f"{NODES_NAME}.b200_fmt")

try:  # ComfyUI progress bar, one tick per window (nodes_adv.py:600,688)
    import comfy.utils as _comfy_utils
except Exception:  # not running under ComfyUI
    _comfy_utils = None


def _progress_bar(total):
    return _comfy_utils.ProgressBar(total) if _comfy_utils is not None else None


# Optional widget both sampler nodes add to the reference's inputs (everything else is identical).  "default" = the FMT_MODE
# environment variable, else bf16.  The reference computes in fp32: "fp32" reproduces it to 1e-4 relative (and passes the
# PSNR >= 40 dB decoded-frame gate); "bf16" is the fastest and within 2e-2 max-abs of the reference latents, which a
# RANDOM-INIT decoder turns into 20-35 dB (profiles/r02_psnr.json); "bf16x3" meets the fp32 mode's gates on the tensor pipe
# (split bf16 operands) - see README.md "Precision".
PRECISION_WIDGET = (("default",) + PRECISION_MODES, {"default": "default", "tooltip": "GEMM operand precision: bf16 (fastest, tcgen05); "
                                                     "fp32 (validation mode, matches the reference to 1e-4, slowest); bf16x3 (matches the "
                                                     "reference like fp32 at tensor-core speed: every GEMM operand is split into two bf16 and "
                                                     "costs three MMAs, so its GEMMs take ~3x their bf16 time, and the first use packs 627 MB more "
                                                     "weights). default = $FMT_MODE or bf16."})


# Second optional widget (SURVEY.md 8f rank 2, second half): the reference moves every tensor back to the CPU between nodes
# (nodes_vadv.py:197,719) and the next node moves it to the GPU again (:692-694).  With keep_on_device the B200 nodes hand CUDA
# tensors to one another - inputs are accepted on either device anyway.  Default False = the reference's behaviour (drop-in);
# FMT_KEEP_ON_DEVICE=1 changes the default.
KEEP_ON_DEVICE_WIDGET = ("BOOLEAN", {"default": False, "tooltip": "Return the result as a CUDA tensor instead of moving it to the CPU "
                                     "(skips the device->host->device round trip between B200 nodes)."})


def keep_on_device_default() -> bool:
    import os
    return os.environ.get("FMT_KEEP_ON_DEVICE", "0") not in ("", "0", "false", "False")


def _hand_over(t: torch.Tensor, keep_on_device) -> torch.Tensor:
    keep = keep_on_device_default() if keep_on_device is None else bool(keep_on_device)
    return t if keep else t.cpu()


def _active_mode(precision, _mode):
    mode = resolve_mode(_mode if _mode is not None else precision)
    logger.info(f"B200 FMT sampler: precision mode {mode}")
    return mode


class FloatSampleMotionSequenceRD_VA:
    UNIQUE_NAME = "FloatSampleMotionSequenceRD_VA"
    DISPLAY_NAME = "Sample Motion Sequence RD"
    DESCRIPTION = ("The core sampling node. It uses the loaded Flow Matching Transformer (FMT) and an ODE solver to generate "
                   "the driven motion latent sequence (r_d). B200-native backend: bf16 tcgen05 GEMMs, one CUDA graph per window.")
    CATEGORY = "FLOAT/Very Advanced"

    @classmethod
    def INPUT_TYPES(cls):
        o = BaseOptions()
        return {
            "required": {
                "r_s_latent": ("TORCH_TENSOR", {"tooltip": "The reference identity latent (wr), derived from the source image."}),
                "wa_latent": ("TORCH_TENSOR", {"tooltip": "The audio conditioning latent (wa)."}),
                "audio_num_frames": ("INT", {"forceInput": True, "tooltip": "Total number of frames to generate."}),
                "we_latent": ("TORCH_TENSOR", {"tooltip": "The emotion conditioning latent (we), (B,1,7) or (B,T,7)."}),
                "float_fmt_model": ("FLOAT_FMT_MODEL", {"tooltip": "The loaded FlowMatchingTransformer model."}),
                "a_cfg_scale": ("FLOAT", {"default": o.a_cfg_scale, "min": 0.0, "max": 10.0, "step": 0.1}),
                "r_cfg_scale": ("FLOAT", {"default": o.r_cfg_scale, "min": 0.0, "max": 10.0, "step": 0.1}),
                "e_cfg_scale": ("FLOAT", {"default": o.e_cfg_scale, "min": 0.0, "max": 10.0, "step": 0.1}),
                "include_r_cfg": ("BOOLEAN", {"default": False}),
                "nfe": ("INT", {"default": o.nfe, "min": 1, "max": 1000}),
                "torchdiffeq_ode_method": (TORCHDIFFEQ_FIXED_STEP_SOLVERS, {"default": o.torchdiffeq_ode_method}),
                "ode_atol": ("FLOAT", {"default": o.ode_atol, "min": 1e-9, "max": 1e-1, "step": 1e-6, "precision": 9}),
                "ode_rtol": ("FLOAT", {"default": o.ode_rtol, "min": 1e-9, "max": 1e-1, "step": 1e-6, "precision": 9}),
                "audio_dropout_prob": ("FLOAT", {"default": o.audio_dropout_prob, "min": 0.0, "max": 1.0, "step": 0.01}),
                "ref_dropout_prob": ("FLOAT", {"default": o.ref_dropout_prob, "min": 0.0, "max": 1.0, "step": 0.01}),
                "emotion_dropout_prob": ("FLOAT", {"default": o.emotion_dropout_prob, "min": 0.0, "max": 1.0, "step": 0.01}),
                "fix_noise_seed": ("BOOLEAN", {"default": o.fix_noise_seed}),
                "seed": ("INT", {"default": o.seed, "min": 0, "max": 0xffffffffffffffff}),
            },
            "optional": {"precision": PRECISION_WIDGET, "keep_on_device": KEEP_ON_DEVICE_WIDGET},
        }

    RETURN_TYPES = ("TORCH_TENSOR", "FLOAT_FMT_MODEL")
    RETURN_NAMES = ("r_d_latents (Wr→D)", "float_fmt_model_out")
    FUNCTION = "sample_rd_sequence_va"

    def sample_rd_sequence_va(self, r_s_latent, wa_latent, we_latent, audio_num_frames, float_fmt_model,
                              a_cfg_scale, r_cfg_scale, e_cfg_scale, include_r_cfg, nfe, torchdiffeq_ode_method,
                              ode_atol, ode_rtol, audio_dropout_prob, ref_dropout_prob, emotion_dropout_prob,
                              fix_noise_seed, seed, precision="default", keep_on_device=None, _mode=None, _noise=None):
        # window geometry from the options the FMT was built with (nodes_vadv.py:627-645)
        src = BaseOptions()
        fco = getattr(float_fmt_model, "final_construction_options", None)
        if isinstance(fco, dict):
            for k, v in fco.items():
                if hasattr(src, k):
                    setattr(src, k, v)
        else:
            logger.error("float_fmt_model does not have 'final_construction_options' dictionary. Using BaseOptions as fallback.")
        num_prev = src.num_prev_frames
        frames_for_clip = int(src.wav2vec_sec * src.fps)
        dim_w = src.dim_w
        target_device = float_fmt_model.target_device

        # validation, identical to nodes_vadv.py:650-656
        if not all(isinstance(t, torch.Tensor) for t in [r_s_latent, wa_latent, we_latent]):
            raise TypeError("All latent inputs must be torch.Tensors.")
        batch_size = wa_latent.shape[0]
        if not (r_s_latent.shape[0] == batch_size and we_latent.shape[0] == batch_size):
            raise ValueError("Batch size mismatch among r_s, wa, we latents.")
        if wa_latent.shape[1] != audio_num_frames:
            logger.warning(f"wa_latent time dim ({wa_latent.shape[1]}) != audio_num_frames ({audio_num_frames}).")

        # the dropout probabilities are set and restored exactly as the reference does (nodes_vadv.py:661-668,722-733);
        # they are no-ops at inference because forward_with_cfv always runs train=False (FMT.py:271-275,372)
        opt = float_fmt_model.opt
        saved = (opt.audio_dropout_prob, opt.ref_dropout_prob, opt.emotion_dropout_prob)
        opt.audio_dropout_prob, opt.ref_dropout_prob, opt.emotion_dropout_prob = audio_dropout_prob, ref_dropout_prob, emotion_dropout_prob
        try:
            # seed policy, nodes_vadv.py:673-689
            noise_gen = None
            if fix_noise_seed or seed != BaseOptions().seed:
                noise_gen = torch.Generator(target_device)
                noise_gen.manual_seed(seed)
            r_s_dev, wa_dev, we_dev = r_s_latent.to(target_device), wa_latent.to(target_device), we_latent.to(target_device)
            n_windows = -(-int(audio_num_frames) // frames_for_clip)
            # the packed weights live in the backend (sampler.backend_for), so the nn.Module never has to move to the GPU
            r_d = perform_ode_sampling_loop(
                fmt_model=float_fmt_model, r_s_latent_dev=r_s_dev, wa_latent_dev=wa_dev, we_latent_dev=we_dev,
                audio_num_frames=audio_num_frames, model_num_prev_frames=num_prev, model_num_frames_for_clip=frames_for_clip,
                model_dim_w=dim_w, ode_nfe=nfe, ode_method=torchdiffeq_ode_method, ode_atol=ode_atol, ode_rtol=ode_rtol,
                target_device=target_device, a_cfg_scale=a_cfg_scale, r_cfg_scale=r_cfg_scale, e_cfg_scale=e_cfg_scale,
                include_r_cfg=include_r_cfg, noise_seed_generator=noise_gen, progress_bar=_progress_bar(n_windows),
                mode=_active_mode(precision, _mode), noise=_noise)
            return (_hand_over(r_d, keep_on_device), float_fmt_model)    # CPU between nodes unless asked otherwise (nodes_vadv.py:719)
        except Exception as e:
            logger.error(f"Error during VA ODE sampling: {e}")
            raise
        finally:
            opt.audio_dropout_prob, opt.ref_dropout_prob, opt.emotion_dropout_prob = saved


class FloatSampleMotionSequenceRD:
    UNIQUE_NAME = "FloatSampleMotionSequenceRD"
    DISPLAY_NAME = "FLOAT Sample Motion Sequence rd"
    DESCRIPTION = "Samples RD using FMT and ODE, with some ODE params from pipe's options."
    CATEGORY = "FLOAT/Advanced"

    @classmethod
    def INPUT_TYPES(cls):
        return {
            "required": {
                "r_s_latent": ("TORCH_TENSOR",),
                "wa_latent": ("TORCH_TENSOR",),
                "audio_num_frames": ("INT", {"forceInput": True}),
                "we_latent": ("TORCH_TENSOR",),
                "float_pipe": ("FLOAT_PIPE",),
                "a_cfg_scale": ("FLOAT", {"default": 2.0, "min": 0.0, "max": 10.0, "step": 0.1}),
                "e_cfg_scale": ("FLOAT", {"default": 1.0, "min": 0.0, "max": 10.0, "step": 0.1}),
                "seed": ("INT", {"default": 62064758300528, "min": 0, "max": 0xffffffffffffffff}),
            },
            "optional": {"precision": PRECISION_WIDGET, "keep_on_device": KEEP_ON_DEVICE_WIDGET},
        }

    RETURN_TYPES = ("TORCH_TENSOR", "FLOAT_PIPE")
    RETURN_NAMES = ("r_d_latents", "float_pipe")
    FUNCTION = "sample_rd_sequence"

    def sample_rd_sequence(self, r_s_latent, wa_latent, audio_num_frames, we_latent, float_pipe, a_cfg_scale, e_cfg_scale, seed,
                           precision="default", keep_on_device=None, _mode=None, _noise=None):
        agent = float_pipe
        opt = agent.opt
        if not all(isinstance(t, torch.Tensor) for t in [r_s_latent, wa_latent, we_latent]):
            raise TypeError("All latent inputs (r_s, wa, we) must be torch.Tensors.")
        batch_size = wa_latent.shape[0]
        if not (r_s_latent.shape[0] == batch_size and we_latent.shape[0] == batch_size):
            raise ValueError(f"Batch size mismatch: wa_latent has {batch_size}, r_s_latent has {r_s_latent.shape[0]}, "
                             f"we_latent has {we_latent.shape[0]}. All must match.")
        if wa_latent.shape[1] != audio_num_frames:
            logger.warning(f"wa_latent time dimension ({wa_latent.shape[1]}) differs from audio_num_frames ({audio_num_frames}).")
        fmt_model = agent.G.fmt
        device = opt.rank
        # seed policy, nodes_adv.py:763-787: seed == -1 means "use opt.seed"
        noise_gen = None
        if opt.fix_noise_seed:
            noise_gen = torch.Generator(device)
            noise_gen.manual_seed(opt.seed if seed == -1 else seed)
        elif seed != -1:
            noise_gen = torch.Generator(device)
            noise_gen.manual_seed(seed)
        r_s_dev, wa_dev, we_dev = r_s_latent.to(device), wa_latent.to(device), we_latent.to(device)
        n_windows = -(-int(audio_num_frames) // int(agent.G.num_frames_for_clip))
        r_d = perform_ode_sampling_loop(
            fmt_model=fmt_model, r_s_latent_dev=r_s_dev, wa_latent_dev=wa_dev, we_latent_dev=we_dev,
            audio_num_frames=audio_num_frames, model_num_prev_frames=agent.G.num_prev_frames,
            model_num_frames_for_clip=agent.G.num_frames_for_clip, model_dim_w=opt.dim_w, ode_nfe=opt.nfe,
            ode_method=opt.torchdiffeq_ode_method, ode_atol=opt.ode_atol, ode_rtol=opt.ode_rtol, target_device=device,
            a_cfg_scale=a_cfg_scale, r_cfg_scale=opt.r_cfg_scale, e_cfg_scale=e_cfg_scale, include_r_cfg=False,
            noise_seed_generator=noise_gen, progress_bar=_progress_bar(n_windows), mode=_active_mode(precision, _mode), noise=_noise)
        return (_hand_over(r_d, keep_on_device), float_pipe)


EMOTIONS = ['none', 'angry', 'disgust', 'fear', 'happy', 'neutral', 'sad', 'surprise']     # nodes.py:27

try:  # VRAM manager the reference wraps the call in (nodes.py:171); absent outside ComfyUI + seconohe
    from seconohe.torch import model_to_target as _model_to_target
except Exception:
    _model_to_target = None


class FloatProcess:
    UNIQUE_NAME = "FloatProcessOpt"
    DISPLAY_NAME = "FLOAT Process (Opt)"
    DESCRIPTION = "Float Processing"
    CATEGORY = "FLOAT"

    @classmethod
    def INPUT_TYPES(cls):
        return {
            "required": {
                "ref_image": ("IMAGE",),
                "ref_audio": ("AUDIO",),
                "float_pipe": ("FLOAT_PIPE",),
                "a_cfg_scale": ("FLOAT", {"default": 2.0, "min": 1.0, "step": 0.1}),
                "e_cfg_scale": ("FLOAT", {"default": 1.0, "min": 1.0, "step": 0.1}),
                "fps": ("FLOAT", {"default": 25, "step": 1}),
                "emotion": (EMOTIONS, {"default": "none"}),
                "face_align": ("BOOLEAN", {"default": True},),
                "seed": ("INT", {"default": 62064758300528, "min": 0, "max": 0xffffffffffffffff}),
            },
            "optional": {"precision": PRECISION_WIDGET},
        }

    RETURN_TYPES = ("IMAGE", "AUDIO", "FLOAT")
    RETURN_NAMES = ("images", "ref_audio", "fps")
    FUNCTION = "floatprocess"

    def floatprocess(self, ref_image, ref_audio, float_pipe, a_cfg_scale, e_cfg_scale, fps, emotion, face_align, seed,
                     precision="default", _mode=None):
        """One (image, audio) pair at a time, the shorter batch repeating its last item, seed + i per pair - as nodes.py:169-222;
        the motion latents of every pair come from libfmt_b200.so instead of eager PyTorch + torchdiffeq."""
        import contextlib
        pipe = float_pipe
        pipe.G.target_device = pipe.rank
        pipe.G.cudnn_benchmark_setting = pipe.opt.cudnn_benchmark_enabled
        vram = _model_to_target(logger, pipe.G) if _model_to_target is not None else contextlib.nullcontext()
        mode = _active_mode(precision, _mode)
        with vram, use_b200_sampler(pipe.G, mode):
            pipe.opt.fps = fps
            wave, rate = ref_audio["waveform"], ref_audio["sample_rate"]
            n_img, n_aud = ref_image.shape[0], wave.shape[0]
            n = max(n_img, n_aud)
            frames, waves = [], []
            for i in range(n):
                img = ref_image[min(i, n_img - 1):min(i, n_img - 1) + 1].to(pipe.rank)
                wav = wave[min(i, n_aud - 1):min(i, n_aud - 1) + 1].to(pipe.rank)
                out = pipe.run_inference(None, img, {"waveform": wav, "sample_rate": rate}, a_cfg_scale=a_cfg_scale,
                                         r_cfg_scale=pipe.opt.r_cfg_scale, e_cfg_scale=e_cfg_scale,
                                         emo=None if emotion == "none" else emotion, no_crop=not face_align, seed=seed + i)
                frames.append(out.cpu())
                waves.append(wav.cpu())
        if n == 1:
            audio_out = ref_audio
        else:   # the audio of every pair, concatenated along time (nodes.py:213-220)
            cat = torch.cat([w.squeeze(0) for w in waves], dim=1).unsqueeze(0).to(wave.device)
            audio_out = {"waveform": cat, "sample_rate": rate}
        return (torch.cat(frames, dim=0), audio_out, fps)


from .audio import FloatApplyAudioProjection  # noqa: E402  (SURVEY.md §8f rank 2: the node in front of the sampler)

NODE_CLASSES = [FloatSampleMotionSequenceRD_VA, FloatSampleMotionSequenceRD, FloatProcess, FloatApplyAudioProjection]
NODE_CLASS_MAPPINGS = {c.UNIQUE_NAME: c for c in NODE_CLASSES}
NODE_DISPLAY_NAME_MAPPINGS = {c.UNIQUE_NAME: c.DISPLAY_NAME for c in NODE_CLASSES}
