"""Audio projection in front of the sampler (SURVEY.md §8f rank 2): ``wa = SiLU(LayerNorm(Linear(wav2vec features)))``.

Replaces what the reference's ``FloatApplyAudioProjection`` node runs (src/nodes/nodes_vadv.py:147-198) on the module that
``LoadAudioProjectionLayer`` builds (src/nodes/nodes_vadv_loader.py:228-257; same layers as ``AudioEncoder.audio_projection``,
src/nodes/models/float/FLOAT.py:338-342): a bf16 tcgen05 GEMM (K = 9216 stacked wav2vec layers, or 768) with fp32
accumulation, then LayerNorm (affine) and SiLU in fp32.  No CPU / eager fallback.
"""
import ctypes as C
import logging
import os
import weakref

import torch

from . import _cabi
from ._cabi import FmtError, check

logger = logging.getLogger("FLOAT_Optimized.b200_fmt")
_MODES = _cabi.MODE_IDS      # "bf16x3" needs in_dim % 64 == 0 (9216 and 768 are)


class AudioProjectionBackend:
    """Packed copy of one projection layer on one CUDA device."""

    def __init__(self, linear_w, linear_b, ln_w, ln_b, ln_eps, device):
        self.lib = _cabi.load_library()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise FmtError(f"projection_layer.target_device is '{self.device}': the B200 audio projection runs on CUDA (sm_100a) only; "
                           "there is no CPU fallback.")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.out_dim, self.in_dim = int(linear_w.shape[0]), int(linear_w.shape[1])
        ts = [t.detach().to(device="cpu", dtype=torch.float32).contiguous() for t in (linear_w, linear_b, ln_w, ln_b)]
        h = C.c_void_p()
        check(self.lib.fmt_proj_create(self.in_dim, self.out_dim, ts[0].data_ptr(), ts[1].data_ptr(), ts[2].data_ptr(), ts[3].data_ptr(),
                                       float(ln_eps), _cabi.FMT_LOC_HOST, self.device.index, C.byref(h)), "fmt_proj_create")
        self._handle = h

    def apply(self, x: torch.Tensor, mode: str = "bf16") -> torch.Tensor:
        """x: (..., in_dim) on this backend's device -> (..., out_dim) fp32 on the same device."""
        if x.shape[-1] != self.in_dim:
            raise ValueError(f"audio projection: last dimension is {x.shape[-1]}, expected {self.in_dim}")
        x2 = x.to(device=self.device, dtype=torch.float32).contiguous().view(-1, self.in_dim)
        out = torch.empty(x2.shape[0], self.out_dim, device=self.device, dtype=torch.float32)
        if x2.shape[0] > 0:
            st = torch.cuda.current_stream(self.device).cuda_stream
            check(self.lib.fmt_proj_apply(self._handle, x2.data_ptr(), x2.shape[0], out.data_ptr(), _MODES[mode], _cabi.FMT_LOC_DEVICE,
                                          C.c_void_p(st)), "fmt_proj_apply")
        return out.view(*x.shape[:-1], self.out_dim)

    def launch_count(self, reset=False) -> int:
        return int(self.lib.fmt_proj_launch_count(self._handle, 1 if reset else 0))

    def close(self):
        if getattr(self, "_handle", None):
            self.lib.fmt_proj_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_BACKENDS = weakref.WeakKeyDictionary()


def _layer_tensors(projection_layer):
    """(linear.weight, linear.bias, ln.weight, ln.bias, ln.eps) of an nn.Sequential(Linear, LayerNorm, SiLU)."""
    sd = projection_layer.state_dict()
    try:
        w, b, g, beta = sd["0.weight"], sd["0.bias"], sd["1.weight"], sd["1.bias"]
    except KeyError as e:
        raise TypeError(f"projection_layer is not Sequential(Linear, LayerNorm, SiLU): missing state-dict key {e}")
    eps = 1e-5
    try:
        eps = float(projection_layer[1].eps)
    except Exception:
        eps = float(getattr(projection_layer, "ln_eps", 1e-5))
    return w, b, g, beta, eps


def projection_backend_for(projection_layer, device) -> AudioProjectionBackend:
    w, b, g, beta, eps = _layer_tensors(projection_layer)
    fp = tuple((t.data_ptr(), getattr(t, "_version", 0), tuple(t.shape)) for t in (w, b, g, beta)) + (eps,)
    device = torch.device(device)
    per = _BACKENDS.setdefault(projection_layer, {})
    hit = per.get(str(device))
    if hit is not None and hit[0] == fp:
        return hit[1]
    if hit is not None:
        hit[1].close()
    be = AudioProjectionBackend(w, b, g, beta, eps, device)
    per[str(device)] = (fp, be)
    return be


class AudioProjectionLayer(torch.nn.Sequential):
    """What ``LoadAudioProjectionLayer`` returns (nodes_vadv_loader.py:233-257): Sequential(Linear, LayerNorm, SiLU) carrying
    ``inferred_input_feature_dim`` and ``target_device``.  For tests, benchmarks and non-ComfyUI hosts."""

    def __init__(self, in_dim: int, dim_a: int = 512, target_device="cuda"):
        super().__init__(torch.nn.Linear(in_dim, dim_a), torch.nn.LayerNorm(dim_a), torch.nn.SiLU())
        self.inferred_input_feature_dim = in_dim
        self.target_device = target_device


class FloatApplyAudioProjection:
    UNIQUE_NAME = "FloatApplyAudioProjection"
    DISPLAY_NAME = "FLOAT Apply Audio Projection"
    DESCRIPTION = ("Applies the loaded audio projection layer to the features extracted from the Wav2Vec model. "
                   "This final step projects the high-dimensional audio features down to the motion latent space, "
                   "producing the final audio conditioning tensor (wa_latent). B200-native backend: bf16 tcgen05 GEMM.")
    CATEGORY = "FLOAT/Very Advanced"

    @classmethod
    def INPUT_TYPES(cls):
        return {
            "required": {
                "wav2vec_features": ("TORCH_TENSOR", {
                    "tooltip": "The batch of interpolated feature tensors output by the Wav2Vec feature extraction node."}),
                "projection_layer": ("AUDIO_PROJECTION_LAYER", {"tooltip": "The loaded audio projection layer module."}),
            },
            # B200 addition: hand wa_latent to the sampler node as a CUDA tensor (default: CPU between nodes, as the reference)
            "optional": {"keep_on_device": ("BOOLEAN", {"default": False, "tooltip": "Return wa_latent as a CUDA tensor instead of moving it to the CPU."})},
        }

    RETURN_TYPES = ("TORCH_TENSOR",)
    RETURN_NAMES = ("wa_latent",)
    FUNCTION = "apply_projection"

    def apply_projection(self, wav2vec_features: torch.Tensor, projection_layer: torch.nn.Module, keep_on_device=None, _mode="bf16"):
        # validation and messages as in nodes_vadv.py:170-181
        if not isinstance(wav2vec_features, torch.Tensor):
            raise TypeError("Input 'wav2vec_features' must be a torch.Tensor.")
        if not isinstance(projection_layer, torch.nn.Module):
            raise TypeError("Input 'projection_layer' must be a torch.nn.Module.")
        if wav2vec_features.ndim != 3:
            raise TypeError("Input 'wav2vec_features' must contain 3 dimensions")
        if wav2vec_features.shape[2] != projection_layer.inferred_input_feature_dim:
            raise TypeError("Input 'wav2vec_features' wrong size has "
                            f"{wav2vec_features.shape[2]}, expected {projection_layer.inferred_input_feature_dim}. "
                            "`only_last_features` mismatch?")
        target_device = projection_layer.target_device
        be = projection_backend_for(projection_layer, target_device)
        features_on_device = wav2vec_features.to(be.device)
        logger.info(f"Applying audio projection layer to features of shape {features_on_device.shape}.")
        wa_latent_gpu = be.apply(features_on_device, mode=_mode)
        logger.info(f"Output wa_latent shape: {wa_latent_gpu.shape}")
        if keep_on_device is None:
            keep_on_device = os.environ.get("FMT_KEEP_ON_DEVICE", "0") not in ("", "0", "false", "False")
        # CPU between nodes, as the reference (nodes_vadv.py:197), unless the device-resident hand-off was asked for
        return (wa_latent_gpu if keep_on_device else wa_latent_gpu.cpu(),)
