"""B200-native FMT motion-latent sampler: drop-in ComfyUI nodes for the sampling path of ComfyUI-FLOAT_Optimized."""
from .nodes import NODE_CLASS_MAPPINGS, NODE_DISPLAY_NAME_MAPPINGS, FloatSampleMotionSequenceRD_VA, FloatSampleMotionSequenceRD, FloatProcess  # noqa: F401
from .audio import AudioProjectionBackend, AudioProjectionLayer, FloatApplyAudioProjection, projection_backend_for  # noqa: F401
from . import synth  # noqa: F401  (seeded synthetic weights / inputs for bench.py, smoke() and the tests)
from .options import BaseOptions, FmtModel, TORCHDIFFEQ_FIXED_STEP_SOLVERS  # noqa: F401
from .sampler import (Dims, FmtBackend, FmtError, backend_for, perform_ode_sampling_loop, float_sample,  # noqa: F401
                      build_schedule, n_branches_for, draw_window_noise, SOLVERS, float_sample_from_audio, use_b200_sampler,
                      resolve_mode, PRECISION_MODES, sample_clips, clip_schedule, clip_noise, ClipSchedule, StreamSampler, Stream,
                      n_evals, plan_schedule, occupancy_slots)

__version__ = "0.1.0"
__all__ = ["NODE_CLASS_MAPPINGS", "NODE_DISPLAY_NAME_MAPPINGS"]
