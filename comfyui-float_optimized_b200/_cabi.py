"""ctypes binding of include/fmt_b200.h.  No fallback: a missing or unloadable library is a hard error."""
import ctypes as C
import os

from .build import LIB_PATH

FMT_W_NUM_GLOBAL = 13
FMT_W_PER_BLOCK = 10
FMT_LOC_DEVICE, FMT_LOC_HOST = 0, 1
FMT_MODE_BF16, FMT_MODE_FP32_VALIDATE, FMT_MODE_BF16X3 = 0, 1, 2
# precision-mode names of sampler.PRECISION_MODES -> FmtPlan.mode / fmt_proj_apply's mode
MODE_IDS = {"bf16": FMT_MODE_BF16, "fp32": FMT_MODE_FP32_VALIDATE, "bf16x3": FMT_MODE_BF16X3}
FMT_MAX_STAGES = 4
FMT_ABI_VERSION = 2

# state-dict key order expected by fmt_create (include/fmt_b200.h enums)
GLOBAL_KEYS = [
    "x_embedder.proj.weight", "x_embedder.proj.bias",
    "t_embedder.mlp.0.weight", "t_embedder.mlp.0.bias", "t_embedder.mlp.2.weight", "t_embedder.mlp.2.bias",
    "c_embedder.weight", "c_embedder.bias", "pos_embed",
    "decoder.adaLN_modulation.1.weight", "decoder.adaLN_modulation.1.bias", "decoder.linear.weight", "decoder.linear.bias",
]
BLOCK_KEYS = [
    "attn.qkv.weight", "attn.qkv.bias", "attn.proj.weight", "attn.proj.bias",
    "mlp.fc1.weight", "mlp.fc1.bias", "mlp.fc2.weight", "mlp.fc2.bias",
    "adaLN_modulation.1.weight", "adaLN_modulation.1.bias",
]


class FmtDims(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("dim_w", "dim_a", "dim_e", "dim_h", "depth", "num_heads", "mlp_hidden",
                                          "num_prev_frames", "frames_per_clip", "attention_window")]


class FmtPlan(C.Structure):
    _fields_ = [("batch", C.c_int32), ("n_branches", C.c_int32), ("we_dynamic", C.c_int32), ("mode", C.c_int32),
                ("n_steps", C.c_int32), ("n_stages", C.c_int32),
                ("t_eval", C.POINTER(C.c_float)), ("dt", C.POINTER(C.c_float)),
                ("rk_a", C.POINTER(C.c_float)), ("rk_b", C.POINTER(C.c_float))]


PROGRESS_FN = C.CFUNCTYPE(None, C.c_int32, C.c_int32, C.c_void_p)


class FmtClip(C.Structure):
    _fields_ = [("location", C.c_int32), ("r_s", C.c_void_p), ("wa", C.c_void_p), ("we", C.c_void_p), ("noise", C.c_void_p),
                ("r_d", C.c_void_p), ("T_wa", C.c_int32), ("T_we", C.c_int32), ("audio_num_frames", C.c_int32),
                ("a_cfg_scale", C.c_float), ("r_cfg_scale", C.c_float), ("e_cfg_scale", C.c_float),
                ("progress", PROGRESS_FN), ("progress_user", C.c_void_p)]


class FmtClipSet(C.Structure):
    _fields_ = [("n_clips", C.c_int32), ("r_s", C.POINTER(C.c_void_p)), ("wa", C.POINTER(C.c_void_p)), ("we", C.POINTER(C.c_void_p)),
                ("noise", C.POINTER(C.c_void_p)), ("r_d", C.POINTER(C.c_void_p)), ("T_wa", C.POINTER(C.c_int32)),
                ("T_we", C.POINTER(C.c_int32)), ("audio_num_frames", C.POINTER(C.c_int32)),
                ("a_cfg_scale", C.c_float), ("r_cfg_scale", C.c_float), ("e_cfg_scale", C.c_float),
                ("progress", PROGRESS_FN), ("progress_user", C.c_void_p)]


class FmtClipGuidance(C.Structure):
    _fields_ = [("a_cfg_scale", C.POINTER(C.c_float)), ("r_cfg_scale", C.POINTER(C.c_float)), ("e_cfg_scale", C.POINTER(C.c_float)),
                ("n_branches", C.POINTER(C.c_int32))]


class FmtWindowSet(C.Structure):
    _fields_ = [("n_streams", C.c_int32)] + [(n, C.POINTER(C.c_void_p)) for n in ("r_s", "wa", "we", "x0", "ctx", "r_d")] + \
               [(n, C.POINTER(C.c_int32)) for n in ("T_wa", "T_we", "n_out", "first_window")]


class FmtClipOde(C.Structure):
    _fields_ = [("n_steps", C.POINTER(C.c_int32)), ("n_stages", C.POINTER(C.c_int32))] + \
               [(n, C.POINTER(C.POINTER(C.c_float))) for n in ("t_eval", "dt", "rk_a", "rk_b")]


class FmtEval(C.Structure):
    _fields_ = [("x", C.c_void_p), ("prev_x", C.c_void_p), ("wa", C.c_void_p), ("prev_wa", C.c_void_p), ("we", C.c_void_p),
                ("prev_we", C.c_void_p), ("r_s", C.c_void_p), ("v_out", C.c_void_p), ("eval_index", C.c_int32),
                ("a_cfg_scale", C.c_float), ("r_cfg_scale", C.c_float), ("e_cfg_scale", C.c_float)]


FMT_EPI_STORE, FMT_EPI_GELU, FMT_EPI_POS, FMT_EPI_GATE_RES = 0, 1, 2, 3


class FmtDebugGemm(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("mode", "kind", "M", "N", "K", "block_n", "ksplit", "ldo", "out_f32", "frames")] + \
               [(n, C.c_void_p) for n in ("A", "W", "bias", "out", "pos", "gate", "urow")] + \
               [("ldg", C.c_int64), ("gate_off", C.c_int64)]


FMT_STAGE_ROW, FMT_STAGE_ATTN, FMT_STAGE_GELU, FMT_STAGE_COMB = 0, 1, 2, 3


class FmtDebugStage(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("kind", "grid", "chunk_rows", "n_branches", "batch", "n_frames", "n_prev", "H", "heads", "window",
                                          "mlp_hidden", "W", "row_mode", "zero_qkv", "parity", "n_stages", "stage", "step")] + \
               [(n, C.c_int64) for n in ("ldt", "gate_off", "shift_off", "scale_off")] + \
               [(n, C.c_float) for n in ("a_scale", "r_scale", "e_scale")] + [("rk_a", C.c_float * 16), ("rk_b", C.c_float * 4)] + \
               [(n, C.c_void_p) for n in ("X", "Pacc", "QKVacc", "Hacc", "Vacc", "A1", "A2", "Hm", "ax", "table", "urow", "bias", "pos",
                                          "x_state", "kbuf", "ddt", "slot_branches", "slot_scales")]


_SIGNATURES = {
    "fmt_abi_version": (C.c_int32, []),
    "fmt_last_error": (C.c_char_p, []),
    "fmt_create": (C.c_int32, [C.POINTER(FmtDims), C.POINTER(C.c_void_p), C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]),
    "fmt_destroy": (C.c_int32, [C.c_void_p]),
    "fmt_configure": (C.c_int32, [C.c_void_p, C.POINTER(FmtPlan), C.c_void_p]),
    "fmt_workspace_bytes": (C.c_int64, [C.c_void_p]),
    "fmt_sample_clip": (C.c_int32, [C.c_void_p, C.POINTER(FmtClip), C.c_void_p]),
    "fmt_sample_clips": (C.c_int32, [C.c_void_p, C.POINTER(FmtClipSet), C.c_void_p]),
    "fmt_sample_clips_guided": (C.c_int32, [C.c_void_p, C.POINTER(FmtClipSet), C.POINTER(FmtClipGuidance), C.c_void_p]),
    "fmt_sample_windows": (C.c_int32, [C.c_void_p, C.POINTER(FmtWindowSet), C.POINTER(FmtClipGuidance), C.c_void_p]),
    "fmt_sample_clips_ode": (C.c_int32, [C.c_void_p, C.POINTER(FmtClipSet), C.POINTER(FmtClipGuidance), C.POINTER(FmtClipOde), C.c_void_p]),
    "fmt_sample_windows_ode": (C.c_int32, [C.c_void_p, C.POINTER(FmtWindowSet), C.POINTER(FmtClipGuidance), C.POINTER(FmtClipOde), C.c_void_p]),
    "fmt_sample_clip_set": (C.c_int32, [C.c_void_p, C.POINTER(FmtClipSet), C.POINTER(FmtClipGuidance), C.POINTER(FmtClipOde),
                                        C.POINTER(C.c_int32), C.c_void_p]),
    "fmt_sample_window_set": (C.c_int32, [C.c_void_p, C.POINTER(FmtWindowSet), C.POINTER(FmtClipGuidance), C.POINTER(FmtClipOde),
                                          C.POINTER(C.c_int32), C.c_void_p]),
    "fmt_occupancy_slots": (C.c_int32, [C.c_int32, C.c_int32]),
    "fmt_last_window_slots": (C.c_int32, [C.c_void_p]),
    "fmt_clip_schedule": (C.c_int32, [C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                      C.POINTER(C.c_int32)]),
    "fmt_velocity": (C.c_int32, [C.c_void_p, C.POINTER(FmtEval), C.c_void_p]),
    "fmt_launch_count": (C.c_int64, [C.c_void_p, C.c_int32]),
    "fmt_graph_kernel_nodes": (C.c_int32, [C.c_void_p]),
    "fmt_ode_graph_kernel_nodes": (C.c_int32, [C.c_void_p]),
    "fmt_window_kernel_status": (C.c_int32, [C.c_void_p]),
    "fmt_debug_window_trace": (C.c_int64, [C.c_void_p, C.c_void_p, C.c_int64]),
    "fmt_debug_condition_rows": (C.c_int32, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "fmt_debug_condition_rows_ode": (C.c_int32, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "fmt_debug_condition_rows_slots": (C.c_int32, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.c_void_p]),
    "fmt_proj_create": (C.c_int32, [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_int32, C.c_int32,
                                    C.POINTER(C.c_void_p)]),
    "fmt_proj_destroy": (C.c_int32, [C.c_void_p]),
    "fmt_proj_apply": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "fmt_proj_launch_count": (C.c_int64, [C.c_void_p, C.c_int32]),
    "fmt_debug_gemm_bf16": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "fmt_debug_gemm_bench": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "fmt_debug_gemm_bf16x3": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "fmt_debug_gemm_bench_bf16x3": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                                C.c_void_p]),
    "fmt_debug_gemm_fp32": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "fmt_debug_gemm_epilogue": (C.c_int32, [C.POINTER(FmtDebugGemm), C.c_void_p]),
    "fmt_debug_lnmod": (C.c_int32, [C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p,
                                    C.c_void_p]),
    "fmt_debug_band_attention": (C.c_int32, [C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32,
                                             C.c_void_p]),
    "fmt_debug_flow_stage": (C.c_int32, [C.POINTER(FmtDebugStage), C.c_void_p]),
    "fmt_debug_window_stage": (C.c_int32, [C.POINTER(FmtDebugStage), C.c_void_p]),
}

_lib = None


class FmtError(RuntimeError):
    pass


def load_library():
    """Loads csrc/libfmt_b200.so.  Raises if it has not been built - there is no Python/torch fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FmtError(f"{LIB_PATH} is missing: build it first (python __graft_entry__.py build, or "
                       f"`python comfyui-float_optimized_b200/build.py`). This node pack has no CPU / eager-PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError if the symbol is not exported
        fn.restype, fn.argtypes = res, args
    if lib.fmt_abi_version() != FMT_ABI_VERSION:
        raise FmtError(f"libfmt_b200.so ABI {lib.fmt_abi_version()} != binding ABI {FMT_ABI_VERSION}: rebuild")
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load_library().fmt_last_error().decode("utf-8", "replace")
        if rc == -1:
            raise ValueError(f"{what}: {msg}")
        raise FmtError(f"{what} failed ({rc}): {msg}")
