"""Host side of the FMT sampler: the reference's window loop and solver schedule, expressed as one C-ABI call.

Mirrors (paths relative to the reference repo):
  * ``_perform_ode_sampling_loop``  src/nodes/nodes_adv.py:545-694   -> :func:`perform_ode_sampling_loop`
  * ``FLOAT.sample`` (from ``wa``/``we`` on)  src/nodes/models/float/FLOAT.py:172-253 -> :func:`float_sample`
  * ``FlowMatchingTransformer.forward_with_cfv``  FMT.py:342-401     -> :meth:`FmtBackend.velocity`
All arithmetic happens in libfmt_b200.so (hand-written CUDA, sm_100a).  PyTorch is used for device memory, the
RNG (one ``torch.randn`` per window, exactly like the reference) and streams.  There is no fallback path.
"""
import ctypes as C
import functools
import math
import numbers
import os
import weakref
from dataclasses import dataclass
from typing import Callable, Dict, List, Mapping, Optional, Sequence

import torch

from . import _cabi
from ._cabi import FmtError

# Butcher tableaux of torchdiffeq's fixed-grid solvers (src/nodes/__init__.py:15-23 lists what the node offers).
# y_i = y0 + dt * sum_j a[i][j] k_j ; t_i = t0 + c[i] * dt ; y1 = y0 + dt * sum_j b[j] k_j
SOLVERS = {
    "euler": dict(c=[0.0], a=[[0.0]], b=[1.0]),
    "midpoint": dict(c=[0.0, 0.5], a=[[0, 0], [0.5, 0]], b=[0.0, 1.0]),
    "heun2": dict(c=[0.0, 1.0], a=[[0, 0], [1.0, 0]], b=[0.5, 0.5]),
    "heun3": dict(c=[0.0, 1 / 3, 2 / 3], a=[[0, 0, 0], [1 / 3, 0, 0], [0, 2 / 3, 0]], b=[0.25, 0.0, 0.75]),
    # torchdiffeq's fixed-grid "rk4" is the 3/8-rule variant (rk4_alt_step_func)
    "rk4": dict(c=[0.0, 1 / 3, 2 / 3, 1.0], a=[[0, 0, 0, 0], [1 / 3, 0, 0, 0], [-1 / 3, 1, 0, 0], [1, -1, 1, 0]],
                b=[0.125, 0.375, 0.375, 0.125]),
}


@dataclass(frozen=True)
class Dims:
    dim_w: int = 512
    dim_a: int = 512
    dim_e: int = 7
    dim_h: int = 1024
    fmt_depth: int = 8
    num_heads: int = 8
    mlp_hidden: int = 4096
    num_prev_frames: int = 10
    frames_per_clip: int = 50
    attention_window: int = 2

    @staticmethod
    def from_options(opt, state_dict=None) -> "Dims":
        """Dims from a BaseOptions-like object (or dict); weight shapes win where both are known
        (the loader infers dim_h/depth/mlp_ratio/dim_a from the checkpoint, nodes_vadv_loader.py:655-866)."""
        get = (lambda k, dflt: opt.get(k, dflt)) if isinstance(opt, dict) else (lambda k, dflt: getattr(opt, k, dflt))
        dim_h = int(get("dim_h", 1024))
        d = dict(dim_w=int(get("dim_w", 512)), dim_a=int(get("dim_a", 512)), dim_e=int(get("dim_e", 7)), dim_h=dim_h,
                 fmt_depth=int(get("fmt_depth", 8)), num_heads=int(get("num_heads", 8)),
                 mlp_hidden=int(dim_h * float(get("mlp_ratio", 4.0))),
                 num_prev_frames=int(get("num_prev_frames", 10)),
                 frames_per_clip=int(float(get("wav2vec_sec", 2.0)) * float(get("fps", 25.0))),
                 attention_window=int(get("attention_window", 2)))
        if state_dict is not None:
            xw = state_dict["x_embedder.proj.weight"]
            d["dim_h"], d["dim_w"] = int(xw.shape[0]), int(xw.shape[1])
            d["mlp_hidden"] = int(state_dict["blocks.0.mlp.fc1.weight"].shape[0])
            d["fmt_depth"] = 1 + max(int(k.split(".")[1]) for k in state_dict if k.startswith("blocks."))
            d["dim_a"] = int(state_dict["c_embedder.weight"].shape[1]) - d["dim_w"] - d["dim_e"]
            if "pos_embed" in state_dict:
                d["frames_per_clip"] = int(state_dict["pos_embed"].shape[-2]) - d["num_prev_frames"]
        return Dims(**d)


def _f32_array(values):
    arr = (C.c_float * max(1, len(values)))()
    for i, v in enumerate(values):
        arr[i] = float(v)
    return arr


def build_schedule(nfe: int, method: str):
    """Time grid of ``torch.linspace(0, 1, nfe)`` (nodes_adv.py:587) walked by a fixed-grid solver:
    nfe points => nfe-1 steps; stage times t0 + c_i*dt evaluated in fp32 like torchdiffeq does.  (Cached: ~0.1 ms of torch scalar
    arithmetic that every sampler call would otherwise repeat.)"""
    return dict(_build_schedule(int(nfe), method))


@functools.lru_cache(maxsize=64)
def _build_schedule(nfe: int, method: str):
    if method not in SOLVERS:
        raise ValueError(f"Unknown fixed-step solver '{method}' (supported: {sorted(SOLVERS)})")
    tab = SOLVERS[method]
    t = torch.linspace(0, 1, int(nfe), dtype=torch.float32)
    dt = (t[1:] - t[:-1])
    stages = len(tab["c"])
    t_eval = []
    for i in range(max(0, int(nfe) - 1)):
        for c in tab["c"]:
            if c == 0.0:
                t_eval.append(float(t[i]))
            elif c == 1.0:
                t_eval.append(float(t[i + 1]) if method == "rk4" else float(t[i] + dt[i]))
            else:
                t_eval.append(float(t[i] + dt[i] * torch.tensor(c, dtype=torch.float32)))
    a_flat = [x for row in tab["a"] for x in row]
    return dict(n_steps=max(0, int(nfe) - 1), n_stages=stages, t_eval=t_eval, dt=[float(x) for x in dt], a=a_flat, b=tab["b"])


def n_evals(nfe: int, method: str) -> int:
    """Model evaluations per window of a fixed-grid solver: (nfe - 1) steps of one evaluation per stage."""
    return max(0, int(nfe) - 1) * len(SOLVERS[method]["c"])


def plan_schedule(schedules: Sequence[tuple], nfe: int, method: str) -> tuple:
    """The (nfe, method) a call of clips with these schedules configures its plan with: a clip's schedule that needs the most
    evaluations per window (:func:`n_evals`); on a tie the call's own (nfe, method) if some clip runs it, else the first in input
    order.  So a call whose clips all run one schedule runs the plan's window graph."""
    most = max(n_evals(*sc) for sc in schedules)
    tied = [sc for sc in schedules if n_evals(*sc) == most]
    return (int(nfe), method) if (int(nfe), method) in tied else tied[0]


PRECISION_MODES = ("bf16", "fp32", "bf16x3")


def resolve_mode(mode: Optional[str] = None) -> str:
    """Operand precision of the GEMMs: "bf16" (tcgen05, fp32 accumulate / residual / softmax / ODE state; latents within 2e-2
    max-abs of the reference), "fp32" (validation mode, fp32 FFMA GEMMs; within 1e-4 relative, the slowest) or "bf16x3" (tcgen05
    on operands split into two bf16 each, x = hi + lo, three MMAs per product; within 1e-4 relative like "fp32", faster than it,
    and the weights are packed once more, 627 MB for the FMT).  An explicit argument wins, then the environment variable
    FMT_MODE, then "bf16".  The reference itself computes in fp32."""
    m = mode if mode not in (None, "", "default") else os.environ.get("FMT_MODE", "bf16")
    m = str(m).lower()
    if m not in PRECISION_MODES:
        raise ValueError(f"precision mode '{m}' is not one of {PRECISION_MODES}")
    return m


def n_branches_for(a_cfg_scale, r_cfg_scale, e_cfg_scale, include_r_cfg) -> int:
    """FMT.py:346,359,380,400: one conditional forward when every scale == 1, else 3 (or 4) batched branches."""
    if a_cfg_scale != 1.0 or r_cfg_scale != 1.0 or e_cfg_scale != 1.0:
        return 4 if include_r_cfg else 3
    return 1


class FmtBackend:
    """Packed weights + workspace + captured window graph for one FMT on one CUDA device (owns an FmtHandle*)."""

    def __init__(self, state_dict: Dict[str, torch.Tensor], dims: Dims, device):
        self.lib = _cabi.load_library()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise FmtError(f"FmtBackend needs a CUDA device (sm_100a); got '{self.device}'. There is no CPU fallback.")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.dims = dims
        self._plan_key = None
        self._n_eval = 0
        self._handle = C.c_void_p()
        keys = list(_cabi.GLOBAL_KEYS) + [f"blocks.{i}.{k}" for i in range(dims.fmt_depth) for k in _cabi.BLOCK_KEYS]
        missing = [k for k in keys if k not in state_dict]
        if missing:
            raise KeyError(f"FMT state dict is missing {missing[:4]}{'...' if len(missing) > 4 else ''}")
        tensors = [state_dict[k].detach() for k in keys]
        on_host = all(t.device.type == "cpu" for t in tensors)
        if on_host:
            tensors = [t.to(torch.float32).contiguous() for t in tensors]
        else:
            tensors = [t.to(device=self.device, dtype=torch.float32).contiguous() for t in tensors]
        self._check_shapes(dict(zip(keys, tensors)))
        ptrs = (C.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])
        cd = _cabi.FmtDims(dims.dim_w, dims.dim_a, dims.dim_e, dims.dim_h, dims.fmt_depth, dims.num_heads, dims.mlp_hidden,
                           dims.num_prev_frames, dims.frames_per_clip, dims.attention_window)
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.fmt_create(C.byref(cd), ptrs, len(tensors),
                                            _cabi.FMT_LOC_HOST if on_host else _cabi.FMT_LOC_DEVICE,
                                            self.device.index, C.byref(self._handle)), "fmt_create")
        self._finalizer = weakref.finalize(self, self.lib.fmt_destroy, self._handle)

    def _check_shapes(self, sd):
        d = self.dims
        H, N = d.dim_h, d.num_prev_frames + d.frames_per_clip
        expect = {"x_embedder.proj.weight": (H, d.dim_w), "c_embedder.weight": (H, d.dim_w + d.dim_a + d.dim_e),
                  "t_embedder.mlp.0.weight": (H, 256), "decoder.linear.weight": (d.dim_w, H),
                  "blocks.0.attn.qkv.weight": (3 * H, H), "blocks.0.mlp.fc1.weight": (d.mlp_hidden, H),
                  "blocks.0.adaLN_modulation.1.weight": (6 * H, H)}
        for k, shp in expect.items():
            if tuple(sd[k].shape) != shp:
                raise ValueError(f"{k}: shape {tuple(sd[k].shape)} != expected {shp} for {d}")
        if sd["pos_embed"].numel() != N * H:
            raise ValueError(f"pos_embed has {sd['pos_embed'].numel()} elements, expected {N}x{H}")

    # ------------------------------------------------------------------------------------------------
    def close(self):
        self._finalizer()

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def configure(self, batch: int, n_branches: int, we_dynamic: bool, nfe: int, method: str = "euler", mode: str = "bf16"):
        mode_id = _cabi.MODE_IDS[resolve_mode(mode)]
        key = (batch, n_branches, bool(we_dynamic), int(nfe), method, mode_id)
        if key == self._plan_key:
            return
        sched = build_schedule(nfe, method)
        t_eval, dt, a, b = (_f32_array(sched[k]) for k in ("t_eval", "dt", "a", "b"))
        plan = _cabi.FmtPlan(batch, n_branches, int(bool(we_dynamic)), mode_id, sched["n_steps"], sched["n_stages"],
                             C.cast(t_eval, C.POINTER(C.c_float)), C.cast(dt, C.POINTER(C.c_float)),
                             C.cast(a, C.POINTER(C.c_float)), C.cast(b, C.POINTER(C.c_float)))
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.fmt_configure(self._handle, C.byref(plan), self._stream()), "fmt_configure")
        self._plan_key = key
        self._n_eval = sched["n_steps"] * sched["n_stages"]

    def workspace_bytes(self) -> int:
        return int(self.lib.fmt_workspace_bytes(self._handle))

    def launch_count(self, reset: bool = False) -> int:
        return int(self.lib.fmt_launch_count(self._handle, int(reset)))

    def window_kernel_status(self) -> int:
        """-1: the current plan runs one kernel per op; 0: the persistent window kernel is in use; >0: it trapped."""
        return int(self.lib.fmt_window_kernel_status(self._handle))

    def graph_kernel_nodes(self) -> int:
        return int(self.lib.fmt_graph_kernel_nodes(self._handle))

    def ode_graph_kernel_nodes(self) -> int:
        """Kernels of the per-slot window graph that calls with per-clip schedules run (0 before the first on this plan)."""
        return int(self.lib.fmt_ode_graph_kernel_nodes(self._handle))

    def last_window_slots(self) -> int:
        """Slots of the window graph the last sampling call replayed: :func:`occupancy_slots` of the plan's slots and the streams of
        the last :meth:`sample_windows`, or the plan's slots (0 before the first call)."""
        return int(self.lib.fmt_last_window_slots(self._handle))

    @staticmethod
    def _clip_ode(schedules, n: int):
        """FmtClipOde of n (nfe, method) pairs, and the ctypes arrays it points into (keep them alive for the call)."""
        if len(schedules) != n:
            raise ValueError(f"schedules needs one (nfe, method) per clip ({n}), got {len(schedules)}")
        sched = []
        for nfe, method in schedules:
            if isinstance(nfe, bool) or not isinstance(nfe, numbers.Integral) or nfe < 1:
                raise ValueError(f"nfe must be an int >= 1 (got {nfe!r})")
            sched.append(build_schedule(nfe, method))
        arrays = [[_f32_array(sc[k]) for sc in sched] for k in ("t_eval", "dt", "a", "b")]
        fptr = C.POINTER(C.c_float)
        ode = _cabi.FmtClipOde((C.c_int32 * n)(*[sc["n_steps"] for sc in sched]), (C.c_int32 * n)(*[sc["n_stages"] for sc in sched]),
                               *[(fptr * n)(*[C.cast(x, fptr) for x in arr]) for arr in arrays])
        return ode, arrays

    # ------------------------------------------------------------------------------------------------
    def _check_clip(self, r_s, wa, we, audio_num_frames, noise, host: bool):
        """Every tensor the C call indexes by the plan's dimensions is checked here (the reference would raise a torch shape
        error inside F.linear / torch.cat; the kernels would read out of bounds)."""
        d = self.dims
        if self._plan_key is None:
            raise FmtError("sample_clip: configure() has not been called")
        B = self._plan_key[0]
        want_dev = "cpu" if host else "cuda"
        for name, t in (("r_s", r_s), ("wa", wa), ("we", we), ("noise", noise)):
            if not torch.is_tensor(t):
                raise TypeError(f"{name} must be a torch.Tensor")
            if t.dtype != torch.float32 or not t.is_contiguous():
                raise ValueError(f"{name} must be contiguous float32 (got {t.dtype}, contiguous={t.is_contiguous()})")
            if t.device.type != want_dev or (not host and t.device != self.device):
                raise ValueError(f"{name} is on {t.device}, expected {'the CPU' if host else self.device}")
        if wa.dim() != 3 or wa.shape[0] != B or wa.shape[2] != d.dim_a or wa.shape[1] < 1:
            raise ValueError(f"wa shape {tuple(wa.shape)} != (B={B}, T>=1, dim_a={d.dim_a})")
        if r_s.numel() != B * d.dim_w or r_s.shape[0] != B:
            raise ValueError(f"r_s shape {tuple(r_s.shape)} != (B={B}, dim_w={d.dim_w})")
        if we.dim() != 3 or we.shape[0] != B or we.shape[2] != d.dim_e or we.shape[1] < 1:
            raise ValueError(f"we shape {tuple(we.shape)} != (B={B}, 1 or T, dim_e={d.dim_e})")
        dynamic = self._plan_key[2]
        if dynamic != (we.shape[1] > 1):
            raise ValueError(f"we has {we.shape[1]} frames but the plan was configured with we_dynamic={dynamic}")
        if int(audio_num_frames) < 1:
            raise ValueError(f"audio_num_frames must be >= 1 (got {audio_num_frames})")
        n_win = -(-int(audio_num_frames) // d.frames_per_clip)
        if tuple(noise.shape) != (n_win, B, d.frames_per_clip, d.dim_w):
            raise ValueError(f"noise shape {tuple(noise.shape)} != {(n_win, B, d.frames_per_clip, d.dim_w)}")

    def sample_clip(self, r_s, wa, we, audio_num_frames: int, noise, a_cfg_scale, r_cfg_scale, e_cfg_scale,
                    progress: Optional[Callable[[int, int], None]] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """All windows of one batch of clips.  Tensors on ``self.device`` (fp32, contiguous); asynchronous."""
        d = self.dims
        self._check_clip(r_s, wa, we, audio_num_frames, noise, host=False)
        B = wa.shape[0]
        if out is None:
            out = torch.empty(B, audio_num_frames, d.dim_w, device=self.device, dtype=torch.float32)
        elif tuple(out.shape) != (B, int(audio_num_frames), d.dim_w) or out.dtype != torch.float32 or not out.is_contiguous() or out.device != self.device:
            raise ValueError(f"out must be a contiguous float32 {(B, int(audio_num_frames), d.dim_w)} tensor on {self.device}")
        cb = _cabi.PROGRESS_FN(lambda w, n, _u: progress(w, n)) if progress is not None else _cabi.PROGRESS_FN(0)
        clip = _cabi.FmtClip(_cabi.FMT_LOC_DEVICE, r_s.data_ptr(), wa.data_ptr(), we.data_ptr(), noise.data_ptr(), out.data_ptr(),
                             wa.shape[1], we.shape[1], int(audio_num_frames), float(a_cfg_scale), float(r_cfg_scale),
                             float(e_cfg_scale), cb, None)
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.fmt_sample_clip(self._handle, C.byref(clip), self._stream()), "fmt_sample_clip")
        return out

    def sample_clip_host(self, r_s, wa, we, audio_num_frames: int, noise, a_cfg_scale, r_cfg_scale, e_cfg_scale) -> torch.Tensor:
        """Same with HOST (CPU, fp32, contiguous) tensors in and out; copies happen inside the C call (synchronous)."""
        d = self.dims
        self._check_clip(r_s, wa, we, audio_num_frames, noise, host=True)
        out = torch.empty(wa.shape[0], audio_num_frames, d.dim_w, dtype=torch.float32)
        clip = _cabi.FmtClip(_cabi.FMT_LOC_HOST, r_s.data_ptr(), wa.data_ptr(), we.data_ptr(), noise.data_ptr(), out.data_ptr(),
                             wa.shape[1], we.shape[1], int(audio_num_frames), float(a_cfg_scale), float(r_cfg_scale),
                             float(e_cfg_scale), _cabi.PROGRESS_FN(0), None)
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.fmt_sample_clip(self._handle, C.byref(clip), self._stream()), "fmt_sample_clip")
        return out

    def sample_clips(self, r_s, wa, we, audio_num_frames, noise, a_cfg_scale, r_cfg_scale, e_cfg_scale,
                     progress: Optional[Callable[[int, int], None]] = None, out: Optional[Sequence[torch.Tensor]] = None,
                     n_branches: Optional[Sequence[int]] = None, schedules: Optional[Sequence[tuple]] = None,
                     we_dynamic: Optional[Sequence[bool]] = None) -> List[torch.Tensor]:
        """Many clips of different lengths in one call on the plan's batch of slots (:func:`clip_schedule`).  Per clip i: r_s[i]
        (1, dim_w), wa[i] (1, T_wa, dim_a), we[i] (1, 1 or T_we, dim_e), noise[i] (n_win_i, L, dim_w) or (n_win_i, 1, L, dim_w), all on
        ``self.device`` (fp32, contiguous).  Returns one (1, audio_num_frames[i], dim_w) tensor per clip (``out[i]`` if given: any
        contiguous fp32 tensor of that many elements); asynchronous.

        Each of the three scales is one float for every clip or a sequence of one float per clip.  ``n_branches[i]`` (1, 3 or 4, at
        most the plan's; default: the plan's for every clip) is the branch count of clip i's guidance, :func:`n_branches_for`.
        ``schedules[i]`` = (nfe, method), at most the plan's evaluations per window (:func:`n_evals`), puts clip i on its own ODE
        schedule; given, the call runs the per-slot window graph (``fmt_sample_clips_ode``), one kernel per op, even where every
        schedule is the plan's.  ``we_dynamic[i]`` (default: the plan's for every clip) is clip i's emotion mode, which its ``we``
        must have: static (1 frame) or dynamic (per frame); clips of both modes share the plan's window graphs."""
        d = self.dims
        if self._plan_key is None:
            raise FmtError("sample_clips: configure() has not been called")
        n = len(wa)
        if n < 1 or not all(len(x) == n for x in (r_s, we, audio_num_frames, noise)) or (out is not None and len(out) != n):
            raise ValueError("sample_clips: r_s, wa, we, audio_num_frames, noise (and out) need one entry per clip")
        scales = []
        for name, v in (("a_cfg_scale", a_cfg_scale), ("r_cfg_scale", r_cfg_scale), ("e_cfg_scale", e_cfg_scale)):
            v = [float(x) for x in v] if isinstance(v, Sequence) else [float(v)] * n
            if len(v) != n:
                raise ValueError(f"sample_clips: {name} needs one float, or one per clip ({n}), got {len(v)}")
            scales.append(v)
        nbr = [self._plan_key[1]] * n if n_branches is None else [int(x) for x in n_branches]
        if len(nbr) != n:
            raise ValueError(f"sample_clips: n_branches needs one entry per clip ({n}), got {len(nbr)}")
        modes = [self._plan_key[2]] * n if we_dynamic is None else [bool(x) for x in we_dynamic]
        if len(modes) != n:
            raise ValueError(f"sample_clips: we_dynamic needs one entry per clip ({n}), got {len(modes)}")
        L = d.frames_per_clip
        outs = []
        for i in range(n):
            for name, t in (("r_s", r_s[i]), ("wa", wa[i]), ("we", we[i]), ("noise", noise[i])):
                if not torch.is_tensor(t):
                    raise TypeError(f"clip {i}: {name} must be a torch.Tensor")
                if t.dtype != torch.float32 or not t.is_contiguous() or t.device != self.device:
                    raise ValueError(f"clip {i}: {name} must be a contiguous float32 tensor on {self.device}")
            T = int(audio_num_frames[i])
            n_win = -(-T // L)
            if T < 1:
                raise ValueError(f"clip {i}: audio_num_frames must be >= 1 (got {T})")
            if wa[i].dim() != 3 or wa[i].shape[0] != 1 or wa[i].shape[2] != d.dim_a or (n_win - 1) * L >= wa[i].shape[1]:
                raise ValueError(f"clip {i}: wa shape {tuple(wa[i].shape)} != (1, T > {(n_win - 1) * L}, dim_a={d.dim_a})")
            if r_s[i].shape[0] != 1 or r_s[i].numel() != d.dim_w:
                raise ValueError(f"clip {i}: r_s shape {tuple(r_s[i].shape)} != (1, dim_w={d.dim_w})")
            if we[i].dim() != 3 or we[i].shape[0] != 1 or we[i].shape[2] != d.dim_e or modes[i] != (we[i].shape[1] > 1):
                raise ValueError(f"clip {i}: we shape {tuple(we[i].shape)} does not match (1, {'T' if modes[i] else 1}, dim_e={d.dim_e})")
            if tuple(noise[i].shape) not in ((n_win, L, d.dim_w), (n_win, 1, L, d.dim_w)):
                raise ValueError(f"clip {i}: noise shape {tuple(noise[i].shape)} != {(n_win, L, d.dim_w)}")
            if out is None:
                outs.append(torch.empty(1, T, d.dim_w, device=self.device, dtype=torch.float32))
            else:
                o = out[i]
                if o.numel() != T * d.dim_w or o.dtype != torch.float32 or not o.is_contiguous() or o.device != self.device:
                    raise ValueError(f"clip {i}: out must be a contiguous float32 tensor of {T} x {d.dim_w} elements on {self.device}")
                outs.append(o)

        def ptrs(ts):
            return (C.c_void_p * n)(*[t.data_ptr() for t in ts])

        def ints(vals):
            return (C.c_int32 * n)(*[int(v) for v in vals])

        def floats(vals):
            return (C.c_float * n)(*vals)

        cb = _cabi.PROGRESS_FN(lambda w, m, _u: progress(w, m)) if progress is not None else _cabi.PROGRESS_FN(0)
        cs = _cabi.FmtClipSet(n, ptrs(r_s), ptrs(wa), ptrs(we), ptrs(noise), ptrs(outs), ints(t.shape[1] for t in wa),
                              ints(t.shape[1] for t in we), ints(audio_num_frames), 1.0, 1.0, 1.0, cb, None)
        g = _cabi.FmtClipGuidance(floats(scales[0]), floats(scales[1]), floats(scales[2]), ints(nbr))
        ode, _keep = self._clip_ode(schedules, n) if schedules is not None else (None, None)
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.fmt_sample_clip_set(self._handle, C.byref(cs), C.byref(g), None if ode is None else C.byref(ode),
                                                     None if we_dynamic is None else ints(modes), self._stream()), "fmt_sample_clip_set")
        return outs

    def sample_windows(self, r_s, wa, we, x0, ctx, out, first_window, a_cfg_scale, r_cfg_scale, e_cfg_scale, n_branches,
                       schedules: Optional[Sequence[tuple]] = None, we_dynamic: Optional[Sequence[bool]] = None) -> None:
        """One window of each of n <= plan batch streams (``fmt_sample_windows``), stream i in slot i.  Per stream i: r_s[i]
        (1, dim_w); wa[i] (T_wa, dim_a) and, dynamic, we[i] (T_we, dim_e) from the window's first context frame (frame 0 in a first
        window), static we[i] (1, 1, dim_e); x0[i] (L, dim_w); ctx[i] (P, dim_w), read unless ``first_window[i]`` and overwritten
        with the window's last P frames; out[i] receives the window's first ``out[i].shape[-2]`` frames.  Scales and n_branches are
        one entry per stream; ``schedules`` (one (nfe, method) per stream) and ``we_dynamic`` (one emotion mode per stream, which
        decides the layout of we[i]) as in :meth:`sample_clips`.  All tensors on ``self.device`` (fp32, contiguous); asynchronous."""
        d = self.dims
        if self._plan_key is None:
            raise FmtError("sample_windows: configure() has not been called")
        n = len(wa)
        groups = (r_s, we, x0, ctx, out, first_window, a_cfg_scale, r_cfg_scale, e_cfg_scale, n_branches)
        if we_dynamic is not None:
            groups += (we_dynamic,)
        if not 1 <= n <= self._plan_key[0] or not all(len(x) == n for x in groups):
            raise ValueError(f"sample_windows: 1 to {self._plan_key[0]} streams, with one entry per stream in every argument")
        for i in range(n):
            for name, t in (("r_s", r_s[i]), ("wa", wa[i]), ("we", we[i]), ("x0", x0[i]), ("ctx", ctx[i]), ("out", out[i])):
                if not torch.is_tensor(t) or t.dtype != torch.float32 or not t.is_contiguous() or t.device != self.device:
                    raise ValueError(f"stream {i}: {name} must be a contiguous float32 tensor on {self.device}")
            if x0[i].numel() != d.frames_per_clip * d.dim_w or ctx[i].numel() != d.num_prev_frames * d.dim_w or r_s[i].numel() != d.dim_w:
                raise ValueError(f"stream {i}: r_s, x0 or ctx does not hold (dim_w), (L, dim_w) or (P, dim_w) elements")
            if wa[i].numel() % d.dim_a or we[i].numel() % d.dim_e or out[i].numel() % d.dim_w:
                raise ValueError(f"stream {i}: wa, we or out is not a whole number of frames")

        def ptrs(ts):
            return (C.c_void_p * n)(*[t.data_ptr() for t in ts])

        def ints(vals):
            return (C.c_int32 * n)(*[int(v) for v in vals])

        ws = _cabi.FmtWindowSet(n, ptrs(r_s), ptrs(wa), ptrs(we), ptrs(x0), ptrs(ctx), ptrs(out), ints(t.numel() // d.dim_a for t in wa),
                                ints(t.numel() // d.dim_e for t in we), ints(t.numel() // d.dim_w for t in out), ints(first_window))
        g = _cabi.FmtClipGuidance(*[(C.c_float * n)(*[float(x) for x in v]) for v in (a_cfg_scale, r_cfg_scale, e_cfg_scale)],
                                  ints(n_branches))
        ode, _keep = self._clip_ode(schedules, n) if schedules is not None else (None, None)
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.fmt_sample_window_set(self._handle, C.byref(ws), C.byref(g), None if ode is None else C.byref(ode),
                                                       None if we_dynamic is None else ints(we_dynamic), self._stream()),
                        "fmt_sample_window_set")

    def velocity(self, eval_index: int, x, wa, r_s, we, prev_x, prev_wa, prev_we, a_cfg_scale, r_cfg_scale, e_cfg_scale) -> torch.Tensor:
        """One ``forward_with_cfv`` (FMT.py:342-401) at plan time ``t_eval[eval_index]``; returns (B, P+L, dim_w)."""
        d = self.dims
        if self._plan_key is None:
            raise FmtError("velocity: configure() has not been called")
        B, L, P = self._plan_key[0], d.frames_per_clip, d.num_prev_frames
        dyn = self._plan_key[2]
        expect = {"x": (B, L, d.dim_w), "wa": (B, L, d.dim_a), "prev_x": (B, P, d.dim_w), "prev_wa": (B, P, d.dim_a),
                  "we": (B, L if dyn else 1, d.dim_e)}
        if dyn:
            if prev_we is None:
                raise ValueError("`we` is dynamic (T>1), but prev_we was not provided with prev_x/prev_wa.")     # FMT.py:304-307
            expect["prev_we"] = (B, P, d.dim_e)
        got = {"x": x, "wa": wa, "prev_x": prev_x, "prev_wa": prev_wa, "we": we, "prev_we": prev_we}
        for name, shp in expect.items():
            t = got[name]
            if not torch.is_tensor(t) or tuple(t.shape) != shp or t.dtype != torch.float32 or not t.is_contiguous() or t.device != self.device:
                raise ValueError(f"{name}: expected a contiguous float32 {shp} tensor on {self.device}, got "
                                 f"{tuple(t.shape) if torch.is_tensor(t) else type(t)}")
        if not torch.is_tensor(r_s) or r_s.numel() != B * d.dim_w or r_s.dtype != torch.float32 or not r_s.is_contiguous() or r_s.device != self.device:
            raise ValueError(f"r_s: expected a contiguous float32 (B={B}, dim_w={d.dim_w}) tensor on {self.device}")
        if not 0 <= int(eval_index) < max(1, self._n_eval):
            raise ValueError(f"eval_index {eval_index} outside the plan's {self._n_eval} evaluations")
        v = torch.empty(x.shape[0], d.num_prev_frames + d.frames_per_clip, d.dim_w, device=self.device, dtype=torch.float32)
        ev = _cabi.FmtEval(x.data_ptr(), prev_x.data_ptr(), wa.data_ptr(), prev_wa.data_ptr(), we.data_ptr(),
                           prev_we.data_ptr() if prev_we is not None else None, r_s.data_ptr(), v.data_ptr(), int(eval_index),
                           float(a_cfg_scale), float(r_cfg_scale), float(e_cfg_scale))
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.fmt_velocity(self._handle, C.byref(ev), self._stream()), "fmt_velocity")
        return v


# ----------------------------------------------------------------------------------------------------
# backend cache: one packed copy per (FMT module, device); rebuilt when the module's weights change
# ----------------------------------------------------------------------------------------------------
_BACKENDS: "weakref.WeakKeyDictionary" = weakref.WeakKeyDictionary()


def _weights_fingerprint(sd) -> tuple:
    return tuple((k, v.data_ptr(), getattr(v, "_version", 0), tuple(v.shape)) for k, v in sd.items() if torch.is_tensor(v))


def _model_dims(fmt_model, sd) -> Dims:
    src = getattr(fmt_model, "final_construction_options", None) or getattr(fmt_model, "opt", None) or {}
    return Dims.from_options(src, sd)


def backend_for(fmt_model, device, dims: Optional[Dims] = None) -> FmtBackend:
    """``fmt_model``: anything with ``state_dict()`` (the reference ``FlowMatchingTransformer`` or :class:`FmtModel`)."""
    device = torch.device(device)
    if device.type != "cuda":
        raise FmtError(f"float_fmt_model.target_device is '{device}': the B200 FMT sampler runs on CUDA (sm_100a) only; "
                       "there is no CPU fallback.")
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    sd = fmt_model.state_dict()
    fp = _weights_fingerprint(sd)
    per_model = _BACKENDS.setdefault(fmt_model, {})
    hit = per_model.get(device)
    if hit is not None and hit[0] == fp:
        return hit[1]
    if dims is None:
        dims = _model_dims(fmt_model, sd)
    if hit is not None:
        hit[1].close()
    be = FmtBackend(sd, dims, device)
    per_model[device] = (fp, be)
    return be


def _as_f32(t: torch.Tensor, device) -> torch.Tensor:
    return t.to(device=device, dtype=torch.float32).contiguous()


def draw_window_noise(batch: int, dims: Dims, n_windows: int, device, generator: Optional[torch.Generator]) -> torch.Tensor:
    """One ``torch.randn(B, L, dim_w)`` per window, in window order, on ``device`` (nodes_adv.py:606)."""
    gen_dev = generator.device if generator is not None else torch.device(device)
    chunks = [torch.randn(batch, dims.frames_per_clip, dims.dim_w, device=gen_dev, generator=generator) for _ in range(n_windows)]
    if not chunks:
        return torch.empty(0, batch, dims.frames_per_clip, dims.dim_w, device=device)
    return torch.stack(chunks, dim=0).to(device)


def perform_ode_sampling_loop(fmt_model, r_s_latent_dev, wa_latent_dev, we_latent_dev, audio_num_frames,
                              model_num_prev_frames, model_num_frames_for_clip, model_dim_w,
                              ode_nfe, ode_method, ode_atol, ode_rtol, target_device,
                              a_cfg_scale, r_cfg_scale, e_cfg_scale, include_r_cfg, noise_seed_generator,
                              progress_bar=None, mode: Optional[str] = None, noise: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Drop-in for ``_perform_ode_sampling_loop`` (nodes_adv.py:545-694): same arguments, returns r_d on ``target_device``.

    ``ode_atol`` / ``ode_rtol`` are accepted and ignored, as torchdiffeq's fixed-grid solvers ignore them.
    ``noise`` (n_windows, B, L, dim_w) optionally injects the per-window x0 instead of drawing it.
    """
    device = torch.device(target_device)
    be = backend_for(fmt_model, device)
    d = be.dims
    if (d.num_prev_frames, d.frames_per_clip, d.dim_w) != (int(model_num_prev_frames), int(model_num_frames_for_clip), int(model_dim_w)):
        raise ValueError(f"window geometry (prev={model_num_prev_frames}, clip={model_num_frames_for_clip}, dim_w={model_dim_w}) "
                         f"does not match the FMT weights ({d.num_prev_frames}, {d.frames_per_clip}, {d.dim_w})")
    mode = resolve_mode(mode)
    # the shape errors the reference raises from inside torch (F.linear on cat[wr, wa, we], FMT.py:327-335) - raised here, before
    # any pointer reaches the kernels
    if wa_latent_dev.dim() != 3 or wa_latent_dev.shape[2] != d.dim_a:
        raise ValueError(f"wa_latent shape {tuple(wa_latent_dev.shape)}: expected (B, T, {d.dim_a}) - e.g. project the wav2vec features first")
    B = wa_latent_dev.shape[0]
    if we_latent_dev.dim() != 3 or we_latent_dev.shape[0] != B or we_latent_dev.shape[2] != d.dim_e:
        raise ValueError(f"we_latent shape {tuple(we_latent_dev.shape)}: expected ({B}, 1 or T, {d.dim_e})")
    if r_s_latent_dev.shape[0] != B or r_s_latent_dev.numel() != B * d.dim_w:
        raise ValueError(f"r_s_latent shape {tuple(r_s_latent_dev.shape)}: expected ({B}, {d.dim_w})")
    if int(audio_num_frames) < 1:
        raise ValueError(f"audio_num_frames must be >= 1 (got {audio_num_frames})")
    dynamic = we_latent_dev.shape[1] > 1
    nb = n_branches_for(a_cfg_scale, r_cfg_scale, e_cfg_scale, include_r_cfg)
    n_win = math.ceil(audio_num_frames / d.frames_per_clip)
    be.configure(B, nb, dynamic, ode_nfe, ode_method, mode)
    r_s, wa, we = _as_f32(r_s_latent_dev, be.device), _as_f32(wa_latent_dev, be.device), _as_f32(we_latent_dev, be.device)
    if noise is None:
        noise = draw_window_noise(B, d, n_win, be.device, noise_seed_generator)
    noise = _as_f32(noise, be.device)
    if noise.shape != (n_win, B, d.frames_per_clip, d.dim_w):
        raise ValueError(f"noise shape {tuple(noise.shape)} != {(n_win, B, d.frames_per_clip, d.dim_w)}")
    progress = (lambda w, n: progress_bar.update(1)) if progress_bar is not None else None
    return be.sample_clip(r_s, wa, we, int(audio_num_frames), noise, a_cfg_scale, r_cfg_scale, e_cfg_scale, progress)


# ----------------------------------------------------------------------------------------------------
# many clips of different lengths in one call: B slots, refilled as clips finish
# ----------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class ClipSchedule:
    slots: int             # S: the plan's batch
    slot: tuple            # slot of every clip, in input order
    start: tuple           # window of the call in which every clip starts (its own window 0)
    makespan: int          # windows the call runs


def clip_schedule(n_windows: Sequence[int], n_slots: int = 0) -> ClipSchedule:
    """Slot schedule of :func:`sample_clips` for clips of ``n_windows[i]`` windows, computed by the library
    (``fmt_clip_schedule``, host-only).  ``n_slots = 0``: the fewest slots (<= 256) that still finish with the longest clip."""
    lib = _cabi.load_library()
    n = len(n_windows)
    nw = (C.c_int32 * max(1, n))(*[int(x) for x in n_windows])
    slot, start, makespan = (C.c_int32 * max(1, n))(), (C.c_int32 * max(1, n))(), C.c_int32()
    S = lib.fmt_clip_schedule(n, nw, int(n_slots), slot, start, C.byref(makespan))
    if S < 0:
        raise ValueError(f"fmt_clip_schedule: bad arguments (n_clips={n}, n_slots={n_slots}, every clip needs >= 1 window)")
    return ClipSchedule(S, tuple(slot[:n]), tuple(start[:n]), makespan.value)


def occupancy_slots(slots: int, n_ready: int) -> int:
    """Slots of the window graph a :class:`StreamSampler` step with ``n_ready`` ready streams runs on a sampler of ``slots`` slots: the
    smallest of 1, 2, 4, ... (the powers of two below ``slots``) and ``slots`` that is >= ``n_ready`` (``fmt_occupancy_slots``,
    host-only).  Raises ValueError unless 1 <= n_ready <= slots <= 256."""
    for name, v in (("slots", slots), ("n_ready", n_ready)):
        if isinstance(v, bool) or not isinstance(v, numbers.Integral):
            raise ValueError(f"{name} must be an int (got {v!r})")
    k = _cabi.load_library().fmt_occupancy_slots(int(slots), int(n_ready))
    if k < 0:
        raise ValueError(f"occupancy_slots: need 1 <= n_ready <= slots <= 256 (got slots={slots}, n_ready={n_ready})")
    return k


def clip_noise(seed: int, dims: Dims, n_windows: int, device) -> torch.Tensor:
    """(n_windows, 1, L, dim_w): the x0 of every window of one clip drawn from its own seed - what the VA node draws for a batch of
    one clip with ``fix_noise_seed`` (a ``torch.Generator`` on the target device, nodes_vadv.py:673-689)."""
    return draw_window_noise(1, dims, n_windows, device, torch.Generator(torch.device(device)).manual_seed(int(seed)))


def _own_guidance(who: str, c: Mapping, a_cfg_scale, r_cfg_scale, e_cfg_scale, include_r_cfg) -> tuple:
    """(a, r, e, n_branches) of one clip or stream: each of its own guidance keys overrides the call's keyword of that name."""
    for k in ("a_cfg_scale", "r_cfg_scale", "e_cfg_scale"):
        if k in c:
            v = c[k]
            if not isinstance(v, numbers.Real) or isinstance(v, bool):
                raise TypeError(f"{who}: {k} must be a number, got {type(v).__name__}")
            if not math.isfinite(v):
                raise ValueError(f"{who}: {k} must be finite (got {v})")
    if "include_r_cfg" in c and not isinstance(c["include_r_cfg"], bool):
        raise TypeError(f"{who}: include_r_cfg must be a bool, got {type(c['include_r_cfg']).__name__}")
    g = tuple(c.get(k, dflt) for k, dflt in (("a_cfg_scale", a_cfg_scale), ("r_cfg_scale", r_cfg_scale), ("e_cfg_scale", e_cfg_scale)))
    return g + (n_branches_for(*g, c.get("include_r_cfg", include_r_cfg)),)


def _own_schedule(who: str, c: Mapping, nfe, method) -> tuple:
    """(nfe, method) of one clip or stream: each of its own keys overrides the call's keyword of that name."""
    if "nfe" in c:
        v = c["nfe"]
        if isinstance(v, bool) or not isinstance(v, numbers.Integral):
            raise TypeError(f"{who}: nfe must be an int, got {type(v).__name__}")
        if v < 1:
            raise ValueError(f"{who}: nfe must be >= 1 (got {v})")
    if "method" in c and (not isinstance(c["method"], str) or c["method"] not in SOLVERS):
        raise ValueError(f"{who}: unknown fixed-step solver {c['method']!r} (supported: {sorted(SOLVERS)})")
    return int(c.get("nfe", nfe)), c.get("method", method)


def sample_clips(fmt_model, clips: Sequence[Mapping], *, nfe: int, method: str = "euler", a_cfg_scale: float = 2.0,
                 r_cfg_scale: float = 1.0, e_cfg_scale: float = 1.0, include_r_cfg: bool = False, mode: Optional[str] = None,
                 we_dynamic: Optional[bool] = None, device=None, progress: Optional[Callable[[int, int], None]] = None) -> List[torch.Tensor]:
    """Many independent clips of different lengths in one call.  Each clip is a mapping with ``r_s`` (1, dim_w), ``wa``
    (1, T_wa, dim_a), ``we`` (1, 1 or T_we, dim_e), optionally ``audio_num_frames`` (default T_wa) and either ``seed`` (its noise is
    :func:`clip_noise`) or ``noise`` (n_win, L, dim_w).  A clip may also hold ``a_cfg_scale``, ``r_cfg_scale``, ``e_cfg_scale``,
    ``include_r_cfg``, ``nfe``, ``method`` and ``we_dynamic``: each overrides the keyword of the same name for that clip.  A clip's
    emotion mode (``we_dynamic``: static, ``we`` of 1 frame, or dynamic, one frame per audio frame) must match its ``we``; with the
    keyword left at None, the clips that do not declare one take the mode of their ``we`` and must all have the same.  Clips of both
    modes share the call's slots and window graphs.  Precision is shared.  The plan runs as many CFG branches as the clip that needs the most (:func:`n_branches_for`); a clip
    that needs fewer combines only its own branches.  Likewise it runs the evaluations per window of the clip that needs the most
    (:func:`n_evals`, :func:`plan_schedule`); a clip that needs fewer runs its own and then idles, and a call whose clips do not all
    run the plan's schedule goes through the per-slot window graph (one kernel per op).  Clip i's result is what
    :func:`perform_ode_sampling_loop` gives for it alone with its settings and noise.  Returns one (1, T_i, dim_w) tensor per clip, in input order, on ``device`` (default: the
    model's ``target_device``).  ``progress(w, makespan)`` is called after each window of the schedule is enqueued."""
    # every check runs before the first device call (the weights are packed only once the clips are known to be valid)
    if not isinstance(clips, (list, tuple)):
        raise TypeError(f"clips must be a list of mappings, got {type(clips).__name__}")
    if not clips:
        raise ValueError("clips is empty")
    d = _model_dims(fmt_model, fmt_model.state_dict())
    L = d.frames_per_clip
    build_schedule(nfe, method)                        # unknown solver -> ValueError
    if int(nfe) < 1:
        raise ValueError(f"nfe must be >= 1 (got {nfe})")
    if we_dynamic is not None and not isinstance(we_dynamic, bool):
        raise TypeError(f"we_dynamic must be a bool or None, got {type(we_dynamic).__name__}")
    mode = resolve_mode(mode)
    T, n_win, dyn, guidance, schedules = [], [], [], [], []
    inferred = set()                                   # modes of the clips that take theirs from the shape of their we      # guidance: (a, r, e, n_branches) of every clip
    for i, c in enumerate(clips):
        if not isinstance(c, Mapping):
            raise TypeError(f"clip {i} must be a mapping (r_s, wa, we, seed or noise), got {type(c).__name__}")
        r_s, wa, we = c.get("r_s"), c.get("wa"), c.get("we")
        if not all(torch.is_tensor(t) for t in (r_s, wa, we)):
            raise TypeError(f"clip {i}: r_s, wa and we must be torch.Tensors")
        if wa.dim() != 3 or we.dim() != 3 or wa.shape[0] != 1 or we.shape[0] != 1 or r_s.shape[0] != 1:
            raise ValueError(f"clip {i}: batch dimension must be 1 (r_s {tuple(r_s.shape)}, wa {tuple(wa.shape)}, we {tuple(we.shape)}); "
                             "a batch of equal-length clips is one clip per entry here")
        if wa.shape[2] != d.dim_a or wa.shape[1] < 1:
            raise ValueError(f"clip {i}: wa shape {tuple(wa.shape)}: expected (1, T, {d.dim_a})")
        if we.shape[2] != d.dim_e or we.shape[1] < 1:
            raise ValueError(f"clip {i}: we shape {tuple(we.shape)}: expected (1, 1 or T, {d.dim_e})")
        if r_s.numel() != d.dim_w:
            raise ValueError(f"clip {i}: r_s shape {tuple(r_s.shape)}: expected (1, {d.dim_w})")
        t = int(c.get("audio_num_frames", wa.shape[1]))
        if t < 1:
            raise ValueError(f"clip {i}: audio_num_frames must be >= 1 (got {t})")
        nw = -(-t // L)
        dynamic = c.get("we_dynamic", we_dynamic)
        if dynamic is None:
            dynamic = we.shape[1] > 1
            inferred.add(dynamic)
        elif not isinstance(dynamic, bool):
            raise TypeError(f"clip {i}: we_dynamic must be a bool, got {type(dynamic).__name__}")
        elif dynamic != (we.shape[1] > 1):
            raise ValueError(f"clip {i}: we_dynamic={dynamic}, but we has {we.shape[1]} frame(s) "
                             f"({'more than one' if dynamic else 'one'} expected)")
        # the reference's F.pad(replicate) needs at least one real frame in every window (nodes_adv.py:614-616)
        if (nw - 1) * L >= wa.shape[1]:
            raise ValueError(f"clip {i}: wa has {wa.shape[1]} frames, but window {nw - 1} of its {t} frames starts at frame {(nw - 1) * L}")
        if dynamic and (nw - 1) * L >= we.shape[1]:
            raise ValueError(f"clip {i}: dynamic we has {we.shape[1]} frames, but window {nw - 1} starts at frame {(nw - 1) * L}")
        has_seed, has_noise = c.get("seed") is not None, c.get("noise") is not None
        if has_seed == has_noise:
            raise ValueError(f"clip {i}: give exactly one of 'seed' and 'noise'")
        if has_noise:
            nz = c["noise"]
            if not torch.is_tensor(nz):
                raise TypeError(f"clip {i}: noise must be a torch.Tensor")
            if tuple(nz.shape) not in ((nw, L, d.dim_w), (nw, 1, L, d.dim_w)):
                raise ValueError(f"clip {i}: noise shape {tuple(nz.shape)} != {(nw, L, d.dim_w)}")
        guidance.append(_own_guidance(f"clip {i}", c, a_cfg_scale, r_cfg_scale, e_cfg_scale, include_r_cfg))
        schedules.append(_own_schedule(f"clip {i}", c, nfe, method))
        T.append(t)
        n_win.append(nw)
        dyn.append(dynamic)
    if len(inferred) > 1:
        raise ValueError("clips mix static (1-frame) and dynamic (per-frame) emotion we; give the clips of one mode we_dynamic "
                         "(or the call the keyword) to sample both in one call")

    if device is None:
        device = getattr(fmt_model, "target_device", None) or "cuda"
    be = backend_for(fmt_model, device, d)
    sched = clip_schedule(n_win)
    a, r, e, nb = zip(*guidance)
    plan = plan_schedule(schedules, nfe, method)
    be.configure(sched.slots, max(nb), dyn[0], *plan, mode)
    dev = be.device
    noise = [_as_f32(c["noise"], dev) if c.get("noise") is not None else clip_noise(c["seed"], d, nw, dev)
             for c, nw in zip(clips, n_win)]
    # the plan's schedule for every clip: the plan's window graph, as without per-clip schedules
    own = {} if all(sc == plan for sc in schedules) else dict(schedules=schedules)
    if any(x != dyn[0] for x in dyn):                  # the plan's emotion mode is clip 0's; the others say theirs only when they differ
        own["we_dynamic"] = dyn
    return be.sample_clips([_as_f32(c["r_s"], dev) for c in clips], [_as_f32(c["wa"], dev) for c in clips],
                           [_as_f32(c["we"], dev) for c in clips], T, noise, a, r, e, progress, n_branches=nb, **own)


# ----------------------------------------------------------------------------------------------------
# streams: clips fed audio in pieces, one window per step on a fixed set of batch slots
# ----------------------------------------------------------------------------------------------------
_GUIDANCE_KEYS = ("a_cfg_scale", "r_cfg_scale", "e_cfg_scale", "include_r_cfg")
_SCHEDULE_KEYS = ("nfe", "method")


class Stream:
    """One clip of a :class:`StreamSampler`, opened by :meth:`StreamSampler.open`.  ``fed`` frames have arrived, ``windows_run``
    windows have been sampled; ``finished`` once :meth:`StreamSampler.finish` was called, ``done`` once its last window ran."""

    def __init__(self, index, L, r_s, we, ctx, wa, we_buf, gen, noise, guidance, schedule, we_dynamic):
        self.index = index                  # open order: breaks ties between windows that became ready at the same tick
        self.L = L
        self.we_dynamic = we_dynamic        # True: we arrives with feed(), one frame per audio frame (we_buf); False: we, from open()
        self.r_s, self.we, self.ctx = r_s, we, ctx
        self.wa, self.we_buf = wa, we_buf   # frames [base, fed): from the next window's first context frame on
        self.base = 0
        self.fed = 0
        self.windows_run = 0
        self.finished = False
        self.ready_at = None                # sampler clock when the next window became ready; None while it is not
        self.gen, self.noise, self.guidance = gen, noise, guidance
        self.schedule = schedule            # (nfe, method)

    @property
    def done(self) -> bool:
        return self.finished and self.windows_run * self.L >= self.fed

    @property
    def buffered_frames(self) -> int:
        """Frames of wa this stream holds on the device."""
        return self.wa.untyped_storage().nbytes() // (self.wa.element_size() * self.wa.shape[1]) if self.wa is not None else 0


class StreamSampler:
    """Clips whose audio arrives in pieces, sampled one window at a time on ``slots`` shared batch slots.

    :meth:`open` starts a stream, :meth:`feed` appends its audio latents, :meth:`finish` ends its audio and :meth:`step` runs one
    window for each of up to ``slots`` streams whose next window is ready: its L frames have arrived, or the stream is finished and
    the window holds its last frames.  The window that has been ready longest goes first (a feed, finish or step that makes
    several windows ready makes them ready at once); ties go in open order.  A stream's frames
    are what :func:`sample_clips` gives for the whole clip (same noise, same guidance, same plan), however the audio was cut.

    The plan (slot count, nfe, solver, precision, and the branch count of the keyword guidance) is fixed at construction.  A step
    with k ready streams runs them in slots 0..k-1 of a window graph captured for :func:`occupancy_slots` ``(slots, k)`` slots - the
    smallest power of two >= k, or ``slots`` - the first time a step needs that graph, so it costs about what a sampler of that many
    slots costs; its idle slots run on zeros.  A stream's frames are the same bits at every occupancy.  Plans whose window graph is
    the persistent window kernel (at most 256 token rows) run their one graph of ``slots`` slots.  A stream may override the four guidance keywords in :meth:`open` as a clip of
    :func:`sample_clips` does, within the plan's branch count, ``we_dynamic`` (static or dynamic emotion) freely, and ``nfe`` and ``method`` within the plan's
    evaluations per window (:func:`n_evals` of the constructor's nfe and method); a step that runs a stream on a schedule other
    than the plan's goes through the per-slot window graph (one kernel per op).  A stream holds on the device its reference latent,
    its last P motion frames and the audio frames from its next window's first context frame on, however long it runs."""

    def __init__(self, fmt_model, *, slots: int, nfe: int, method: str = "euler", mode: Optional[str] = None, a_cfg_scale: float = 2.0,
                 r_cfg_scale: float = 1.0, e_cfg_scale: float = 1.0, include_r_cfg: bool = False, we_dynamic: bool = False, device=None):
        if isinstance(slots, bool) or not isinstance(slots, numbers.Integral) or not 1 <= slots <= 256:
            raise ValueError(f"slots must be an int in [1, 256] (got {slots!r})")
        build_schedule(nfe, method)                        # unknown solver -> ValueError
        if int(nfe) < 1:
            raise ValueError(f"nfe must be >= 1 (got {nfe})")
        if not isinstance(we_dynamic, bool):
            raise TypeError(f"we_dynamic must be a bool, got {type(we_dynamic).__name__}")
        self._mode = resolve_mode(mode)
        self._keywords = (a_cfg_scale, r_cfg_scale, e_cfg_scale, include_r_cfg)
        # CFG branches of the plan: those of the keyword guidance
        self.n_branches = _own_guidance("StreamSampler", dict(zip(_GUIDANCE_KEYS, self._keywords)), *self._keywords)[3]
        self.dims = _model_dims(fmt_model, fmt_model.state_dict())
        if device is None:
            device = getattr(fmt_model, "target_device", None) or "cuda"
        self.slots, self.nfe, self.method, self.we_dynamic = int(slots), int(nfe), method, we_dynamic
        self.capacity = n_evals(nfe, method)               # evaluations per window a stream may need
        self._be = backend_for(fmt_model, device, self.dims)
        self.device = self._be.device
        self._configure()
        self._streams: List[Stream] = []
        self._opened = 0
        self._clock = 0                                    # ticks once per feed(), finish() and step()

    def _configure(self):
        self._be.configure(self.slots, self.n_branches, self.we_dynamic, self.nfe, self.method, self._mode)

    def _check_tensor(self, who, name, t, shape):
        if not torch.is_tensor(t):
            raise TypeError(f"{who}: {name} must be a torch.Tensor")
        if not t.is_floating_point():
            raise TypeError(f"{who}: {name} must be a floating-point tensor (got {t.dtype})")
        if t.dim() != len(shape) or any(want is not None and got != want for got, want in zip(t.shape, shape)):
            raise ValueError(f"{who}: {name} shape {tuple(t.shape)} != {tuple('T' if x is None else x for x in shape)}")

    def _own(self, stream) -> Stream:
        if not isinstance(stream, Stream) or stream not in self._streams:
            raise ValueError("not an open stream of this sampler")
        return stream

    def open(self, r_s, we=None, seed: Optional[int] = None, noise: Optional[torch.Tensor] = None, we_dynamic: Optional[bool] = None,
             **guidance) -> Stream:
        """A new stream with reference latent ``r_s`` (1, dim_w) and, for static emotion, ``we`` (1, 1, dim_e) (dynamic emotion
        arrives with :meth:`feed`).  ``we_dynamic`` (default: the sampler's) is the stream's emotion mode.  Its noise is :func:`clip_noise` of ``seed``, drawn one window at a time, or ``noise``
        (n_win, L, dim_w) for a clip of exactly n_win windows.  ``guidance`` may hold ``a_cfg_scale``, ``r_cfg_scale``,
        ``e_cfg_scale``, ``include_r_cfg``, ``nfe`` and ``method``, each overriding the sampler's keyword for this stream."""
        d, L = self.dims, self.dims.frames_per_clip
        unknown = sorted(set(guidance) - set(_GUIDANCE_KEYS) - set(_SCHEDULE_KEYS))
        if unknown:
            raise TypeError(f"open: unexpected keyword(s) {unknown}")
        self._check_tensor("open", "r_s", r_s, (1, d.dim_w))
        if we_dynamic is None:
            we_dynamic = self.we_dynamic
        elif not isinstance(we_dynamic, bool):
            raise TypeError(f"open: we_dynamic must be a bool, got {type(we_dynamic).__name__}")
        if we_dynamic:
            if we is not None:
                raise ValueError("open: this stream has dynamic emotion: we arrives with feed(), one frame per audio frame")
        else:
            if we is None:
                raise ValueError("open: this stream has static emotion: give we (1, 1, dim_e) here")
            self._check_tensor("open", "we", we, (1, 1, d.dim_e))
        if (seed is None) == (noise is None):
            raise ValueError("open: give exactly one of 'seed' and 'noise'")
        if noise is not None:
            self._check_tensor("open", "noise", noise, (None, L, d.dim_w) if torch.is_tensor(noise) and noise.dim() == 3 else (None, 1, L, d.dim_w))
            if noise.shape[0] < 1:
                raise ValueError("open: noise holds no window")
        g = _own_guidance("open", guidance, *self._keywords)
        if g[3] > self.n_branches:
            raise ValueError(f"open: this stream's guidance needs {g[3]} CFG branches, the sampler's plan runs {self.n_branches} "
                             "(construct it with the guidance of the stream that needs the most)")
        sc = _own_schedule("open", guidance, self.nfe, self.method)
        if n_evals(*sc) > self.capacity:
            raise ValueError(f"open: nfe={sc[0]} with {sc[1]} needs {n_evals(*sc)} evaluations per window, the sampler's plan runs "
                             f"{self.capacity} (construct it with the nfe and method of the stream that needs the most)")
        dev = self.device
        gen = torch.Generator(dev).manual_seed(int(seed)) if seed is not None else None
        st = Stream(self._opened, L, _as_f32(r_s, dev).clone(), None if we is None else _as_f32(we, dev).clone(),
                    torch.zeros(d.num_prev_frames, d.dim_w, device=dev), torch.empty(0, d.dim_a, device=dev),
                    torch.empty(0, d.dim_e, device=dev) if we_dynamic else None, gen,
                    None if noise is None else noise.reshape(noise.shape[0], L, d.dim_w), g, sc, we_dynamic)
        self._opened += 1
        self._streams.append(st)
        return st

    def feed(self, stream: Stream, wa, we=None) -> None:
        """Appends audio latents ``wa`` (1, t, dim_a), t >= 1, and, to a stream with dynamic emotion, as many ``we`` frames
        (1, t, dim_e)."""
        st, d = self._own(stream), self.dims
        if st.finished:
            raise ValueError("feed: the stream is finished")
        self._check_tensor("feed", "wa", wa, (1, None, d.dim_a))
        t = wa.shape[1]
        if t < 1:
            raise ValueError("feed: wa holds no frame")
        if st.we_dynamic:
            if we is None:
                raise ValueError("feed: this stream has dynamic emotion: give we (1, t, dim_e) with every wa")
            self._check_tensor("feed", "we", we, (1, t, d.dim_e))
        elif we is not None:
            raise ValueError("feed: this stream has static emotion, given to open(); feed takes wa only")
        if st.noise is not None and -(-(st.fed + t) // d.frames_per_clip) > st.noise.shape[0]:
            raise ValueError(f"feed: {st.fed + t} frames need more windows than the stream's {st.noise.shape[0]} windows of noise")
        st.wa = torch.cat([st.wa, wa[0].to(device=self.device, dtype=torch.float32)])
        if st.we_dynamic:
            st.we_buf = torch.cat([st.we_buf, we[0].to(device=self.device, dtype=torch.float32)])
        st.fed += t
        self._clock += 1
        self._refresh(st)

    def finish(self, stream: Stream) -> None:
        """No more audio comes for this stream: its clip has as many frames as were fed."""
        st, L = self._own(stream), self.dims.frames_per_clip
        if st.finished:
            raise ValueError("finish: the stream is already finished")
        if st.fed < 1:
            raise ValueError("finish: no audio was fed to the stream")
        if st.noise is not None and st.noise.shape[0] != -(-st.fed // L):
            raise ValueError(f"finish: {st.fed} frames are {-(-st.fed // L)} windows, but the stream's noise holds {st.noise.shape[0]}")
        st.finished = True
        self._clock += 1
        self._refresh(st)

    def close(self, stream: Stream) -> None:
        """Forgets the stream and frees its buffers, whether or not all its windows ran."""
        st = self._own(stream)
        self._streams.remove(st)
        st.wa = st.we_buf = st.ctx = st.r_s = st.we = st.gen = st.noise = None
        st.ready_at = None

    def _ready(self, st: Stream) -> bool:
        L, w = self.dims.frames_per_clip, st.windows_run
        return st.fed >= (w + 1) * L or (st.finished and w * L < st.fed)

    def _refresh(self, st: Stream):
        if st.ready_at is None and self._ready(st):
            st.ready_at = self._clock

    def ready(self) -> List[Stream]:
        """The streams the next :meth:`step` runs, in slot order."""
        waiting = [st for st in self._streams if st.ready_at is not None]
        return sorted(waiting, key=lambda st: (st.ready_at, st.index))[:self.slots]

    def step(self) -> Dict[Stream, torch.Tensor]:
        """One window of each of up to ``slots`` ready streams; returns their new frames, (1, n, dim_w) each, on the device.
        Asynchronous, like :func:`sample_clips`.  Returns {} when no stream is ready."""
        run = self.ready()
        if not run:
            return {}
        d, dev = self.dims, self.device
        L, P = d.frames_per_clip, d.num_prev_frames
        self._configure()                                  # no-op unless the backend ran another plan in between
        x0, outs = [], []
        for st in run:
            w = st.windows_run
            x0.append(torch.randn(1, L, d.dim_w, device=dev, generator=st.gen) if st.gen is not None
                      else st.noise[w].to(device=dev, dtype=torch.float32).contiguous())
            outs.append(torch.empty(1, min(L, st.fed - w * L), d.dim_w, device=dev))
        schedules = [st.schedule for st in run]
        own = {} if all(sc == (self.nfe, self.method) for sc in schedules) else dict(schedules=schedules)
        if any(st.we_dynamic != self.we_dynamic for st in run):
            own["we_dynamic"] = [st.we_dynamic for st in run]
        self._be.sample_windows([st.r_s for st in run], [st.wa for st in run],
                                [st.we_buf if st.we_dynamic else st.we for st in run], x0, [st.ctx for st in run], outs,
                                [int(st.windows_run == 0) for st in run], *zip(*[st.guidance for st in run]), **own)
        self._clock += 1
        for st in run:
            st.windows_run += 1
            st.ready_at = None
            # keep frames from the next window's first context frame on (copied, so the dropped frames are freed)
            keep = st.windows_run * L - P - st.base
            st.wa = st.wa[keep:].clone()
            if st.we_dynamic:
                st.we_buf = st.we_buf[keep:].clone()
            st.base += keep
            self._refresh(st)
        return dict(zip(run, outs))


def float_sample(fmt_model, opt, r_s, wa, we, a_cfg_scale=1.0, r_cfg_scale=1.0, e_cfg_scale=1.0, seed=None,
                 mode: Optional[str] = None, noise: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Drop-in for the sampling part of ``FLOAT.sample`` (FLOAT.py:172-253) once ``wa`` (B,T,dim_a) and ``we`` (B,1,dim_e;
    float or the int64 one-hot of :200) exist.  Uses ``opt.nfe`` (the method's own ``nfe`` argument is ignored by the
    reference, :188), static emotion, 3 CFG branches at most, Euler (``opt.torchdiffeq_ode_method``)."""
    device = torch.device(opt.rank)
    g = None
    if getattr(opt, "fix_noise_seed", True):
        g = torch.Generator(device)
        g.manual_seed(opt.seed if seed is None else seed)
    be = backend_for(fmt_model, device)
    d = be.dims
    return perform_ode_sampling_loop(fmt_model, r_s, wa, we.to(torch.float32), wa.shape[1], d.num_prev_frames, d.frames_per_clip,
                                     d.dim_w, opt.nfe, getattr(opt, "torchdiffeq_ode_method", "euler"), getattr(opt, "ode_atol", 1e-5),
                                     getattr(opt, "ode_rtol", 1e-5), device, a_cfg_scale, r_cfg_scale, e_cfg_scale, False, g,
                                     mode=mode, noise=noise)


def float_sample_from_audio(agent_G, data, a_cfg_scale=1.0, r_cfg_scale=1.0, e_cfg_scale=1.0, emo=None, nfe=10, seed=None,
                            mode: Optional[str] = None, noise: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Drop-in for the WHOLE of ``FLOAT.sample`` (FLOAT.py:172-253), bound in place of the method by
    :func:`use_b200_sampler`.  The conditioning front end keeps running the reference's own encoders (north_star): the audio
    encoder on the whole waveform (:191-194) and either the SER prediction or the forced int64 one-hot emotion (:196-200);
    the window loop + FMT + ODE solver behind it run in libfmt_b200.so.  ``nfe`` is accepted and ignored exactly as the
    reference ignores it (:188 uses ``self.opt.nfe``)."""
    import torch.nn.functional as F
    opt = agent_G.opt
    r_s = data["r_s"]
    a = data["a"].to(opt.rank)
    T = math.ceil(a.shape[-1] * opt.fps / opt.sampling_rate)
    wa = agent_G.audio_encoder.inference(a, seq_len=T)
    emo_idx = agent_G.emotion_encoder.label2id.get(str(emo).lower(), None)
    if emo_idx is None:
        we = agent_G.emotion_encoder.predict_emotion(a).unsqueeze(1)
    else:
        we = F.one_hot(torch.tensor(emo_idx, device=a.device), num_classes=opt.dim_e).unsqueeze(0).unsqueeze(0)
    return float_sample(agent_G.fmt, opt, r_s, wa, we, a_cfg_scale, r_cfg_scale, e_cfg_scale, seed=seed, mode=mode, noise=noise)


class use_b200_sampler:
    """``with use_b200_sampler(float_pipe.G):`` - inside the block ``G.sample`` (called by ``G.inference``, FLOAT.py:255-300) is
    this backend; the instance attribute is removed again on exit, so the reference module is left as it was."""

    def __init__(self, agent_G, mode: Optional[str] = None):
        self.G, self.mode = agent_G, mode

    def __enter__(self):
        G, mode = self.G, self.mode
        self._had = "sample" in vars(G)
        self._old = vars(G).get("sample")

        def sample(data, a_cfg_scale=1.0, r_cfg_scale=1.0, e_cfg_scale=1.0, emo=None, nfe=10, seed=None):
            return float_sample_from_audio(G, data, a_cfg_scale, r_cfg_scale, e_cfg_scale, emo, nfe, seed, mode=mode)
        try:
            object.__setattr__(G, "sample", sample)
        except Exception:
            G.sample = sample
        return G

    def __exit__(self, *exc):
        if self._had:
            object.__setattr__(self.G, "sample", self._old)
        else:
            try:
                object.__delattr__(self.G, "sample")
            except AttributeError:
                pass
        return False
